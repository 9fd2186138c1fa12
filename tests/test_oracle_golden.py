"""Pin oracle/nst_oracle.py against vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py, generated in the build container from /root/reference)."""
import os

import numpy as np
import pytest
import torch

from oracle import nst_oracle as O

torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))


def rand_img(seed, shape):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g)


@pytest.fixture(scope="module")
def ev(golden_dir):
    return np.load(os.path.join(golden_dir, "eval_48x64.npz"))


@pytest.fixture(scope="module")
def traj(golden_dir):
    return np.load(os.path.join(golden_dir, "nst_traj.npz"))


def test_weights_checksum(ev, vgg_weights):
    tot = sum(float(w.double().abs().sum()) + float(b.double().abs().sum()) for w, b in vgg_weights)
    assert tot == pytest.approx(float(ev["weights_abs_sum"]), rel=1e-12)


def test_vgg_features_gram_stats(ev, vgg_weights):
    H, W = 48, 64
    c = rand_img(11, (2, 3, H, W))
    with torch.no_grad():
        p5, c_f, s_f = O.vgg19_forward(c, vgg_weights, full=True)
    np.testing.assert_allclose(p5.numpy(), ev["eval_pool5"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose([float(f.double().sum()) for f in c_f], ev["eval_content_feat_sum"], rtol=1e-5)
    for i, f in enumerate(s_f):
        G = O.gram_matrix(f)
        if "eval_gram_c_%d" % i in ev.files:
            np.testing.assert_allclose(G.numpy(), ev["eval_gram_c_%d" % i], rtol=1e-5, atol=1e-9)
        np.testing.assert_allclose(G[:, :32, -32:].numpy(), ev["eval_gram_c_%d_corner" % i], rtol=1e-5, atol=1e-9)
        sums = [float(G.double().sum()), float(G.double().abs().sum()), float((G.double() ** 2).sum())]
        np.testing.assert_allclose(sums, ev["eval_gram_c_%d_sums" % i], rtol=1e-5)
    np.testing.assert_allclose(O.style_features(s_f).numpy(), ev["eval_style_features"], rtol=1e-5, atol=1e-7)
    # unbatched GramMatrix normalises by H*W (SURVEY note N3)
    np.testing.assert_allclose(O.gram_matrix(s_f[1][0]).numpy(), ev["eval_gram_unbatched"], rtol=1e-5, atol=1e-9)
    # 5-layer variant (relu5_1 tap)
    with torch.no_grad():
        _, _, s5 = O.vgg19_forward(c, vgg_weights, style_layers=list(O.DEFAULT_STYLE) + ["relu5_1"], full=False)
    G5 = O.gram_matrix(s5[4])
    np.testing.assert_allclose(G5[:, :32, -32:].numpy(), ev["eval_gram5_c_4_corner"], rtol=1e-5, atol=1e-9)


def test_conv_tap_aliases_relu(vgg_weights):
    """SURVEY note N2: a conv* tap is the post-ReLU tensor."""
    c = rand_img(3, (1, 3, 16, 16))
    with torch.no_grad():
        _, _, a = O.vgg19_forward(c, vgg_weights, style_layers=["conv2_1"], full=False)
        _, _, b = O.vgg19_forward(c, vgg_weights, style_layers=["relu2_1"], full=False)
    assert torch.equal(a[0], b[0]) and float(a[0].min()) >= 0.0


@pytest.mark.parametrize("name,BN", [("gram", False), ("bn", True)])
def test_losses_and_gradient(ev, vgg_weights, name, BN):
    H, W = 48, 64
    c, s, xq = rand_img(11, (2, 3, H, W)), rand_img(12, (2, 3, H, W)), rand_img(13, (2, 3, H, W))
    with torch.no_grad():
        _, c_f, _ = O.vgg19_forward(c, vgg_weights, full=False)
        _, _, s_t = O.vgg19_forward(s, vgg_weights, full=False)
    targets = ([t.mean(dim=(-2, -1)) for t in s_t], [t.std(dim=(-2, -1)) for t in s_t]) if BN else [O.gram_matrix(t) for t in s_t]
    cl, sl, g = O.nst_eval(xq, c_f, targets, vgg_weights, BN, 1.0, 1e6)
    assert cl == pytest.approx(float(ev["eval_%s_c_loss" % name]), rel=1e-5)
    assert sl == pytest.approx(float(ev["eval_%s_s_loss" % name]), rel=1e-5)
    ref = ev["eval_%s_grad" % name]
    assert np.abs(g.numpy() - ref).max() <= 1e-5 * np.abs(ref).max()


@pytest.fixture(scope="module")
def otraj(golden_dir):
    return np.load(os.path.join(golden_dir, "nst_traj_oracle.npz"))


def _check_traj(traj, tag, x, c_hist, s_hist, exact=True, otraj=None):
    """`traj`: the reference's run of the case; `otraj`: the oracle's recorded run (make_golden_oracle_traj.py)."""
    # against the reference on any host: the same number of evaluations, the first evaluation, and the first L-BFGS
    # steps (the 1/|g|_1-scaled first step, the two-loop directions, the history), which host rounding moves by < 1e-4
    # over evaluations 0-2 and < 1e-2 over 0-10 before the run's chaos amplifies it
    assert len(c_hist) == len(s_hist) == len(traj[tag + "_c_hist"]) == len(traj[tag + "_s_hist"])
    np.testing.assert_allclose([c_hist[0], s_hist[0]], [traj[tag + "_c_hist"][0], traj[tag + "_s_hist"][0]],
                               rtol=1e-5, atol=1e-12)
    for n, rtol in ((3, 1e-4), (11, 1e-2)):
        np.testing.assert_allclose(c_hist[:n], traj[tag + "_c_hist"][:n], rtol=rtol, atol=1e-12)
        np.testing.assert_allclose(s_hist[:n], traj[tag + "_s_hist"][:n], rtol=rtol, atol=1e-12)
    # the whole run: float32 L-BFGS grows the host's rounding over the run, so it is pinned to a run on a recorded host
    assert len(c_hist) == len(otraj[tag + "_c_hist"])
    tol = dict(rtol=1e-6, atol=1e-12) if exact else dict(rtol=1e-3, atol=1e-9)
    np.testing.assert_allclose(c_hist, otraj[tag + "_c_hist"], **tol)
    np.testing.assert_allclose(s_hist, otraj[tag + "_s_hist"], **tol)
    k = int(otraj[tag + "_x_stride"])
    np.testing.assert_allclose(x.numpy()[..., ::k, ::k], otraj[tag + "_x"], atol=1e-6 if exact else 1e-3)


def test_nst_gram_b1(traj, otraj, vgg_weights):
    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    x, xh, ch, sh = O.nst(c1, s1, vgg_weights, BN_loss=False, s_loss_weight=1e6, epochs=50)
    assert len(ch) == 60  # ceil(50/20)*20 (SURVEY §0.1)
    _check_traj(traj, "gram_b1", x, ch, sh, otraj=otraj)
    assert len(xh) == 60 and not torch.equal(xh[0], xh[-1])  # per-eval copies (CUDA semantics of pipelines.py:93)


def test_nst_bn_b1(traj, otraj, vgg_weights):
    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    x, _, ch, sh = O.nst(c1, s1, vgg_weights, BN_loss=True, s_loss_weight=1e4, epochs=40)
    _check_traj(traj, "bn_b1", x, ch, sh, otraj=otraj)


def test_nst_batched_is_one_problem(traj, otraj, vgg_weights):
    c, s = rand_img(11, (2, 3, 48, 64)), rand_img(12, (2, 3, 48, 64))
    x, _, ch, sh = O.nst(c, s, vgg_weights, BN_loss=False, s_loss_weight=1e6, epochs=20)
    _check_traj(traj, "gram_b2_coupled", x, ch, sh, otraj=otraj)
    x, _, ch, sh = O.nst(c, s[:1], vgg_weights, BN_loss=False, s_loss_weight=1e6, epochs=20)
    _check_traj(traj, "gram_b2_style1", x, ch, sh, otraj=otraj)


def test_nst_rand_init(traj, otraj, vgg_weights):
    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    torch.manual_seed(123)
    x0 = torch.rand(c1.shape)  # pipelines.py:54 under the same seed as make_golden
    x, _, ch, sh = O.nst(c1, s1, vgg_weights, clone_content=False, x0=x0, BN_loss=False, s_loss_weight=1e6, epochs=20)
    _check_traj(traj, "gram_rand_init", x, ch, sh, otraj=otraj)


def test_nst_degenerate_never_moves(traj, otraj, vgg_weights):
    """|g|inf < tolerance_grad with alpha=beta=1 (SURVEY trap H1): one eval per optim.step, x fixed."""
    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    x, _, ch, sh = O.nst(c1, s1, vgg_weights, BN_loss=False, s_loss_weight=1.0, epochs=5)
    assert len(ch) == 5 and torch.equal(x, c1)
    _check_traj(traj, "degenerate", x, ch, sh, otraj=otraj)


def test_nst_unbatched_style(traj, otraj, vgg_weights):
    """…2020.py:103-104 passes a (1,H,W) style image (SURVEY note N3)."""
    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    x, _, ch, sh = O.nst(c1, s1[0, :1], vgg_weights, BN_loss=False, s_loss_weight=1e6, epochs=20)
    _check_traj(traj, "gram_unbatched_style", x, ch, sh, exact=False, otraj=otraj)
    x, _, ch, sh = O.nst(c1, s1[0, :1], vgg_weights, BN_loss=True, s_loss_weight=1e4, epochs=20)
    _check_traj(traj, "bn_unbatched_style", x, ch, sh, otraj=otraj)


def test_nst_long_history(traj, otraj, vgg_weights):
    c3, s3 = rand_img(31, (1, 3, 32, 32)), rand_img(32, (1, 3, 32, 32))
    x, _, ch, sh = O.nst(c3, s3, vgg_weights, BN_loss=False, s_loss_weight=1e6, epochs=130)
    assert len(ch) == 140
    _check_traj(traj, "gram_long", x, ch, sh, otraj=otraj)


@pytest.fixture(scope="module")
def traj2(golden_dir):
    return np.load(os.path.join(golden_dir, "nst_traj_r2.npz"))


@pytest.mark.parametrize("tag,BN,s4d", [("gram_c3d_s3d", False, False), ("bn_c3d_s3d", True, False),
                                        ("gram_c3d_s4d", False, True)])
def test_nst_unbatched_content(traj2, otraj, vgg_weights, tag, BN, s4d):
    """The notebook's call: nst(c (3,H,W), s (3,H,W)) returns (3,H,W); GramMatrix divides by H*W for an unbatched
    map and by C*H*W for a batched one (utils.py:253-254), so c3d x s4d mixes the two normalisers like the reference."""
    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    x, _, ch, sh = O.nst(c1[0], s1 if s4d else s1[0], vgg_weights, BN_loss=BN, s_loss_weight=1e4, epochs=20)
    assert tuple(x.shape) == tuple(traj2[tag + "_x_shape"]) == (3, 48, 64)
    _check_traj(traj2, tag, x, ch, sh, exact=False, otraj=otraj)


def test_nst_iris224_bn_coupled_batch(traj2, otraj, vgg_weights):
    """…2019.py:93-100: a batch of 224x224 iris crops, default StyleLoss_BN, the batch as ONE L-BFGS problem."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("isx_synthetic", os.path.join(
        os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "iris-style-transfer_b200", "synthetic.py"))
    syn = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(syn)
    ic = torch.from_numpy(syn.synthetic_iris_crops([1, 2, 3, 4, 11, 12, 13, 14], 224))
    x, _, ch, sh = O.nst(ic[:4], ic[4:], vgg_weights, BN_loss=True, s_loss_weight=1e4, epochs=40, keep_hist=False)
    _check_traj(traj2, "bn_iris224_b4", x, ch, sh, exact=False, otraj=otraj)


def test_mask_bbox(golden_dir):
    import importlib.util
    import sys

    m = np.load(os.path.join(golden_dir, "mask_bbox.npz"))
    sys.path.insert(0, os.path.join(os.path.dirname(golden_dir), "..", "iris-style-transfer_b200"))
    import synthetic

    for k, (seed, h, w) in enumerate([(5, 640, 400), (6, 400, 640), (7, 64, 48)]):
        frame, seg = synthetic.synthetic_eye(seed, h, w)
        xc, mc, x0, y0, x1, y1 = O.mask_and_crop(frame, seg)
        assert [x0, y0, x1, y1] == list(m["syn%d_bbox" % k])
        assert int(mc.sum()) == int(m["syn%d_mask_count" % k])
        assert list(xc.shape) == list(m["syn%d_crop_shape" % k])
        assert float(xc.astype(np.float64).sum()) == pytest.approx(float(m["syn%d_crop_sum" % k]), rel=1e-12)
    # real eye PNGs through the shipped RITnet: notebook cell 2 prints [171, 206] for the first
    for k in range(2):
        if "real%d_bbox" % k not in m.files:
            pytest.skip("real-image fixtures absent")
        shape = tuple(m["real%d_shape" % k])
        n = int(np.prod(shape))
        iris = np.unpackbits(m["real%d_iris_bits" % k])[:n].reshape(shape).astype(bool)
        nog = np.unpackbits(m["real%d_noglint_bits" % k])[:n].reshape(shape).astype(bool)
        mm = iris & nog
        # pixels are > 0 wherever the mask is set in these frames, so bbox(mask) == bbox(x*m)
        bb = O.crop_bbox(mm.astype(np.float32))
        assert list(bb) == list(m["real%d_bbox" % k])
    assert list(m["real0_bbox"]) == [223, 92, 393, 297]
    assert (393 - 223 + 1, 297 - 92 + 1) == (171, 206)


def test_crop_bbox_edge_cases():
    with pytest.raises(Exception):
        O.crop_bbox(np.zeros((2, 4, 4), np.float32))  # utils.py:66 'image shape wrong'
    with pytest.raises(RuntimeError):
        O.crop_bbox(np.zeros((1, 4, 4), np.float32))  # empty -> torch min() error in the reference
    a = np.zeros((5, 7), np.float32)
    a[2, 3] = 1e-30
    assert O.crop_bbox(a) == (2, 3, 2, 3)
    a[4, 0] = -1.0
    assert O.crop_bbox(a) == (2, 0, 4, 3)


def test_composite_and_resize(golden_dir):
    import sys

    k = np.load(os.path.join(golden_dir, "composite.npz"))
    sys.path.insert(0, os.path.join(os.path.dirname(golden_dir), "..", "iris-style-transfer_b200"))
    import synthetic

    for idx, (seed, h, w) in enumerate([(5, 640, 400), (6, 400, 640)]):
        frame, seg = synthetic.synthetic_eye(seed, h, w)
        m = (seg == 2) & (frame <= np.float32(0.8))
        bbox = O.crop_bbox(frame * m)
        assert list(bbox) == list(k["comp%d_bbox" % idx])
        new_rgb = rand_img(40 + idx, (1, 3, 224, 224)).numpy()[0]
        out = O.composite(frame, new_rgb, m, bbox)
        x_min, y_min = bbox[0], bbox[1]
        np.testing.assert_allclose(out[:, x_min:x_min + 24, y_min + 40:y_min + 64], k["comp%d_patch" % idx], atol=2e-6)
        np.testing.assert_allclose(out, k["comp%d_out" % idx].astype(np.float32), atol=1e-3)
        assert float(out.astype(np.float64).sum()) == pytest.approx(float(k["comp%d_out_sum" % idx]), rel=1e-6)
        crop = (frame * m)[:, bbox[0]:bbox[2] + 1, bbox[1]:bbox[3] + 1]
        r = O.resize_bilinear_aa(crop, 224, 224)
        np.testing.assert_allclose(r[:, 100:116, 100:116], k["resize%d_224_patch" % idx], atol=2e-6)
        assert float(r.astype(np.float64).sum()) == pytest.approx(float(k["resize%d_224_sum" % idx]), rel=1e-6)
