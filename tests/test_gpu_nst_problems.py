"""Several coupled L-BFGS problems in one nst() call (problem_size=g, per-problem weights and styles) on the B200.

Per-image losses are accumulated with double atomicAdd, whose order varies from run to run, so loss values that should be
identical are compared to 1e-12; images, gradients and evaluation counts are compared bit for bit."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def rand_img(seed, shape):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g)


@pytest.fixture(scope="module")
def mods():
    import iris_b200
    from iris_b200 import _lib, engine, pipelines, synthetic, vgg
    from oracle import nst_oracle as O

    _lib.load()
    weights = O.random_vgg19_weights(0)
    return dict(engine=engine, pipelines=pipelines, vgg=vgg.VGG19(weights=weights), synthetic=synthetic, api=iris_b200)


@pytest.fixture(scope="module")
def crops(mods):
    return torch.from_numpy(mods["synthetic"].synthetic_iris_crops([1, 2, 3, 4, 11, 12, 13, 14], 224))


def _run(mods, c, s, **kw):
    kw.setdefault("x_hist_stride", 0)
    x, _, ch, sh = mods["pipelines"].nst(c, s, vgg=mods["vgg"], use_tqdm=False, device="cuda:0", **kw)
    torch.cuda.synchronize()
    info = dict(mods["pipelines"].last_info)
    return x.cpu(), np.array(ch), np.array(sh), info


def _same_run(a, b):
    xa, cha, sha, ia = a
    xb, chb, shb, ib = b
    assert torch.equal(xa, xb)
    assert torch.equal(ia["evals_per_problem"], ib["evals_per_problem"]) and len(sha) == len(shb)
    np.testing.assert_allclose(cha, chb, rtol=1e-12, atol=0)
    np.testing.assert_allclose(shb, sha, rtol=1e-12, atol=0)


# ------------------------------------------------------------------------------------------------
# 1. problem_size=B is the default layout, problem_size=1 is independent=True
# ------------------------------------------------------------------------------------------------
def test_problem_size_b_and_1_equal_existing_layouts_224_bn(mods, crops):
    c, s = crops[:4], crops[4:]
    kw = dict(BN_loss=True, s_loss_weight=1e4, epochs=20)
    _same_run(_run(mods, c, s, **kw), _run(mods, c, s, problem_size=4, **kw))
    _same_run(_run(mods, c, s, independent=True, **kw), _run(mods, c, s, problem_size=1, **kw))


def test_problem_size_b_and_1_equal_existing_layouts_640_gram(mods):
    import bench

    c, s = bench.make_inputs(2, 1)
    kw = dict(BN_loss=False, s_loss_weight=1e6, epochs=10)
    _same_run(_run(mods, c, s, **kw), _run(mods, c, s, problem_size=2, **kw))
    _same_run(_run(mods, c, s, independent=True, **kw), _run(mods, c, s, problem_size=1, **kw))


# ------------------------------------------------------------------------------------------------
# 2. one evaluation: per-problem weights scale exactly like the scalar weights of isx_nst_eval
# ------------------------------------------------------------------------------------------------
def _engine(mods, c, s, BN, content_w):
    E, net = mods["engine"], mods["vgg"]
    dev = torch.device("cuda:0")
    packed = net.packed(dev)
    B, xc, H, W = c.shape
    cc, sc = net.content_convs, net.style_convs
    eng = E.NstEngine(packed, B, H, W, xc, cc, sc, style_mode=1 if BN else 0, content_w=[content_w] * len(cc),
                      coupled=True)
    eng.forward(c)
    eng.set_content_targets([eng.tap(i) for i in cc])
    seng = E.NstEngine(packed, s.shape[0], H, W, xc, cc, sc)
    seng.forward(s)
    feats = [seng.tap_view(i) for i in sc]
    if BN:
        st = [E.stats_of(f) for f in feats]
        eng.set_bn_targets([m for m, _ in st], [v for _, v in st])
    else:
        eng.set_gram_targets([E.gram_of(f) for f in feats])
    return eng


@pytest.mark.parametrize("BN", [False, True])
@pytest.mark.parametrize("style_batch", ["one", "problems", "images"])
def test_eval_problems_scales_like_scalar_eval(mods, BN, style_batch):
    g, P = 2, 2                                      # g, P powers of two: the content denominators agree exactly
    B = g * P
    dev = torch.device("cuda:0")
    c = rand_img(61, (B, 3, 64, 64)).to(dev)
    x = (c + 0.05 * rand_img(62, (B, 3, 64, 64)).to(dev)).clamp(0, 1).contiguous()
    s_all = rand_img(63, (B, 3, 64, 64)).to(dev)
    s = {"one": s_all[:1], "problems": s_all[:P], "images": s_all}[style_batch]
    s_per_image = s if s.shape[0] in (1, B) else s.repeat_interleave(g, dim=0)
    alpha, beta = [1.5, 0.375], [1e4, 3e5]

    eng = _engine(mods, c, s, BN, content_w=1.0)    # F.mse_loss over g images: denominator per_image * g
    eng.set_problems(g, torch.tensor(alpha, device=dev, dtype=torch.float64), torch.tensor(beta, device=dev, dtype=torch.float64))
    grad = torch.empty_like(x)
    eng.eval(x, grad)
    torch.cuda.synchronize()
    lc, ls = eng.loss_c.cpu(), eng.loss_s.cpu()
    for p in range(P):
        # scalar isx_nst_eval on the same batch: coupled content loss over B = P * g images, content_w = P gives the same
        # per_image * g denominator exactly
        ref = _engine(mods, c, s_per_image.contiguous(), BN, content_w=float(P))
        ref.cfg.c_weight, ref.cfg.s_weight = alpha[p], beta[p]
        rgrad = torch.empty_like(x)
        ref.eval(x, rgrad)
        torch.cuda.synchronize()
        sl = slice(p * g, (p + 1) * g)
        assert torch.equal(grad[sl], rgrad[sl]), p
        np.testing.assert_allclose(lc[sl].numpy(), ref.loss_c.cpu()[sl].numpy(), rtol=1e-12, atol=0)
        np.testing.assert_allclose(ls[sl].numpy(), ref.loss_s.cpu()[sl].numpy(), rtol=1e-12, atol=0)
        assert float(lc[sl].abs().sum()) > 0 and float(ls[sl].abs().sum()) > 0


# ------------------------------------------------------------------------------------------------
# 3. each problem is the reference's call: the golden 224x224 BN trajectory, twice in one job
# ------------------------------------------------------------------------------------------------
def test_two_problems_each_meet_the_reference_golden(mods, crops, golden_dir):
    """The bars test_gpu_parity_r2 applies to bn_iris224_b4: exact evaluation count, first two losses, final image within
    the calibrated bound of the golden.  Its strict 1e-2 is not asserted here: at B = 8 the kernels pick other split
    counts than at B = 4, and the reference optimiser itself moves this final image by up to 0.016 when its gradient is
    perturbed by 2^-9 (calibration_r2.json), so 1e-2 depends on the summation order.  Both problems see the same inputs
    and must end bit-identical: nothing leaks from one problem into the other."""
    traj2 = np.load(os.path.join(golden_dir, "nst_traj_r2.npz"))
    calib = json.load(open(os.path.join(golden_dir, "calibration_r2.json")))
    tag = "bn_iris224_b4"
    rs = traj2[tag + "_s_hist"]
    ref_x = torch.from_numpy(traj2[tag + "_x"])
    cal = calib[tag]
    bound = max(1e-2, 1.5 * max([cal["sens_bf16"]] + list(cal["sens_noise"])))
    c, s = torch.cat([crops[:4], crops[:4]]), torch.cat([crops[4:], crops[4:]])     # per-image style batch B = 8
    x, _, _, info = _run(mods, c, s, BN_loss=True, s_loss_weight=1e4, epochs=40, problem_size=4)
    hs = info["s_loss_per_problem"].numpy()
    for p in range(2):
        mae = float((x[4 * p:4 * p + 4] - ref_x).abs().mean())
        print("problem %d: evals %d/%d s %.5g/%.5g %.5g/%.5g final MAE %.5f (bound %.5f)" % (
            p, int(info["evals_per_problem"][p]), len(rs), hs[0, p], rs[0], hs[1, p], rs[1], mae, bound))
        assert int(info["evals_per_problem"][p]) == len(rs) == 40
        assert hs[0, p] == pytest.approx(rs[0], rel=1e-2) and hs[1, p] == pytest.approx(rs[1], rel=2e-2)
        assert mae <= bound
    assert torch.equal(x[:4], x[4:])


# ------------------------------------------------------------------------------------------------
# 4. a weight sweep in one job == the separate calls
# ------------------------------------------------------------------------------------------------
def test_beta_sweep_in_one_job_matches_separate_calls(mods, crops):
    betas = [1e3, 1e4, 1e5]
    c, s = crops[:4], crops[4:]
    x, ch, sh, info = _run(mods, c.repeat(3, 1, 1, 1), s.repeat(3, 1, 1, 1), BN_loss=True, s_loss_weight=betas, epochs=20,
                           problem_size=4)
    hc, hs = info["c_loss_per_problem"].numpy(), info["s_loss_per_problem"].numpy()
    assert info["problems"] == 3 and hs.shape[1] == 3
    np.testing.assert_allclose(sh, hs.sum(axis=1), rtol=1e-12)
    np.testing.assert_allclose(ch, hc.mean(axis=1), rtol=1e-12)
    for p, beta in enumerate(betas):
        xp, chp, shp, _ = _run(mods, c, s, BN_loss=True, s_loss_weight=beta, epochs=20)
        e = int(info["evals_per_problem"][p])
        print("beta %g: evals %d/%d s %.5g/%.5g %.5g/%.5g MAE vs separate %.2e" % (
            beta, e, len(shp), hs[0, p], shp[0], hs[1, p], shp[1], float((x[4 * p:4 * p + 4] - xp).abs().mean())))
        assert e == len(shp)
        assert hs[0, p] == pytest.approx(shp[0], rel=1e-2) and hs[1, p] == pytest.approx(shp[1], rel=2e-2)
        assert hc[0, p] == pytest.approx(chp[0], abs=1e-12)


# ------------------------------------------------------------------------------------------------
# 5. every problem has its own exit tests
# ------------------------------------------------------------------------------------------------
def test_degenerate_problem_exits_alone(mods):
    """alpha = beta = 1 with random-init VGG: |g|inf < tolerance_grad, so that problem makes one evaluation per
    optimizer.step and never moves, while the problem beside it runs its own course."""
    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    c2, s2 = rand_img(11, (2, 3, 48, 64)), rand_img(12, (2, 3, 48, 64))
    c, s = torch.cat([c1, c1, c2]), torch.cat([s1, s1, s2])
    epochs = 5
    x, _, _, info = _run(mods, c, s, BN_loss=False, c_loss_weight=[1.0, 1.0], s_loss_weight=[1.0, 1e6], epochs=epochs,
                         problem_size=2)
    xa, cha, sha, ia = _run(mods, c2, s2, BN_loss=False, s_loss_weight=1e6, epochs=epochs)
    ev = info["evals_per_problem"].tolist()
    hc, hs = info["c_loss_per_problem"].numpy(), info["s_loss_per_problem"].numpy()
    print("evals per problem %s, alone %d" % (ev, len(sha)))
    assert ev[0] == epochs
    assert torch.equal(x[:2], c[:2])
    assert ev[1] == len(sha) >= epochs
    assert hs[0, 1] == pytest.approx(sha[0], rel=1e-2) and hs[1, 1] == pytest.approx(sha[1], rel=2e-2)
    assert hc[0, 1] == pytest.approx(cha[0], abs=1e-12)
    assert float((x[2:] - c2).abs().mean()) > 1e-4


# ------------------------------------------------------------------------------------------------
# 6. a captured tick reads the per-problem weights from the device
# ------------------------------------------------------------------------------------------------
def test_cuda_graph_with_per_problem_weights_equals_eager(mods, crops):
    c, s = torch.cat([crops[:4], crops[:4]]), crops[4:6]      # style batch P = 2: one style per problem
    kw = dict(BN_loss=True, c_loss_weight=[1.0, 2.0], s_loss_weight=[1e4, 1e5], epochs=20, problem_size=4)
    _same_run(_run(mods, c, s, **kw), _run(mods, c, s, cuda_graph=True, **kw))
