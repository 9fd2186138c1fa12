"""Coupled L-BFGS problems of unequal size in one nst() call (problem_sizes=...) and one problem per driver batch in
stylize_frames (frames_per_problem=g), on the B200.

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
    return dict(engine=engine, pipelines=pipelines, vgg=vgg.VGG19(weights=weights), synthetic=synthetic, api=iris_b200,
                lib=_lib)


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
# 1. equal sizes are the existing layouts, bit for bit
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hdt", [torch.float32, torch.bfloat16])
def test_equal_sizes_equal_existing_layouts_224_bn(mods, crops, hdt):
    c, s = crops[:4], crops[4:]
    kw = dict(BN_loss=True, s_loss_weight=1e4, epochs=20, history_dtype=hdt)
    _same_run(_run(mods, c, s, problem_size=2, **kw), _run(mods, c, s, problem_sizes=[2, 2], **kw))
    _same_run(_run(mods, c, s, **kw), _run(mods, c, s, problem_sizes=[4], **kw))
    _same_run(_run(mods, c, s, independent=True, **kw), _run(mods, c, s, problem_sizes=[1] * 4, **kw))


@pytest.mark.parametrize("hdt", [torch.float32, torch.bfloat16])
def test_equal_sizes_equal_existing_layouts_640_gram(mods, hdt):
    import bench

    c, s = bench.make_inputs(4, 1)
    kw = dict(BN_loss=False, s_loss_weight=1e6, epochs=10, history_dtype=hdt)
    _same_run(_run(mods, c, s, problem_size=2, **kw), _run(mods, c, s, problem_sizes=[2, 2], **kw))
    _same_run(_run(mods, c, s, **kw), _run(mods, c, s, problem_sizes=[4], **kw))
    _same_run(_run(mods, c, s, independent=True, **kw), _run(mods, c, s, problem_sizes=[1] * 4, **kw))


# ------------------------------------------------------------------------------------------------
# 2. one evaluation: problem p scales like g_p single-image problems with alpha_p / g_p
# ------------------------------------------------------------------------------------------------
def _engine(mods, c, s, BN):
    E, net = mods["engine"], mods["vgg"]
    dev = torch.device("cuda:0")
    packed = net.packed(dev)
    B, xc, H, W = c.shape
    cc, sc = net.content_convs, net.style_convs
    eng = E.NstEngine(packed, B, H, W, xc, cc, sc, style_mode=1 if BN else 0, coupled=True)
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
def test_eval_ranges_scales_like_single_image_problems(mods, BN, style_batch):
    sizes = [1, 2, 4, 1]                       # powers of two: alpha_p / g_p and the content denominators are exact
    P, B = len(sizes), sum(sizes)
    first = [sum(sizes[:p]) for p in range(P + 1)]
    dev = torch.device("cuda:0")
    c = rand_img(71, (B, 3, 64, 64)).to(dev)
    x = (c + 0.05 * rand_img(72, (B, 3, 64, 64)).to(dev)).clamp(0, 1).contiguous()
    s_all = rand_img(73, (B, 3, 64, 64)).to(dev)
    s = {"one": s_all[:1], "problems": s_all[:P], "images": s_all}[style_batch].contiguous()
    g_img = torch.tensor(sizes).repeat_interleave(torch.tensor(sizes))
    s_per_image = s if s.shape[0] in (1, B) else s.repeat_interleave(torch.tensor(sizes, device=dev), dim=0)
    alpha, beta = [1.5, 0.375, 3.0, 0.75], [1e4, 3e5, 2e3, 5e4]
    f64 = dict(device=dev, dtype=torch.float64)

    eng = _engine(mods, c, s, BN)
    eng.set_problem_ranges(first, torch.tensor(alpha, **f64), torch.tensor(beta, **f64))
    grad = torch.empty_like(x)
    eng.eval(x, grad)

    ref = _engine(mods, c, s_per_image.contiguous(), BN)   # B single-image problems, alpha_p / g_p, beta_p
    a_img = torch.tensor([alpha[p] / sizes[p] for p in range(P) for _ in range(sizes[p])], **f64)
    b_img = torch.tensor([beta[p] for p in range(P) for _ in range(sizes[p])], **f64)
    ref.set_problems(1, a_img, b_img)
    rgrad = torch.empty_like(x)
    ref.eval(x, rgrad)
    torch.cuda.synchronize()
    assert torch.equal(grad, rgrad)
    lc, ls = eng.loss_c.cpu(), eng.loss_s.cpu()
    # the content loss of an image in a problem of g_p images is the single-image loss / g_p (F.mse_loss over g_p images)
    np.testing.assert_allclose((lc * g_img).numpy(), ref.loss_c.cpu().numpy(), rtol=1e-12, atol=0)
    np.testing.assert_allclose(ls.numpy(), ref.loss_s.cpu().numpy(), rtol=1e-12, atol=0)
    assert float(lc.abs().min()) > 0 and float(ls.abs().min()) > 0


# ------------------------------------------------------------------------------------------------
# 3. isolation: the golden 224x224 BN problem twice, around a problem of another size
# ------------------------------------------------------------------------------------------------
def test_golden_problem_twice_around_another_size(mods, crops, golden_dir):
    """Layout [4, 3, 4]: bn_iris224_b4, three other crops, bn_iris224_b4 again.  The bars of
    test_two_problems_each_meet_the_reference_golden: exact evaluation count, first two losses, final image within the
    calibrated bound; both copies end bit-identical, so nothing leaks between problems of different sizes."""
    traj2 = np.load(os.path.join(golden_dir, "nst_traj_r2.npz"))
    calib = json.load(open(os.path.join(golden_dir, "calibration_r2.json")))
    tag = "bn_iris224_b4"
    rs = traj2[tag + "_s_hist"]
    ref_x = torch.from_numpy(traj2[tag + "_x"])
    cal = calib[tag]
    bound = max(1e-2, 1.5 * max([cal["sens_bf16"]] + list(cal["sens_noise"])))
    other_c = torch.from_numpy(mods["synthetic"].synthetic_iris_crops([21, 22, 23], 224))
    other_s = torch.from_numpy(mods["synthetic"].synthetic_iris_crops([31, 32, 33], 224))
    c = torch.cat([crops[:4], other_c, crops[:4]])
    s = torch.cat([crops[4:], other_s, crops[4:]])             # per-image style batch B = 11
    x, _, _, info = _run(mods, c, s, BN_loss=True, s_loss_weight=1e4, epochs=40, problem_sizes=[4, 3, 4])
    hs = info["s_loss_per_problem"].numpy()
    assert info["problems"] == 3
    for p, lo in ((0, 0), (2, 7)):
        mae = float((x[lo:lo + 4] - ref_x).abs().mean())
        print("problem %d: evals %d/%d s %.5g/%.5g %.5g/%.5g final MAE %.5f (bound %.5f)" % (
            p, int(info["evals_per_problem"][p]), len(rs), hs[0, p], rs[0], hs[1, p], rs[1], mae, bound))
        assert int(info["evals_per_problem"][p]) == len(rs) == 40
        assert hs[0, p] == pytest.approx(rs[0], rel=1e-2) and hs[1, p] == pytest.approx(rs[1], rel=2e-2)
        assert mae <= bound
    assert torch.equal(x[:4], x[7:])


# ------------------------------------------------------------------------------------------------
# 4. very unequal sizes: nothing is read outside a problem's own slices
# ------------------------------------------------------------------------------------------------
def _drive(job):
    """The loop of nst(), checking after every tick that no history holds more pairs than iterations were made."""
    while job.ticks < job.max_ticks:
        job.tick()
        counts = job.history_counts()
        assert int(counts.max()) <= min(job.ticks - 1, job.cfg.history), (job.ticks, counts.tolist())
        if job.ticks >= job.epochs and bool((job.evals_done() > 0).all().item()):
            break
    return job.finish()


@pytest.mark.parametrize("sizes", [[1, 31], [31, 1]])
def test_very_unequal_sizes_read_only_their_own_slices(mods, sizes):
    B, epochs = sum(sizes), 10
    c, s = rand_img(81, (B, 3, 48, 64)), rand_img(82, (B, 3, 48, 64))
    dev = torch.device("cuda:0")
    with torch.no_grad():
        job = mods["pipelines"].NstJob(c, s, mods["vgg"], dev, BN_loss=False, s_loss_weight=1e6, epochs=epochs,
                                       problem_sizes=sizes)
        for t in (job.Sh, job.Yh, job.grad_prev, job.grad):
            t.fill_(float("nan"))
        job.scratch.fill_(0xFF)                                 # NaN as float and as double
        x, n_evals, evals, hc, hs = _drive(job)
        torch.cuda.synchronize()
    assert torch.isfinite(x).all() and torch.isfinite(job.grad).all()
    assert torch.isfinite(hc).all() and torch.isfinite(hs).all()
    lo = 0
    for p, g in enumerate(sizes):
        xa, cha, sha, _ = _run(mods, c[lo:lo + g], s[lo:lo + g], BN_loss=False, s_loss_weight=1e6, epochs=epochs)
        print("problem %d (%d images): evals %d, alone %d; s %.6g/%.6g %.6g/%.6g" % (
            p, g, int(evals[p]), len(sha), hs[0, p], sha[0], hs[1, p], sha[1]))
        assert int(evals[p]) == len(sha)
        assert float(hs[0, p]) == pytest.approx(sha[0], rel=1e-2) and float(hs[1, p]) == pytest.approx(sha[1], rel=2e-2)
        assert float(hc[0, p]) == pytest.approx(cha[0], abs=1e-12)
        lo += g


# ------------------------------------------------------------------------------------------------
# 5. every problem has its own exit tests
# ------------------------------------------------------------------------------------------------
def test_degenerate_problem_exits_alone_between_unequal_neighbours(mods):
    """alpha = beta = 1 with random-init VGG: |g|inf < tolerance_grad, so the single-image problem makes one evaluation
    per optimizer.step and never moves, while the problems of 2 and 3 images beside it run their own course."""
    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    c2, s2 = rand_img(11, (2, 3, 48, 64)), rand_img(12, (2, 3, 48, 64))
    c3, s3 = rand_img(13, (3, 3, 48, 64)), rand_img(14, (3, 3, 48, 64))
    c, s = torch.cat([c2, c1, c3]), torch.cat([s2, s1, s3])
    epochs = 5
    x, _, _, info = _run(mods, c, s, BN_loss=False, c_loss_weight=[1.0, 1.0, 1.0], s_loss_weight=[1e6, 1.0, 1e6],
                         epochs=epochs, problem_sizes=[2, 1, 3])
    ev = info["evals_per_problem"].tolist()
    hc, hs = info["c_loss_per_problem"].numpy(), info["s_loss_per_problem"].numpy()
    assert ev[1] == epochs
    assert torch.equal(x[2:3], c1)
    for p, (cp, sp, lo) in ((0, (c2, s2, 0)), (2, (c3, s3, 3))):
        xa, cha, sha, _ = _run(mods, cp, sp, BN_loss=False, s_loss_weight=1e6, epochs=epochs)
        print("problem %d: evals %d, alone %d" % (p, ev[p], len(sha)))
        assert ev[p] == len(sha) >= epochs
        assert hs[0, p] == pytest.approx(sha[0], rel=1e-2) and hs[1, p] == pytest.approx(sha[1], rel=2e-2)
        assert hc[0, p] == pytest.approx(cha[0], abs=1e-12)
        assert float((x[lo:lo + cp.shape[0]] - cp).abs().mean()) > 1e-4


# ------------------------------------------------------------------------------------------------
# 6. a captured tick carries the offsets by value
# ------------------------------------------------------------------------------------------------
def test_cuda_graph_of_unequal_problems_equals_eager(mods, crops):
    c, s = crops, crops[4:7]                                    # style batch P = 3: one style per problem
    kw = dict(BN_loss=True, c_loss_weight=[1.0, 2.0, 0.5], s_loss_weight=[1e4, 1e5, 3e4], epochs=20,
              problem_sizes=[3, 1, 4])
    _same_run(_run(mods, c, s, **kw), _run(mods, c, s, cuda_graph=True, **kw))


# ------------------------------------------------------------------------------------------------
# 7. stylize_frames: one coupled problem per driver batch, frames without an iris and a short last batch
# ------------------------------------------------------------------------------------------------
def test_stylize_frames_one_problem_per_run(mods):
    api, syn, P = mods["api"], mods["synthetic"], mods["pipelines"]
    dev = torch.device("cuda:0")
    B, g = 29, 8                                                # runs of 8, 8, 8 and 5 frames
    seeds = [500 + i for i in range(B)]
    fr, sg = syn.synthetic_batch(seeds, 400, 640)
    erased = [10, 13] + list(range(16, 24))                     # two frames of run 1, every frame of run 2
    for i in erased:
        sg[i, 0] = syn.synthetic_label_map(seeds[i], 400, 640, drop=(2,))
    frames, segs = torch.from_numpy(fr).to(dev), torch.from_numpy(sg).to(dev)
    sf, ss = syn.synthetic_eye(777, 400, 640)
    sx, sseg = torch.from_numpy(sf).to(dev)[None], torch.from_numpy(ss).to(dev)[None]
    smask, sbb = P.iris_masks_and_bboxes(sx, sseg)
    style = P.crop_resize_irises(sx, smask, sbb, size=(64, 64))[0, :1].contiguous()
    kw = dict(vgg=mods["vgg"], s_loss_weight=1e4, epochs=20, BN_loss=True, size=(64, 64), device="cuda:0")

    out, info = api.stylize_frames(frames, style, segs=segs, frames_per_problem=g, **kw)
    torch.cuda.synchronize()
    assert info["problem_sizes"] == [8, 6, 0, 5]
    assert info["evals_per_run"][2] == 0
    for i in erased:
        assert torch.equal(out[i], frames[i]), i

    # the manual chain
    x = frames.clone()
    masks, bboxes = P.iris_masks_and_bboxes(x, segs)
    cr = P.crop_resize_irises(x, masks, bboxes, size=(64, 64))
    idx = torch.nonzero(bboxes[:, 2] >= 0).flatten()
    new, _, _, _ = P.nst(cr[idx], style, BN_loss=True, s_loss_weight=1e4, epochs=20, vgg=mods["vgg"], use_tqdm=False,
                         device="cuda:0", x_hist_stride=0, problem_sizes=[8, 6, 5])
    sub = x[idx]
    P.composite_irises(sub, new, masks[idx], bboxes[idx])
    x[idx] = sub
    torch.cuda.synchronize()
    assert torch.equal(out, x)

    # each run against its own call
    hc, hs = info["c_loss_per_run"].numpy(), info["s_loss_per_run"].numpy()
    for k in (0, 1, 3):
        lo, hi = g * k, min(B, g * (k + 1))
        ok, oinfo = api.stylize_frames(frames[lo:hi], style, segs=segs[lo:hi], **kw)
        torch.cuda.synchronize()
        ch, sh = oinfo["c_loss_hist"], oinfo["s_loss_hist"]
        print("run %d: evals %d/%d s %.5g/%.5g %.5g/%.5g final-frame MAE vs its own call %.3e" % (
            k, info["evals_per_run"][k], len(sh), hs[0, k], sh[0], hs[1, k], sh[1],
            float((out[lo:hi] - ok).abs().mean())))
        assert info["evals_per_run"][k] == len(sh)
        assert hs[0, k] == pytest.approx(sh[0], rel=1e-2) and hs[1, k] == pytest.approx(sh[1], rel=2e-2)
        assert hc[0, k] == pytest.approx(ch[0], abs=1e-12)
