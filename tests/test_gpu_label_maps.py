"""uint8 label maps on the B200, from the segmenter to every consumer: RITnet(label_dtype=torch.uint8) ->
mask / bbox (isx_mask_bbox_typed) -> cal_IoUs (isx_seg_iou_typed) -> extract_eye_landmarks_batch, with no widening pass.
Index work: every result is asserted EQUAL to the int64 path on the widened maps."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env(golden_dir):
    import iris_b200
    from oracle import metrics_oracle as M

    gold = np.load(os.path.join(golden_dir, "ritnet.npz"))
    sd = {k[2:]: torch.from_numpy(gold[k]) for k in gold.files if k.startswith("w:")}
    return dict(ib=iris_b200, M=M, gold=gold, rit64=iris_b200.RITnet(state_dict=sd),
                rit8=iris_b200.RITnet(state_dict=sd, label_dtype=torch.uint8),
                mgold=np.load(os.path.join(golden_dir, "metrics.npz")))


@pytest.fixture
def calls(env, monkeypatch):
    """Record every libisx call: name and, for tensor arguments, (data_ptr, dtype)."""
    lib = env["ib"]._lib
    log, call = [], lib.call

    def rec(name, *args):
        log.append((name, [(a.data_ptr(), a.dtype) if isinstance(a, torch.Tensor) else a for a in args]))
        return call(name, *args)

    monkeypatch.setattr(lib, "call", rec)
    return log


@pytest.mark.parametrize("k,seed,h,w", [(0, 5, 640, 400), (1, 6, 400, 640), (2, 7, 64, 48), (3, 8, 160, 96)])
def test_ritnet_uint8_labels_equal_reference(env, k, seed, h, w):
    ib, gold = env["ib"], env["gold"]
    x = torch.from_numpy(ib.synthetic.synthetic_eye(seed, h, w)[0]).cuda()
    lab, logits = env["rit8"](x, return_logits=True)
    assert lab.dtype == torch.uint8 and tuple(lab.shape) == (1, h, w) and lab.is_cuda
    assert np.array_equal(lab.cpu().numpy(), gold["syn%d_labels" % k])
    lab64, logits64 = env["rit64"](x, return_logits=True)
    assert torch.equal(logits, logits64)


def test_ritnet_uint8_batch_equals_int64(env):
    frames, _ = env["ib"].synthetic.synthetic_batch([5, 9, 10, 11, 12], 400, 640)
    x = torch.from_numpy(frames).cuda()
    a = env["rit64"](x)
    b = env["rit8"](x)
    assert b.dtype == torch.uint8 and torch.equal(b, a.to(torch.uint8))


def _mask_bbox(lib, x, seg, dt, label, thr):
    B, _, H, W = x.shape
    mask = torch.empty(B, 1, H, W, device="cuda", dtype=torch.uint8)
    xm = torch.empty_like(x)
    bbox = torch.empty(B, 4, device="cuda", dtype=torch.int32)
    if dt is None:
        lib.call("isx_mask_bbox", x, seg, label, int(thr), lib.f32(0.8), mask, xm, bbox, B, H, W, lib.stream_ptr())
    else:
        lib.call("isx_mask_bbox_typed", x, seg, dt, label, int(thr), lib.f32(0.8), mask, xm, bbox, B, H, W, lib.stream_ptr())
    torch.cuda.synchronize()
    return mask, xm, bbox


@pytest.mark.parametrize("B,H,W,offset", [(3, 640, 400, 0), (2, 400, 640, 0), (3, 37, 53, 0), (2, 64, 48, 1), (1, 400, 640, 0),
                                          (2, 400, 640, 1)])
def test_mask_bbox_uint8_equals_int64(env, B, H, W, offset):
    """Vector path (W % 4 == 0, 4-byte aligned uint8 rows) and scalar path (W % 4 != 0, or a seg view one byte off)."""
    ib = env["ib"]
    g = torch.Generator().manual_seed(B * H + W + offset)
    x = torch.rand(B, 1, H, W, generator=g).cuda()
    lab = torch.randint(0, 4, (B, 1, H, W), generator=g)
    lab[torch.rand(B, 1, H, W, generator=g) < 0.05] = 255
    lab[0][lab[0] == 2] = 0                                 # frame 0 has no iris: row_max = -1 for label 2
    flat = torch.zeros(B * H * W + offset, dtype=torch.uint8)
    flat[offset:] = lab.reshape(-1).to(torch.uint8)
    seg8 = flat.cuda()[offset:].view(B, 1, H, W)            # offset 1: not 4-byte aligned -> VEC = 1
    assert (seg8.data_ptr() % 4 == 0) == (offset == 0)
    seg64 = lab.cuda()
    for label in (0, 2, 3, 255, 300):
        for thr in (False, True):
            want = _mask_bbox(ib._lib, x, seg64, None, label, thr)
            got = _mask_bbox(ib._lib, x, seg8, 1, label, thr)
            for a, b in zip(got, want):
                assert torch.equal(a, b), (label, thr)
            if label == 2:
                assert int(want[2][0, 2]) == -1
            if label == 300:
                assert int(want[0].sum()) == 0 and bool((want[2][:, 2] == -1).all())


def test_mask_and_crop_and_iris_masks_read_uint8(env, calls):
    ib = env["ib"]
    frames, segs = ib.synthetic.synthetic_batch([21, 22, 23], 640, 400)
    x, s64 = torch.from_numpy(frames).cuda(), torch.from_numpy(segs).cuda()
    s8 = s64.to(torch.uint8)
    assert all(torch.equal(a, b) for a, b in zip(ib.iris_masks_and_bboxes(x, s8), ib.iris_masks_and_bboxes(x, s64)))
    r8 = ib.mask_and_crop_iris(x[0], seg=s8[0])
    r64 = ib.mask_and_crop_iris(x[0], seg=s64[0])
    assert torch.equal(r8[0], r64[0]) and torch.equal(r8[1], r64[1]) and r8[2:] == r64[2:]
    mb = [a for n, a in calls if n == "isx_mask_bbox_typed"]
    assert [a[2] for a in mb] == [1, 0, 1, 0]
    assert mb[0][1] == (s8.data_ptr(), torch.uint8) and mb[2][1] == (s8.data_ptr(), torch.uint8)   # no widening copy


def _ious(ib, p, t, nc=4):
    per_class, miou = ib.cal_IoUs(p, t, num_class=nc)
    return torch.stack(per_class, dim=1).cpu(), miou.cpu()


@pytest.mark.parametrize("name,shape", [("2019", (640, 400)), ("small", (37, 53))])
def test_ious_uint8_equal_reference_golden(env, name, shape):
    ib, gold = env["ib"], env["mgold"]
    p, t = ib.synthetic.iou_case(shape)
    p8, t8 = torch.from_numpy(p).to(torch.uint8).cuda(), torch.from_numpy(t).to(torch.uint8).cuda()
    iou, miou = _ious(ib, p8, t8)
    assert np.array_equal(iou.numpy(), gold["iou_" + name])
    i64, m64 = _ious(ib, torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda())
    assert torch.equal(iou, i64) and torch.equal(miou, m64)


def test_ious_uint8_shapes_classes_alignment(env, calls):
    ib, M = env["ib"], env["M"]
    rng = np.random.default_rng(5)
    cases = [(1, 1, 1, 4), (3, 5, 7, 2), (2, 33, 31, 8), (7, 64, 96, 4), (1, 400, 640, 4), (2, 17, 1025, 3), (16, 400, 640, 4),
             (5, 37, 53, 1), (3, 16, 16, 5), (2, 3, 17, 6), (4, 31, 33, 7)]
    for (b, h, w, nc) in cases:
        p = rng.integers(0, 256, size=(b, h, w), dtype=np.uint8)      # labels 0..255: most are "no class"
        t = rng.integers(0, 256, size=(b, h, w), dtype=np.uint8)
        dense = rng.random((b, h, w)) < 0.7                             # and a dense share inside 0..nc-1
        p[dense] = rng.integers(0, nc, size=int(dense.sum()))
        t[dense] = np.where(rng.random(int(dense.sum())) < 0.8, p[dense], rng.integers(0, nc, size=int(dense.sum())))
        P8, T8 = torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda()
        i8, m8 = _ious(ib, P8, T8, nc)
        i64, m64 = _ious(ib, P8.long(), T8.long(), nc)
        assert torch.equal(i8, i64) and torch.equal(m8, m64), (b, h, w, nc)
        iou_ref, _ = M.cal_ious(p.astype(np.int64), t.astype(np.int64), nc)
        assert np.array_equal(i8.numpy(), iou_ref), (b, h, w, nc)
        # misaligned views: one map one byte off (the maps' alignments differ) and both one byte off (scalar head and tail)
        for op, ot in ((1, 0), (0, 1), (1, 1), (3, 3)):
            fp = torch.zeros(p.size + op, dtype=torch.uint8, device="cuda")
            ft = torch.zeros(t.size + ot, dtype=torch.uint8, device="cuda")
            fp[op:] = P8.reshape(-1)
            ft[ot:] = T8.reshape(-1)
            iv, mv = _ious(ib, fp[op:].view(b, h, w), ft[ot:].view(b, h, w), nc)
            assert torch.equal(iv, i64) and torch.equal(mv, m64), (b, h, w, nc, op, ot)
    codes = [a[2] for n, a in calls if n == "isx_seg_iou_typed"]
    assert codes == [1, 0, 1, 1, 1, 1] * len(cases)                  # uint8 pairs read as uint8, no widening


def test_ious_mixed_dtypes_widen(env):
    """uint8 against int64 widens the uint8 map: an int64 value >= 256 stays "no class" instead of wrapping to 0..255."""
    ib, M = env["ib"], env["M"]
    rng = np.random.default_rng(8)
    p = rng.integers(0, 4, size=(3, 37, 53))
    t = p.copy()
    t[rng.random(t.shape) < 0.3] += 256                                  # 256 + c: no class, but c after a uint8 cast
    a, ma = _ious(ib, torch.from_numpy(p).to(torch.uint8).cuda(), torch.from_numpy(t).cuda())
    b, mb = _ious(ib, torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda())
    assert torch.equal(a, b) and torch.equal(ma, mb)
    assert np.array_equal(a.numpy(), M.cal_ious(p, t, 4)[0])
    assert not torch.equal(a, _ious(ib, torch.from_numpy(p).to(torch.uint8).cuda(), torch.from_numpy(t).to(torch.uint8).cuda())[0])


def test_stylize_frames_uint8_segs(env, vgg_weights):
    """uint8 segs from the device and from pinned host memory == the int64 call: frames, masks, bboxes."""
    ib = env["ib"]
    vgg = ib.VGG19(weights=vgg_weights)
    frames, segs = ib.synthetic.synthetic_batch([31, 32, 33], 400, 640)
    style = torch.from_numpy(ib.synthetic.synthetic_iris_crops([34], 64)[0, :1]).cuda()
    kw = dict(vgg=vgg, s_loss_weight=1e4, epochs=10, size=(64, 64))
    fr = torch.from_numpy(frames).cuda()
    s64 = torch.from_numpy(segs)
    ref, rinfo = ib.stylize_frames(fr, style, segs=s64.cuda(), **kw)
    ref2, _ = ib.stylize_frames(fr, style, segs=s64.cuda(), **kw)
    for segs8 in (s64.to(torch.uint8).cuda(), s64.to(torch.uint8).pin_memory()):
        out, info = ib.stylize_frames(fr, style, segs=segs8, **kw)
        torch.cuda.synchronize()
        assert torch.equal(info["masks"], rinfo["masks"]) and torch.equal(info["bboxes"], rinfo["bboxes"])
        assert torch.equal(info["valid"], rinfo["valid"])
        if torch.equal(ref, ref2):          # the NST is bit-reproducible run to run: the uint8 call must be bit-identical
            assert torch.equal(out, ref)
        else:                               # otherwise within the int64 call's own run-to-run spread
            assert float((out - ref).abs().max()) <= 2 * float((ref2 - ref).abs().max())


def test_driver_chain_uint8_segmenter(env, calls):
    """RITnet(label_dtype=torch.uint8) as the segmenter: mask / crop -> cal_IoUs -> extract_eye_landmarks_batch ->
    GazeEstimator1 equal the default int64 chain, and the uint8 maps reach every kernel as they are."""
    ib = env["ib"]
    rit8, rit64 = env["rit8"], env["rit64"]
    frames, _ = ib.synthetic.synthetic_batch([41, 42, 43, 44], 400, 640)
    x = torch.from_numpy(frames).cuda()
    post_x = x.flip(-1).contiguous()                        # a second set of frames for the pre / post IoU
    r8 = ib.mask_and_crop_iris(x[0], ritnet=rit8)
    r64 = ib.mask_and_crop_iris(x[0], ritnet=rit64)
    assert torch.equal(r8[0], r64[0]) and torch.equal(r8[1], r64[1]) and r8[2:] == r64[2:]
    pre8, post8 = rit8(x), rit8(post_x)
    pre64, post64 = rit64(x), rit64(post_x)
    assert pre8.dtype == torch.uint8 and torch.equal(pre8, pre64.to(torch.uint8))
    del calls[:]
    i8, m8 = _ious(ib, post8, pre8)
    lm8 = ib.extract_eye_landmarks_batch(pre8)
    log8 = list(calls)
    i64, m64 = _ious(ib, post64, pre64)
    assert torch.equal(i8, i64) and torch.equal(m8, m64)
    assert torch.equal(lm8, ib.extract_eye_landmarks_batch(pre64))
    params, _ = ib.synthetic.gaze_head_case(19)
    names = ["model.0.weight", "model.0.bias", "model.3.weight", "model.3.bias", "model.6.weight", "model.6.bias"]
    net = ib.GazeEstimator1(extract_feature=True, state_dict={k: torch.from_numpy(p) for k, p in zip(names, params)}).to("cuda:0")
    assert torch.equal(net(pre8), net(pre64))
    # no widening pass: the kernels read RITnet's own uint8 buffers
    iou_call = [a for n, a in log8 if n == "isx_seg_iou_typed"][0]
    assert iou_call[0] == (post8.data_ptr(), torch.uint8) and iou_call[1] == (pre8.data_ptr(), torch.uint8) and iou_call[2] == 1
    lm_call = [a for n, a in log8 if n == "isx_eye_landmarks"][0]
    assert lm_call[0] == (pre8.data_ptr(), torch.uint8) and lm_call[1] == 1
