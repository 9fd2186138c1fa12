"""The per-batch body of the reference's experiment drivers, batched on the device
(iris_style_transfer_openeds2019.py:64-79,93-100,111-137; iris_style_transfer_openeds2020.py:78-139):

    iris mask = (label map == 2) & (frame <= glint threshold)   -> bbox of the masked frame
    crop to the bbox, Resize(224x224, antialiased), repeat to 3 channels
    nst(content irises, style iris(es))                          -> new irises
    rgb_to_grayscale -> Resize(bbox shape) -> * mask -> paste into the frame

The reference loops over the batch in Python for the crop and for the composite; here each of the three image
stages is ONE kernel launch for the whole batch with ragged per-image windows (isx_mask_bbox,
isx_crop_resize_masked, isx_composite) and nothing synchronises with the host except the validity read of the
bounding boxes.  The segmenter (the mask PRODUCER) is the caller's: pass its label maps as `segs`, or a callable
`segmenter(frames) -> label maps` such as iris_b200.RITnet (the 2019 driver's segmenter on the GPU)."""
from __future__ import annotations

from typing import Callable, Dict, Optional

import torch

from . import _lib
from .pipelines import composite_irises, crop_resize_irises, iris_masks_and_bboxes, nst


def _ev(dev):
    e = torch.cuda.Event(enable_timing=True)
    e.record(torch.cuda.current_stream(dev))
    return e


@torch.no_grad()
def stylize_frames(frames: torch.Tensor,
                   style_iris: torch.Tensor,
                   segs: Optional[torch.Tensor] = None,
                   segmenter: Optional[Callable[[torch.Tensor], torch.Tensor]] = None,
                   vgg=None,
                   c_loss_weight: float = 1,
                   s_loss_weight: float = 1,
                   epochs: int = 200,
                   BN_loss: bool = True,
                   glint_threshold: float = 0.8,
                   label: int = 2,
                   size=(224, 224),
                   device: str = 'cuda:0',
                   independent: bool = False,
                   inplace: bool = False,
                   **nst_kw):
    """frames: [B,1,H,W] fp32 eye frames (host or device); style_iris: what the drivers hand to nst() as the style --
    (1,h,w) / (3,h,w) unbatched like …2020.py:103-104, or [B|1,1|3,h,w]; segs: label maps [B,1,H,W], host or device
    (int64 and uint8 are read as they are, uint8 moves 1 B per pixel; or `segmenter`, e.g. iris_b200.RITnet).  Returns (new_frames [B,1,H,W] on the device, info) with info = {masks, bboxes, valid, irises,
    c_loss_hist, s_loss_hist, evals, timings_ms}.  Frames without a single iris pixel are returned unchanged
    (valid[i] False; the reference would fail in crop_image).  nst()'s `problem_size` is not accepted: dropping the frames
    without an iris would leave problems of unequal size."""
    if "problem_size" in nst_kw:
        raise ValueError("stylize_frames does not take problem_size: frames without an iris are dropped from the NST batch, "
                         "so its problems would not all have the same size")
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise _lib.IsxError("iris_b200.stylize_frames runs on a CUDA B200 only; there is no CPU path")
    if dev.index is None:
        dev = torch.device('cuda', torch.cuda.current_device())
    with torch.cuda.device(dev):
        t0 = _ev(dev)
        x = frames.to(dev, torch.float32, non_blocking=True)
        if x.dim() == 3:
            x = x[:, None]
        x = x.contiguous() if inplace else x.clone().contiguous()
        B, _, H, W = x.shape
        if segs is None:
            if segmenter is None:
                raise ValueError("stylize_frames: pass `segs` (label maps) or `segmenter` (callable: frames -> label maps)")
            segs = segmenter(x)
        segs = segs.to(dev, non_blocking=True).reshape(B, 1, H, W)
        t1 = _ev(dev)
        masks, bboxes = iris_masks_and_bboxes(x, segs, glint_threshold=glint_threshold, label=label)
        t2 = _ev(dev)
        crops = crop_resize_irises(x, masks, bboxes, size=size)
        t3 = _ev(dev)
        valid = (bboxes[:, 2] >= 0)
        valid_h = valid.cpu()                      # the one host synchronisation: which frames have an iris at all
        idx = torch.nonzero(valid_h).flatten()
        info: Dict[str, object] = dict(masks=masks, bboxes=bboxes, valid=valid_h)
        if idx.numel() == 0:
            info.update(irises=crops, c_loss_hist=[], s_loss_hist=[], evals=0, timings_ms={})
            return x, info
        all_valid = idx.numel() == B
        c_in = crops if all_valid else crops[idx.to(dev)]
        s_in = style_iris
        if s_in.dim() == 4 and s_in.shape[0] == B and not all_valid:
            s_in = s_in[idx.to(s_in.device)]
        if s_in.dim() == 4 and s_in.shape[1] == 1:
            s_in = s_in.repeat(1, 3, 1, 1)          # …2019.py:94 `s_irises.repeat(1, 3, 1, 1)`
        new, _, c_hist, s_hist = nst(c_in, s_in, BN_loss=BN_loss, c_loss_weight=c_loss_weight, s_loss_weight=s_loss_weight,
                                     epochs=epochs, vgg=vgg, use_tqdm=False, device=str(dev), independent=independent,
                                     x_hist_stride=nst_kw.pop("x_hist_stride", 0), **nst_kw)
        t4 = _ev(dev)
        if all_valid:
            composite_irises(x, new, masks, bboxes)
        else:
            sub = x[idx.to(dev)]
            composite_irises(sub, new, masks[idx.to(dev)], bboxes[idx.to(dev)])
            x[idx.to(dev)] = sub
        t5 = _ev(dev)
        torch.cuda.current_stream(dev).synchronize()
        info.update(irises=new, c_loss_hist=c_hist, s_loss_hist=s_hist, evals=len(s_hist),
                    timings_ms=dict(upload_segment=t0.elapsed_time(t1), mask_bbox=t1.elapsed_time(t2),
                                    crop_resize=t2.elapsed_time(t3), nst=t3.elapsed_time(t4), composite=t4.elapsed_time(t5)))
    return x, info


# ---------------------------------------------------------------------------------------------------------------
# BASELINE config[3]: OpenEDS2020-shaped synthetic eye sequences, privacy-masking NST, sharded over the GPUs of a box
# ---------------------------------------------------------------------------------------------------------------
def bench_frames2020(args, dev, vgg, world: int, rank: int, dump=None):
    """One JSON line for `bench.py --config frames2020`: every rank stylises its own batches of 128 synthetic 400x640
    frames (the 2020 driver's batch size, …2020.py:211) against ONE fixed 224x224 style iris (…2020.py:238-249), default
    StyleLoss_BN, the batch as one L-BFGS problem, 200 evaluations, from pinned host frames + label maps to pinned host
    frames -- mask, bbox, crop, resize, NST, composite all inside the timed region.  One step = one batch (`--steps`).
    `dump(frames)`, if given, receives the stylised frames of the last batch (pinned host memory)."""
    import time

    import numpy as np
    import torch.distributed as dist

    from . import synthetic

    Hf, Wf = 400, 640                                   # OpenEDS2020 frames are (1,400,640) (gaze_estimators.py:121)
    B = args.batch or 128
    n_batches = args.steps
    epochs = 200
    fr, sg = synthetic.synthetic_batch([50000 * rank + i for i in range(B)], Hf, Wf)
    frames_h = torch.from_numpy(fr).pin_memory()
    segs_h = torch.from_numpy(sg).pin_memory()
    sf, ss = synthetic.synthetic_eye(777, Hf, Wf)       # the one-for-all style frame
    sx, sseg = torch.from_numpy(sf).to(dev)[None], torch.from_numpy(ss).to(dev)[None]
    smask, sbb = iris_masks_and_bboxes(sx, sseg)
    s_iris = crop_resize_irises(sx, smask, sbb)[0, :1].contiguous()          # (1,224,224), unbatched like …2020.py:103
    out_h = torch.empty_like(frames_h).pin_memory()
    kw = dict(vgg=vgg, c_loss_weight=1.0, s_loss_weight=1e4, epochs=epochs, BN_loss=True, device=str(dev))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stylize_frames(frames_h, s_iris, segs=segs_h, **dict(kw, epochs=20))     # warm-up: workspaces, allocator
    barrier()
    t0 = time.perf_counter()
    stages: Dict[str, float] = {}
    evals = 0
    for _ in range(n_batches):
        out, info = stylize_frames(frames_h, s_iris, segs=segs_h, **kw)
        out_h.copy_(out, non_blocking=True)
        for k, v in info["timings_ms"].items():
            stages[k] = stages.get(k, 0.0) + v
        evals = info["evals"]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if dump is not None:
        dump(out_h)
    t = torch.tensor([dt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    n_frames = world * B * n_batches
    px = Hf * Wf
    # algorithmic bytes of the three image stages per frame: labels 8 B + pixel 4 B read, mask 1 B written;
    # crop: window read (<= px * 5 B) + 3*224*224*4 written; composite: 3*224*224*4 read + window read-modify-write
    gbs = lambda bytes_, ms: (bytes_ * B * n_batches / (ms / 1e3) / 1e9) if ms > 0 else None
    moved = float((out_h - frames_h).abs().mean())
    return {
        "metric": "privacy-masking NST image-steps/sec, OpenEDS2020-shaped 400x640 frames end to end", "value": n_frames * evals / dt,
        "unit": "image-steps/s", "n_gpus": world, "steps": n_batches, "warmup": 1, "ms_per_step": 1e3 * dt / n_batches,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "BASELINE config[3]: %d batches of %d synthetic OpenEDS2020-shaped 400x640 frames per GPU, one fixed "
                               "224x224 style iris, mask -> bbox -> crop -> resize -> nst(BN loss, batch as one problem, %d evaluations) "
                               "-> composite, host frames in / host frames out" % (n_batches, B, epochs),
                   "name": "frames2020", "batch_per_gpu": B, "image": "1x%dx%d -> 3x224x224" % (Hf, Wf)},
        "frames_per_s": n_frames / dt, "evals_per_frame": evals,
        "stages_ms_rank0": stages,
        "image_ops_gbs_rank0": {"mask_bbox": gbs(px * 13.0, stages.get("mask_bbox", 0.0)),
                                "crop_resize": gbs(3 * 224 * 224 * 4.0 + 0.1 * px * 5.0, stages.get("crop_resize", 0.0)),
                                "composite": gbs(3 * 224 * 224 * 4.0 + 0.1 * px * 9.0, stages.get("composite", 0.0))},
        "sanity": {"frames_changed_mae": moved, "valid_frames": int(info["valid"].sum())},
    }
