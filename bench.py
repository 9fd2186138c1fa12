#!/usr/bin/env python
"""bench.py -- masked-NST image-steps/s @640x400 VGG-19 (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: a closure evaluation (VGG-19 forward to the deepest tap,
style + content losses, backward to the image) plus one L-BFGS iteration for every image of the batch.
Default workload = BASELINE config[1]: 64 synthetic OpenEDS2019-shaped 640x400 eyes per GPU, iris-masked, random-init
VGG-19, Gram style loss, each image its own problem.  N > 1: one process per GPU (torchrun), each rank owns its own
batch (weak scaling), no collective on the inner loop; timing = max over ranks.

What a step costs does NOT depend on --steps: before the timed region the L-BFGS history is filled to its 100
pairs with untimed ticks (a 300-step job spends 2/3 of its life there), and `history_pairs_min/max` of the timed
region are printed.  The end-to-end leg always runs the whole BASELINE job (300 evaluations).

Prints ONE JSON line (rank 0).  `value`: inputs resident in HBM, CUDA-event timed.  `e2e`: the job through the public
API `iris_b200.nst()` from pinned HOST tensors to HOST results (H2D / D2H inside the timed region).  `roofline`: the
tcgen05 conv kernel family, CUDA-event timed inside the timed region.  `cpu_baseline`: the CPU oracle (a port of the
reference path, oracle/nst_oracle.py) on this box's host cores (N = 1 only).  `gpu_library_baseline`: the reference's
own library calls (torchvision VGG-19 through cuDNN, torch.optim.LBFGS) on the same GPU, reported beside it.
`--impl reference` times the CPU path alone with the same metric/config.

--config: nst640 (default, BASELINE config[1]) | nst640_5tap (style taps relu1_1..relu5_1) | masked_gram (row G':
mask-weighted Gram via c_mask / s_mask) | nst224 (64 iris crops 224x224, default BN loss, the batch as one problem:
what the reference's drivers call) | nst1024 (BASELINE config[4]: 1024x1024 RGB, Gram loss) | feat4 / feat5
(BASELINE config[2]: style-feature extraction only, 4 / 5 taps) | frames2020 (BASELINE config[3]: OpenEDS2020-shaped
400x640 frames end to end: mask -> crop -> resize -> NST -> composite) | landmarks (SURVEY §8f row 4: 400x640 label maps
-> 19 eye landmarks -> GazeEstimator1; frames/s, roofline of the bit-plane kernel, cv2 on one host core beside it).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "masked-NST image-steps/sec @640x400 VGG-19"
UNIT = "image-steps/s"
H, W = 640, 400
# SURVEY.md §8(d), per image-step: fwd->deepest tap + dgrad + Gram fwd/bwd (FLOPs = 2*9*Cin*Cout*H*W per conv, 2*C^2*HW per Gram)
FLOPS_640 = {"4tap": 301.66e9, "5tap": 387.65e9}
STYLE4 = ["relu1_1", "relu2_1", "relu3_1", "relu4_1"]
STYLE5 = STYLE4 + ["relu5_1"]


def flops_per_image_step(h, w, taps5=False, gram=True):
    """Same arithmetic as SURVEY.md §8(d) for any frame size (floor division of the pooled sizes like the network)."""
    cfg = [(3, 64), (64, 64), "M", (64, 128), (128, 128), "M", (128, 256), (256, 256), (256, 256), (256, 256), "M",
           (256, 512), (512, 512), (512, 512), (512, 512), "M", (512, 512)]
    last = 13 if taps5 else 10   # number of convs up to relu5_1 / relu4_2
    tap_after = {1: 64, 3: 128, 5: 256, 9: 512, 13: 512} if taps5 else {1: 64, 3: 128, 5: 256, 9: 512}
    fl, n, hh, ww = 0.0, 0, h, w
    for v in cfg:
        if v == "M":
            hh, ww = hh // 2, ww // 2
            continue
        n += 1
        if n > last:
            break
        fl += 2.0 * 2 * 9 * v[0] * v[1] * hh * ww          # forward + dgrad
        if gram and n in tap_after:
            fl += 2.0 * 2 * tap_after[n] ** 2 * hh * ww     # Gram forward + backward
    return fl


def make_inputs(batch, seed0, h=H, w=W):
    """Iris-masked synthetic eyes: frame * ((seg == 2) & (frame <= 0.8)), replicated to 3 channels."""
    import numpy as np
    import torch

    from iris_b200 import synthetic

    def masked(seeds):
        frames, segs = synthetic.synthetic_batch(seeds, h, w)
        m = (segs == 2) & (frames <= np.float32(0.8))
        return torch.from_numpy(frames * m).repeat(1, 3, 1, 1).contiguous()

    c = masked([seed0 + i for i in range(batch)])
    s = masked([seed0 + 100000 + i for i in range(batch)])
    return c, s


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.samples:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the reference path's CPU implementation (oracle port)
# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_rate(steps, warmup, threads=None, dump_dir=None):
    """B = 1 closure evaluations + L-BFGS on one 640x400 masked eye (BASELINE config[0] shape), all host threads.
    The forward runs the WHOLE vgg19.features stack to pool5 like the reference does (models/vgg/vgg.py:87),
    although nothing past relu4_2 is consumed.  Returns image-steps/s."""
    import torch

    from oracle import nst_oracle as O

    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    weights = O.random_vgg19_weights(0)
    c, s = make_inputs(1, 1)
    with torch.no_grad():
        _, c_feats, _ = O.vgg19_forward(c, weights, full=True)
        _, _, s_feats = O.vgg19_forward(s, weights, full=True)
        t_gram = [O.gram_matrix(t) for t in s_feats]
    x = c.clone()
    opt = O.LBFGS(x, lr=1.0)
    count = [0]
    t0 = [None]
    total = warmup + steps

    class Done(Exception):
        """Raised by the closure after the last timed evaluation: opt.step() runs up to 20 of them per call."""

    def closure():
        if count[0] == warmup:
            t0[0] = time.perf_counter()
        if count[0] == total:
            raise Done
        with torch.no_grad():
            x.clamp_(0, 1)
        xv = x.detach().requires_grad_(True)
        with torch.enable_grad():
            _, x_c, x_s = O.vgg19_forward(xv, weights, full=True)
            cl = O.content_loss_l2(x_c, c_feats)
            sl = O.style_loss_gram(x_s, t_gram)
            loss = cl + 1e6 * sl
            (g,) = torch.autograd.grad(loss, xv)
        count[0] += 1
        return float(loss), g.reshape(-1)

    try:
        while True:
            opt.step(closure)
    except Done:
        pass
    dt = time.perf_counter() - t0[0]
    if dump_dir:   # the image an nst() caller would receive after the last timed evaluation's update
        dump_outputs(dump_dir, {"x": x.clamp(0, 1)})
    return steps / dt, steps, dt, threads


def run_reference(args, rank):
    if rank != 0:
        return
    if args.config == "landmarks":      # row f4: the reference's own per-frame OpenCV path on one host thread
        import numpy as np

        sys.path.insert(0, os.path.join(ROOT, "iris-style-transfer_b200"))
        import synthetic

        labs = np.stack([synthetic.synthetic_label_map(i, speck=0.002 * (i % 4)) for i in range(32)])
        rate, n = cv2_landmark_rate(labs, seconds=10.0)
        print(json.dumps({"impl": "reference", "metric": "eye-landmark frames/sec @400x640 label maps (extract_eye_landmarks + GazeEstimator1)",
                          "value": rate, "unit": "frames/s", "n_gpus": args.gpus, "steps": n, "warmup": 1, "ms_per_step": 1e3 / rate,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8 / f64", "data": "synthetic",
                          "config": {"workload": "row f4: synthetic 400x640 label maps, 0-0.6 % stray pixels, one frame per step", "name": "landmarks"},
                          "cpu_baseline": {"value": rate, "unit": "frames/s", "cores": 1, "kind": "reference",
                                           "sample": "%d frames through cv2.findContours / contourArea / fitEllipse + np.where" % n},
                          "e2e": {"value": rate, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}),
              flush=True)
        return
    steps = max(1, args.steps)
    rate, done, dt, threads = cpu_reference_rate(steps, args.warmup, dump_dir=args.dump_outputs)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / done, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "iris-masked Gatys NST, 640x400 synthetic eyes, random-init VGG-19, Gram style loss "
                               "(s_loss_weight 1e6), L-BFGS; reference arm: one image per step on the host CPU, "
                               "full vgg19.features forward to pool5 like models/vgg/vgg.py:87"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d closure evaluations + L-BFGS iterations of one 640x400 image (oracle/nst_oracle.py, "
                                   "torch CPU fp32, %d threads)" % (done, threads)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# GPU library comparator: the reference's own library calls on the same B200 (SURVEY §8d "second baseline")
# ---------------------------------------------------------------------------------------------------------------
def gpu_library_rate(dev, c, s, mode, evals=20, history_copy=True):
    """pipelines.py:44-103 restated with the SAME library calls the reference makes -- torchvision vgg19.features
    (all 37 modules to pool5), F.mse_loss, bmm Gram, torch.optim.LBFGS([x], lr=1), the batch as ONE problem -- on
    `dev`.  mode 'tf32': fp32 tensors, PyTorch defaults (cuDNN convs may use TF32, matmul fp32).  mode 'bf16':
    channels_last + autocast(bfloat16), the strongest stock configuration.  history_copy: keep the reference's
    per-evaluation `x.cpu()` + two `.item()` (pipelines.py:93-95).  Returns image-steps/s over `evals` evaluations
    after one warm-up optimizer.step."""
    import torch
    import torch.nn.functional as F
    import torchvision

    torch.manual_seed(0)
    net = torchvision.models.vgg19(weights=None).features.to(dev).eval()
    for p in net.parameters():
        p.requires_grad_(False)
    if mode == "bf16":
        net = net.to(memory_format=torch.channels_last)
    mean = torch.tensor([0.485, 0.456, 0.406], device=dev).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225], device=dev).view(1, 3, 1, 1)
    style_idx, content_idx = (1, 6, 11, 20), (22,)

    def vgg(x):
        h = (x - mean) / std
        if mode == "bf16":
            h = h.contiguous(memory_format=torch.channels_last)
        feats = {}
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16")):
            for i, m in enumerate(net):
                h = m(h)
                if i in style_idx or i in content_idx:
                    feats[i] = h
        return [feats[i].float() for i in content_idx], [feats[i].float() for i in style_idx]

    def gram(f):
        f = f.flatten(start_dim=-2)
        return (f @ f.transpose(-2, -1)) / f[0].numel()

    c, s = c.to(dev), s.to(dev)
    with torch.no_grad():
        c_t, _ = vgg(c)
        _, s_f = vgg(s)
        s_t = [gram(f) for f in s_f]
    x = c.clone().contiguous().requires_grad_(True)
    opt = torch.optim.LBFGS([x], lr=1)
    n = [0]
    hist = []

    def closure():
        with torch.no_grad():
            x.clamp_(0, 1)
        opt.zero_grad()
        x_c, x_s = vgg(x)
        cl = sum(F.mse_loss(p, t) for p, t in zip(x_c, c_t)) * 0.5
        sl = sum(((gram(p) - t) ** 2).sum() for p, t in zip(x_s, s_t)) * 0.25
        loss = cl + 1e6 * sl
        loss.backward()
        if history_copy:
            hist.append(x.detach().cpu())
            cl.item()
            sl.item()
        n[0] += 1
        return loss

    opt.step(closure)          # warm-up: cuDNN algorithm selection, allocator
    torch.cuda.synchronize(dev)
    n[0] = 0
    hist.clear()
    t0 = time.perf_counter()
    while n[0] < evals:
        opt.step(closure)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    return c.shape[0] * n[0] / dt, n[0]


# ---------------------------------------------------------------------------------------------------------------
# device-resident NST leg
# ---------------------------------------------------------------------------------------------------------------
def nst_leg(args, dev, vgg, c_dev, s_dev, BN_loss, independent, K, Wm, world, rank, local, lib, c_mask=None,
            s_mask=None, s_weight=1e6):
    import ctypes

    import torch
    import torch.distributed as dist

    from iris_b200 import _lib, pipelines

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    hist = 100
    prefill = 0 if args.no_prefill else hist + 2
    with torch.cuda.device(dev), torch.no_grad():
        jkw = dict(clone_content=True, BN_loss=BN_loss, c_loss_weight=1.0, s_loss_weight=s_weight, lr=1.0,
                   epochs=prefill + K + Wm + 40, independent=independent, history_size=hist,
                   history_dtype=torch.bfloat16 if args.history_bf16 else torch.float32, c_mask=c_mask, s_mask=s_mask)
        if args.streams > 1 and independent:
            job = pipelines.NstJobGroup(c_dev, s_dev, vgg, dev, streams=args.streams, overlap=args.overlap, **jkw)
            subjobs = job.jobs
        else:
            job = pipelines.NstJob(c_dev, s_dev, vgg, dev, **jkw)
            subjobs = [job]
        torch.cuda.synchronize()
        x0 = torch.cat([j.x for j in subjobs]).clone()
        if args.streams > 1 and independent:
            job.fork(dev)
        for _ in range(prefill + Wm):      # untimed: fills the L-BFGS ring, warms clocks / allocator / L2
            job.tick()
        if args.streams > 1 and independent:
            job.join(dev)
        barrier()
        pairs0 = torch.cat([j.history_counts() for j in subjobs])
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        lib.isx_prof_enable(1)
        launches0 = lib.isx_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if args.streams > 1 and independent:
            job.fork(dev)
        for _ in range(K):
            job.tick()
        if args.streams > 1 and independent:
            job.join(dev)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = int(lib.isx_launch_count() - launches0)
        prof = (ctypes.c_double * 12)()
        _lib.call("isx_prof_collect", prof, 12)
        lib.isx_prof_enable(0)
        clocks = sampler.stop() if rank == 0 else None
        pairs1 = torch.cat([j.history_counts() for j in subjobs])
        if args.dump_outputs and rank == 0:
            # what nst() hands back after the last timed step: the images clamped to [0, 1] and each problem's losses
            # (a problem that stopped early keeps its own last logged losses, as in NstJob.finish)
            x, idx = dump_sample(torch.cat([j.x for j in subjobs]).clamp(0, 1), DUMP_BUDGET - (1 << 20))
            c_loss, s_loss = [], []
            for j in subjobs:
                e = j.evals_done().to(j.hist_c.device).long()      # 0 while a problem still runs
                rows = torch.where(e > 0, e - 1, j.ticks - 1)
                cols = torch.arange(j.P, device=rows.device)
                c_loss.append(j.hist_c[rows, cols])
                s_loss.append(j.hist_s[rows, cols])
            dump_outputs(args.dump_outputs, {"x": x, "x_image_index": idx.double(), "c_loss": torch.cat(c_loss),
                                             "s_loss": torch.cat(s_loss)})
        moved = float((torch.cat([j.x for j in subjobs]) - x0).abs().mean())
        loss_first = float(sum(j.hist_s[0].sum() for j in subjobs))
        loss_last = float(sum(j.hist_s[j.ticks - 1].sum() for j in subjobs))
        evals_alive = int(sum(int((j.evals_done() == 0).sum()) for j in subjobs))
        P = sum(j.P for j in subjobs)
        del job, subjobs
        torch.cuda.empty_cache()
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return dict(ms=ms, ms_max=float(t.item()), launches=launches, prof=list(prof), clocks=clocks, moved=moved,
                loss_first=loss_first, loss_last=loss_last, pairs_min=int(min(pairs0.min(), pairs1.min())),
                pairs_max=int(max(pairs0.max(), pairs1.max())),
                pairs_mean=0.5 * (float(pairs0.float().mean()) + float(pairs1.float().mean())), problems=P, problems_running=evals_alive,
                prefill=prefill)


def feature_leg(dev, vgg, taps5, n_per_gpu, world, batch=32, passes=1, dump_dir=None):
    """BASELINE config[2]: style features (mean/std + Gram upper triangles of the style taps) of synthetic eyes for the
    iris classifier, image list sharded contiguously over the ranks, rows exchanged over NVLink (sharding.PeerRows).
    `passes` timed passes over the image list; `dump_dir`: the rows of the last one (rank 0)."""
    import torch
    import torch.distributed as dist

    import iris_b200
    from iris_b200 import features

    n_total = n_per_gpu * world
    base, _ = iris_b200.synthetic.synthetic_batch(list(range(16)), H, W)   # 16 distinct eyes, tiled
    base = torch.from_numpy(base).pin_memory()

    class Tiled:
        """n_total eyes = the 16 synthetic frames repeated; a slice is served from pinned memory (cached per phase)."""

        def __init__(self):
            self.cache = {}

        def __len__(self):
            return n_total

        def __getitem__(self, sl):
            key = (sl.start % base.shape[0], sl.stop - sl.start)
            if key not in self.cache:
                idx = torch.arange(sl.start, sl.stop) % base.shape[0]
                self.cache[key] = base[idx].pin_memory()
            return self.cache[key]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    imgs = Tiled()
    layers = STYLE5 if taps5 else STYLE4
    vgg_feat = iris_b200.VGG19(content_layers=[], style_layers=layers, weights=vgg.host_weights)
    features.extract_features_sharded(vgg_feat, imgs, batch=batch, device=dev)  # warm-up (workspaces, NCCL)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(passes):
        rows = features.extract_features_sharded(vgg_feat, imgs, batch=batch, device=dev)
    f1.record()
    barrier()
    if dump_dir and (world == 1 or dist.get_rank() == 0):
        r, idx = dump_sample(rows, DUMP_BUDGET - (1 << 20))
        dump_outputs(dump_dir, {"rows": r, "row_index": idx.double()})
    tf = torch.tensor([f0.elapsed_time(f1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tf, op=dist.ReduceOp.MAX)
    fl = 193.82e9 if taps5 else 131.96e9
    rate = passes * n_total / (float(tf.item()) / 1e3)
    out = {"metric": "Gram-feature images/sec @640x400 (%s: mean/std + Gram upper triangles)" % ("relu1_1..relu5_1" if taps5 else "relu1_1..relu4_1"),
           "value": rate, "unit": "images/s", "n_images": n_total, "feature_dim": int(rows.shape[1]),
           "all_gather_bytes": int(rows.numel() * 4), "flops_per_image": fl,
           "model_tflops_per_gpu": rate * fl / 1e12 / world,
           "note": "host (pinned) -> device copies of the frames inside the timed region; rows pushed into every rank over NVLink peer memory (copy engines; NCCL all-gather fallback)"}
    del rows
    torch.cuda.empty_cache()
    return out


DUMP_BUDGET = 64 << 20


def dump_sample(t, budget, seed=0):
    """(rows, row_index) of a (N, ...) tensor within `budget` bytes: all of it, else a seeded subset of rows, so that two
    builds run with the same arguments dump the same rows."""
    import torch

    t = t.detach().cpu()
    n = t.shape[0]
    per_row = max(1, t[:1].numel() * t.element_size())
    keep = min(n, max(1, budget // per_row))
    idx = torch.arange(n) if keep == n else torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:keep].sort().values
    return t[idx], idx


def dump_outputs(d, arrays):
    """Write {name: tensor} as d/<name>.npy in float32 (float64 stays float64); the total must fit DUMP_BUDGET."""
    import numpy as np
    import torch

    os.makedirs(d, exist_ok=True)
    out = {}
    for name, t in arrays.items():
        t = torch.as_tensor(t).detach().cpu()
        out[name] = t.numpy() if t.dtype == torch.float64 else t.float().numpy()
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_BUDGET:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte budget" % (total, DUMP_BUDGET))
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), a)


def measured_peaks():
    """HBM peak for the roofline legs: the driver-written MEASURED_PEAKS.json, else the profiling guide's fallback."""
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        if pk.get("hbm_gbs"):
            return {"hbm_gbs": float(pk["hbm_gbs"]), "source": "MEASURED_PEAKS.json hbm_gbs (of measured)"}
    except Exception:
        pass
    return {"hbm_gbs": 6650.0, "source": "B200_PROFILING.md fallback (of fallback)"}


def cv2_landmark_rate(labs, seconds=8.0):
    """The reference's own CPU path for row f4: per frame the three OpenCV calls per class + np.where that
    gaze_estimators.py:55-178 executes (cv2 is the third-party library the reference calls), one host thread like the
    reference's per-frame Python loop.  Returns (frames/s, frames timed)."""
    import cv2
    import numpy as np

    def one(seg):
        s8 = seg.astype(np.uint8)
        for cls in (3, 2):
            cs, _ = cv2.findContours((s8 == cls).astype(np.uint8), cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
            if cs:
                c = max(cs, key=cv2.contourArea)
                if len(c) >= 5:
                    cv2.fitEllipse(c)
        ys, xs = np.where((s8 == 1) > 0)
        return (xs.min(), xs.max(), ys.min(), ys.max()) if len(xs) else None

    one(labs[0])
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        one(labs[n % len(labs)])
        n += 1
    return n / (time.perf_counter() - t0), n


def landmarks_leg(args, dev, lib, world, rank, local):
    """`--config landmarks` (SURVEY.md §8f row 4): 128 OpenEDS2020-shaped 400x640 label maps per GPU and step -> 19 eye
    landmarks (extract_eye_landmarks) -> GazeEstimator1 gaze vectors.  A quarter of the maps each carry 0 / 0.2 / 0.4 / 0.6 %
    randomly relabelled pixels (up to ~450 stray contours per class)."""
    import ctypes

    import numpy as np
    import torch
    import torch.distributed as dist

    import iris_b200
    from iris_b200 import _lib

    B = args.batch or 128
    K, Wm = args.steps, args.warmup
    labs = np.stack([iris_b200.synthetic.synthetic_label_map(100000 * rank + i, speck=0.002 * (i % 4)) for i in range(B)])
    seg_h = torch.from_numpy(labs).pin_memory()
    seg = seg_h.to(dev)
    net = iris_b200.GazeEstimator1(extract_feature=True).to(dev)
    out_h = torch.empty(B, 3).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(Wm):
        net(seg)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.isx_prof_enable(1)
    launches0 = lib.isx_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for e0, e1 in ev:
        flush.zero_()                       # 256 MB written between steps: the label maps (262 MB) come from HBM
        e0.record()
        g = net(seg)
        e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"gaze": g})
    launches = int(lib.isx_launch_count() - launches0)
    prof = (ctypes.c_double * 12)()
    _lib.call("isx_prof_collect", prof, 12)
    lib.isx_prof_enable(0)
    ms = sum(e0.elapsed_time(e1) for e0, e1 in ev)
    # end to end: pinned host label maps -> device -> landmarks -> gaze vectors -> pinned host
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        g = net(seg_h.to(dev, non_blocking=True))
        out_h.copy_(g, non_blocking=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms, dt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, dt = float(t[0]), float(t[1])
    if rank != 0:
        return None
    from oracle import landmarks_oracle as L                      # checker only: the timed results against the oracle
    lm = iris_b200.extract_eye_landmarks_batch(seg[:4]).cpu().numpy()
    err = float(max(np.abs(lm[i] - L.extract_eye_landmarks(labs[i])).max() for i in range(4)))
    peaks = measured_peaks()
    plane_ms, plane_bytes = prof[3 * 3 + 1], prof[3 * 3 + 2]
    achieved = plane_bytes / (plane_ms / 1e3) / 1e9 if plane_ms > 0 else None
    traffic, traffic_src = None, "not measured in this run (ncu is not available inside the timed run)"
    try:      # DRAM traffic per launch: only from an ncu capture of this round committed under profiles/
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_landmarks_traffic.json")))
        if tr.get("batch") == B:
            traffic, traffic_src = tr["dram_bytes_per_launch"], tr["source"]
    except Exception:
        pass
    line = {"metric": "eye-landmark frames/sec @400x640 label maps (extract_eye_landmarks + GazeEstimator1)",
            "value": world * B * K / (ms / 1e3), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8 labels / int32 contours / f64 fit",
            "data": "synthetic",
            "config": {"workload": "row f4: %d synthetic OpenEDS2020-shaped 400x640 int64 label maps per GPU and step, 0-0.6 %% stray "
                                   "pixels, -> 19 landmarks -> GazeEstimator1 (19-64-64-3)" % B, "name": "landmarks", "batch_per_gpu": B,
                       "l2": "256 MB written between steps; the maps of one step are 262 MB"},
            "e2e": {"value": world * B * K / dt, "unit": "frames/s", "h2d_bytes_per_step": int(seg_h.numel() * 8),
                    "d2h_bytes_per_step": int(out_h.numel() * 4)},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": {"kernel": "lm_planes_kernel (labels -> pupil / iris bit planes + sclera bounding box)", "bound": "hbm",
                         "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": (achieved / peaks["hbm_gbs"]) if achieved else None, "traffic": traffic,
                         "traffic_source": traffic_src, "algorithmic_bytes_per_launch": plane_bytes / max(prof[3 * 3], 1.0),
                         "peak_source": peaks["source"], "share_of_step": plane_ms / ms if ms > 0 else None,
                         "note": "the rest of a step is lm_contour_kernel: one CTA per frame and class following borders out of "
                                 "shared memory -- latency-bound serial index work, no roofline applies"},
            "sanity": {"max_abs_diff_vs_oracle_first4": err}}
    if not args.no_cpu_baseline:
        rate, n = cv2_landmark_rate(labs)
        line["cpu_baseline"] = {"value": rate, "unit": "frames/s", "cores": 1, "kind": "reference",
                                "sample": "%d frames of the same batch through cv2.findContours / contourArea / fitEllipse + np.where "
                                          "(what gaze_estimators.py:55-178 executes per frame), one thread like the reference's loop" % n}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="isx", choices=["isx", "reference"])
    ap.add_argument("--config", default="nst640", choices=["nst640", "nst640_5tap", "masked_gram", "nst224", "nst1024",
                                                           "feat4", "feat5", "frames2020", "landmarks"])
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-library", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-features", action="store_true")
    ap.add_argument("--no-prefill", action="store_true", help="do not fill the L-BFGS history before timing (diagnostic)")
    ap.add_argument("--streams", type=int, default=1, help="sub-batches on separate CUDA streams (overlap L-BFGS and convs)")
    ap.add_argument("--overlap", action="store_true", help="with --streams > 1: L-BFGS passes on low-priority streams beside the convs")
    ap.add_argument("--smem-reserve-kb", type=int, default=0, help="shared memory per SM the persistent conv CTAs leave free")
    ap.add_argument("--history-bf16", action="store_true", help="opt-in: store the L-BFGS (s, y) history in bf16")
    ap.add_argument("--feature-images", type=int, default=512, help="images per GPU of the feature-extraction leg")
    ap.add_argument("--feature-batch", type=int, default=64, help="images per forward pass of the feature-extraction leg")
    ap.add_argument("--opt", action="append", default=[], help="name=value: libisx kernel-selection option (isx_set_option), repeatable")
    ap.add_argument("--e2e-evals", type=int, default=300, help="evaluations of the end-to-end job (BASELINE config[1]: 300)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (at most 64 MB, "
                         "a seeded sample of the images or rows when larger) to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference" and args.config == "landmarks":
        raise SystemExit("--dump-outputs: the landmarks reference arm times cv2 calls and keeps none of their results")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 40
        run_reference(args, rank)
        return
    if args.steps is None:   # a step: one tick of an NST job, one pass over the feature images, one batch of frames
        args.steps = {"feat4": 1, "feat5": 1, "frames2020": 2}.get(args.config, 100)
    if args.warmup < 3:
        args.warmup = 3

    import ctypes

    import torch
    import torch.distributed as dist

    import iris_b200
    from iris_b200 import _lib, sharding

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        sharding.init_from_env("nccl")
    lib = _lib.load()
    lib.isx_launch_count.restype = ctypes.c_ulonglong
    _lib.call("isx_device_check", local)
    if args.smem_reserve_kb:
        lib.isx_set_option(b"smem_reserve_kb", int(args.smem_reserve_kb))
    for kv in args.opt:
        name, val = kv.split("=")
        if lib.isx_set_option(name.encode(), int(val)) != 0:
            raise SystemExit("unknown libisx option %r" % name)

    def finish():
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()

    K, Wm = args.steps, args.warmup
    cfgname = args.config
    vgg = iris_b200.VGG19(weights="random", seed=0)

    # ------------------------------------------------------------------ feature-only configs
    if cfgname in ("feat4", "feat5"):
        feat = feature_leg(dev, vgg, cfgname == "feat5", args.feature_images, world, batch=args.feature_batch, passes=K,
                           dump_dir=args.dump_outputs)
        if rank == 0:
            line = {"metric": feat["metric"], "value": feat["value"], "unit": "images/s", "n_gpus": world, "steps": K,
                    "warmup": 1, "ms_per_step": 1e3 * feat["n_images"] / feat["value"], "higher_is_better": True,
                    "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                    "config": {"workload": "BASELINE config[2]: %d synthetic 640x400 eyes per GPU -> style features, sharded, "
                                           "all-gathered" % args.feature_images}, "detail": feat}
            print(json.dumps(line), flush=True)
        finish()
        return
    if cfgname == "landmarks":
        line = landmarks_leg(args, dev, lib, world, rank, local)
        if rank == 0:
            print(json.dumps(line), flush=True)
        finish()
        return
    if cfgname == "frames2020":
        from iris_b200 import frames as frames_mod

        def dump_frames(frames):
            f, idx = dump_sample(frames, DUMP_BUDGET - (1 << 20))
            dump_outputs(args.dump_outputs, {"frames": f, "frame_index": idx.double()})

        line = frames_mod.bench_frames2020(args, dev, vgg, world, rank,
                                           dump=dump_frames if args.dump_outputs and rank == 0 else None)
        if rank == 0:
            print(json.dumps(line), flush=True)
        finish()
        return

    # ------------------------------------------------------------------ NST configs
    h, w, B = H, W, args.batch or 64
    BN_loss, independent, s_weight = False, True, 1e6
    c_mask = s_mask = None
    taps5 = False
    if cfgname == "nst640_5tap":
        taps5 = True
        vgg = iris_b200.VGG19(style_layers=STYLE5, weights=vgg.host_weights)
    if cfgname == "nst1024":
        h, w, B = 1024, 1024, args.batch or 16
    if cfgname == "nst224":
        h, w, BN_loss, independent, s_weight = 224, 224, True, False, 1e4
    if cfgname == "nst224":
        ic = torch.from_numpy(iris_b200.synthetic.synthetic_iris_crops(list(range(1000 * rank + 1, 1000 * rank + 1 + 2 * B)), 224))
        c_host, s_host = ic[:B].contiguous(), ic[B:].contiguous()
    elif cfgname == "nst1024":
        g = torch.Generator().manual_seed(1000 * rank + 1)      # tubingen x starry-night SHAPES, synthetic pixels
        import torch.nn.functional as F
        c_host = F.interpolate(torch.rand(B, 3, 64, 64, generator=g), size=(h, w), mode="bilinear").clamp(0, 1).contiguous()
        s_host = F.interpolate(torch.rand(B, 3, 128, 128, generator=g), size=(h, w), mode="bilinear").clamp(0, 1).contiguous()
    elif cfgname == "masked_gram":
        import numpy as np
        fr_c, sg_c = iris_b200.synthetic.synthetic_batch([1000 * rank + 1 + i for i in range(B)], h, w)
        fr_s, sg_s = iris_b200.synthetic.synthetic_batch([1000 * rank + 100001 + i for i in range(B)], h, w)
        c_host = torch.from_numpy(fr_c).repeat(1, 3, 1, 1).contiguous()
        s_host = torch.from_numpy(fr_s).repeat(1, 3, 1, 1).contiguous()
        c_mask = torch.from_numpy(((sg_c == 2) & (fr_c <= np.float32(0.8))).astype(np.float32)).to(dev)
        s_mask = torch.from_numpy(((sg_s == 2) & (fr_s <= np.float32(0.8))).astype(np.float32)).to(dev)
    else:
        c_host, s_host = make_inputs(B, 1000 * rank + 1, h, w)
    c_host, s_host = c_host.pin_memory(), s_host.pin_memory()
    flops = flops_per_image_step(h, w, taps5=taps5, gram=not BN_loss)
    if (h, w) == (H, W) and not BN_loss:
        flops = FLOPS_640["5tap" if taps5 else "4tap"]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    r = nst_leg(args, dev, vgg, c_host.to(dev), s_host.to(dev), BN_loss, independent, K, Wm, world, rank, local, lib,
                c_mask=c_mask, s_mask=s_mask, s_weight=s_weight)
    ms, ms_max, prof = r["ms"], r["ms_max"], r["prof"]
    value = world * B * K / (ms_max / 1e3)

    # ------------------------------------------------------------------ end-to-end leg (public API, host buffers)
    e2e = None
    e2e_hist = None
    nkw = dict(BN_loss=BN_loss, c_loss_weight=1.0, s_loss_weight=s_weight, vgg=vgg, use_tqdm=False, device=str(dev),
               independent=independent, streams=args.streams, overlap=args.overlap, c_mask=c_mask, s_mask=s_mask,
               history_dtype=torch.bfloat16 if args.history_bf16 else torch.float32)
    if not args.no_e2e:
        x_host = torch.empty_like(c_host).pin_memory()

        def e2e_run(epochs, stride):
            barrier()
            t0 = time.perf_counter()
            x, xh, c_hist, s_hist = iris_b200.nst(c_host, s_host, epochs=epochs, x_hist_stride=stride, **nkw)
            x_host.copy_(x, non_blocking=True)  # result image back into pinned host memory
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            n = len(s_hist)
            nh = len(xh)
            del x, xh
            return float(t.item()), n, nh

        dt_max, evals, _ = e2e_run(args.e2e_evals, 0)
        h2d = c_host.numel() * 4 + s_host.numel() * 4
        d2h = x_host.numel() * 4 + 2 * evals * B * 8
        e2e = {"value": world * B * evals / dt_max, "unit": UNIT, "h2d_bytes_per_step": h2d / evals,
               "d2h_bytes_per_step": d2h / evals, "evals": evals,
               "note": "iris_b200.nst() from pinned host tensors to host results: targets, %d evaluations (the whole BASELINE "
                       "job, independent of --steps), final image and per-evaluation losses copied back; wall clock" % evals}
        torch.cuda.empty_cache()
        if world == 1 and cfgname == "nst640":
            # the reference's DEFAULT semantics: every evaluated image also lands in x_hist on the host (pipelines.py:93);
            # 40-evaluation jobs (7.9 GB of history), stride 0 vs stride 1, after one warm-up call that populates the
            # pinned-host allocator cache like a long-running service
            e2e_run(40, 1)
            t_off, n_off, _ = e2e_run(40, 0)
            t_on, n_on, n_hist = e2e_run(40, 1)
            e2e_hist = {"evals": n_on, "x_hist_entries": n_hist, "x_hist_bytes": n_hist * c_host.numel() * 4,
                        "value_x_hist_off": B * n_off / t_off, "value_x_hist_on": B * n_on / t_on, "unit": UNIT,
                        "ratio_on_over_off": (B * n_on / t_on) / (B * n_off / t_off),
                        "note": "nst(..., x_hist_stride=1) = the reference's default history: device snapshot + side-stream "
                                "D2H into pinned host tensors, no host synchronisation per evaluation"}
            torch.cuda.empty_cache()

    # ------------------------------------------------------------------ secondary metric: Gram-feature images/s
    feat = feat5 = None
    if not args.no_features and cfgname == "nst640":
        feat = feature_leg(dev, vgg, False, args.feature_images, world, batch=args.feature_batch)
        feat5 = feature_leg(dev, vgg, True, args.feature_images, world, batch=args.feature_batch)

    if rank != 0:
        finish()
        return

    # ------------------------------------------------------------------ roofline + baselines
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained")
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)"
    if not peak_tf:
        peak_tf, peak_src = 1400.0, "B200_PROFILING.md fallback, sustained (of fallback)"
    # L-BFGS passes: algorithmic HBM bytes (SURVEY.md §8d) = history streamed twice (16*m*N) + 36*N per image-step, with
    # m = number of stored pairs (constant = the full ring in the timed region when prefilled)
    N_img = 3 * h * w
    esz = 2 if args.history_bf16 else 4
    m_avg = r["pairs_mean"]
    lbfgs_bytes = K * B * N_img * (4.0 * esz * m_avg + 36.0)
    hbm_peak = peaks.get("hbm_gbs") or 6650.0
    lbfgs_gbs = lbfgs_bytes / (prof[7] / 1e3) / 1e9 if prof[7] > 0 else None
    # DRAM traffic of the conv family per launch: only from an ncu capture of THIS round committed under profiles/
    traffic, traffic_src = None, "not measured in this run (ncu is not available inside the timed run)"
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_conv_traffic.json")))
        if tr.get("batch") == B and tr.get("config") == cfgname:
            traffic = tr["dram_bytes_per_conv_launch"]
            traffic_src = ("ncu capture of this command (dram__bytes_read.sum + dram__bytes_write.sum per launch, "
                           "profiles/r02_ncu_launches_bench_b64.csv), averaged over the conv launches of one evaluation: "
                           "profiles/r02_conv_traffic.json")
    except Exception:
        pass
    conv_n, conv_ms, conv_flops = prof[0], prof[1], prof[2]
    achieved = conv_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else None
    roofline = {
        "kernel": "conv family: conv_halo / conv_c64 / conv_tc / conv1_1 head+tail (tcgen05 implicit-GEMM conv fwd/dgrad/Gram-bwd)", "bound": "tensor",
        "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf if achieved else None,
        "traffic": traffic, "traffic_source": traffic_src,
        # algorithmic DRAM bytes of the 19 conv launches of one evaluation (bf16 NHWC in + out, ReLU-mask and Gram-operand
        # reads of the dgrads): 587 MB per 640x400 image (DESIGN.md §2)
        "algorithmic_dram_bytes_per_launch": 587e6 * B / 19.0 * (h * w) / (H * W),
        "peak_source": peak_src, "launches": int(conv_n), "avg_launch_ms": conv_ms / max(conv_n, 1),
        "share_of_step": conv_ms / ms,
        "other": {"gram_tc_ms_share": prof[4] / ms, "lbfgs_ms_share": prof[7] / ms,
                  "gram_tflops": prof[5] / (prof[4] / 1e3) / 1e12 if prof[4] > 0 else None,
                  "lbfgs_hbm": {"bound": "hbm", "achieved": lbfgs_gbs, "peak": hbm_peak, "unit": "GB/s",
                                "frac": lbfgs_gbs / hbm_peak if lbfgs_gbs else None,
                                "note": "lbfgs_dots + reduce + control + lbfgs_update, algorithmic bytes / CUDA-event time"}},
    }
    if args.streams > 1:
        roofline["note"] = "streams > 1: per-family CUDA-event times overlap across streams and are not additive"
    cpu = None
    if not args.no_cpu_baseline and world == 1 and cfgname == "nst640":
        rate, done, dtc, threads = cpu_reference_rate(30, 2)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "%d closure evaluations + L-BFGS iterations of ONE 640x400 masked eye (%.1f s; oracle/nst_oracle.py, "
                         "torch CPU fp32, %d threads, full vgg19.features forward like the reference)" % (done, dtc, threads)}
    elif world > 1:
        cpu = {"value": None, "unit": UNIT, "cores": None, "kind": "port",
               "sample": "skipped under torchrun (N > 1): the host cores are shared by N ranks; see the N = 1 line"}
    gpu_lib = None
    if not args.no_gpu_library and world == 1 and cfgname == "nst640":
        try:
            cl, sl = make_inputs(16, 1)
            gpu_lib = {"unit": UNIT, "batch": 16,
                       "what": "the reference's own library calls on this B200: torchvision vgg19.features (all 37 modules) "
                               "through cuDNN, bmm Gram, torch.optim.LBFGS, 16 images as ONE problem, 20 evaluations"}
            for mode in ("tf32", "bf16"):
                rate, n = gpu_library_rate(dev, cl, sl, mode, evals=20, history_copy=True)
                gpu_lib["fp32_tf32_convs" if mode == "tf32" else "bf16_autocast_channels_last"] = rate
                rate2, _ = gpu_library_rate(dev, cl, sl, mode, evals=20, history_copy=False)
                gpu_lib[("fp32_tf32_convs" if mode == "tf32" else "bf16_autocast_channels_last") + "_no_history_copy"] = rate2
                torch.cuda.empty_cache()
        except Exception as e:  # a comparator failure must not lose the measurement
            gpu_lib = {"error": repr(e)[:300]}
    workload = {
        "nst640": "BASELINE config[1]: batch of %d synthetic OpenEDS2019-shaped 640x400 eyes per GPU, iris-masked, 3-channel, "
                  "random-init VGG-19, Gram style loss (relu1_1..relu4_1) + content relu4_2, alpha=1 beta=1e6, "
                  "L-BFGS(lr=1, history 100), every image its own problem" % B,
        "nst640_5tap": "as config[1] with the 5-tap Gatys style set relu1_1..relu5_1 (forward/backward to conv5_1), batch %d" % B,
        "masked_gram": "as config[1] on UNMASKED frames with the mask-weighted Gram loss (row G': c_mask / s_mask = iris masks), batch %d" % B,
        "nst224": "what the reference's drivers call: %d iris crops 224x224, default StyleLoss_BN, alpha=1 beta=1e4, the batch as ONE "
                  "L-BFGS problem (iris_style_transfer_openeds2019.py:93-100)" % B,
        "nst1024": "BASELINE config[4]: %d RGB images 1024x1024 per GPU (tubingen x starry-night shapes, synthetic pixels), unmasked Gram "
                   "loss, every image its own problem" % B,
    }[cfgname]
    line = {
        "metric": METRIC if cfgname == "nst640" else "NST image-steps/sec (%s)" % cfgname, "value": value, "unit": UNIT,
        "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": workload, "name": cfgname,
                   "batch_per_gpu": B, "image": "3x%dx%d" % (h, w), "l2": "inputs larger than L2 (activations %.1f GB per step)"
                   % (B * 139e6 * (h * w) / (H * W) / 1e9), "history_slots": 100,
                   "history_pairs_min": r["pairs_min"], "history_pairs_max": r["pairs_max"], "history_pairs_mean": r["pairs_mean"],
                   "untimed_prefill_ticks": r["prefill"] + Wm, "problems": r["problems"],
                   "problems_still_running_at_end": r["problems_running"],
                   "history_dtype": "bf16" if args.history_bf16 else "f32", "streams": args.streams,
                   "overlap": bool(args.overlap), "smem_reserve_kb": args.smem_reserve_kb,
                   "flops_per_image_step": flops,
                   "model_tflops": value * flops / 1e12 / world},
        "e2e": e2e, "e2e_default_api": e2e_hist, "secondary": feat, "secondary_5tap": feat5, "gpu_launches": r["launches"],
        "clocks": r["clocks"], "roofline": roofline, "cpu_baseline": cpu, "gpu_library_baseline": gpu_lib,
        "sanity": {"image_moved_mae": r["moved"], "s_loss_first": r["loss_first"], "s_loss_last": r["loss_last"]},
    }
    print(json.dumps(line), flush=True)
    finish()


if __name__ == "__main__":
    main()
