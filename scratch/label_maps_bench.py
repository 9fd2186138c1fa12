"""int64 against uint8 label maps on the three kernels that read or write them and on the landmark path; prints one JSON line.

    python scratch/label_maps_bench.py [--seconds 1.0] [--rounds 3] [--out FILE]

128 frames of 400x640 (the 2020 driver's batch and frame shape).  Per workload the int64 and the uint8 call alternate in the
same process, `--rounds` windows of >= `--seconds` of CUDA events each after a warm-up; the median window is reported.
  mask_bbox   isx_mask_bbox / isx_mask_bbox_typed(uint8), mask output only (as iris_masks_and_bboxes): 13 / 6 B per pixel
  seg_iou     isx_seg_iou / isx_seg_iou_typed(uint8), four classes: 16 / 2 B per pixel
  ritnet      isx_ritnet_forward / _typed(uint8), whole forward; rit_classify_kernel alone from torch.profiler in a separate
              pass (128 B of features in, 8 / 1 B of label out per pixel)
  landmarks   extract_eye_landmarks_batch + GazeEstimator1 end to end from pinned host label maps (host clock around a
              synchronised loop, like bench.py --config landmarks), frames/s
Inputs rotate over enough copies that a window's working set exceeds the 126 MB L2 twice over.  Bytes over kernel time is
compared with the 7.7 TB/s data-sheet HBM rate.  Card name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import iris_b200  # noqa: E402
from iris_b200 import _lib  # noqa: E402

HBM_TBS = 7.7
B, H, W = 128, 400, 640
L2_BYTES = 126 << 20


def window_ms(fn, seconds):
    """ms per call over one window of >= `seconds`."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    n = max(3, int(seconds * 1000 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def alternate(fns, seconds, rounds):
    """{name: median ms per call} with the workloads' windows interleaved."""
    for f in fns.values():
        f(); f()
    torch.cuda.synchronize()
    res = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            res[k].append(window_ms(f, seconds))
    return {k: {"ms": statistics.median(v), "windows_ms": v} for k, v in res.items()}


def rotating(make, bytes_per_call):
    """Enough copies of an input that one pass over them is >= 2x the L2; returns a callable giving the next copy."""
    n = max(1, -(-2 * L2_BYTES // bytes_per_call))
    copies = [make() for _ in range(n)]
    state = [0]

    def nxt():
        state[0] = (state[0] + 1) % n
        return copies[state[0]]
    return nxt, n


def roof(bytes_per_call, ms):
    tbs = bytes_per_call / (ms * 1e-3) / 1e12
    return {"bytes_per_call": bytes_per_call, "TB_per_s": tbs, "frac_of_7.7TBs": tbs / HBM_TBS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("label_maps_bench.py measures on a CUDA device; there is none")
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "batch": B, "frame": [H, W],
           "seconds_per_window": a.seconds, "rounds": a.rounds}
    npx = B * H * W
    labs = np.stack([iris_b200.synthetic.synthetic_label_map(i, speck=0.002 * (i % 4)) for i in range(B)])
    lab64 = torch.from_numpy(labs).to(dev)
    lab8 = lab64.to(torch.uint8)
    s = _lib.stream_ptr()

    # ---- mask / bbox ----
    x = torch.rand(B, 1, H, W, device=dev)
    mask = torch.empty(B, 1, H, W, device=dev, dtype=torch.uint8)
    bbox = torch.empty(B, 4, device=dev, dtype=torch.int32)
    nx64, n64 = rotating(lambda: (x.clone(), lab64.clone()), npx * 13)
    nx8, n8 = rotating(lambda: (x.clone(), lab8.clone()), npx * 6)

    def mb64():
        xx, ss = nx64()
        _lib.call("isx_mask_bbox", xx, ss, 2, 1, _lib.f32(0.8), mask, None, bbox, B, H, W, s)

    def mb8():
        xx, ss = nx8()
        _lib.call("isx_mask_bbox_typed", xx, ss, 1, 2, 1, _lib.f32(0.8), mask, None, bbox, B, H, W, s)
    r = alternate({"int64": mb64, "uint8": mb8}, a.seconds, a.rounds)
    r["int64"].update(roof(npx * 13, r["int64"]["ms"]), copies=n64)
    r["uint8"].update(roof(npx * 6, r["uint8"]["ms"]), copies=n8)
    res["mask_bbox"] = r
    del nx64, nx8

    # ---- IoU ----
    pred64 = lab64.clone()
    pred64[:, ::7] = (pred64[:, ::7] + 1) % 4
    counts = torch.empty(B, 4, 2, device=dev, dtype=torch.int32)
    iou = torch.empty(B, 4, device=dev)
    miou = torch.empty(B, device=dev)
    ni64, n64 = rotating(lambda: (pred64.clone(), lab64.clone()), npx * 16)
    ni8, n8 = rotating(lambda: (pred64.to(torch.uint8), lab8.clone()), npx * 2)

    def iou64():
        p, t = ni64()
        _lib.call("isx_seg_iou", p, t, B, _lib.i64(H * W), 4, _lib.f32(1e-6), counts, iou, miou, s)

    def iou8():
        p, t = ni8()
        _lib.call("isx_seg_iou_typed", p, t, 1, B, _lib.i64(H * W), 4, _lib.f32(1e-6), counts, iou, miou, s)
    iou64(); ref = iou.clone(); iou8(); torch.cuda.synchronize()
    r = alternate({"int64": iou64, "uint8": iou8}, a.seconds, a.rounds)
    r["int64"].update(roof(npx * 16, r["int64"]["ms"]), copies=n64)
    r["uint8"].update(roof(npx * 2, r["uint8"]["ms"]), copies=n8)
    r["uint8_equals_int64"] = bool(torch.equal(iou, ref))
    res["seg_iou"] = r
    del ni64, ni8

    # ---- RITnet ----
    gold = np.load(os.path.join(ROOT, "tests", "golden", "ritnet.npz"))
    sd = {k[2:]: torch.from_numpy(gold[k]) for k in gold.files if k.startswith("w:")}
    rit64 = iris_b200.RITnet(state_dict=sd)
    rit8 = iris_b200.RITnet(state_dict=sd, label_dtype=torch.uint8)
    fr, _ = iris_b200.synthetic.synthetic_batch(list(range(8)), H, W)
    frames = torch.from_numpy(fr).to(dev).repeat(B // 8, 1, 1, 1).contiguous()
    l64, l8 = rit64(frames), rit8(frames)
    torch.cuda.synchronize()
    r = alternate({"int64": lambda: rit64(frames), "uint8": lambda: rit8(frames)}, a.seconds, a.rounds)
    r["uint8_equals_int64"] = bool(torch.equal(l8, l64.to(torch.uint8)))
    from torch.profiler import ProfilerActivity, profile
    cls = {}
    for name, net in (("int64", rit64), ("uint8", rit8)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                net(frames)
            torch.cuda.synchronize()
        ev = [e for e in prof.key_averages() if "rit_classify_kernel" in e.key]
        us = sum(e.device_time_total for e in ev) / max(1, sum(e.count for e in ev))
        nbytes = npx * (128 + (8 if name == "int64" else 1))
        cls[name] = dict(us=us, **roof(nbytes, us / 1e3))
    r["rit_classify_kernel"] = cls
    res["ritnet_forward"] = r
    del frames, l64, l8

    # ---- landmarks + GazeEstimator1 end to end from pinned host label maps ----
    net = iris_b200.GazeEstimator1(extract_feature=True).to(dev)
    h64 = torch.from_numpy(labs).pin_memory()
    h8 = h64.to(torch.uint8).pin_memory()
    out_h = torch.empty(B, 3).pin_memory()
    g64, g8 = net(h64.to(dev)), net(h8.to(dev))
    torch.cuda.synchronize()
    same = bool(torch.equal(g64, g8))

    def e2e(hsrc, seconds):
        for _ in range(3):
            net(hsrc.to(dev, non_blocking=True))
        torch.cuda.synchronize()
        t0, k = time.perf_counter(), 0
        while True:
            for _ in range(10):
                g = net(hsrc.to(dev, non_blocking=True))
                out_h.copy_(g, non_blocking=True)
            torch.cuda.synchronize()
            k += 10
            dt = time.perf_counter() - t0
            if dt >= seconds:
                return B * k / dt
    rates = {"int64": [], "uint8": []}
    for _ in range(a.rounds):
        rates["int64"].append(e2e(h64, a.seconds))
        rates["uint8"].append(e2e(h8, a.seconds))
    res["landmarks_e2e_pinned_host"] = {
        k: {"frames_per_s": statistics.median(v), "windows": v, "h2d_bytes_per_step": npx * (8 if k == "int64" else 1)}
        for k, v in rates.items()}
    res["landmarks_e2e_pinned_host"]["gaze_uint8_equals_int64"] = same
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
