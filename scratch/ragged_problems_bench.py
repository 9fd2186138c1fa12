"""Coupled problems of unequal size in one job against one call per problem; prints one JSON line.

    python scratch/ragged_problems_bench.py [--rounds 3] [--epochs 200] [--out FILE]

  driver      the drivers' loop over four DataLoader batches of synthetic 400x640 frames, of 128, 128, 128 and 64 frames
              (a short last batch), the iris erased from the label maps of 8 frames in each batch (blinks: these frames
              leave the NST batch and come back unchanged); one fixed 224x224 style iris, StyleLoss_BN, beta = 1e4,
              `--epochs` evaluations.  One stylize_frames(frames_per_problem=128) call on the 448 frames (problems of 120,
              120, 120 and 56 crops in one job) against four sequential stylize_frames calls, one per batch.
  regression  256 crops of 224x224: nst(problem_sizes=[64] * 4) against nst(problem_size=64), the same problems through
              the ranged and the equal-size entry points; the final images must be identical.
The arms alternate in the same process, `--rounds` times after a warm-up of each; every timed window is a whole arm
(several seconds), host clock around synchronised calls, host frames in, device frames out.  frames/s counts every frame
handed in; image-steps/s = sum over problems of evaluations x crops / seconds.  The median window is reported, with all
windows.  Card name and power limit are read in the same run."""
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
from iris_b200 import pipelines, synthetic  # noqa: E402

BATCHES = [128, 128, 128, 64]
ERASED = 8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--epochs", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_problems_bench.py measures on a CUDA device; there is none")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "epochs": a.epochs,
           "rounds": a.rounds}
    dev = torch.device("cuda:0")
    vgg = iris_b200.VGG19(weights="random", seed=0)

    # ---- driver workload ----
    B = sum(BATCHES)
    seeds = list(range(20000, 20000 + B))
    fr, sg = synthetic.synthetic_batch(seeds, 400, 640)
    bounds = np.cumsum([0] + BATCHES)
    erased = [int(lo) + 3 + j * n // ERASED for lo, n in zip(bounds[:-1], BATCHES) for j in range(ERASED)]  # spread out
    for i in erased:
        sg[i, 0] = synthetic.synthetic_label_map(seeds[i], 400, 640, drop=(2,))
    frames_h, segs_h = torch.from_numpy(fr).pin_memory(), torch.from_numpy(sg).pin_memory()
    sf, ss = synthetic.synthetic_eye(777, 400, 640)
    sx, sseg = torch.from_numpy(sf).to(dev)[None], torch.from_numpy(ss).to(dev)[None]
    smask, sbb = pipelines.iris_masks_and_bboxes(sx, sseg)
    s_iris = pipelines.crop_resize_irises(sx, smask, sbb)[0, :1].contiguous()       # (1,224,224) like …2020.py:103
    kw = dict(vgg=vgg, c_loss_weight=1.0, s_loss_weight=1e4, epochs=a.epochs, BN_loss=True, device="cuda:0")

    def one_call():
        out, info = iris_b200.stylize_frames(frames_h, s_iris, segs=segs_h, frames_per_problem=BATCHES[0], **kw)
        return [out], sum(e * g for e, g in zip(info["evals_per_run"], info["problem_sizes"]))

    def separate_calls():
        outs, steps = [], 0
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            out, info = iris_b200.stylize_frames(frames_h[lo:hi], s_iris, segs=segs_h[lo:hi], **kw)
            outs.append(out)
            steps += info["evals"] * int(info["valid"].sum())
        return outs, steps

    # ---- regression workload ----
    crops = torch.from_numpy(synthetic.synthetic_iris_crops(list(range(1, 513)), 224))
    c_all, s_all = crops[:256].pin_memory(), crops[256:].pin_memory()

    def nst_call(**lay):
        x, _, _, _ = iris_b200.nst(c_all, s_all, vgg=vgg, s_loss_weight=1e4, epochs=a.epochs, use_tqdm=False,
                                   device="cuda:0", x_hist_stride=0, **lay)
        return [x], int(pipelines.last_info["evals_per_problem"].sum()) * 64

    workloads = {
        "driver": {"one_call": one_call, "separate_calls": separate_calls},
        "regression": {"ranged": lambda: nst_call(problem_sizes=[64] * 4),
                       "equal_size": lambda: nst_call(problem_size=64)},
    }

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        outs, steps = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, steps, outs

    for name, arms in workloads.items():
        outs = {}
        for k, fn in arms.items():                       # warm-up (module loads, allocator) + outputs for the comparison
            _, _, xs = timed(fn)
            outs[k] = torch.cat([x.cpu() for x in xs])
        wins = {k: [] for k in arms}
        steps = {}
        for _ in range(a.rounds):
            for k, fn in arms.items():
                dt, steps[k], _ = timed(fn)
                wins[k].append(dt)
        r = {}
        for k in arms:
            sec = statistics.median(wins[k])
            r[k] = {"seconds": sec, "windows_s": wins[k], "image_steps": steps[k], "image_steps_per_s": steps[k] / sec}
        k0, k1 = list(arms)
        r["ratio_%s_over_%s" % (k0, k1)] = r[k0]["image_steps_per_s"] / r[k1]["image_steps_per_s"]
        if name == "driver":
            for k in arms:
                r[k]["frames_per_s"] = B / r[k]["seconds"]
            d = (outs[k0] - outs[k1]).abs()
            r["final_frame_mae_per_batch_vs_separate"] = [float(d[lo:hi].mean()) for lo, hi in zip(bounds[:-1], bounds[1:])]
            r["final_frame_max_abs_diff_vs_separate"] = float(d.max())
            r["erased_frames_unchanged"] = bool(torch.equal(outs[k0][erased], frames_h[erased]))
            r["batches"], r["erased_per_batch"], r["frame"], r["crop"] = BATCHES, ERASED, [1, 400, 640], [3, 224, 224]
        else:
            r["images_identical"] = bool(torch.equal(outs[k0], outs[k1]))
            r["crops"], r["layout"] = 256, "ranged: nst(problem_sizes=[64] * 4), equal_size: nst(problem_size=64)"
        res[name] = r
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
