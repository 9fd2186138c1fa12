"""Several coupled problems in one nst() call against one call per problem; prints one JSON line.

    python scratch/nst_problems_bench.py [--rounds 3] [--epochs 200] [--out FILE]

Both workloads are the reference drivers' call: 224x224 iris crops, default StyleLoss_BN, alpha = 1, 64 crops per
problem, `--epochs` evaluations (…2019.py:93-100,215).
  layout  4 problems of 64 different crops (four driver batches): one nst(problem_size=64) call on 256 crops against four
          sequential calls of 64; beta = 1e4.
  sweep   4 betas {1e3, 1e4, 1e5, 1e6} on the same 64 crops: one nst(problem_size=64, s_loss_weight=[...]) call on the batch
          repeated four times against four calls, one per beta.
The one-call arm and the four-call arm alternate in the same process, `--rounds` times after a warm-up of each; every
timed window is a whole arm (>= 1 s: a call of 64 crops and 200 evaluations is well over a second), host clock around
synchronised calls, target features and result copies included.  image-steps/s = sum over problems of evaluations x
images / seconds; the median window is reported.  Each problem's final image in the one-call arm is compared with its
separate call (kernel choices depend on the batch, so summation order differs: not bit-identical).  Card name and power
limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import iris_b200  # noqa: E402
from iris_b200 import pipelines  # noqa: E402

G, P = 64, 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--epochs", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nst_problems_bench.py measures on a CUDA device; there is none")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "images_per_problem": G,
           "problems": P, "image": [3, 224, 224], "BN_loss": True, "epochs": a.epochs, "rounds": a.rounds}
    vgg = iris_b200.VGG19(weights="random", seed=0)
    crops = torch.from_numpy(iris_b200.synthetic.synthetic_iris_crops(list(range(1, 2 * G * P + 1)), 224))
    c_all, s_all = crops[:G * P].pin_memory(), crops[G * P:].pin_memory()
    betas = [1e3, 1e4, 1e5, 1e6]

    def call(c, s, **kw):
        x, _, _, _ = iris_b200.nst(c, s, vgg=vgg, epochs=a.epochs, use_tqdm=False, device="cuda:0", x_hist_stride=0, **kw)
        ev = pipelines.last_info["evals_per_problem"]
        return x, int(ev.sum()) * (c.shape[0] // ev.numel())

    arms = {
        "layout": {
            "one_call": lambda: [call(c_all, s_all, s_loss_weight=1e4, problem_size=G)],
            "separate_calls": lambda: [call(c_all[i * G:(i + 1) * G], s_all[i * G:(i + 1) * G], s_loss_weight=1e4)
                                       for i in range(P)],
        },
        "sweep": {
            "one_call": lambda: [call(c_all[:G].repeat(P, 1, 1, 1), s_all[:G].repeat(P, 1, 1, 1), s_loss_weight=betas,
                                      problem_size=G)],
            "separate_calls": lambda: [call(c_all[:G], s_all[:G], s_loss_weight=b) for b in betas],
        },
    }

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return dt, sum(n for _, n in out), [x for x, _ in out]

    for name, arm in arms.items():
        outs = {}
        for k, fn in arm.items():                       # warm-up (module loads, allocator) + outputs for the comparison
            _, steps, xs = timed(fn)
            outs[k] = torch.cat([x.cpu() for x in xs])
        d = (outs["one_call"] - outs["separate_calls"]).abs().view(P, -1)
        wins = {k: [] for k in arm}
        steps = {}
        for _ in range(a.rounds):
            for k, fn in arm.items():
                dt, steps[k], _ = timed(fn)
                wins[k].append(dt)
        r = {}
        for k in arm:
            sec = statistics.median(wins[k])
            r[k] = {"seconds": sec, "windows_s": wins[k], "image_steps": steps[k], "image_steps_per_s": steps[k] / sec}
        r["speedup_one_call"] = r["one_call"]["image_steps_per_s"] / r["separate_calls"]["image_steps_per_s"]
        r["final_image_mae_per_problem_vs_separate"] = d.mean(dim=1).tolist()
        r["final_image_max_abs_diff_vs_separate"] = float(d.max())
        res[name] = r
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
