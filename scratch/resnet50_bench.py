"""Throughput of iris_b200.ResNet50 (the GazeEstimator2 feature extractor) against torchvision on cuDNN; prints one JSON line.

    python scratch/resnet50_bench.py [--seconds 1.5] [--out FILE]

Workloads: 128 frames of 400x640 per step (one channel, the 2020 driver's batch and frame shape) and 256 images of 224x224
(three channels).  Per workload: device-resident frames/s of ResNet50 (CUDA events around >= --seconds of steps after a
warm-up), per-stage CUDA-event times of the same chain launched entry point by entry point, the conv family's achieved
TFLOP/s from the library's event profiler (family 0, algorithmic FLOPs over kernel time) against the sustained 1410.9, the
algorithmic FLOPs from the layer shapes, torchvision resnet50 (same weights, fc dropped) in fp32 (TF32 off) and in bf16
autocast + channels_last, and the output differences.  Card name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import iris_b200  # noqa: E402
from iris_b200 import _lib  # noqa: E402
from iris_b200 import resnet as R  # noqa: E402

SUSTAINED_TFLOPS = 1410.9


def timed(fn, seconds):
    """ms per call over a window of >= `seconds` (calls counted from a calibration run), after two warm-up calls."""
    fn(); fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    n = max(3, int(seconds * 1000 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def algorithmic_flops(H, W):
    """2 * MACs of the 53 convolutions for one H x W image, walking the blocks like isx_resnet50_forward."""
    h, w = (H + 1) // 2, (W + 1) // 2
    total = 2 * 147 * 64 * h * w
    h, w, cin = (h + 1) // 2, (w + 1) // 2, 64
    for st, (planes, blocks) in enumerate(R.STAGES):
        for blk in range(blocks):
            stride = 2 if (st > 0 and blk == 0) else 1
            ho, wo = (h + stride - 1) // stride, (w + stride - 1) // stride
            total += 2 * (cin * planes * h * w + 9 * planes * planes * ho * wo + planes * 4 * planes * ho * wo)
            if blk == 0:
                total += 2 * cin * planes * 4 * ho * wo
            h, w, cin = ho, wo, planes * 4
    return total


def staged(net, x):
    """The driver's chain launched entry point by entry point, CUDA events between the stages: (features, {stage: ms})."""
    pk = net.packed(x.device)
    B, xc, H, W = x.shape
    s = _lib.stream_ptr()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
    names = ["stem", "maxpool", "layer1", "layer2", "layer3", "layer4", "avgpool"]
    h, w = (H + 1) // 2, (W + 1) // 2
    bf = dict(device=x.device, dtype=torch.bfloat16)
    t0 = torch.cuda.Event(enable_timing=True)
    t0.record()
    y = torch.empty(B, h, w, 64, **bf)
    _lib.call("isx_resnet_stem_fwd", x, xc, pk.w[0], pk.bias[0], y, B, H, W, s)
    ev[0].record()
    h2, w2 = (h + 1) // 2, (w + 1) // 2
    cur = torch.empty(B, h2, w2, 64, **bf)
    _lib.call("isx_maxpool3x3s2_fwd", y, cur, B, h, w, 64, s)
    ev[1].record()
    h, w, cin, li = h2, w2, 64, 1
    for st, (planes, blocks) in enumerate(R.STAGES):
        for blk in range(blocks):
            stride = 2 if (st > 0 and blk == 0) else 1
            ho, wo = (h + stride - 1) // stride, (w + stride - 1) // stride
            t1 = torch.empty(B, h, w, planes, **bf)
            _lib.call("isx_conv_bias_act_fwd", cur, pk.w[li], pk.bias[li], None, t1, B, h, w, cin, planes, 1, 1, 1, s)
            t2 = torch.empty(B, ho, wo, planes, **bf)
            _lib.call("isx_conv_bias_act_fwd", t1, pk.w[li + 1], pk.bias[li + 1], None, t2, B, h, w, planes, planes, 3, stride, 1, s)
            sc = cur
            if blk == 0:
                sc = torch.empty(B, ho, wo, planes * 4, **bf)
                _lib.call("isx_conv_bias_act_fwd", cur, pk.w[li + 3], pk.bias[li + 3], None, sc, B, h, w, cin, planes * 4, 1, stride, 0, s)
            out = torch.empty(B, ho, wo, planes * 4, **bf)
            _lib.call("isx_conv_bias_act_fwd", t2, pk.w[li + 2], pk.bias[li + 2], sc, out, B, ho, wo, planes, planes * 4, 1, 1, 1, s)
            cur, h, w, cin = out, ho, wo, planes * 4
            li += 4 if blk == 0 else 3
        ev[2 + st].record()
    feat = torch.empty(B, 2048, device=x.device, dtype=torch.float32)
    _lib.call("isx_global_avgpool", cur, feat, B, h * w, 2048, s)
    ev[6].record()
    torch.cuda.synchronize()
    prev, ms = t0, {}
    for n, e in zip(names, ev):
        ms[n] = prev.elapsed_time(e)
        prev = e
    return feat, ms


def trunk_tv(model, x):
    h = model.maxpool(model.relu(model.bn1(model.conv1(x))))
    h = model.layer4(model.layer3(model.layer2(model.layer1(h))))
    return torch.flatten(model.avgpool(h), 1)


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("resnet50_bench: needs a CUDA device (B200); nothing is measured on the CPU")
    dev = torch.device("cuda:0")
    lib = _lib.load()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "workloads": []}
    model = R.random_resnet50(0).to(dev)
    net = iris_b200.ResNet50(weights=model)
    for B, xc, H, W in ((128, 1, 400, 640), (256, 3, 224, 224)):
        g = torch.Generator(device=dev).manual_seed(B)
        x = torch.rand(B, xc, H, W, device=dev, generator=g)
        x3 = x.repeat(1, 3, 1, 1) if xc == 1 else x
        flops = algorithmic_flops(H, W)
        r = {"B": B, "xc": xc, "H": H, "W": W, "gflop_per_image": flops / 1e9, "chunk": net.chunk_size(B, H, W)}
        with torch.no_grad():
            feat = net(x)
            ms, n = timed(lambda: net(x), args.seconds)
            r.update(isx_ms_per_step=ms, isx_steps_timed=n, isx_frames_per_s=B * 1000 / ms,
                     isx_end_to_end_tflops=flops * B / ms / 1e9)
            lib.isx_prof_enable(1)
            net(x)
            torch.cuda.synchronize()
            prof = (ctypes.c_double * 12)()
            _lib.call("isx_prof_collect", prof, 12)
            lib.isx_prof_enable(0)
            r["conv_family"] = {"launches": prof[0], "ms": prof[1], "gflop": prof[2] / 1e9,
                                "tflops": prof[2] / prof[1] / 1e9 if prof[1] else None}
            r["conv_family"]["share_of_sustained"] = (r["conv_family"]["tflops"] or 0) / SUSTAINED_TFLOPS
            staged(net, x)
            f2, stages = staged(net, x)
            r["stage_ms"] = stages
            r["staged_equals_driver"] = bool(torch.equal(f2, feat))
            torch.backends.cudnn.allow_tf32 = False
            torch.backends.cuda.matmul.allow_tf32 = False
            ref = trunk_tv(model, x3)
            ms32, _ = timed(lambda: trunk_tv(model, x3), args.seconds)
            r.update(cudnn_fp32_ms=ms32, cudnn_fp32_frames_per_s=B * 1000 / ms32)
            model_cl = model.to(memory_format=torch.channels_last)
            xcl = x3.contiguous(memory_format=torch.channels_last)

            def tv_bf16():
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    return trunk_tv(model_cl, xcl)

            out16 = tv_bf16().float()
            ms16, _ = timed(tv_bf16, args.seconds)
            model.to(memory_format=torch.contiguous_format)
            r.update(cudnn_bf16_cl_ms=ms16, cudnn_bf16_cl_frames_per_s=B * 1000 / ms16,
                     isx_over_cudnn_bf16_cl=(B * 1000 / ms) / (B * 1000 / ms16),
                     isx_rel_l2_vs_fp32=rel(feat, ref), cudnn_bf16_rel_l2_vs_fp32=rel(out16, ref))
        res["workloads"].append(r)
        del x, x3, ref, feat, out16
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
