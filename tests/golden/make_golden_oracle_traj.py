"""Trajectories of the CPU oracle (oracle/nst_oracle.py) for the cases of tests/test_oracle_golden.py:
    python tests/golden/make_golden_oracle_traj.py        -> tests/golden/nst_traj_oracle.npz

A float32 L-BFGS run of 20-140 evaluations carries the rounding of every convolution and matrix product, and that
rounding depends on the host: oneDNN and MKL choose their kernels and reduction splits from the CPU and the thread
count, and L-BFGS grows a 1e-7 difference of one evaluation into 1e-3 over a run.  The reference's own runs
(nst_traj.npz, nst_traj_r2.npz) were recorded on an 8-vCPU AMD EPYC; on other hosts the oracle agrees with them in
the evaluation count and the first evaluation only.  These runs were recorded with torch 2.11 (oneDNN 3.10, MKL 2024.2)
on an 8-vCPU x86-64 Intel Xeon (AVX-512) with 8 threads, the thread count the tests set.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iris-style-transfer_b200"))
from oracle import nst_oracle as O  # noqa: E402
import synthetic  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
torch.set_num_threads(8)


def rand_img(seed, shape):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g)


def main():
    w = O.random_vgg19_weights(0)
    t = {}

    def run(tag, c_img, s_img, x_stride=1, **kw):
        x, _, c_hist, s_hist = O.nst(c_img, s_img, w, keep_hist=False, **kw)
        t[tag + "_x"] = x.numpy()[..., ::x_stride, ::x_stride]   # every x_stride-th row and column: files stay < 1 MB
        t[tag + "_x_stride"] = np.int64(x_stride)
        t[tag + "_c_hist"] = np.array(c_hist)
        t[tag + "_s_hist"] = np.array(s_hist)
        print(tag, tuple(x.shape), len(c_hist), "evals", flush=True)

    c1, s1 = rand_img(21, (1, 3, 48, 64)), rand_img(22, (1, 3, 48, 64))
    run("gram_b1", c1, s1, BN_loss=False, s_loss_weight=1e6, epochs=50)
    run("bn_b1", c1, s1, BN_loss=True, s_loss_weight=1e4, epochs=40)
    c, s = rand_img(11, (2, 3, 48, 64)), rand_img(12, (2, 3, 48, 64))
    run("gram_b2_coupled", c, s, BN_loss=False, s_loss_weight=1e6, epochs=20)
    run("gram_b2_style1", c, s[:1], BN_loss=False, s_loss_weight=1e6, epochs=20)
    torch.manual_seed(123)
    x0 = torch.rand(c1.shape)
    run("gram_rand_init", c1, s1, clone_content=False, x0=x0, BN_loss=False, s_loss_weight=1e6, epochs=20)
    run("gram_unbatched_style", c1, s1[0, :1], BN_loss=False, s_loss_weight=1e6, epochs=20)
    run("bn_unbatched_style", c1, s1[0, :1], BN_loss=True, s_loss_weight=1e4, epochs=20)
    run("degenerate", c1, s1, BN_loss=False, s_loss_weight=1.0, epochs=5)
    c3, s3 = rand_img(31, (1, 3, 32, 32)), rand_img(32, (1, 3, 32, 32))
    run("gram_long", c3, s3, BN_loss=False, s_loss_weight=1e6, epochs=130)
    run("gram_c3d_s3d", c1[0], s1[0], BN_loss=False, s_loss_weight=1e4, epochs=20)
    run("bn_c3d_s3d", c1[0], s1[0], BN_loss=True, s_loss_weight=1e4, epochs=20)
    run("gram_c3d_s4d", c1[0], s1, BN_loss=False, s_loss_weight=1e4, epochs=20)
    ic = torch.from_numpy(synthetic.synthetic_iris_crops([1, 2, 3, 4, 11, 12, 13, 14], 224))
    run("bn_iris224_b4", ic[:4], ic[4:], BN_loss=True, s_loss_weight=1e4, epochs=40, x_stride=4)
    path = os.path.join(OUT, "nst_traj_oracle.npz")
    np.savez_compressed(path, **t)
    print(os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
