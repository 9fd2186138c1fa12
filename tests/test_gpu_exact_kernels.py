"""Bit-exact tests of the tcgen05 convolution, Gram and fused-pool kernels on exactly representable operands.

Activations are small integers stored in bf16 ({0..3} after a ReLU, {-3..3} for gradients), weights and Gram gradients
are k/64 with k in {-4..4}, biases, residuals and affine coefficients are multiples of 2^-6 no larger than 2.  Every
product and every partial sum of such operands is a multiple of the smallest product LSB and stays far below 2^24 of
them, so fp32 accumulation is exact whatever the summation order, the split-K or the TMEM accumulation: the one rounding
left is the kernel's final fp32 -> bf16 conversion.  The expected output is therefore fully determined,

    float64 reference (exact) -> float32 (exact) -> bfloat16 (round to nearest even),

and the kernels must match it bit for bit (the sign of a zero is not compared).  `exact_budget` checks for every
test that the operands round-trip through bf16 and that the largest sum of |terms| stays below 2^22 LSBs, so a test
that silently loses exactness fails instead of passing loosely.  This also checks the premise that tcgen05 kind::f16
accumulation into fp32 drops no bits on such operands: every convolution here would fail if it did.

The integer activations make equal window maxima and exact zeros common: the input on which the fused pools' tie rule
(first maximum, 4 where the maximum is <= 0) and the `act > 0` masks of the dgrad epilogues go wrong.  The routing
bytes are compared with a reference written here, not with another kernel of the library.

Routes: the kernel-selection options force conv_c64, conv_sweep, conv_halo or the generic conv_tc kernel, and are
restored to the values they had.  After every call the test records the same call by stream capture into a CUDA graph
(not executed) and asserts the names of its kernel nodes, so a route that quietly falls back to the generic kernel
fails.  A graph holds every launch, so this identification cannot miss one.

The conv1_1 head and image-gradient tail normalise the image by the ImageNet mean / std, which no exact operand
survives; they are checked against float64 with an error bound that scales with the sum of |terms| instead."""
import contextlib
import ctypes
import math
import re

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
EXACT_LIMIT = 2.0 ** 22


@pytest.fixture(scope="module")
def isx():
    import iris_b200  # noqa: F401
    from iris_b200 import _lib

    _lib.load()
    _lib.call("isx_device_check", 0)
    return _lib


# ---- exact operands ----------------------------------------------------------------------------------------------------
def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def ints(shape, lo, hi, g):
    """float64 tensor of integers drawn uniformly from [lo, hi]"""
    return torch.randint(lo, hi + 1, tuple(shape), generator=g, device=DEV).double()


def act_bf16(shape, g):
    return ints(shape, 0, 3, g).to(torch.bfloat16)


def grad_bf16(shape, g):
    return ints(shape, -3, 3, g).to(torch.bfloat16)


def weights(shape, g, kmax=4):
    return (ints(shape, -kmax, kmax, g) / 64).float()


def symmetric_D(B, C, g):
    """bf16 [B,C,C] symmetric, entries k/64 with k in {-4..4}: what the Gram backward receives"""
    k = ints((B, C, C), -4, 4, g).triu()
    D = ((k + k.transpose(1, 2).tril(-1)) / 64).to(torch.bfloat16)
    assert torch.equal(D, D.transpose(1, 2))
    return D


def fine(shape, g):
    """fp32 multiples of 2^-6 with |.| <= 2"""
    return (ints(shape, -128, 128, g) / 64).float()


def assert_bf16_exact(**operands):
    for name, t in operands.items():
        if t is None:
            continue
        d = t.double()
        assert torch.equal(d.to(torch.bfloat16).double(), d), "operand %s is not exact in bf16" % name


def exact_budget(abssum_max, lsb, what):
    """Largest sum of |terms| in units of the smallest product LSB: below 2^22, fp32 accumulation is exact."""
    units = float(abssum_max) / lsb
    assert units < EXACT_LIMIT, "%s: sum of |terms| is %.3g LSBs, not exact in fp32" % (what, units)


def snap(ref, lsb, what):
    """The float64 reference is a multiple of `lsb` (a float64 algorithm may leave ~1e-16 of noise): return it exactly."""
    q = torch.round(ref / lsb)
    assert float((ref / lsb - q).abs().max()) < 1e-6, "%s: the reference is not a multiple of the LSB" % what
    return q * lsb


def rn_bf16(ref):
    """float64 holding an fp32-exact value -> bf16, rounded to nearest even"""
    return ref.float().to(torch.bfloat16)


def assert_bits(got, exp, what):
    """bf16 results equal, element for element (NaN never equals; -0 == +0)"""
    g, e = got.float(), exp.float()
    assert g.shape == e.shape, "%s: shape %s, expected %s" % (what, tuple(g.shape), tuple(e.shape))
    bad = g != e
    n = int(bad.sum())
    if n:
        idx = bad.nonzero()[:4].tolist()
        ex = ", ".join("%s got %r want %r" % (tuple(i), g[tuple(i)].item(), e[tuple(i)].item()) for i in idx)
        pytest.fail("%s: %d / %d elements differ (%s)" % (what, n, g.numel(), ex))


def max_abs_row_sum(w2d):
    """max over output rows of sum |w|: with |x| <= xmax, every dot product's sum of |terms| is <= xmax * this"""
    return float(w2d.double().abs().sum(dim=1).max())


# ---- float64 references ------------------------------------------------------------------------------------------------
def conv3x3_nhwc(x, w):
    """3x3, pad 1, stride 1 convolution of NHWC x with OIHW w in float64, as nine DGEMMs (exact on these operands)"""
    B, H, W, Cin = x.shape
    xp = F.pad(x.double(), (0, 0, 1, 1, 1, 1))
    wd = w.double()
    out = torch.zeros(B * H * W, wd.shape[0], dtype=torch.float64, device=DEV)
    for ky in range(3):
        for kx in range(3):
            out += xp[:, ky:ky + H, kx:kx + W, :].reshape(-1, Cin) @ wd[:, :, ky, kx].t()
    return out.reshape(B, H, W, -1)


def dgrad3x3_nhwc(dy, w):
    """dx of the forward conv with OIHW w (Cout x Cin): conv of dy with the rotated, transposed filter"""
    return conv3x3_nhwc(dy, w.transpose(0, 1).flip(2, 3))


def pool_reference(a):
    """MaxPool2d(2, 2) of the bf16 NHWC map a and the routing bytes of its backward: the position of the FIRST maximum in
    window order (0,0), (0,1), (1,0), (1,1), and 4 where the maximum is <= 0"""
    B, H, W, C = a.shape
    Hp, Wp = H // 2, W // 2
    v = a[:, :2 * Hp, :2 * Wp].float().reshape(B, Hp, 2, Wp, 2, C).permute(0, 1, 3, 5, 2, 4).reshape(B, Hp, Wp, C, 4)
    m = v.amax(dim=-1)
    eq = v == m[..., None]
    code = torch.where(eq[..., 0], 0, torch.where(eq[..., 1], 1, torch.where(eq[..., 2], 2, 3)))
    code = torch.where(m > 0, code, 4).to(torch.uint8)
    pooled = F.max_pool2d(a.float().permute(0, 3, 1, 2), 2, 2).permute(0, 2, 3, 1)
    return pooled, code


# ---- kernel routes -----------------------------------------------------------------------------------------------------
def get_option(lib, name):
    v = ctypes.c_int(-1)
    assert lib.isx_get_option(name.encode(), ctypes.byref(v)) == 0
    return v.value


@contextlib.contextmanager
def options(isx, **kw):
    """Set kernel-selection options and restore the values they had, whatever happens inside."""
    lib = isx.load()
    saved = {k: get_option(lib, k) for k in kw}
    try:
        for k, v in kw.items():
            assert lib.isx_set_option(k.encode(), v) == 0
        yield
    finally:
        for k, v in saved.items():
            lib.isx_set_option(k.encode(), v)


ROUTES = {
    # route: (options, the kernel that must run)
    "generic": (dict(c64=0, sweep64=0, halo2=0), "conv_tc_kernel"),
    "c64": (dict(c64=2, sweep64=0, halo2=0), "conv_c64_kernel"),
    "sweep": (dict(sweep64=2, c64=0, halo2=0), "conv_sweep64_kernel"),
    "halo": (dict(halo2=2, c64=0, sweep64=0), "conv_halo_kernel"),
    "default": ({}, None),
}
CONV_KERNELS = ("conv_tc_kernel", "conv_c64_kernel", "conv_sweep64_kernel", "conv_halo_kernel", "conv1_1_tail_kernel")


class KernelNodeParams(ctypes.Structure):
    """CUDA_KERNEL_NODE_PARAMS_v2 (cuda.h)"""
    _fields_ = [("func", ctypes.c_void_p), ("gridDimX", ctypes.c_uint), ("gridDimY", ctypes.c_uint),
                ("gridDimZ", ctypes.c_uint), ("blockDimX", ctypes.c_uint), ("blockDimY", ctypes.c_uint),
                ("blockDimZ", ctypes.c_uint), ("sharedMemBytes", ctypes.c_uint), ("kernelParams", ctypes.c_void_p),
                ("extra", ctypes.c_void_p), ("kern", ctypes.c_void_p), ("ctx", ctypes.c_void_p)]


_DRIVER = []


def cu(name, *args):
    """call a CUDA driver API function, raise on an error"""
    if not _DRIVER:
        _DRIVER.append(ctypes.CDLL("libcuda.so.1"))
    rc = getattr(_DRIVER[0], name)(*args)
    if rc != 0:
        err = ctypes.c_char_p()
        _DRIVER[0].cuGetErrorName(rc, ctypes.byref(err))
        raise RuntimeError("%s failed: %s" % (name, err.value))


def launched(fn):
    """Run fn, then return the names of the kernels it launches, in launch order.

    The names come from a stream capture of a second call (recorded into a CUDA graph, not executed): the graph's kernel
    nodes are exactly the launches, so no record can be lost.  The library picks its kernels from the arguments and the
    options alone, so the second call launches what the first one ran.  fn must take the stream from isx.stream_ptr()
    when it is called."""
    fn()
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    h = ctypes.c_void_p(stream.cuda_stream)
    graph = ctypes.c_void_p()
    with torch.cuda.stream(stream):
        cu("cuStreamBeginCapture_v2", h, 2)   # CU_STREAM_CAPTURE_MODE_RELAXED
        try:
            fn()
        finally:
            cu("cuStreamEndCapture", h, ctypes.byref(graph))
    names = []
    try:
        n = ctypes.c_size_t(0)
        cu("cuGraphGetNodes", graph, None, ctypes.byref(n))
        nodes = (ctypes.c_void_p * n.value)()
        cu("cuGraphGetNodes", graph, nodes, ctypes.byref(n))
        # cuGraphGetNodes lists nodes in creation order; a single stream creates them in launch order
        for node in nodes:
            kind = ctypes.c_int(-1)
            cu("cuGraphNodeGetType", ctypes.c_void_p(node), ctypes.byref(kind))
            if kind.value != 0:    # CU_GRAPH_NODE_TYPE_KERNEL
                continue
            p = KernelNodeParams()
            cu("cuGraphKernelNodeGetParams_v2", ctypes.c_void_p(node), ctypes.byref(p))
            name = ctypes.c_char_p()
            if p.func:
                cu("cuFuncGetName", ctypes.byref(name), ctypes.c_void_p(p.func))
            else:
                cu("cuKernelGetName", ctypes.byref(name), ctypes.c_void_p(p.kern))
            names.append(name.value.decode())
    finally:
        cu("cuGraphDestroy", graph)
    return names


def kernel_args(name, family):
    """template arguments of a kernel name, mangled (conv_tc_kernelILi64ELi2ELi0EE...) or not (conv_tc_kernel<64, 2, 0>)"""
    m = re.search(re.escape(family) + r"(?:<([^>]*)>|I(.*?)EE)", name)
    return tuple(int(v) for v in re.findall(r"\d+", (m.group(1) or m.group(2)))) if m else None


def run_on_route(isx, route, fn, what, expect=None):
    """Call fn with the route's options; assert that the route's convolution kernel (or `expect`) ran, and return the names
    of all kernels launched."""
    opts, kernel = ROUTES[route]
    kernel = expect or kernel
    with options(isx, **opts):
        names = launched(fn)
    convs = [n for n in names if any(k in n for k in CONV_KERNELS)]
    assert convs, "%s: no convolution kernel launched (launched: %s)" % (what, names)
    if kernel is not None:
        assert all(kernel in n for n in convs), "%s: route %s expected %s, ran %s" % (what, route, kernel, convs)
    return names


def generic_tile(names):
    """(BN, MT) of the generic kernel that ran"""
    for n in names:
        a = kernel_args(n, "conv_tc_kernel")
        if a:
            return a[0], a[1]
    return None


# ---- the patch shapes of the generic kernel (conv_tc.cu, choose_patch) -------------------------------------------------
def choose_patch(B, H, W, one_image_per_tile=False):
    best = None
    tw = 128
    while tw >= 1:
        th = 128 // tw
        while th >= 1:
            tb = 128 // (tw * th)
            if not (one_image_per_tile and tb != 1):
                padded = (-(-W // tw) * tw) * (-(-H // th) * th) * (-(-B // tb) * tb)
                if best is None or padded < best[0]:
                    best = (padded, tw, th, tb)
            th //= 2
        tw //= 2
    return best[1:]


ALL_PATCHES = [(tw, th, 128 // (tw * th)) for tw in (128, 64, 32, 16, 8, 4, 2, 1) for th in (1, 2, 4, 8, 16, 32, 64, 128)
               if tw * th <= 128]
VGG_PAIRS = [(64, 64), (64, 128), (128, 128), (128, 256), (256, 256), (256, 512), (512, 512)]
# every patch shape choose_patch can return, each on the image batch it fits exactly (TB > 1: several images per tile)
PATCH_CASES = [(tb, th, tw) + VGG_PAIRS[i % len(VGG_PAIRS)] for i, (tw, th, tb) in enumerate(ALL_PATCHES)]


# ---- 1. 3x3 convolution forward ----------------------------------------------------------------------------------------
def conv_fwd_case(isx, route, B, H, W, Cin, Cout, relu, cfg=0, seed=0, expect=None):
    g = gen(seed * 7919 + B * 1009 + H * 31 + W + Cin + Cout)
    x = act_bf16((B, H, W, Cin), g)
    w = weights((Cout, Cin, 3, 3), g)
    bias = fine((Cout,), g)
    assert_bf16_exact(x=x, w=w, bias=bias)
    exact_budget(3 * max_abs_row_sum(w.reshape(Cout, -1)) + 2, 2.0 ** -6, "conv fwd")
    wf = torch.empty(9, Cout, Cin, device=DEV, dtype=torch.bfloat16)
    isx.call("isx_pack_conv3x3_weights", w, Cout, Cin, wf, None, isx.stream_ptr())
    out = torch.full((B, H, W, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    what = "conv fwd %s B%d %dx%d %d->%d relu%d cfg%d" % (route, B, H, W, Cin, Cout, relu, cfg)
    names = run_on_route(isx, route, lambda: isx.call("isx_conv3x3_bias_relu_fwd", x, wf, bias, out, B, H, W, Cin, Cout,
                                                      relu, cfg, isx.stream_ptr()), what, expect)
    ref = snap(conv3x3_nhwc(x, w) + bias.double(), 2.0 ** -6, what)
    if relu:
        ref = ref.clamp_min(0)
    assert_bits(out, rn_bf16(ref), what)
    return names


TILE_CFGS = [bn * 100 + mt * 10 + st for bn in (64, 128, 256) for mt in (1, 2) for st in (0, 3)]


@pytest.mark.parametrize("shape", [(3, 13, 9, 256, 256), (5, 6, 10, 64, 256)])
@pytest.mark.parametrize("cfg", TILE_CFGS)
def test_conv_fwd_generic_tiles(isx, cfg, shape):
    names = conv_fwd_case(isx, "generic", *shape, relu=cfg % 2, cfg=cfg, seed=cfg)
    assert generic_tile(names) == (cfg // 100, (cfg // 10) % 10), names


@pytest.mark.parametrize("case", PATCH_CASES, ids=["TW%dTH%dTB%d" % p for p in ALL_PATCHES])
def test_conv_fwd_generic_patch_shapes(isx, case):
    B, H, W, Cin, Cout = case
    assert len(ALL_PATCHES) == 36 and choose_patch(B, H, W) == (W, H, B)
    conv_fwd_case(isx, "generic", B, H, W, Cin, Cout, relu=(H + W) % 2)


EDGE_HW = [(1, 1), (1, 2), (2, 1), (2, 2), (3, 3), (1, 130), (130, 1), (3, 257), (17, 129), (16, 128), (7, 11), (13, 31)]


@pytest.mark.parametrize("pair", VGG_PAIRS)
@pytest.mark.parametrize("relu", [0, 1])
def test_conv_fwd_generic_vgg_pairs(isx, pair, relu):
    conv_fwd_case(isx, "generic", 2, 17, 23, *pair, relu=relu, seed=relu)


@pytest.mark.parametrize("hw", EDGE_HW)
def test_conv_fwd_generic_edges(isx, hw):
    conv_fwd_case(isx, "generic", 2, *hw, 128, 128, relu=hw[0] % 2)


C64_SHAPES = [(2, 20, 24), (3, 13, 9), (4, 160, 200), (2, 41, 37), (1, 1, 1), (1, 2, 3), (2, 3, 2), (1, 16, 8), (1, 17, 9),
              (2, 16, 7), (1, 48, 128)]
SWEEP_SHAPES = [(2, 20, 24), (3, 13, 9), (2, 41, 37), (1, 256, 40), (2, 128, 230), (4, 160, 200), (1, 300, 128), (1, 1, 1),
                (1, 2, 2), (1, 3, 129), (2, 129, 3), (1, 2, 128), (1, 131, 2)]
HALO_SHAPES = [(2, 20, 24, 64, 64), (3, 13, 9, 128, 128), (1, 50, 80, 128, 256), (2, 37, 41, 256, 128),
               (2, 100, 200, 64, 128), (3, 160, 100, 128, 64), (1, 25, 40, 512, 512), (1, 1, 1, 64, 128), (1, 2, 3, 128, 64),
               (2, 3, 1, 64, 64), (1, 16, 16, 256, 256), (1, 17, 17, 64, 64), (1, 32, 8, 128, 128), (1, 33, 9, 64, 128),
               (1, 11, 13, 256, 512), (1, 9, 7, 512, 256)]


@pytest.mark.parametrize("shape", C64_SHAPES)
def test_conv_fwd_c64(isx, shape):
    conv_fwd_case(isx, "c64", *shape, 64, 64, relu=shape[1] % 2)


@pytest.mark.parametrize("shape", SWEEP_SHAPES)
def test_conv_fwd_sweep(isx, shape):
    conv_fwd_case(isx, "sweep", *shape, 64, 64, relu=shape[1] % 2)


@pytest.mark.parametrize("shape", HALO_SHAPES)
def test_conv_fwd_halo(isx, shape):
    conv_fwd_case(isx, "halo", *shape, relu=shape[1] % 2)


@pytest.mark.parametrize("pair", VGG_PAIRS)
def test_conv_fwd_halo_vgg_pairs(isx, pair):
    conv_fwd_case(isx, "halo", 2, 19, 35, *pair, relu=1)


@pytest.mark.parametrize("B", [1, 2])
def test_conv_fwd_bench_frame(isx, B):
    """a 400 x 640 eye frame at 64 channels on the library's own choice of kernel, then forced onto conv_c64 and conv_sweep"""
    conv_fwd_case(isx, "default", B, 400, 640, 64, 64, relu=1)
    conv_fwd_case(isx, "c64", B, 400, 640, 64, 64, relu=0)
    conv_fwd_case(isx, "sweep", B, 400, 640, 64, 64, relu=0)


# ---- 2. the fused pool and its routing bytes ---------------------------------------------------------------------------
def pool_case(isx, route, B, H, W, Cin, Cout, cfg=0, plateau=False, seed=0):
    g = gen(seed * 131 + B * 1009 + H * 31 + W + Cin + 7 * Cout)
    if plateau:
        # constant input and a filter with the centre tap alone: every pixel of a channel has the same value, so every
        # window ties (and the channels whose bias drives them negative are blocked by the ReLU: code 4)
        x = torch.full((B, H, W, Cin), 2.0, device=DEV, dtype=torch.bfloat16)
        w = torch.zeros(Cout, Cin, 3, 3, device=DEV)
        w[:, :, 1, 1] = weights((Cout, Cin), g, kmax=1)
    else:
        x = act_bf16((B, H, W, Cin), g)
        w = weights((Cout, Cin, 3, 3), g)
    bias = fine((Cout,), g)
    assert_bf16_exact(x=x, w=w, bias=bias)
    exact_budget(3 * max_abs_row_sum(w.reshape(Cout, -1)) + 2, 2.0 ** -6, "conv fwd + pool")
    wf = torch.empty(9, Cout, Cin, device=DEV, dtype=torch.bfloat16)
    isx.call("isx_pack_conv3x3_weights", w, Cout, Cin, wf, None, isx.stream_ptr())
    what = "conv + pool %s B%d %dx%d %d->%d cfg%d%s" % (route, B, H, W, Cin, Cout, cfg, " plateau" if plateau else "")
    pre = rn_bf16(snap(conv3x3_nhwc(x, w) + bias.double(), 2.0 ** -6, what))
    act = pre.clamp_min(0)
    ref_pool, ref_code = pool_reference(act)
    Hp, Wp = H // 2, W // 2
    if plateau:
        assert bool((ref_code == 0).any()) and bool((ref_code == 4).any())
    out = torch.full((B, H, W, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    pool = torch.full((B, Hp, Wp, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    run_on_route(isx, route, lambda: isx.call("isx_conv3x3_bias_relu_pool_fwd", x, wf, bias, out, pool, B, H, W, Cin, Cout,
                                              cfg, isx.stream_ptr()), what)
    assert_bits(out, act, what + ": full-resolution output")
    assert_bits(pool, ref_pool, what + ": pooled map")
    sentinel = 0x7FC1   # bits of a bf16 NaN that no kernel writes
    codes = {}
    for skip in (0, 1):
        out2 = torch.full((B, H, W, Cout), sentinel, device=DEV, dtype=torch.int16).view(torch.bfloat16)
        pool2 = torch.full((B, Hp, Wp, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
        idx = torch.full((B, Hp, Wp, Cout), 255, device=DEV, dtype=torch.uint8)
        names = run_on_route(isx, route, lambda: isx.call("isx_conv3x3_bias_relu_pool_idx_fwd", x, wf, bias, out2, pool2, idx,
                                                          skip, B, H, W, Cin, Cout, cfg, isx.stream_ptr()), what)
        assert_bits(pool2, ref_pool, "%s skip_out %d: pooled map" % (what, skip))
        bad = idx != ref_code
        if bool(bad.any()):
            i = tuple(bad.nonzero()[0].tolist())
            pytest.fail("%s skip_out %d: %d / %d routing bytes differ, e.g. at %s: %d, want %d" % (
                what, skip, int(bad.sum()), idx.numel(), i, int(idx[i]), int(ref_code[i])))
        fused = not any("maxpool" in n for n in names)
        if skip and fused:
            assert bool((out2.view(torch.int16) == sentinel).all()), \
                "%s: skip_out 1 wrote the full-resolution buffer" % what
        else:   # no skip, or the generic kernel's unfused fallback, which stores the map for the separate pool launch
            assert_bits(out2, act, "%s skip_out %d: full-resolution output" % (what, skip))
        codes[skip] = idx
    return pre, codes[0]


POOL_CASES = [
    ("generic", (2, 20, 24, 64, 64), 0), ("generic", (3, 13, 9, 128, 128), 6410), ("generic", (2, 41, 37, 64, 128), 12820),
    ("generic", (5, 6, 10, 64, 64), 0), ("generic", (1, 2, 2, 128, 256), 25610), ("generic", (3, 7, 5, 256, 256), 25623),
    ("generic", (1, 3, 128, 64, 64), 0),     # 128 x 1 patch: pooled by the separate kernel after the conv
    ("generic", (2, 25, 40, 512, 512), 0),
] + [("c64", s, 0) for s in [(2, 20, 24), (3, 13, 9), (4, 160, 200), (2, 41, 37), (1, 2, 2), (1, 3, 5), (1, 17, 9)]] \
  + [("sweep", s, 0) for s in [(2, 20, 24), (3, 13, 9), (2, 41, 37), (1, 256, 40), (2, 128, 230), (4, 160, 200), (1, 2, 2),
                                (1, 3, 129), (2, 131, 5)]] \
  + [("halo", s, 0) for s in [(2, 20, 24, 64, 64), (3, 13, 9, 128, 128), (2, 37, 41, 256, 128), (2, 100, 200, 64, 128),
                               (3, 160, 100, 128, 64), (1, 25, 40, 512, 512), (1, 2, 3, 64, 128), (1, 33, 17, 128, 256)]]


def _pool_id(c):
    return "%s-%s-%d" % (c[0], "x".join(map(str, c[1])), c[2])


def _full(shape):
    return tuple(shape) if len(shape) == 5 else tuple(shape) + (64, 64)


@pytest.mark.parametrize("case", POOL_CASES, ids=[_pool_id(c) for c in POOL_CASES])
def test_conv_fused_pool(isx, case):
    route, shape, cfg = case
    pool_case(isx, route, *_full(shape), cfg=cfg)


@pytest.mark.parametrize("route,shape", [("generic", (2, 8, 10, 64, 128)), ("generic", (1, 3, 128, 64, 64)),
                                         ("c64", (2, 19, 17, 64, 64)), ("sweep", (2, 20, 130, 64, 64)),
                                         ("sweep", (1, 131, 6, 64, 64)), ("halo", (2, 18, 33, 128, 128))])
def test_conv_fused_pool_plateau(isx, route, shape):
    """every window ties: the first position must win, a window whose maximum is <= 0 routes nothing"""
    pool_case(isx, route, *shape, plateau=True)


# ---- 3. the pool backward through the epilogue's routing bytes ---------------------------------------------------------
@pytest.mark.parametrize("route,shape", [("generic", (2, 20, 24, 64, 128)), ("c64", (2, 41, 37, 64, 64)),
                                         ("sweep", (2, 41, 37, 64, 64)), ("halo", (2, 37, 41, 128, 128)),
                                         ("halo", (1, 16, 16, 64, 64))])
def test_pool_bwd_from_epilogue_codes(isx, route, shape):
    """isx_maxpool2x2_bwd_idx on the fused epilogue's bytes == torch autograd of relu -> max_pool2d, bit for bit"""
    B, H, W, Cin, Cout = shape
    pre, codes = pool_case(isx, route, *shape, plateau=route == "halo" and H == 16, seed=3)
    dyp = grad_bf16((B, H // 2, W // 2, Cout), gen(H * W))
    dx = torch.full((B, H, W, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    isx.call("isx_maxpool2x2_bwd_idx", dyp, codes, dx, B, H, W, Cout, isx.stream_ptr())
    torch.cuda.synchronize()
    z = pre.float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    F.max_pool2d(F.relu(z), 2, 2).backward(dyp.float().permute(0, 3, 1, 2).contiguous())
    assert_bits(dx, z.grad.permute(0, 2, 3, 1), "pool bwd %s %s" % (route, shape))


# ---- 4. 3x3 dgrad, its epilogues and the fused Gram tap gradient -------------------------------------------------------
def dgrad_case(isx, route, B, H, W, Cin, Cout, mode, cfg=0, seed=0):
    """dgrad of the forward conv Cin -> Cout: dy [.., Cout] -> dx [.., Cin]"""
    g = gen(seed * 17 + B * 1009 + H * 31 + W + 3 * Cin + Cout + len(mode))
    dy = grad_bf16((B, H, W, Cout), g)
    w = weights((Cout, Cin, 3, 3), g)
    act = act_bf16((B, H, W, Cin), g)
    add = fine((B, H, W, Cin), g).to(torch.bfloat16) if mode == "mask_add" else None
    aa = fine((B, Cin), g) if mode == "mask_affine" else None
    ab = fine((B, Cin), g) if mode == "mask_affine" else None
    D = None
    if mode == "gram":
        D = symmetric_D(B, Cin, g)
    assert_bf16_exact(dy=dy, w=w, act=act, add=add, aa=aa, ab=ab, D=D)
    budget = 3 * max_abs_row_sum(w.transpose(0, 1).reshape(Cin, -1)) + 2 + 2 + 2 * 3
    if D is not None:
        budget += 3 * max_abs_row_sum(D[0] if B == 1 else D.reshape(-1, Cin))
    exact_budget(budget, 2.0 ** -6, "dgrad")
    wd = torch.empty(9, Cin, Cout, device=DEV, dtype=torch.bfloat16)
    isx.call("isx_pack_conv3x3_weights", w, Cout, Cin, None, wd, isx.stream_ptr())
    dx = torch.full((B, H, W, Cin), float("nan"), device=DEV, dtype=torch.bfloat16)
    what = "dgrad %s %s B%d %dx%d %d->%d cfg%d" % (route, mode, B, H, W, Cin, Cout, cfg)
    if mode == "gram":
        fn = lambda: isx.call("isx_conv3x3_dgrad_gram", dy, wd, dx, B, H, W, Cin, Cout, act, D,  # noqa: E731
                              isx.stream_ptr())
    else:
        fn = lambda: isx.call("isx_conv3x3_dgrad", dy, wd, dx, B, H, W, Cin, Cout, None if mode == "plain" else act,  # noqa: E731
                              add, aa, ab, cfg, isx.stream_ptr())
    names = run_on_route(isx, route, fn, what)
    ref = dgrad3x3_nhwc(dy, w)
    if mode == "mask_add":
        ref = ref + add.double()
    if mode == "mask_affine":
        ref = ref + aa.double()[:, None, None, :] + ab.double()[:, None, None, :] * act.double()
    if mode == "gram":
        ref = ref + torch.bmm(act.double().reshape(B, H * W, Cin), D.double()).reshape(B, H, W, Cin)
    if mode != "plain":
        ref = torch.where(act.double() > 0, ref, torch.zeros_like(ref))
    assert_bits(dx, rn_bf16(snap(ref, 2.0 ** -6, what)), what)
    return names


DGRAD_MODES = ["plain", "mask", "mask_add", "mask_affine", "gram"]
REVERSED_PAIRS = [(cout, cin) for cin, cout in VGG_PAIRS]   # dgrad GEMMs run the VGG layers backwards: K = Cout, N = Cin


@pytest.mark.parametrize("pair", VGG_PAIRS)
@pytest.mark.parametrize("mode", DGRAD_MODES)
def test_dgrad_generic_vgg_pairs(isx, pair, mode):
    dgrad_case(isx, "generic", 2, 17, 23, *pair, mode=mode)


@pytest.mark.parametrize("cfg", [6410, 6423, 12811, 12820, 25612, 25620])
@pytest.mark.parametrize("mode", ["mask", "mask_affine"])
def test_dgrad_generic_tiles(isx, cfg, mode):
    names = dgrad_case(isx, "generic", 3, 13, 9, 256, 256, mode=mode, cfg=cfg)
    assert generic_tile(names) == (cfg // 100, (cfg // 10) % 10), names


@pytest.mark.parametrize("hw", [(1, 1), (2, 3), (3, 2), (1, 130), (17, 129), (16, 128)])
@pytest.mark.parametrize("mode", ["mask_affine", "gram"])
def test_dgrad_generic_edges(isx, hw, mode):
    dgrad_case(isx, "generic", 2, *hw, 64, 128, mode=mode)


@pytest.mark.parametrize("shape", C64_SHAPES)
@pytest.mark.parametrize("mode", DGRAD_MODES)
def test_dgrad_c64(isx, shape, mode):
    dgrad_case(isx, "c64", *shape, 64, 64, mode=mode)


@pytest.mark.parametrize("shape", SWEEP_SHAPES)
@pytest.mark.parametrize("mode", DGRAD_MODES)
def test_dgrad_sweep(isx, shape, mode):
    dgrad_case(isx, "sweep", *shape, 64, 64, mode=mode)


@pytest.mark.parametrize("shape", HALO_SHAPES)
@pytest.mark.parametrize("mode", DGRAD_MODES)
def test_dgrad_halo(isx, shape, mode):
    dgrad_case(isx, "halo", *shape, mode=mode)


@pytest.mark.parametrize("pair", REVERSED_PAIRS)
@pytest.mark.parametrize("mode", ["mask_affine", "gram"])
def test_dgrad_halo_vgg_pairs(isx, pair, mode):
    dgrad_case(isx, "halo", 2, 19, 35, pair[1], pair[0], mode=mode)


# ---- 5. Gram ----------------------------------------------------------------------------------------------------------
def gram_pick_splits(B, HW, C, sms):
    """conv-side replica of gram_tc.cu's split choice, to aim tests at its extremes"""
    n_units = {64: 1, 128: 1, 256: 2, 512: 6}[C]
    kp = 64 if C <= 128 else 32
    per_sm = 4 if C >= 256 else 6
    want = (per_sm * sms) // (B * n_units)
    want = max(1, min(want, max(1, HW // (kp * 4))))
    chunk = (-(-HW // want) + kp - 1) // kp * kp
    return -(-HW // chunk), (per_sm * sms) // (B * n_units)


def gram_case(isx, B, HW, C, mask_b=0, seed=0):
    g = gen(seed + B * 7 + HW * 3 + C)
    f = act_bf16((B, HW, C), g)
    Fd = f.double()
    lsb = 1.0
    m = None
    if mask_b:
        # quarter steps, and a run of zero pixels long enough to empty whole K blocks (the kernel skips those)
        m = ints((mask_b, HW), 0, 4, g) / 4
        m[:, HW // 4: HW // 4 + max(HW // 2, 1)] = 0
        m = m.float()
        Fd = Fd * m.double().reshape(mask_b, HW, 1)
        lsb = 1.0 / 16
    assert_bf16_exact(f=f, fm=Fd, m=m)
    exact_budget(HW * float(Fd.abs().max()) ** 2 + 1e-30, lsb, "gram")
    inv_n = 2.0 ** -math.ceil(math.log2(C * HW))
    grad_scale, loss_scale = 8.0, 0.25
    S = torch.bmm(Fd.transpose(1, 2), Fd)
    G_exact = S * inv_n
    # T = G - k * LSB_G with |k| < 2^10: G - T, its square and the kernel's per-thread sums of eight squares are exact in
    # fp32, and grad_scale * (G - T) has 10 significant bits, so D is rounded to bf16 (ties to even included)
    k = ints((B, C, C), -1023, 1023, g)
    lsb_g = lsb * inv_n
    T = G_exact - k * lsb_g
    assert torch.equal(T.float().double(), T)
    T = T.float()
    sms = isx.load().isx_sm_count()
    splits, _ = gram_pick_splits(B, HW, C, sms)
    ws_bytes = isx.call_i64("isx_gram_workspace_bytes", B, HW, C)
    assert ws_bytes == splits * B * C * C * 4, (ws_bytes, splits)
    ws = torch.empty(ws_bytes, device=DEV, dtype=torch.uint8)
    G = torch.full((B, C, C), float("nan"), device=DEV)
    D = torch.full((B, C, C), float("nan"), device=DEV, dtype=torch.bfloat16)
    loss = torch.zeros(B, device=DEV, dtype=torch.float64)
    s = isx.stream_ptr()
    what = "gram B%d HW%d C%d mask_b%d splits%d" % (B, HW, C, mask_b, splits)
    if mask_b:
        fl = torch.empty(max(16, isx.call_i64("isx_gram_mask_flags_bytes", mask_b, HW, C)), device=DEV, dtype=torch.uint8)
        fm2 = torch.full((B, HW, C), float("nan"), device=DEV, dtype=torch.bfloat16)
        isx.call("isx_gram_masked_fwd", f, B, HW, C, m, mask_b, fl, fm2, isx.f32(inv_n), ws, G, T, B, isx.f64(loss_scale),
                 loss, isx.f32(grad_scale), D, s)
    else:
        isx.call("isx_gram_fwd", f, B, HW, C, isx.f32(inv_n), ws, G, T, B, isx.f64(loss_scale), loss, isx.f32(grad_scale), D, s)
    torch.cuda.synchronize()
    bad = G.double() != G_exact
    assert not bool(bad.any()), "%s: %d / %d Gram entries differ, e.g. %s" % (what, int(bad.sum()), G.numel(),
                                                                               bad.nonzero()[0].tolist())
    assert torch.equal(G, G.transpose(1, 2)), what + ": G is not symmetric"
    assert_bits(D, rn_bf16(grad_scale * k * lsb_g), what + ": D")
    ref_loss = loss_scale * ((k * lsb_g) ** 2).sum(dim=(1, 2))
    assert torch.allclose(loss, ref_loss, rtol=1e-12, atol=0), (what, loss.tolist(), ref_loss.tolist())
    if mask_b:
        fm2_ref = (f.double() * m.double().reshape(mask_b, HW, 1) ** 2).to(torch.bfloat16)
        assert_bits(fm2, fm2_ref, what + ": F * m^2")
    return splits


GRAM_SMALL_HW = [1, 63, 65, 127, 129]


@pytest.mark.parametrize("C", [64, 128, 256, 512])
@pytest.mark.parametrize("HW", GRAM_SMALL_HW)
def test_gram_fwd_small_hw(isx, C, HW):
    """HW that is no multiple of the K block, down to a single pixel: one split"""
    assert gram_case(isx, 2, HW, C) == 1


@pytest.mark.parametrize("C,HW", [(64, 400 * 640), (128, 400 * 640), (256, 200 * 200), (512, 100 * 160)])
def test_gram_fwd_most_splits(isx, C, HW):
    """one image large enough that the split count is bounded by the SM count, not by HW"""
    sms = isx.load().isx_sm_count()
    splits, cap = gram_pick_splits(1, HW, C, sms)
    assert HW // ((64 if C <= 128 else 32) * 4) >= cap
    assert gram_case(isx, 1, HW, C) == splits > 1


@pytest.mark.parametrize("C", [64, 128, 256, 512])
@pytest.mark.parametrize("HW,mask_b", [(63, 1), (129, 2), (1, 1), (4000, 2)])
def test_gram_masked_fwd(isx, C, HW, mask_b):
    gram_case(isx, 2, HW, C, mask_b=mask_b)


@pytest.mark.parametrize("C", [64, 128, 256, 512])
@pytest.mark.parametrize("relu", [False, True])
def test_gram_bwd(isx, C, relu):
    B, H, W = 2, 13, 17
    g = gen(C + relu)
    f = act_bf16((B, H, W, C), g)
    D = symmetric_D(B, C, g)
    assert_bf16_exact(f=f, D=D)
    exact_budget(3 * max_abs_row_sum(D.reshape(-1, C)), 2.0 ** -6, "gram bwd")
    dF = torch.full((B, H, W, C), float("nan"), device=DEV, dtype=torch.bfloat16)
    names = launched(lambda: isx.call("isx_gram_bwd", f, D, dF, B, H, W, C, f if relu else None, isx.stream_ptr()))
    assert names and all("conv_tc_kernel" in n for n in names), names
    ref = torch.bmm(f.double().reshape(B, H * W, C), D.double()).reshape(B, H, W, C)
    if relu:
        ref = torch.where(f.double() > 0, ref, torch.zeros_like(ref))
    assert_bits(dF, rn_bf16(snap(ref, 2.0 ** -6, "gram bwd")), "gram bwd C%d relu%d" % (C, relu))


# ---- 7. the same conv_tc, other callers ------------------------------------------------------------------------------
CBA_CASES = [
    # k, stride, Cin, Cout, B, H, W, residual, relu
    (1, 1, 64, 256, 3, 25, 33, True, True),
    (1, 2, 256, 512, 2, 25, 33, False, False),
    (3, 2, 128, 128, 3, 25, 33, True, True),
    (3, 1, 64, 64, 1, 31, 17, True, False),
    (3, 2, 64, 128, 5, 9, 11, False, True),
    (1, 1, 2048, 512, 2, 7, 9, True, True),
    (3, 1, 256, 256, 2, 1, 3, False, True),
    (1, 2, 1024, 2048, 1, 13, 17, True, False),
]


@pytest.mark.parametrize("case", CBA_CASES)
def test_conv_bias_act(isx, case):
    k, stride, Cin, Cout, B, H, W, res, relu = case
    g = gen(sum(case[:7]))
    x = act_bf16((B, H, W, Cin), g)
    w = weights((Cout, Cin, k, k), g)
    bias = fine((Cout,), g)
    Ho, Wo = (H + stride - 1) // stride, (W + stride - 1) // stride
    r = fine((B, Ho, Wo, Cout), g).to(torch.bfloat16) if res else None
    assert_bf16_exact(x=x, w=w, bias=bias, r=r)
    exact_budget(3 * max_abs_row_sum(w.reshape(Cout, -1)) + 4, 2.0 ** -6, "conv_bias_act")
    s = isx.stream_ptr()
    if k == 1:
        wp = torch.empty(Cout, Cin, device=DEV, dtype=torch.bfloat16)
        isx.call("isx_pack_conv1x1_weights", w.reshape(Cout, Cin).contiguous(), Cout, Cin, wp, s)
    else:
        wp = torch.empty(9, Cout, Cin, device=DEV, dtype=torch.bfloat16)
        isx.call("isx_pack_conv3x3_weights", w, Cout, Cin, wp, None, s)
    out = torch.full((B, Ho, Wo, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    names = launched(lambda: isx.call("isx_conv_bias_act_fwd", x, wp, bias, r, out, B, H, W, Cin, Cout, k, stride, int(relu),
                                      isx.stream_ptr()))
    assert names and all("conv_tc_kernel" in n for n in names), names
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), w.double(), bias.double(), stride=stride, padding=k // 2).permute(0, 2, 3, 1)
    if res:
        ref = ref + r.double()
    if relu:
        ref = ref.clamp_min(0)
    exp = rn_bf16(snap(ref, 2.0 ** -6, "conv_bias_act"))
    assert_bits(out, exp, "conv_bias_act %s" % (case,))
    for rep in range(2):   # the same call again, into a fresh buffer: the result must not depend on the run
        out.fill_(float("nan"))
        isx.call("isx_conv_bias_act_fwd", x, wp, bias, r, out, B, H, W, Cin, Cout, k, stride, int(relu), isx.stream_ptr())
        torch.cuda.synchronize()
        assert_bits(out, exp, "conv_bias_act %s, repeated call %d" % (case, rep + 1))


@pytest.mark.parametrize("B,xc,H,W", [(3, 3, 97, 131), (1, 1, 64, 64), (2, 3, 33, 32), (1, 3, 7, 9)])
def test_resnet_stem(isx, B, xc, H, W):
    g = gen(B * 7 + H)
    x = (ints((B, xc, H, W), 0, 256, g) / 256).float()     # k / 256: exact in bf16, as the stem stages it
    w = weights((64, 3, 7, 7), g)
    bias = fine((64,), g)
    assert_bf16_exact(x=x, w=w, bias=bias)
    exact_budget(max_abs_row_sum(w.reshape(64, -1)) + 2, 2.0 ** -14, "stem")
    s = isx.stream_ptr()
    wp = torch.empty(64, 192, device=DEV, dtype=torch.bfloat16)
    isx.call("isx_pack_resnet_stem_weights", w, wp, s)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    out = torch.full((B, Ho, Wo, 64), float("nan"), device=DEV, dtype=torch.bfloat16)
    isx.call("isx_resnet_stem_fwd", x, xc, wp, bias, out, B, H, W, s)
    torch.cuda.synchronize()
    ref = F.conv2d(x.double().repeat(1, 3 // xc, 1, 1), w.double(), bias.double(), stride=2, padding=3).clamp_min(0)
    assert_bits(out, rn_bf16(snap(ref.permute(0, 2, 3, 1), 2.0 ** -14, "stem")), "stem B%d xc%d %dx%d" % (B, xc, H, W))


def linear_layer(isx, Xp, W, bias, M, Mpad, N, Npad, relu, lsb, what):
    """isx_linear_pack + isx_linear_fwd; returns out^T [Npad, Mpad] and the exact expected out^T.  lsb: the smallest
    product LSB of the operands"""
    K = W.shape[1]
    s = isx.stream_ptr()
    Wp = torch.full((Npad, K + 64), float("nan"), device=DEV, dtype=torch.bfloat16)
    isx.call("isx_linear_pack", W, bias, N, K, Npad, Wp, s)
    outT = torch.full((Npad, Mpad), float("nan"), device=DEV, dtype=torch.bfloat16)
    names = launched(lambda: isx.call("isx_linear_fwd", Xp, Wp, outT, Mpad, Npad, K + 64, relu, isx.stream_ptr()))
    assert names and all("conv_tc_kernel" in n for n in names), names
    Wd = torch.zeros(Npad, K + 64, dtype=torch.float64, device=DEV)
    Wd[:N, :K] = W.double()
    Wd[:N, K] = bias.double()
    assert torch.equal(Wp.double(), Wd), what + ": packed weights"
    X = Xp.double()
    exact_budget(float((X.abs() @ Wd.abs().t()).max()), lsb, what)
    ref = X @ Wd.t()
    if relu:
        ref = ref.clamp_min(0)
    ref = rn_bf16(snap(ref, lsb, what)).t()
    assert_bits(outT, ref, what + ": out^T")
    return outT, ref


@pytest.mark.parametrize("M,Mpad", [(50, 64), (200, 256)])
def test_classifier_chain_rows(isx, M, Mpad):
    """Linear(25088, 320) + ReLU -> Linear(320, 100): rows_pack, linear_fwd, transpose_pack, linear_fwd, transpose_out"""
    K, N1, N2 = 25088, 320, 100
    g = gen(M)
    src = ints((M, K), -3, 3, g).float()
    W1, b1 = weights((N1, K), g, kmax=2), fine((N1,), g)
    W2, b2 = weights((N2, N1), g), fine((N2,), g)
    s = isx.stream_ptr()
    X1 = torch.full((Mpad, K + 64), float("nan"), device=DEV, dtype=torch.bfloat16)
    isx.call("isx_rows_pack", src, K, M, K, Mpad, X1, s)
    X1ref = torch.zeros(Mpad, K + 64, dtype=torch.float64, device=DEV)
    X1ref[:M, :K] = src.double()
    X1ref[:M, K] = 1
    assert torch.equal(X1.double(), X1ref), "rows_pack"
    out1, ref1 = linear_layer(isx, X1, W1, b1, M, Mpad, N1, 384, 1, 2.0 ** -6, "layer 1 M%d" % M)
    X2 = torch.full((Mpad, N1 + 64), float("nan"), device=DEV, dtype=torch.bfloat16)
    isx.call("isx_transpose_pack", out1, N1, Mpad, M, X2, s)
    X2ref = torch.zeros(Mpad, N1 + 64, dtype=torch.float64, device=DEV)
    X2ref[:M, :N1] = ref1[:N1, :M].t().double()
    X2ref[:M, N1] = 1
    torch.cuda.synchronize()
    assert torch.equal(X2.double(), X2ref), "transpose_pack"
    out2, ref2 = linear_layer(isx, X2, W2, b2, M, Mpad, N2, 128, 0, 2.0 ** -12, "layer 2 M%d" % M)
    logits = torch.full((M, N2), float("nan"), device=DEV)
    isx.call("isx_transpose_out", out2, N2, Mpad, M, logits, s)
    torch.cuda.synchronize()
    assert torch.equal(logits, ref2[:N2, :M].t().float()), "transpose_out"


@pytest.mark.parametrize("B,h,w,Mpad", [(3, 14, 14, 64), (70, 14, 28, 256)])
def test_classifier_chain_pool7(isx, B, h, w, Mpad):
    """AdaptiveAvgPool2d(7,7) + Flatten over bins of 4 / 8 pixels (exact divisions) -> Linear(25088, 320)"""
    C, N1 = 512, 320
    g = gen(B + h + w)
    p5 = act_bf16((B, h, w, C), g)
    X = torch.full((Mpad, C * 49 + 64), float("nan"), device=DEV, dtype=torch.bfloat16)
    isx.call("isx_pool7_flatten_pack", p5, B, h, w, C, Mpad, X, isx.stream_ptr())
    Xref = torch.zeros(Mpad, C * 49 + 64, dtype=torch.float64, device=DEV)
    Xref[:B, :C * 49] = F.adaptive_avg_pool2d(p5.double().permute(0, 3, 1, 2), (7, 7)).flatten(1)
    Xref[:B, C * 49] = 1
    torch.cuda.synchronize()
    assert torch.equal(Xref.to(torch.bfloat16).double(), Xref)
    assert torch.equal(X.double(), Xref), "pool7_flatten_pack"
    W1, b1 = weights((N1, C * 49), g, kmax=2), fine((N1,), g)
    area = (h // 7) * (w // 7)
    linear_layer(isx, X, W1, b1, B, Mpad, N1, N1, 1, 2.0 ** -6 / area, "pool7 layer B%d" % B)


# ---- 8. conv1_1 head and image-gradient tail: float64 with a sum-of-|terms| bound ---------------------------------------
MEAN = torch.tensor([0.485, 0.456, 0.406], dtype=torch.float32).double().view(1, 3, 1, 1)
STD = torch.tensor([0.229, 0.224, 0.225], dtype=torch.float32).double().view(1, 3, 1, 1)


MASKS = {"none": 0, "shared": 1, "per_image": -1}   # mask batch: none, 1, B


def conv1_1_operands(B, H, W, xc, mask_b, seed):
    g = gen(seed + B * 101 + H * 13 + W)
    x = torch.rand(B, xc, H, W, device=DEV, generator=g)
    w = torch.randn(64, 3, 3, 3, device=DEV, generator=g) * 0.2
    bias = torch.randn(64, device=DEV, generator=g) * 0.1
    mask = (ints((mask_b, 1, H, W), 0, 4, g) / 4).float() if mask_b else None
    return x, w, bias, mask


def normalised(x, mask):
    xn = (x.double().expand(-1, 3, -1, -1) - MEAN.to(DEV)) / STD.to(DEV)
    return xn * mask.double() if mask is not None else xn


def assert_within(got, ref, abssum, rel, abs_units, what):
    err = (got.double() - ref).abs()
    bound = rel * ref.abs() + abs_units * abssum + 1e-30
    worst = float((err / bound).max())
    print("%s: max |err| %.3g, worst err / bound %.3f" % (what, float(err.max()), worst))
    assert worst <= 1.0, "%s: error %.3f x the bound" % (what, worst)


CONV1_1_SHAPES = [(1, 1, 1), (2, 3, 5), (1, 17, 129), (3, 15, 29), (2, 64, 40)]


@pytest.mark.parametrize("B,H,W", CONV1_1_SHAPES)
@pytest.mark.parametrize("xc", [1, 3])
@pytest.mark.parametrize("mask", list(MASKS))
def test_conv1_1_fwd(isx, B, H, W, xc, mask):
    """bf16 outputs within 2^-8 |ref| + 1e-5 sum|terms| of float64 (the old tests allow 2^-7 |ref| + 2 % of the mean)"""
    mask_b = MASKS[mask] if MASKS[mask] >= 0 else B
    x, w, bias, mask = conv1_1_operands(B, H, W, xc, mask_b, 1)
    s = isx.stream_ptr()
    xn = normalised(x, mask)
    for kind in ("cuda_core", "tc"):
        out = torch.full((B, H, W, 64), float("nan"), device=DEV, dtype=torch.bfloat16)
        if kind == "cuda_core":
            wr = w.double()
            isx.call("isx_conv1_1_fwd", x, xc, mask, mask_b, w, bias, out, B, H, W, s)
        else:
            wr = w.to(torch.bfloat16).double()
            w0p = torch.empty(64, 64, device=DEV, dtype=torch.bfloat16)
            isx.call("isx_pack_conv1_1_fwd", w, w0p, s)
            isx.call("isx_conv1_1_fwd_tc", x, xc, mask, mask_b, w0p, bias, out, B, H, W, s)
        torch.cuda.synchronize()
        ref = F.conv2d(xn, wr, bias.double(), padding=1).clamp_min(0).permute(0, 2, 3, 1)
        abssum = (F.conv2d(xn.abs(), wr.abs(), padding=1) + bias.double().abs().view(1, 64, 1, 1)).permute(0, 2, 3, 1)
        assert_within(out, ref, abssum, 2.0 ** -8, 1e-5, "conv1_1 fwd %s B%d %dx%d xc%d mask_b%d" % (kind, B, H, W, xc, mask_b))


CONV1_1_TAILS = {
    # kernel options, kernel, its first template argument (BN = 16: the image-gradient tail)
    "tail_n": (dict(tail_n=1, c64=1), "conv1_1_tail_kernel", None),
    "generic": (dict(tail_n=0, c64=1), "conv_tc_kernel", 16),
    "c64": (dict(tail_n=1, c64=2), "conv_c64_kernel", 16),
}


@pytest.mark.parametrize("B,H,W", CONV1_1_SHAPES)
@pytest.mark.parametrize("xc", [1, 3])
@pytest.mark.parametrize("mask", list(MASKS))
def test_conv1_1_dgrad(isx, B, H, W, xc, mask):
    """fp32 image gradients within 8 fp32 ulps of sum|terms| (+ 2^-22 |ref| for the 1/std and mask products) of float64,
    from the CUDA-core tail and each tensor-core tail"""
    mask_b = MASKS[mask] if MASKS[mask] >= 0 else B
    x, w, bias, mask = conv1_1_operands(B, H, W, xc, mask_b, 2)
    dy = grad_bf16((B, H, W, 64), gen(B * H * W + xc))
    s = isx.stream_ptr()
    md = mask.double() if mask is not None else torch.ones(1, 1, H, W, dtype=torch.float64, device=DEV)

    def reference(wr):
        dyn = dy.double().permute(0, 3, 1, 2)
        gx = F.conv_transpose2d(dyn, wr, padding=1) * md / STD.to(DEV)
        ab = F.conv_transpose2d(dyn.abs(), wr.abs(), padding=1) * md.abs() / STD.to(DEV)
        if xc == 1:
            gx, ab = gx.sum(dim=1, keepdim=True), ab.sum(dim=1, keepdim=True)
        return gx, ab

    dx = torch.full((B, xc, H, W), float("nan"), device=DEV)
    isx.call("isx_conv1_1_dgrad", dy, w, mask, mask_b, dx, xc, B, H, W, s)
    torch.cuda.synchronize()
    ref, ab = reference(w.double())
    what = "conv1_1 dgrad B%d %dx%d xc%d mask_b%d" % (B, H, W, xc, mask_b)
    assert_within(dx, ref, ab, 2.0 ** -22, 8 * 2.0 ** -24, what + " cuda_core")
    wd0 = torch.empty(9, 16, 64, device=DEV, dtype=torch.bfloat16)
    isx.call("isx_pack_conv1_1_dgrad", w, wd0, s)
    ref, ab = reference(w.to(torch.bfloat16).double())
    for name, (opts, kernel, args) in CONV1_1_TAILS.items():
        dx2 = torch.full((B, xc, H, W), float("nan"), device=DEV)
        with options(isx, **opts):
            names = launched(lambda: isx.call("isx_conv1_1_dgrad_tc", dy, wd0, mask, mask_b, dx2, xc, B, H, W, isx.stream_ptr()))
        assert names and all(kernel in n and (args is None or kernel_args(n, kernel)[0] == args) for n in names), (name, names)
        assert_within(dx2, ref, ab, 2.0 ** -22, 8 * 2.0 ** -24, what + " " + name)
