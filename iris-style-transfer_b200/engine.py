"""Host-side plumbing around libisx's fused NST driver (isx_nst_forward / isx_nst_eval /
isx_lbfgs_tick): ctypes mirrors of the C structs, weight packing, workspace ownership.
PyTorch supplies device memory and streams only -- no torch op touches the data path."""
from __future__ import annotations

import ctypes
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib

MAX_TAPS = 8
N_CONVS = 16
TAP_POOL0 = 16          # tap ids: 0..15 = ReLU output of conv i, 16..20 = output of pool 0..4 (include/isx.h ISX_TAP_POOL0)
N_TAPS = 21
FWD_LAST_POOL, FWD_LEAN = 1, 2   # include/isx.h ISX_FWD_*
CONV_BEFORE_POOL = [1, 3, 7, 11, 15]

# models/vgg/vgg.py:6-10 (torchvision vgg19.features indices)
VGG19_CFG = [64, 64, "M", 128, 128, "M", 256, 256, 256, 256, "M", 512, 512, 512, 512, "M", 512, 512, 512, 512, "M"]
VGG19_LAYERS: Dict[str, int] = {}
CONV_OF_FEATURE_INDEX: Dict[int, int] = {}   # features index (conv or relu) -> conv ordinal 0..15
POOL_OF_FEATURE_INDEX: Dict[int, int] = {}   # features index of a pool -> pool ordinal 0..4
_i, _blk, _sub, _c, _p = 0, 1, 1, 0, 0
for _v in VGG19_CFG:
    if _v == "M":
        VGG19_LAYERS["pool%d" % _blk] = _i
        POOL_OF_FEATURE_INDEX[_i] = _p
        _p += 1
        _i += 1
        _blk += 1
        _sub = 1
    else:
        VGG19_LAYERS["conv%d_%d" % (_blk, _sub)] = _i
        VGG19_LAYERS["relu%d_%d" % (_blk, _sub)] = _i + 1
        CONV_OF_FEATURE_INDEX[_i] = _c       # in-place ReLU: a conv tap aliases the ReLU output (SURVEY N2)
        CONV_OF_FEATURE_INDEX[_i + 1] = _c
        _c += 1
        _i += 2
        _sub += 1
CONV_COUT = [v for v in VGG19_CFG if v != "M"]


class NstConfig(ctypes.Structure):
    _fields_ = [
        ("B", ctypes.c_int32), ("H", ctypes.c_int32), ("W", ctypes.c_int32), ("xc", ctypes.c_int32),
        ("n_conv", ctypes.c_int32), ("style_mode", ctypes.c_int32),
        ("n_style", ctypes.c_int32), ("style_conv", ctypes.c_int32 * MAX_TAPS), ("style_w", ctypes.c_float * MAX_TAPS),
        ("n_content", ctypes.c_int32), ("content_conv", ctypes.c_int32 * MAX_TAPS),
        ("content_w", ctypes.c_float * MAX_TAPS),
        ("style_target_b", ctypes.c_int32), ("content_target_b", ctypes.c_int32),
        ("coupled", ctypes.c_int32), ("mask_b", ctypes.c_int32),
        ("style_mask_b", ctypes.c_int32), ("pred_unbatched", ctypes.c_int32),
        ("c_weight", ctypes.c_double), ("s_weight", ctypes.c_double),
    ]


class NstBuffers(ctypes.Structure):
    _fields_ = [
        ("w0", ctypes.c_void_p),
        ("w0_fwd", ctypes.c_void_p),
        ("w0_dgrad", ctypes.c_void_p),
        ("bias", ctypes.c_void_p * N_CONVS),
        ("w_fwd", ctypes.c_void_p * N_CONVS),
        ("w_dgrad", ctypes.c_void_p * N_CONVS),
        ("workspace", ctypes.c_void_p),
        ("content_target", ctypes.c_void_p * MAX_TAPS),
        ("gram_target", ctypes.c_void_p * MAX_TAPS),
        ("bn_target_mean", ctypes.c_void_p * MAX_TAPS),
        ("bn_target_std", ctypes.c_void_p * MAX_TAPS),
        ("input_mask", ctypes.c_void_p),
        ("style_mask", ctypes.c_void_p * MAX_TAPS),
    ]


class LbfgsConfig(ctypes.Structure):
    _fields_ = [
        ("epochs", ctypes.c_int32), ("max_iter", ctypes.c_int32), ("max_eval", ctypes.c_int32),
        ("history", ctypes.c_int32), ("history_bf16", ctypes.c_int32), ("reserved_", ctypes.c_int32),
        ("lr", ctypes.c_double), ("tolerance_grad", ctypes.c_double),
        ("tolerance_change", ctypes.c_double), ("c_weight", ctypes.c_double), ("s_weight", ctypes.c_double),
    ]


class NstProblems(ctypes.Structure):
    _fields_ = [
        ("images_per_problem", ctypes.c_int32), ("style_target_b", ctypes.c_int32),
        ("c_weight", ctypes.c_void_p), ("s_weight", ctypes.c_void_p),
    ]


class NstProblemRanges(ctypes.Structure):
    _fields_ = [
        ("n_problems", ctypes.c_int32), ("style_target_b", ctypes.c_int32),
        ("first_image", ctypes.c_void_p), ("c_weight", ctypes.c_void_p), ("s_weight", ctypes.c_void_p),
    ]


def problem_ranges(first_image: Sequence[int], c_weight: torch.Tensor, s_weight: torch.Tensor):
    """isx_nst_problem_ranges for the offsets first_image [P+1] (a host int32 array, returned with the struct: it must
    outlive every call that reads the struct) and the device float64 [P] weights."""
    P = len(first_image) - 1
    for w in (c_weight, s_weight):
        assert w.is_cuda and w.dtype == torch.float64 and w.is_contiguous() and w.shape == (P,)
    offsets = (ctypes.c_int32 * (P + 1))(*[int(v) for v in first_image])
    pr = NstProblemRanges()
    pr.n_problems = P
    pr.first_image = ctypes.cast(offsets, ctypes.c_void_p).value
    pr.c_weight, pr.s_weight = c_weight.data_ptr(), s_weight.data_ptr()
    return pr, offsets


class PackedVGG:
    """VGG-19 conv parameters packed once for the device kernels (isx_pack_conv3x3_weights)."""

    def __init__(self, weights: Sequence[Tuple[torch.Tensor, torch.Tensor]], device: torch.device):
        assert len(weights) == N_CONVS, "expected the 16 (weight, bias) pairs of vgg19.features"
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.IsxError("iris_b200 runs on a CUDA B200 only (device=%s); there is no CPU path" % device)
        _lib.call("isx_device_check", self.device.index or 0)
        self.w0 = weights[0][0].detach().to(self.device, torch.float32).contiguous()
        self.bias = [b.detach().to(self.device, torch.float32).contiguous() for _, b in weights]
        self.w_fwd: List[Optional[torch.Tensor]] = [None]
        self.w_dgrad: List[Optional[torch.Tensor]] = [None]
        with torch.cuda.device(self.device):
            self.w0_dgrad = torch.empty(9, 16, 64, device=self.device, dtype=torch.bfloat16)
            _lib.call("isx_pack_conv1_1_dgrad", self.w0, self.w0_dgrad, _lib.stream_ptr())
            self.w0_fwd = torch.empty(64, 64, device=self.device, dtype=torch.bfloat16)
            _lib.call("isx_pack_conv1_1_fwd", self.w0, self.w0_fwd, _lib.stream_ptr())
            for i in range(1, N_CONVS):
                w = weights[i][0].detach().to(self.device, torch.float32).contiguous()
                cout, cin = w.shape[:2]
                wf = torch.empty(9, cout, cin, device=self.device, dtype=torch.bfloat16)
                wd = torch.empty(9, cin, cout, device=self.device, dtype=torch.bfloat16)
                _lib.call("isx_pack_conv3x3_weights", w, cout, cin, wf, wd, _lib.stream_ptr())
                self.w_fwd.append(wf)
                self.w_dgrad.append(wd)
            torch.cuda.current_stream().synchronize()


class NstEngine:
    """One (batch shape, tap set) instance of the fused driver.  Owns the workspace."""

    def __init__(self, packed: PackedVGG, B: int, H: int, W: int, xc: int, content_convs: Sequence[int],
                 style_convs: Sequence[int], style_mode: int = 0, content_w: Optional[Sequence[float]] = None,
                 style_w: Optional[Sequence[float]] = None, c_weight: float = 1.0, s_weight: float = 1.0,
                 coupled: bool = False, n_conv: Optional[int] = None, style_mask_b: int = 0,
                 pred_unbatched: bool = False):
        self.packed = packed
        self.device = packed.device
        cfg = NstConfig()
        cfg.B, cfg.H, cfg.W, cfg.xc = B, H, W, xc
        taps = list(content_convs) + list(style_convs)
        cfg.n_conv = n_conv if n_conv is not None else (max(tap_conv(t) for t in taps) + 1 if taps else N_CONVS)
        cfg.style_mode = style_mode
        if len(style_convs) > MAX_TAPS or len(content_convs) > MAX_TAPS:
            raise ValueError("at most %d style and %d content layers" % (MAX_TAPS, MAX_TAPS))
        cfg.n_style = len(style_convs)
        cfg.n_content = len(content_convs)
        for t, c in enumerate(style_convs):
            cfg.style_conv[t] = c
            cfg.style_w[t] = 1.0 if style_w is None else float(style_w[t])
        for t, c in enumerate(content_convs):
            cfg.content_conv[t] = c
            cfg.content_w[t] = 1.0 if content_w is None else float(content_w[t])
        cfg.style_target_b = B
        cfg.content_target_b = B
        cfg.coupled = int(coupled)
        cfg.mask_b = 0
        cfg.style_mask_b = int(style_mask_b)
        cfg.pred_unbatched = int(pred_unbatched)
        cfg.c_weight, cfg.s_weight = float(c_weight), float(s_weight)
        self.cfg = cfg
        nbytes = _lib.call_i64("isx_nst_workspace_bytes", ctypes.byref(cfg))
        if nbytes < 0:
            raise _lib.IsxError("isx_nst_workspace_bytes: " + _lib.load().isx_last_error().decode())
        self.workspace = torch.empty(nbytes, device=self.device, dtype=torch.uint8)
        bufs = NstBuffers()
        bufs.w0 = packed.w0.data_ptr()
        bufs.w0_dgrad = packed.w0_dgrad.data_ptr()
        bufs.w0_fwd = packed.w0_fwd.data_ptr()
        for i in range(N_CONVS):
            bufs.bias[i] = packed.bias[i].data_ptr()
            bufs.w_fwd[i] = packed.w_fwd[i].data_ptr() if packed.w_fwd[i] is not None else None
            bufs.w_dgrad[i] = packed.w_dgrad[i].data_ptr() if packed.w_dgrad[i] is not None else None
        bufs.workspace = self.workspace.data_ptr()
        self.bufs = bufs
        self._keep: List[torch.Tensor] = []  # targets referenced by raw pointer
        self.loss_c = torch.zeros(B, device=self.device, dtype=torch.float64)
        self.loss_s = torch.zeros(B, device=self.device, dtype=torch.float64)
        self.problems: Optional[NstProblems] = None
        self.ranges: Optional[NstProblemRanges] = None

    def set_problems(self, images_per_problem: int, c_weight: torch.Tensor, s_weight: torch.Tensor):
        """Evaluate the batch as B / images_per_problem coupled problems (isx_nst_eval_problems) with per-problem alpha /
        beta: device float64 [P] tensors, read on every eval (they may be updated in place between evals)."""
        for w in (c_weight, s_weight):
            assert w.is_cuda and w.dtype == torch.float64 and w.is_contiguous()
            assert w.shape == (self.cfg.B // images_per_problem,)
        self._keep += [c_weight, s_weight]
        pr = NstProblems()
        pr.images_per_problem = int(images_per_problem)
        pr.c_weight, pr.s_weight = c_weight.data_ptr(), s_weight.data_ptr()
        self.problems = pr

    def set_problem_ranges(self, first_image: Sequence[int], c_weight: torch.Tensor, s_weight: torch.Tensor):
        """Evaluate the batch as P coupled problems of unequal size (isx_nst_eval_ranges): problem p is the images
        [first_image[p], first_image[p+1]), with per-problem alpha / beta as device float64 [P] tensors read on every
        eval.  The offsets are checked by the library on every call."""
        self.ranges, self._offsets = problem_ranges(first_image, c_weight, s_weight)
        self._keep += [c_weight, s_weight]

    # ---- targets -------------------------------------------------------------------------
    def set_input_mask(self, mask: Optional[torch.Tensor]):
        if mask is None:
            self.cfg.mask_b = 0
            self.bufs.input_mask = None
            return
        m = mask.detach().to(self.device, torch.float32).contiguous()
        if m.dim() == 3:
            m = m[None]
        assert m.shape[-2:] == (self.cfg.H, self.cfg.W) and m.shape[0] in (1, self.cfg.B)
        self._keep.append(m)
        self.cfg.mask_b = m.shape[0]
        self.bufs.input_mask = m.data_ptr()

    def set_style_masks(self, masks: Sequence[torch.Tensor]):
        """Row G': one fp32 mask [style_mask_b, h_l, w_l] per style tap (see mask_pyramid)."""
        assert self.cfg.style_mask_b > 0 and len(masks) == self.cfg.n_style
        for t, m in enumerate(masks):
            m = m.detach().to(self.device, torch.float32).contiguous()
            assert m.shape[0] == self.cfg.style_mask_b
            self._keep.append(m)
            self.bufs.style_mask[t] = m.data_ptr()
        with torch.cuda.device(self.device):
            _lib.call("isx_nst_prepare_style_masks", ctypes.byref(self.cfg), ctypes.byref(self.bufs), _lib.stream_ptr())

    def set_content_targets(self, feats: Sequence[torch.Tensor]):
        for t, f in enumerate(feats):
            f = f.contiguous()
            self._keep.append(f)
            self.bufs.content_target[t] = f.data_ptr()
        if feats:
            self.cfg.content_target_b = feats[0].shape[0]

    def set_gram_targets(self, grams: Sequence[torch.Tensor]):
        for t, g in enumerate(grams):
            g = g.to(torch.float32).contiguous()
            self._keep.append(g)
            self.bufs.gram_target[t] = g.data_ptr()
        if grams:
            self.cfg.style_target_b = grams[0].shape[0] if grams[0].dim() == 3 else 1

    def set_bn_targets(self, means: Sequence[torch.Tensor], stds: Sequence[torch.Tensor]):
        for t, (m, s) in enumerate(zip(means, stds)):
            m, s = m.to(torch.float32).contiguous(), s.to(torch.float32).contiguous()
            self._keep += [m, s]
            self.bufs.bn_target_mean[t] = m.data_ptr()
            self.bufs.bn_target_std[t] = s.data_ptr()
        if means:
            self.cfg.style_target_b = means[0].shape[0] if means[0].dim() == 2 else 1

    # ---- compute -------------------------------------------------------------------------
    def forward(self, x: torch.Tensor, with_last_pool: bool = False, lean: bool = False):
        """lean (ISX_FWD_LEAN): pre-pool ReLU outputs that are not taps are not written to memory -- only their pooled maps and
        the routing bytes of the pool's backward; feature_view(0, i) of such a conv is undefined afterwards."""
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
        assert tuple(x.shape) == (self.cfg.B, self.cfg.xc, self.cfg.H, self.cfg.W), (tuple(x.shape), self.cfg.B)
        flags = (FWD_LAST_POOL if with_last_pool else 0) | (FWD_LEAN if lean else 0)
        _lib.call("isx_nst_forward", ctypes.byref(self.cfg), ctypes.byref(self.bufs), x, flags, _lib.stream_ptr())

    def feature(self, kind: int, idx: int) -> torch.Tensor:
        """bf16 NHWC COPY of a stored activation: kind 0 = conv idx's ReLU output, 1 = pool idx."""
        return self.feature_view(kind, idx).clone()

    def style_features(self, out: torch.Tensor, stats: bool = True, gram: bool = True):
        """Rows of style features of the batch of the last forward(), written in place into `out` [B, >= D] fp32
        (isx_nst_style_features): mean | unbiased std per style tap, then the Gram upper triangles."""
        assert out.is_cuda and out.dtype == torch.float32 and out.stride(1) == 1 and out.shape[0] == self.cfg.B
        _lib.call("isx_nst_style_features", ctypes.byref(self.cfg), ctypes.byref(self.bufs), int(stats), int(gram), out,
                  _lib.i64(out.stride(0)), _lib.stream_ptr())

    def tap_view(self, tap: int) -> torch.Tensor:
        """bf16 NHWC view of tap id `tap` (conv ReLU output 0..15 or pool output 16..20)."""
        return self.feature_view(1, tap - TAP_POOL0) if tap >= TAP_POOL0 else self.feature_view(0, tap)

    def tap(self, tap: int) -> torch.Tensor:
        return self.tap_view(tap).clone()

    def feature_view(self, kind: int, idx: int) -> torch.Tensor:
        """bf16 NHWC VIEW into the workspace (valid until the next forward / eval on this engine)."""
        ptr = ctypes.c_void_p()
        h, w, c = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        _lib.call("isx_nst_feature", ctypes.byref(self.cfg), ctypes.byref(self.bufs), kind, idx, ctypes.byref(ptr),
                  ctypes.byref(h), ctypes.byref(w), ctypes.byref(c))
        off = ptr.value - self.workspace.data_ptr()
        n = self.cfg.B * h.value * w.value * c.value
        return self.workspace[off:off + 2 * n].view(torch.bfloat16).view(self.cfg.B, h.value, w.value, c.value)

    def backward(self, feat_grads: Dict[int, torch.Tensor], last_pool_grad: Optional[torch.Tensor], grad: torch.Tensor):
        """isx_nst_backward: feat_grads {tap id: bf16 NHWC gradient w.r.t. that tap}; uses the activations of
        the forward() that ran last on this engine."""
        arr = (ctypes.c_void_p * N_TAPS)()
        keep = []
        for j, g in feat_grads.items():
            g = g.contiguous()
            keep.append(g)
            arr[j] = g.data_ptr()
        lp = last_pool_grad.contiguous() if last_pool_grad is not None else None
        _lib.call("isx_nst_backward", ctypes.byref(self.cfg), ctypes.byref(self.bufs), arr, lp, grad, _lib.stream_ptr())

    def eval(self, x: torch.Tensor, grad: torch.Tensor):
        if self.ranges is not None:
            self.ranges.style_target_b = self.cfg.style_target_b   # the batch of the targets set last
            _lib.call("isx_nst_eval_ranges", ctypes.byref(self.cfg), ctypes.byref(self.bufs), ctypes.byref(self.ranges),
                      x, self.loss_c, self.loss_s, grad, _lib.stream_ptr())
            return
        if self.problems is not None:
            self.problems.style_target_b = self.cfg.style_target_b   # the batch of the targets set last
            _lib.call("isx_nst_eval_problems", ctypes.byref(self.cfg), ctypes.byref(self.bufs), ctypes.byref(self.problems),
                      x, self.loss_c, self.loss_s, grad, _lib.stream_ptr())
            return
        _lib.call("isx_nst_eval", ctypes.byref(self.cfg), ctypes.byref(self.bufs), x, self.loss_c, self.loss_s, grad,
                  _lib.stream_ptr())


def mask_pyramid(mask: torch.Tensor, levels: Sequence[int]) -> List[torch.Tensor]:
    """SURVEY.md note N5: m_1 = iris mask at frame resolution, m_{l+1} = 2x2 stride-2 average pool of m_l.
    mask: [Bm,1,H,W] or [Bm,H,W] (bool / float) on the device; returns fp32 [Bm,h,w] per requested level."""
    m = mask.detach().to(torch.float32)
    if m.dim() == 4:
        m = m[:, 0]
    m = m.contiguous()
    out, cur, lvl = {}, m, 0
    for want in sorted(set(levels)):
        while lvl < want:
            Bm, H, W = cur.shape
            nxt = torch.empty(Bm, H // 2, W // 2, device=cur.device, dtype=torch.float32)
            _lib.call("isx_avgpool2x2_f32", cur, nxt, Bm, H, W, _lib.stream_ptr())
            cur, lvl = nxt, lvl + 1
        out[want] = cur
    return [out[l] for l in levels]


def masked_gram_of(feat_nhwc: torch.Tensor, m: torch.Tensor, inv_n: Optional[float] = None) -> torch.Tensor:
    """Row G': utils.GramMatrix(F * m) with m fp32 [Bm,h,w] (Bm in {1,B}) via isx_gram_masked_fwd -- the weights are
    applied to the operand tiles inside the Gram kernel, all-zero K blocks are skipped."""
    B, H, W, C = feat_nhwc.shape
    HW = H * W
    if inv_n is None:
        inv_n = 1.0 / (C * HW)
    dev = feat_nhwc.device
    m = m.to(dev, torch.float32).contiguous()
    ws = torch.empty(max(256, _lib.call_i64("isx_gram_workspace_bytes", B, HW, C)), device=dev, dtype=torch.uint8)
    fl = torch.empty(max(256, _lib.call_i64("isx_gram_mask_flags_bytes", m.shape[0], HW, C)), device=dev, dtype=torch.uint8)
    fm2 = torch.empty_like(feat_nhwc)
    G = torch.empty(B, C, C, device=dev, dtype=torch.float32)
    _lib.call("isx_gram_masked_fwd", feat_nhwc, B, HW, C, m, m.shape[0], fl, fm2, _lib.f32(inv_n), ws, G, None, 1,
              _lib.f64(0.0), None, _lib.f32(0.0), None, _lib.stream_ptr())
    return G


def masked_features(feat_nhwc: torch.Tensor, m: torch.Tensor) -> torch.Tensor:
    B, H, W, C = feat_nhwc.shape
    fm = torch.empty_like(feat_nhwc)
    _lib.call("isx_mask_features", feat_nhwc, m.contiguous(), m.shape[0], fm, None, B, _lib.i64(H * W), C,
              _lib.stream_ptr())
    return fm


CONV_LEVEL = [0, 0, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4]  # number of 2x2 pools before each conv
CONV_LEVEL += [1, 2, 3, 4, 5]                                   # ... and before the output of pool 0..4 (tap ids 16..20)


def tap_conv(tap: int) -> int:
    """The conv that must have run for tap id `tap` to exist."""
    return CONV_BEFORE_POOL[tap - TAP_POOL0] if tap >= TAP_POOL0 else tap


def tap_channels(tap: int) -> int:
    return CONV_COUT[tap_conv(tap)]


def gram_of(feat_nhwc: torch.Tensor, inv_n: Optional[float] = None) -> torch.Tensor:
    """utils.GramMatrix on a bf16 NHWC feature map via isx_gram_fwd -> fp32 [B,C,C]."""
    B, H, W, C = feat_nhwc.shape
    HW = H * W
    if inv_n is None:
        inv_n = 1.0 / (C * HW)
    ws = torch.empty(max(256, _lib.call_i64("isx_gram_workspace_bytes", B, HW, C)), device=feat_nhwc.device,
                     dtype=torch.uint8)
    G = torch.empty(B, C, C, device=feat_nhwc.device, dtype=torch.float32)
    _lib.call("isx_gram_fwd", feat_nhwc, B, HW, C, _lib.f32(inv_n), ws, G, None, 1, _lib.f64(0.0), None,
              _lib.f32(0.0), None, _lib.stream_ptr())
    return G


def masked_stats_of(feat_nhwc: torch.Tensor, m: torch.Tensor):
    """mean / unbiased std over (H,W) of F * m (m fp32 [Bm,h,w], Bm in {1,B}) via isx_bn_stats_masked_fwd."""
    B, H, W, C = feat_nhwc.shape
    dev = feat_nhwc.device
    m = m.to(dev, torch.float32).contiguous()
    sums = torch.empty(B, C, 2, device=dev, dtype=torch.float64)
    mean = torch.empty(B, C, device=dev, dtype=torch.float32)
    std = torch.empty(B, C, device=dev, dtype=torch.float32)
    _lib.call("isx_bn_stats_masked_fwd", feat_nhwc, m, m.shape[0], B, _lib.i64(H * W), C, sums, mean, std, _lib.stream_ptr())
    return mean, std


def stats_of(feat_nhwc: torch.Tensor):
    """Per-(image, channel) mean and unbiased std over (H,W) via isx_bn_stats_fwd -> fp32 [B,C] each."""
    B, H, W, C = feat_nhwc.shape
    sums = torch.empty(B, C, 2, device=feat_nhwc.device, dtype=torch.float64)
    mean = torch.empty(B, C, device=feat_nhwc.device, dtype=torch.float32)
    std = torch.empty(B, C, device=feat_nhwc.device, dtype=torch.float32)
    _lib.call("isx_bn_stats_fwd", feat_nhwc, B, _lib.i64(H * W), C, sums, mean, std, None, None, 1, _lib.f64(0.0),
              _lib.f64(0.0), None, None, None, _lib.stream_ptr())
    return mean, std
