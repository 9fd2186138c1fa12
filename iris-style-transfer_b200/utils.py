"""Drop-ins for the hot-path symbols of the reference's utils.py: GramMatrix (242-257),
ContentLoss_L2 (259-290), StyleLoss_Gram (292-322), StyleLoss_BN (324-355), crop_image (44-72).
Inputs are fp32 NCHW CUDA tensors as in the reference; arithmetic runs in libisx."""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch

from . import _lib
from .engine import gram_of, stats_of


def _to_nhwc_bf16(x: torch.Tensor) -> torch.Tensor:
    if not x.is_cuda:
        raise _lib.IsxError("iris_b200 needs CUDA tensors (B200); there is no CPU path")
    if x.dim() == 3:
        x = x[None]
    return x.detach().permute(0, 2, 3, 1).to(torch.bfloat16).contiguous()


class _GramFunction(torch.autograd.Function):
    """G = F F^T / n on tcgen05 (isx_gram_fwd); backward dF = (dG + dG^T) F / n through the 1x1 tcgen05 path (isx_gram_bwd)."""

    @staticmethod
    def forward(ctx, x):
        unbatched = x.dim() == 3
        f = _to_nhwc_bf16(x)
        B, H, W, C = f.shape
        inv_n = 1.0 / (H * W) if unbatched else 1.0 / (C * H * W)
        G = gram_of(f, inv_n)
        ctx.save_for_backward(f)
        ctx.inv_n, ctx.unbatched = inv_n, unbatched
        return G[0] if unbatched else G

    @staticmethod
    def backward(ctx, dG):
        (f,) = ctx.saved_tensors
        B, H, W, C = f.shape
        if ctx.unbatched:
            dG = dG[None]
        D = ((dG + dG.transpose(-2, -1)) * ctx.inv_n).to(torch.bfloat16).contiguous()
        dF = torch.empty_like(f)
        with torch.cuda.device(f.device):
            _lib.call("isx_gram_bwd", f, D, dF, B, H, W, C, None, _lib.stream_ptr())
        g = dF.permute(0, 3, 1, 2).float()
        return g[0] if ctx.unbatched else g


def GramMatrix(x: torch.Tensor) -> torch.Tensor:
    """utils.py:242-257: flatten (H,W), x @ x^T / n with n = x[0].numel() after the flatten, i.e.
    C*H*W for a batched (B,C,H,W) input and H*W for an unbatched (C,H,W) one (SURVEY note N3).
    Differentiable (custom autograd Function) when x requires grad."""
    if torch.is_grad_enabled() and x.requires_grad:
        return _GramFunction.apply(x)
    unbatched = x.dim() == 3
    f = _to_nhwc_bf16(x)
    B, H, W, C = f.shape
    inv_n = 1.0 / (H * W) if unbatched else 1.0 / (C * H * W)
    G = gram_of(f, inv_n)
    return G[0] if unbatched else G


class _MseFunction(torch.autograd.Function):
    """F.mse_loss(p, t) (mean over ALL elements, utils.py:288) with its gradient from ONE kernel pass (isx_mse_fwd_bwd)."""

    @staticmethod
    def forward(ctx, p, t):
        unb = p.dim() == 3
        pn, tn = _to_nhwc_bf16(p), _to_nhwc_bf16(t)
        B = pn.shape[0]
        per_image = pn[0].numel()
        n = float(per_image * B)
        loss = torch.zeros(B, device=p.device, dtype=torch.float64)
        grad = torch.empty_like(pn)
        with torch.cuda.device(p.device):
            _lib.call("isx_mse_fwd_bwd", pn, tn, tn.shape[0], grad, B, _lib.i64(per_image), _lib.f64(1.0 / n),
                      _lib.f32(2.0 / n), 0, loss, _lib.stream_ptr())
        ctx.save_for_backward(grad)
        ctx.unb = unb
        return loss.sum().float()

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        d = grad.permute(0, 3, 1, 2).float() * g
        return (d[0] if ctx.unb else d), None


class _ChannelStatsFunction(torch.autograd.Function):
    """(mean, unbiased std) over (H,W) per (image, channel) -- utils.py:337-338, classifiers.py:71 -- from isx_bn_stats_fwd;
    the backward is affine in the feature map, dF = g_mean/n + g_std (F - mean) / ((n-1) std), one pass of isx_channel_affine."""

    @staticmethod
    def forward(ctx, p):
        unb = p.dim() == 3
        f = _to_nhwc_bf16(p)
        mean, std = stats_of(f)
        ctx.save_for_backward(f, mean, std)
        ctx.unb = unb
        return (mean[0], std[0]) if unb else (mean, std)

    @staticmethod
    def backward(ctx, g_mean, g_std):
        f, mean, std = ctx.saved_tensors
        B, H, W, C = f.shape
        n = float(H * W)
        if ctx.unb:
            g_mean, g_std = g_mean[None], g_std[None]
        bcoef = torch.where(std > 0, g_std.float() / ((n - 1.0) * std), torch.zeros_like(std))
        acoef = (g_mean.float() / n - bcoef * mean).contiguous()
        out = torch.empty_like(f)
        with torch.cuda.device(f.device):
            _lib.call("isx_channel_affine", f, acoef, bcoef.contiguous(), out, B, _lib.i64(H * W), C, 0, _lib.stream_ptr())
        d = out.permute(0, 3, 1, 2).float()
        return d[0] if ctx.unb else d


class ContentLoss_L2(torch.nn.Module):
    """utils.py:259-290; differentiable through _MseFunction (nst() itself uses the fused driver)."""

    def __init__(self, targets: List[torch.Tensor] = None, weights: List[float] = None) -> None:
        super().__init__()
        self.targets = targets
        self.weights = [1.0] * len(targets) if weights is None else weights

    def forward(self, preds: List[torch.Tensor]) -> torch.Tensor:
        if torch.is_grad_enabled() and any(p.requires_grad for p in preds):
            loss = 0  # utils.py:285-290 with the mse and its gradient computed by libisx
            for p, t, w in zip(preds, self.targets, self.weights):
                loss = loss + _MseFunction.apply(p, t) * w
            return loss * 0.5
        with torch.no_grad():
            return self._forward_kernels(preds)

    def _forward_kernels(self, preds: List[torch.Tensor]) -> torch.Tensor:
        total = torch.zeros((), device=preds[0].device, dtype=torch.float64)
        for p, t, w in zip(preds, self.targets, self.weights):
            pn, tn = _to_nhwc_bf16(p), _to_nhwc_bf16(t)
            B = pn.shape[0]
            per_image = pn[0].numel()
            loss = torch.zeros(B, device=p.device, dtype=torch.float64)
            _lib.call("isx_content_mse_fwd_bwd", pn, tn, tn.shape[0], None, B, _lib.i64(per_image),
                      _lib.f64(1.0 / (per_image * B)), _lib.f32(0.0), loss, _lib.stream_ptr())
            total = total + loss.sum() * w
        return (total * 0.5).float()


class StyleLoss_Gram(torch.nn.Module):
    """utils.py:292-322."""

    def __init__(self, targets: List[torch.Tensor] = None, weights: List[float] = None) -> None:
        super().__init__()
        self.targets = [GramMatrix(t) for t in targets]
        self.weights = [1.0] * len(targets) if weights is None else weights

    def forward(self, preds: List[torch.Tensor]) -> torch.Tensor:
        # utils.py:317-322; GramMatrix carries its own backward, the C x C arithmetic is plain torch
        total = torch.zeros((), device=preds[0].device, dtype=torch.float64)
        for p, t, w in zip(preds, self.targets, self.weights):
            total = total + ((GramMatrix(p) - t).double() ** 2).sum() * w
        return (total * 0.25).float()


class StyleLoss_BN(torch.nn.Module):
    """utils.py:324-355 (the reference's default style loss, pipelines.py:11,65-66)."""

    def __init__(self, targets: List[torch.Tensor] = None, weights: List[float] = None) -> None:
        super().__init__()
        stats = [stats_of(_to_nhwc_bf16(t)) for t in targets]
        self.targets_mean = [m if t.dim() == 4 else m[0] for (m, _), t in zip(stats, targets)]
        self.targets_std = [s if t.dim() == 4 else s[0] for (_, s), t in zip(stats, targets)]
        self.weights = [1.0] * len(targets) if weights is None else weights

    def forward(self, preds: List[torch.Tensor]) -> torch.Tensor:
        if torch.is_grad_enabled() and any(p.requires_grad for p in preds):
            loss = 0  # utils.py:350-355; the statistics and their backward run in libisx, the (B,C) arithmetic is plain torch
            for p, tm, ts, w in zip(preds, self.targets_mean, self.targets_std, self.weights):
                pm, ps = _ChannelStatsFunction.apply(p)
                loss = loss + ((pm - tm) ** 2 + (ps - ts) ** 2).sum() * w / pm.shape[-1]
            return loss
        with torch.no_grad():
            return self._forward_kernels(preds)

    def _forward_kernels(self, preds: List[torch.Tensor]) -> torch.Tensor:
        total = torch.zeros((), device=preds[0].device, dtype=torch.float64)
        for p, tm, ts, w in zip(preds, self.targets_mean, self.targets_std, self.weights):
            pm, ps = stats_of(_to_nhwc_bf16(p))
            total = total + ((pm - tm).double() ** 2 + (ps - ts).double() ** 2).sum() * w / pm.shape[-1]
        return total.float()


def style_features(style_feats: Sequence[torch.Tensor]) -> torch.Tensor:
    """Classifier2's reduction (models/classifiers/classifiers.py:71): per layer cat(mean, std_unbiased)
    over (H,W), concatenated -> (B, 2*sum C_l).  Accepts fp32 NCHW or bf16 NHWC (from features_nhwc)."""
    out = []
    for f in style_feats:
        fn = f if f.dtype == torch.bfloat16 else _to_nhwc_bf16(f)
        m, s = stats_of(fn)
        out += [m, s]
    return torch.cat(out, dim=1)


_SEG_DTYPES = {torch.int64: 0, torch.uint8: 1}    # label-map dtypes the mask / bbox and IoU kernels read natively


def _bbox_of(image: torch.Tensor, seg: Optional[torch.Tensor] = None, label: int = 2,
             threshold: Optional[float] = None, want_mask: bool = False, want_masked: bool = False):
    """isx_mask_bbox_typed on a batch [B,1,H,W]: returns (bbox int32 [B,4] on device, mask or None, x*m or None).  int64 and
    uint8 label maps are read as they are; any other dtype is widened to int64 first."""
    if not image.is_cuda:
        raise _lib.IsxError("iris_b200 needs CUDA tensors (B200); there is no CPU path")
    x = image.detach().to(torch.float32).contiguous()
    B, _, H, W = x.shape
    bbox = torch.empty(B, 4, device=x.device, dtype=torch.int32)
    mask = torch.empty(B, 1, H, W, device=x.device, dtype=torch.uint8) if want_mask else None
    xm = torch.empty_like(x) if want_masked else None
    segc = None
    if seg is not None:
        segc = seg.detach().to(x.device, seg.dtype if seg.dtype in _SEG_DTYPES else torch.int64).contiguous()
    with torch.cuda.device(x.device):
        _lib.call("isx_mask_bbox_typed", x, segc, _SEG_DTYPES[segc.dtype] if segc is not None else 0, int(label),
                  int(threshold is not None),
                  _lib.f32(threshold if threshold is not None else 0.0), mask, xm, bbox, B, H, W, _lib.stream_ptr())
    return bbox, mask, xm


def crop_image(image: torch.Tensor, return_idx: bool = False):
    """utils.py:44-72: trim the black border -- bbox of the NONZERO PIXELS, (x_min, y_min, x_max, y_max) =
    (row_min, col_min, row_max, col_max) inclusive; `image` is (h,w) or (1,h,w)."""
    if image.dim() == 2:
        img3 = image[None]
    elif image.dim() == 3 and image.shape[0] == 1:
        img3 = image
    else:
        raise Exception('image shape wrong:', image.shape)  # utils.py:66
    bbox, _, _ = _bbox_of(img3[None])
    x_min, y_min, x_max, y_max = bbox[0].tolist()
    if x_max < 0:
        raise RuntimeError("crop_image: image has no nonzero pixel (the reference fails in min() of an empty tensor)")
    if return_idx:
        return x_min, y_min, x_max, y_max
    return img3[:, x_min: x_max + 1, y_min: y_max + 1]


def cal_IoUs(preds: torch.Tensor, targets: torch.Tensor, num_class: int = 4, eps: float = 1e-6, device="cuda:0"):
    """utils.py:163-194: IoU per image and class and their mean for label maps of shape (b, h, w).  One fused pass over the
    two maps (`isx_seg_iou_typed`: exact counts) instead of the reference's ~30 elementwise passes; returns
    (iou_per_class: list of num_class tensors [b], miou [b]) on the device, bit-identical to the reference.  Two uint8 maps
    are read as they are (2 B per pixel); any other combination, mixed dtypes included, is widened to int64 first, so a
    value >= 256 in an int64 map keeps meaning "no class"."""
    if preds.shape != targets.shape:      # the reference broadcasts (data_preprocessing.py:168 passes (1,h,w) vs (1,h,w))
        preds, targets = torch.broadcast_tensors(preds, targets)
    if preds.dim() != 3:
        raise ValueError("label maps must be (b, h, w), got %s" % (tuple(preds.shape),))
    dev = preds.device if preds.is_cuda else (targets.device if targets.is_cuda else torch.device(device))
    dt = torch.uint8 if preds.dtype == targets.dtype == torch.uint8 else torch.int64
    p = preds.detach().to(dev, dt).contiguous()
    t = targets.detach().to(dev, dt).contiguous()
    B, H, W = p.shape
    with torch.cuda.device(dev):
        counts = torch.empty(B, num_class, 2, device=dev, dtype=torch.int32)
        iou = torch.empty(B, num_class, device=dev, dtype=torch.float32)
        miou = torch.empty(B, device=dev, dtype=torch.float32)
        _lib.call("isx_seg_iou_typed", p, t, _SEG_DTYPES[dt], B, _lib.i64(H * W), int(num_class), _lib.f32(eps), counts, iou, miou, _lib.stream_ptr())
    return [iou[:, c] for c in range(num_class)], miou


def angular_distance(v1: torch.Tensor, v2: torch.Tensor, device="cuda:0"):
    """utils.py:216-240: radian and degree distance between rows of two sets of unit vectors (N, 3)."""
    dev = v1.device if v1.is_cuda else (v2.device if v2.is_cuda else torch.device(device))
    a = v1.detach().to(dev, torch.float32).contiguous()
    b = v2.detach().to(dev, torch.float32).contiguous()
    if a.shape != b.shape or a.dim() != 2:
        raise ValueError("expected two (N, d) tensors, got %s and %s" % (tuple(v1.shape), tuple(v2.shape)))
    n, d = a.shape
    rad = torch.empty(n, device=dev, dtype=torch.float32)
    deg = torch.empty(n, device=dev, dtype=torch.float32)
    if n:
        with torch.cuda.device(dev):
            _lib.call("isx_angular_distance", a, b, n, d, rad, deg, _lib.stream_ptr())
    return rad, deg
