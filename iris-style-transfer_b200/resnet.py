"""ResNet-50 feature extractor of GazeEstimator2 (models/gaze_estimators/gaze_estimators.py:180-223, models/resnet/resnet.py)
on the device: the torchvision resnet50 trunk in eval mode, conv1 -> bn1 -> relu -> maxpool -> layer1..layer4 -> avgpool ->
flatten, computed by libisx (isx_resnet50_forward: bf16 tcgen05 convolutions with BatchNorm folded in, fp32 accumulation)."""
from __future__ import annotations

import ctypes
from typing import Dict, List, Tuple

import torch

from . import _lib
from .vgg import fold_batchnorm

N_CONVS = 53
STAGES = ((64, 3), (128, 4), (256, 6), (512, 3))   # (planes, blocks) of layer1..layer4; out channels = 4 * planes
FEATURE_DIM = 2048
WORKSPACE_BUDGET = 8 << 30   # bytes of activations per forward call: larger batches run in chunks of this size


def conv_specs() -> List[Tuple[str, str, int, int, int, int]]:
    """The 53 convolutions in torchvision module order (isx_resnet50_weights order):
    (conv parameter prefix, BatchNorm prefix, Cin, Cout, kernel size, stride)."""
    specs = [("conv1", "bn1", 3, 64, 7, 2)]
    cin = 64
    for li, (planes, blocks) in enumerate(STAGES):
        for blk in range(blocks):
            stride = 2 if (li > 0 and blk == 0) else 1
            p = "layer%d.%d." % (li + 1, blk)
            specs += [(p + "conv1", p + "bn1", cin, planes, 1, 1), (p + "conv2", p + "bn2", planes, planes, 3, stride),
                      (p + "conv3", p + "bn3", planes, planes * 4, 1, 1)]
            if blk == 0:
                specs.append((p + "downsample.0", p + "downsample.1", cin, planes * 4, 1, stride))
            cin = planes * 4
    assert len(specs) == N_CONVS
    return specs


def plan_shapes(H: int, W: int) -> Dict[str, Tuple[int, int, int]]:
    """(C, h, w) after each stage for an H x W input, as torchvision computes them (every stride-2 layer rounds up)."""
    up = lambda n: (n + 1) // 2  # noqa: E731
    h, w = up(H), up(W)
    out = {"conv1": (64, h, w)}
    h, w = up(h), up(w)
    out["maxpool"] = (64, h, w)
    for li, (planes, _) in enumerate(STAGES):
        if li > 0:
            h, w = up(h), up(w)
        out["layer%d" % (li + 1)] = (planes * 4, h, w)
    return out


def expected_keys() -> List[str]:
    """State-dict keys of a torchvision resnet50 trunk (no fc)."""
    keys = []
    for conv, bn, *_ in conv_specs():
        keys.append(conv + ".weight")
        keys += [bn + "." + k for k in ("weight", "bias", "running_mean", "running_var", "num_batches_tracked")]
    return keys


def fold_state_dict(state_dict: Dict[str, torch.Tensor]) -> List[Tuple[torch.Tensor, torch.Tensor]]:
    """The 53 folded fp32 (weight, bias) pairs of a torchvision resnet50 state dict.  Keys are checked strictly: `fc.*` is
    ignored, any other missing or unexpected key raises."""
    want = set(expected_keys())
    have = {k for k in state_dict if not k.startswith("fc.")}
    missing, unexpected = sorted(want - have), sorted(have - want)
    if missing or unexpected:
        raise KeyError("not a torchvision resnet50 state dict: missing %s, unexpected %s" % (missing[:8], unexpected[:8]))
    out = []
    for conv, bn, cin, cout, k, _ in conv_specs():
        w = state_dict[conv + ".weight"].detach().cpu()
        if tuple(w.shape) != (cout, cin, k, k):
            raise ValueError("%s.weight has shape %s, expected %s" % (conv, tuple(w.shape), (cout, cin, k, k)))
        g = lambda n: state_dict[bn + "." + n].detach().cpu()  # noqa: E731
        out.append(fold_batchnorm(w, torch.zeros(cout, dtype=torch.float64), g("weight"), g("bias"), g("running_mean"),
                                  g("running_var")))
    return out


def random_resnet50(seed: int = 0) -> torch.nn.Module:
    """torchvision resnet50(weights=None) under torch.manual_seed(seed), in eval mode."""
    import torchvision.models as tvm

    torch.manual_seed(seed)
    return tvm.resnet50(weights=None).eval()


class ResNet50Weights(ctypes.Structure):
    """ctypes mirror of isx_resnet50_weights (include/isx.h)."""
    _fields_ = [("w", ctypes.c_void_p * N_CONVS), ("bias", ctypes.c_void_p * N_CONVS)]


class PackedResNet50:
    """The folded weights packed once for one device (isx_pack_resnet_stem_weights / isx_pack_conv1x1_weights /
    isx_pack_conv3x3_weights) and the weights struct pointing at them."""

    def __init__(self, folded: List[Tuple[torch.Tensor, torch.Tensor]], device: torch.device):
        self.device = torch.device(device)
        _lib.call("isx_device_check", self.device.index or 0)
        self.w: List[torch.Tensor] = []
        self.bias: List[torch.Tensor] = []
        self.struct = ResNet50Weights()
        with torch.cuda.device(self.device):
            s = _lib.stream_ptr()
            for i, ((w, b), (_, _, cin, cout, k, _)) in enumerate(zip(folded, conv_specs())):
                w32 = w.to(self.device, torch.float32).contiguous()
                if k == 7:
                    wp = torch.empty(64, 192, device=self.device, dtype=torch.bfloat16)
                    _lib.call("isx_pack_resnet_stem_weights", w32, wp, s)
                elif k == 3:
                    wp = torch.empty(9, cout, cin, device=self.device, dtype=torch.bfloat16)
                    _lib.call("isx_pack_conv3x3_weights", w32, cout, cin, wp, None, s)
                else:
                    wp = torch.empty(cout, cin, device=self.device, dtype=torch.bfloat16)
                    _lib.call("isx_pack_conv1x1_weights", w32, cout, cin, wp, s)
                self.w.append(wp)
                self.bias.append(b.to(self.device, torch.float32).contiguous())
                self.struct.w[i] = wp.data_ptr()
                self.struct.bias[i] = self.bias[-1].data_ptr()
            torch.cuda.current_stream().synchronize()


class ResNet50(torch.nn.Module):
    """torchvision resnet50 trunk (eval mode, no fc) on the B200: x fp32 [B, xc, H, W] -> features fp32 [B, 2048].

    `weights`: 'random' (torchvision resnet50(weights=None) under torch.manual_seed(seed)), a torchvision resnet50 module, or
    its state dict (fc.* is ignored; any other missing or unexpected key raises).  The library never downloads anything:
    a caller with ImageNet weights passes the module or its state dict.

    The module does NO input normalisation -- preprocessing (e.g. the ImageNet mean / std) stays with the caller.  xc = 1
    broadcasts to three channels (forward(x) == forward(x.repeat(1, 3, 1, 1))); H and W >= 32, any parity.  Inference only:
    forward raises in .train() mode.  Batches larger than the workspace budget run in chunks; every image's features are
    independent of the batch it is in (bit for bit)."""

    def __init__(self, weights="random", seed: int = 0) -> None:
        super().__init__()
        if isinstance(weights, str):
            if weights != "random":
                raise ValueError("weights must be 'random', a torchvision resnet50 module or its state dict (no downloads: "
                                 "pass ImageNet weights as a module or state dict)")
            weights = random_resnet50(seed)
        if isinstance(weights, torch.nn.Module):
            weights = weights.state_dict()
        if not isinstance(weights, dict):
            raise TypeError("weights must be 'random', a torchvision resnet50 module or its state dict")
        self.host_weights = fold_state_dict(weights)
        self._packed: Dict[str, PackedResNet50] = {}
        self._workspace: Dict[str, torch.Tensor] = {}
        self._device = torch.device("cuda:0")
        self.eval()

    def to(self, device=None, *args, **kwargs):  # noqa: D401  (like VGG19.to: chooses the device of the packed weights)
        if device is not None:
            self._device = torch.device(device)
        return self

    def packed(self, device=None) -> PackedResNet50:
        dev = torch.device(device if device is not None else self._device)
        if dev.type != "cuda":
            raise _lib.IsxError("iris_b200.ResNet50 runs on CUDA (B200) only; got device %s" % dev)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        key = str(dev)
        if key not in self._packed:
            self._packed[key] = PackedResNet50(self.host_weights, dev)
        return self._packed[key]

    def chunk_size(self, B: int, H: int, W: int) -> int:
        """Images per isx_resnet50_forward call: the largest count whose workspace fits WORKSPACE_BUDGET (at least 1)."""
        per_image = _lib.call_i64("isx_resnet50_workspace_bytes", 1, H, W)
        if per_image < 0:
            raise ValueError(_lib.load().isx_last_error().decode())
        return max(1, min(B, WORKSPACE_BUDGET // per_image))

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if self.training:
            raise RuntimeError("iris_b200.ResNet50 is the eval-mode forward (folded BatchNorm); training stays with the caller")
        if x.dim() != 4:
            raise ValueError("expected images [B, xc, H, W], got %s" % (tuple(x.shape),))
        B, xc, H, W = x.shape
        if xc not in (1, 3):
            raise ValueError("images must have 1 or 3 channels, got %d" % xc)
        if H < 32 or W < 32:
            raise ValueError("images must be at least 32 x 32, got %d x %d" % (H, W))
        dev = x.device if x.is_cuda else self._device
        pk = self.packed(dev)
        dev = pk.device
        x = x.detach().to(dev, torch.float32).contiguous()
        out = torch.empty(B, FEATURE_DIM, device=dev, dtype=torch.float32)
        if B == 0:
            return out
        with torch.cuda.device(dev):
            n = self.chunk_size(B, H, W)
            nbytes = _lib.call_i64("isx_resnet50_workspace_bytes", n, H, W)
            ws = self._workspace.get(str(dev))
            if ws is None or ws.numel() < nbytes:
                self._workspace[str(dev)] = ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            for s in range(0, B, n):
                m = min(n, B - s)
                _lib.call("isx_resnet50_forward", ctypes.byref(pk.struct), x[s:s + m], xc, m, H, W, ws, out[s:s + m],
                          _lib.stream_ptr())
        return out
