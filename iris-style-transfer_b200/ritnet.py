"""Drop-in for models/ritnet/ritnet.py: `RITnet(...)(x)` -> int64 (or uint8) label map (2 = iris), entirely on the device.

The reference pushes every frame through the CPU (uint8 conversion, cv2.LUT, cv2 CLAHE, ritnet.py:88-98) and runs the
DenseNet2D one image at a time (…2019.py:155, data_preprocessing.py:165).  Here RITnet_transform is three byte kernels
(bit-exact with the OpenCV round trip) and the network is hand-written fp32 CUDA (csrc/ritnet.cu), batched."""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch

from . import _lib

_DOWN = ("conv1", "conv21", "conv22", "conv31", "conv32")
_UP = ("conv11", "conv12", "conv21", "conv22")


def pack_ritnet_params(sd: Dict[str, torch.Tensor]) -> torch.Tensor:
    """DenseNet2D state dict (ritnet.py:165-207) -> the flat fp32 blob isx_ritnet_forward reads (include/isx.h)."""
    out = []

    def conv(name):
        w = sd[name + ".weight"].detach().to(torch.float32).cpu()          # [32, Cin, kh, kw]
        out.append(w.permute(2, 3, 1, 0).contiguous().reshape(-1))         # [kh*kw][Cin][32]
        out.append(sd[name + ".bias"].detach().to(torch.float32).cpu().reshape(-1))

    for k in range(1, 6):
        for c in _DOWN:
            conv("down_block%d.%s" % (k, c))
        p = "down_block%d.bn." % k
        mean, var = sd[p + "running_mean"].double().cpu(), sd[p + "running_var"].double().cpu()
        scale = sd[p + "weight"].double().cpu() / torch.sqrt(var + 1e-5)   # BatchNorm2d in eval mode (ritnet.py:135), eps default
        shift = sd[p + "bias"].double().cpu() - mean * scale
        out += [scale.float(), shift.float()]
    for k in range(1, 5):
        for c in _UP:
            conv("up_block%d.%s" % (k, c))
    out.append(sd["out_conv1.weight"].detach().to(torch.float32).cpu().reshape(4, 32).reshape(-1))
    out.append(sd["out_conv1.bias"].detach().to(torch.float32).cpu().reshape(-1))
    blob = torch.cat(out).contiguous()
    want = _lib.call_i64("isx_ritnet_param_floats")
    if blob.numel() != want:
        raise ValueError("RITnet state dict packs to %d floats, libisx expects %d" % (blob.numel(), want))
    return blob


def gamma_table_u8() -> np.ndarray:
    """ritnet.py:72 `255.0 * (np.linspace(0, 1, 256)**0.8)`, looked up by cv2.LUT and truncated by np.uint8 (ritnet.py:93-94)."""
    return np.uint8(255.0 * (np.linspace(0, 1, 256) ** 0.8))


def normalize_table_f32() -> np.ndarray:
    """What ToImage -> ToDtype(float32, scale=True) -> Normalize([0.5],[0.5]) (ritnet.py:73-77) makes of each uint8 value,
    computed with torchvision itself (plumbing: 256 values, once)."""
    import torchvision.transforms.v2 as transforms

    t = transforms.Compose([transforms.ToImage(), transforms.ToDtype(torch.float32, scale=True),
                            transforms.Normalize([0.5], [0.5])])
    return t(np.arange(256, dtype=np.uint8).reshape(16, 16)).reshape(-1).numpy().copy()


_LABEL_DTYPES = {torch.int64: 0, torch.uint8: 1}


class RITnet(torch.nn.Module):
    """models/ritnet/ritnet.py:8-58.  Same constructor arguments; `state_dict=` (a DenseNet2D state dict) replaces the
    pickle on disk.  forward(x): x (1,h,w) / (h,w) like the reference, or a batch (B,1,h,w) -> labels (B,h,w) of
    `label_dtype` on x's device.  `label_dtype=torch.uint8` gives the same values at 1 B per pixel, which the mask / bbox,
    IoU and landmark kernels read without widening; the default is the reference's int64.  Inference only (the reference
    freezes the model, ritnet.py:31-34); dropout is the identity."""

    def __init__(self, dropout: bool = True, prob: float = 0.2, load_pretrained: bool = True,
                 pretrained_path: str = 'models/weights/ritnet_pretrained.pkl',
                 state_dict: Optional[Dict[str, torch.Tensor]] = None, label_dtype: torch.dtype = torch.int64) -> None:
        super().__init__()
        if label_dtype not in _LABEL_DTYPES:
            raise ValueError("RITnet: label_dtype must be torch.int64 or torch.uint8, got %s" % (label_dtype,))
        self.label_dtype = label_dtype
        if state_dict is None:
            if not load_pretrained:
                raise ValueError("iris_b200.RITnet is an inference engine: pass `state_dict` or keep load_pretrained=True")
            state_dict = torch.load(pretrained_path, weights_only=True, map_location='cpu')   # ritnet.py:29
        self._blob_host = pack_ritnet_params(state_dict)
        self._gamma_host = torch.from_numpy(gamma_table_u8().copy())
        self._norm_host = torch.from_numpy(normalize_table_f32())
        self._dev: Dict[str, tuple] = {}
        self._device = torch.device("cuda:0")

    def to(self, device=None, *args, **kwargs):   # the drivers call ritnet.to(device) (…2019.py:233)
        if device is not None:
            self._device = torch.device(device)
        return self

    def _tables(self, dev):
        key = str(dev)
        if key not in self._dev:
            self._dev[key] = (self._blob_host.to(dev), self._gamma_host.to(dev), self._norm_host.to(dev))
        return self._dev[key]

    @torch.no_grad()
    def transform(self, x: torch.Tensor) -> torch.Tensor:
        """RITnet_transform (ritnet.py:79-98) for a batch [B,1,h,w] (any size >= 8) on the device: the network's input."""
        if x.dim() == 3:
            x = x[None]
        dev = x.device if x.is_cuda else self._device
        x = x.detach().to(dev, torch.float32).contiguous()
        B, _, H, W = x.shape
        _, gamma, norm = self._tables(dev)
        with torch.cuda.device(dev):
            ws = torch.empty(_lib.call_i64("isx_ritnet_transform_workspace_bytes", B, H, W), device=dev, dtype=torch.uint8)
            out = torch.empty_like(x)
            _lib.call("isx_ritnet_transform", x, gamma, norm, ws, out, B, H, W, _lib.stream_ptr())
        return out

    @torch.no_grad()
    def forward(self, x: torch.Tensor, return_logits: bool = False):
        if x.dim() == 2:
            x = x[None]
        if x.dim() == 3:
            x = x[None]                                   # (1,h,w) image -> batch of one (ritnet.py:86-87)
        dev = x.device if x.is_cuda else self._device
        if dev.type != "cuda":
            raise _lib.IsxError("iris_b200.RITnet runs on a CUDA B200 only; there is no CPU path")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        x = x.detach().to(dev, torch.float32).contiguous()
        B, C, H, W = x.shape
        if C != 1:
            raise ValueError("RITnet expects one-channel eye frames, got %d channels" % C)
        nbytes = _lib.call_i64("isx_ritnet_workspace_bytes", B, H, W)
        if nbytes < 0:
            raise ValueError("RITnet: frame %dx%d must be a multiple of 16 in both dimensions" % (H, W))
        blob, gamma, norm = self._tables(dev)
        with torch.cuda.device(dev):
            ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            labels = torch.empty(B, H, W, device=dev, dtype=self.label_dtype)
            logits = torch.empty(B, 4, H, W, device=dev, dtype=torch.float32) if return_logits else None
            _lib.call("isx_ritnet_forward_typed", x, blob, gamma, norm, ws, labels, _LABEL_DTYPES[self.label_dtype], logits,
                      B, H, W, _lib.stream_ptr())
        return (labels, logits) if return_logits else labels
