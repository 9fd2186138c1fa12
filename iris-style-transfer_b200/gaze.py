"""Drop-ins for models/gaze_estimators/gaze_estimators.py (SURVEY.md §8f row 4, inference): `extract_eye_landmarks` on the
device for whole batches of label maps, and the GazeEstimator1 / GazeEstimator2 heads in eval mode (csrc/landmarks.cu).

The reference extracts the 19 landmarks one frame at a time with a `.cpu().numpy()` round trip and three OpenCV calls per
class (gaze_estimators.py:49,127-137); here a batch is three kernel launches and never leaves the device.  Training the
heads (gaze_estimation.py, Adam) and the EfficientNet segmenter stay with the caller (SURVEY.md §2).
`GazeEstimator2(extract_feature=True)` takes its feature extractor as `resnet=`: `iris_b200.ResNet50` keeps frames ->
features -> head -> unit vectors on the device."""
from __future__ import annotations

from typing import Callable, Dict, Optional

import torch

from . import _lib

_DTYPES = {torch.int64: 0, torch.uint8: 1, torch.int32: 2}
FLAG_NOT_OPENCV = 1     # five-point or rank-deficient contour: cv2.fitEllipse perturbs / switches algorithm there (isx.h)
FLAG_TOO_MANY_POINTS = 2


def extract_eye_landmarks_batch(segs: torch.Tensor, epsilon: float = 1e-6, max_points: int = 16384, return_info: bool = False,
                                device="cuda:0"):
    """Label maps [B,H,W] or [B,1,H,W] (int64 as a segmenter's arg-max emits them, or uint8 / int32) -> landmarks fp32
    [B,19] on the device, in the order of gaze_estimators.py:154-174.  info int32 [B,8]: see isx_eye_landmarks."""
    if segs.dim() == 4 and segs.shape[1] == 1:
        segs = segs[:, 0]
    if segs.dim() != 3:
        raise ValueError("label maps must be [B,H,W] or [B,1,H,W], got %s" % (tuple(segs.shape),))
    if not segs.is_cuda:
        segs = segs.to(device)
    if segs.dtype not in _DTYPES:
        segs = segs.to(torch.int64)
    segs = segs.contiguous()
    B, H, W = segs.shape
    dev = segs.device
    with torch.cuda.device(dev):
        nbytes = _lib.call_i64("isx_eye_landmarks_workspace_bytes", B, H, W, int(max_points))
        if nbytes < 0:
            raise ValueError("bad landmark shape B=%d H=%d W=%d max_points=%d" % (B, H, W, max_points))
        ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        out = torch.empty(B, 19, device=dev, dtype=torch.float32)
        info = torch.empty(B, 8, device=dev, dtype=torch.int32)
        _lib.call("isx_eye_landmarks", segs, _DTYPES[segs.dtype], B, H, W, _lib.f64(epsilon), int(max_points), ws, out, info,
                  _lib.stream_ptr())
    return (out, info) if return_info else out


def extract_eye_landmarks(segmentation: torch.Tensor, epsilon: float = 1e-6) -> torch.Tensor:
    """gaze_estimators.py:108-178: one (400, 640) label map -> the 19 landmark features, on the map's device."""
    assert segmentation.shape == (400, 640)          # gaze_estimators.py:121
    out, info = extract_eye_landmarks_batch(segmentation[None], epsilon, return_info=True)
    if bool((info[0, [2, 5]] & FLAG_TOO_MANY_POINTS).any()):
        raise _lib.IsxError("extract_eye_landmarks: a contour has more than 16384 points; use extract_eye_landmarks_batch(max_points=)")
    return out[0]


class _GazeHead(torch.nn.Module):
    """in_dim -> hidden -> hidden -> out_dim with ReLU (+ Dropout, the identity in eval mode) between, then x / ||x||.
    Parameters are kept in a `model` Sequential with the reference's layout so that its state dicts load unchanged
    (`model.0.*`, `model.3.*`, `model.6.*`)."""

    def __init__(self, in_dim: int, hidden_dim: int, output_dim: int, state_dict: Optional[Dict[str, torch.Tensor]] = None):
        super().__init__()
        self.model = torch.nn.Sequential(
            torch.nn.Linear(in_dim, hidden_dim), torch.nn.ReLU(inplace=True), torch.nn.Dropout(0.5),
            torch.nn.Linear(hidden_dim, hidden_dim), torch.nn.ReLU(inplace=True), torch.nn.Dropout(0.5),
            torch.nn.Linear(hidden_dim, output_dim))
        self.in_dim, self.hidden_dim, self.output_dim = in_dim, hidden_dim, output_dim
        if state_dict is not None:
            self.load_state_dict({k: v for k, v in state_dict.items() if k.startswith("model.")}, strict=True)
        self.eval()

    @torch.no_grad()
    def _head(self, x: torch.Tensor) -> torch.Tensor:
        if self.training:
            raise RuntimeError("the device head is the eval-mode forward (Dropout = identity); training stays with the caller")
        l1, l2, l3 = self.model[0], self.model[3], self.model[6]
        dev = l1.weight.device
        if dev.type != "cuda":
            raise _lib.IsxError("gaze head parameters are on %s: move the module to the B200 (.to('cuda:0')); there is no CPU path" % dev)
        x = x.to(device=dev, dtype=torch.float32)
        if x.dim() != 2 or x.shape[1] != self.in_dim:
            raise ValueError("expected features [B,%d], got %s" % (self.in_dim, tuple(x.shape)))
        if x.stride(1) != 1:
            x = x.contiguous()
        B = x.shape[0]
        out = torch.empty(B, self.output_dim, device=dev, dtype=torch.float32)
        if B == 0:
            return out
        with torch.cuda.device(dev):
            _lib.call("isx_gaze_head_fwd", x, _lib.i64(x.stride(0)), B, self.in_dim, self.hidden_dim, self.output_dim,
                      l1.weight.contiguous(), l1.bias.contiguous(), l2.weight.contiguous(), l2.bias.contiguous(),
                      l3.weight.contiguous(), l3.bias.contiguous(), out, _lib.stream_ptr())
        return out


class GazeEstimator1(_GazeHead):
    """gaze_estimators.py:8-53: the model-based estimator on the 19 eye landmarks."""

    def __init__(self, extract_feature: bool = False, landmark_dim: int = 19, hidden_dim: int = 64, output_dim: int = 3,
                 state_dict: Optional[Dict[str, torch.Tensor]] = None):
        super().__init__(landmark_dim, hidden_dim, output_dim, state_dict)
        self.extract_feature = extract_feature

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: label maps (b,400,640) / (b,1,400,640) when extract_feature, else landmark features (b,19)."""
        if x.dim() == 3:
            x = x.unsqueeze(1)                          # gaze_estimators.py:45-46
        if self.extract_feature:
            assert tuple(x.shape[-2:]) == (400, 640)    # extract_eye_landmarks asserts it per frame (:121)
            x = extract_eye_landmarks_batch(x, device=self.model[0].weight.device)
        return self._head(x)


class GazeEstimator2(_GazeHead):
    """gaze_estimators.py:180-223: the appearance-based estimator on 2048 ResNet50 features.  With extract_feature the
    feature extractor (models/resnet/resnet.py) is passed as `resnet=`, e.g. `iris_b200.ResNet50(weights=<torchvision
    resnet50 module or state dict>)`; it applies no input normalisation, so frames arrive preprocessed."""

    def __init__(self, extract_feature: bool = False, freeze_resnet: bool = True, hidden_dim: int = 64, output_dim: int = 3,
                 state_dict: Optional[Dict[str, torch.Tensor]] = None, resnet: Optional[Callable] = None):
        super().__init__(2048, hidden_dim, output_dim, state_dict)
        self.extract_feature = extract_feature
        if extract_feature and resnet is None:
            raise ValueError("GazeEstimator2(extract_feature=True) needs resnet=<callable image -> [B,2048] features>, e.g. "
                             "iris_b200.ResNet50(weights=<torchvision resnet50 module or state dict>)")
        self._resnet = resnet

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if self.extract_feature:
            x = self._resnet(x)
        return self._head(x)
