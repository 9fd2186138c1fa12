"""Reference for iris_b200.ResNet50: the torchvision resnet50 trunk (eval mode, no fc) -- the feature extractor of
GazeEstimator2 (models/gaze_estimators/gaze_estimators.py:180-223, models/resnet/resnet.py) -- written out layer by layer
from the torchvision modules, with an EMULATION of the device's storage precision.

`operand_dtype` = torch.float32: BatchNorm folded into each convolution (in float64), everything else fp32 -- the
torchvision forward up to rounding.  torch.bfloat16: what the device kernels store is rounded to bf16 exactly where they
store it -- the input image (the stem's operand), every folded conv weight, every conv output (after bias, residual and
ReLU; the projection shortcut too), the max-pool output (a max of bf16 values) -- with fp32 accumulation and fp32 biases.
The tests use the emulation's own distance from fp32 torchvision as the yardstick of the device's error.

Runs on whatever device `x` is on; TF32 is switched off for the duration, so a CUDA run is a real fp32 computation."""
from __future__ import annotations

import contextlib
from typing import Iterator

import torch
import torch.nn.functional as F


@contextlib.contextmanager
def _no_tf32() -> Iterator[None]:
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


@torch.no_grad()
def torchvision_features(model: torch.nn.Module, x: torch.Tensor) -> torch.Tensor:
    """The unmodified torchvision trunk in eval mode: conv1 .. avgpool -> flatten, fp32 [B, 2048] (xc = 1 is repeated)."""
    model = model.eval().to(x.device)
    if x.shape[1] == 1:
        x = x.repeat(1, 3, 1, 1)
    with _no_tf32():
        h = model.maxpool(model.relu(model.bn1(model.conv1(x.float()))))
        h = model.layer4(model.layer3(model.layer2(model.layer1(h))))
        return torch.flatten(model.avgpool(h), 1)


def fold(conv: torch.nn.Conv2d, bn: torch.nn.BatchNorm2d):
    """Eval-mode Conv2d (no bias) + BatchNorm2d -> one (weight, bias), folded in float64, returned as fp32."""
    scale = bn.weight.double() / torch.sqrt(bn.running_var.double() + bn.eps)
    w = conv.weight.double() * scale[:, None, None, None]
    b = bn.bias.double() - bn.running_mean.double() * scale
    return w.float(), b.float()


@torch.no_grad()
def resnet50_forward(model: torch.nn.Module, x: torch.Tensor, operand_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """The folded trunk with the storage precision of the device kernels emulated (see the module docstring)."""
    model = model.eval().to(x.device)
    if x.shape[1] == 1:
        x = x.repeat(1, 3, 1, 1)

    def rnd(t):
        return t.to(operand_dtype).float()

    def conv(h, c, bn, relu=True, residual=None):
        w, b = fold(c, bn)
        y = F.conv2d(h, rnd(w), b, stride=c.stride, padding=c.padding)
        if residual is not None:
            y = y + residual
        return rnd(F.relu(y) if relu else y)

    with _no_tf32():
        h = conv(rnd(x.float()), model.conv1, model.bn1)
        h = F.max_pool2d(h, 3, 2, 1)
        for layer in (model.layer1, model.layer2, model.layer3, model.layer4):
            for blk in layer:
                t = conv(h, blk.conv1, blk.bn1)
                t = conv(t, blk.conv2, blk.bn2)
                sc = h if blk.downsample is None else conv(h, blk.downsample[0], blk.downsample[1], relu=False)
                h = conv(t, blk.conv3, blk.bn3, residual=sc)
        return h.mean(dim=(2, 3))
