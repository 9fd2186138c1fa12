"""CPU tier of the uint8 label maps: the typed entry points (isx_ritnet_forward_typed, isx_mask_bbox_typed,
isx_seg_iou_typed) are exported and refuse a bad dtype code, a null pointer or a bad shape on the host, before any device
work; RITnet refuses a label dtype other than int64 / uint8."""
import ctypes
import os

import numpy as np
import pytest
import torch

import iris_b200
from iris_b200 import _lib

TYPED = ("isx_ritnet_forward_typed", "isx_mask_bbox_typed", "isx_seg_iou_typed")
D = ctypes.c_void_p(256)                   # never dereferenced: the checks come first


def test_typed_entry_points_are_exported():
    lib = _lib.load()
    names = _lib.declared_symbols()
    for n in TYPED:
        assert n in names and hasattr(lib, n), n


def _ritnet(dt, labels=D, B=1, H=64, W=64):
    _lib.call("isx_ritnet_forward_typed", D, D, D, D, D, labels, dt, None, B, H, W, None)


def _mask_bbox(dt, x=D, bbox=D, B=1, H=8, W=8):
    _lib.call("isx_mask_bbox_typed", x, D, dt, 2, 1, _lib.f32(0.8), D, D, bbox, B, H, W, None)


def _seg_iou(dt, p=D, t=D, B=1, HW=16, nc=4):
    _lib.call("isx_seg_iou_typed", p, t, dt, B, _lib.i64(HW), nc, _lib.f32(1e-6), D, D, D, None)


@pytest.mark.parametrize("fn", [_ritnet, _mask_bbox, _seg_iou])
@pytest.mark.parametrize("dt", [2, 7, -1])
def test_typed_entry_points_reject_unknown_dtype_codes(fn, dt):
    with pytest.raises(_lib.IsxError):
        fn(dt)
    assert b"dtype" in _lib.load().isx_last_error()


@pytest.mark.parametrize("dt", [0, 1])
def test_typed_entry_points_validate_pointers_and_shapes(dt):
    lib = _lib.load()
    bad = [
        lambda: _ritnet(dt, labels=None),
        lambda: _ritnet(dt, H=40),                         # not a multiple of 16
        lambda: _ritnet(dt, B=0),
        lambda: _mask_bbox(dt, x=None),
        lambda: _mask_bbox(dt, bbox=None),
        lambda: _mask_bbox(dt, B=0),
        lambda: _mask_bbox(dt, W=0),
        lambda: _seg_iou(dt, p=None),
        lambda: _seg_iou(dt, t=None),
        lambda: _seg_iou(dt, HW=0),
        lambda: _seg_iou(dt, B=70000),
        lambda: _seg_iou(dt, nc=9),
        lambda: _seg_iou(dt, nc=0),
    ]
    for i, f in enumerate(bad):
        with pytest.raises(_lib.IsxError):
            f()
        assert lib.isx_last_error(), i
    with pytest.raises(_lib.IsxError):
        _seg_iou(dt, nc=9)
    assert b"num_class" in lib.isx_last_error()


def test_ritnet_label_dtype_is_int64_or_uint8(golden_dir):
    gold = np.load(os.path.join(golden_dir, "ritnet.npz"))
    sd = {k[2:]: torch.from_numpy(gold[k]) for k in gold.files if k.startswith("w:")}
    for bad in (torch.float32, torch.int32, torch.int8, torch.bool):
        with pytest.raises(ValueError):
            iris_b200.RITnet(state_dict=sd, label_dtype=bad)
    assert iris_b200.RITnet(state_dict=sd).label_dtype == torch.int64
    assert iris_b200.RITnet(state_dict=sd, label_dtype=torch.uint8).label_dtype == torch.uint8
