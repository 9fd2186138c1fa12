"""ctypes binding of libisx.so (include/isx.h).  PyTorch is used only for device memory and streams;
every compute call goes through the C ABI with raw device pointers.  There is NO fallback: if the
library is missing or a call fails, an exception is raised."""
from __future__ import annotations

import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libisx.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "isx.h")

_lib = None


class IsxError(RuntimeError):
    pass


def declared_symbols(header: str = HEADER_PATH):
    """Every function name declared in include/isx.h (used by the CPU export test)."""
    txt = open(header).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(isx_[a-z0-9_]+)\s*\(", txt)))


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IsxError("libisx.so not built (%s missing): run `python build.py` or __graft_entry__.build(); "
                       "there is no CPU / PyTorch fallback for this path" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.isx_last_error.restype = ctypes.c_char_p
    lib.isx_gram_workspace_bytes.restype = ctypes.c_int64
    for name in ("isx_nst_workspace_bytes", "isx_lbfgs_state_bytes", "isx_lbfgs_workspace_bytes"):
        if hasattr(lib, name):
            getattr(lib, name).restype = ctypes.c_int64
    _lib = lib
    return lib


def _conv(a):
    if a is None:
        return ctypes.c_void_p(0)
    if isinstance(a, bool):
        return ctypes.c_int(int(a))
    if isinstance(a, int):
        return ctypes.c_int64(a) if abs(a) >= 2 ** 31 else ctypes.c_int(a)
    if isinstance(a, float):
        raise TypeError("pass floats explicitly as f32()/f64()")
    if hasattr(a, "data_ptr"):
        return ctypes.c_void_p(a.data_ptr())
    return a


def f32(v):
    return ctypes.c_float(float(v))


def f64(v):
    return ctypes.c_double(float(v))


def i64(v):
    return ctypes.c_int64(int(v))


def stream_ptr():
    import torch

    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def call(name: str, *args):
    """Call an int-returning C-ABI function; tensors -> device pointers; raise on failure."""
    lib = load()
    fn = getattr(lib, name)
    rc = fn(*[_conv(a) for a in args])
    if rc != 0:
        raise IsxError("%s failed (rc=%d): %s" % (name, rc, lib.isx_last_error().decode()))
    return rc


def call_i64(name: str, *args) -> int:
    lib = load()
    fn = getattr(lib, name)
    fn.restype = ctypes.c_int64
    return int(fn(*[_conv(a) for a in args]))


class Handle:
    """isx_create / isx_make_current / isx_destroy: a library context (options, launch counter, profiler, SM count) for
    hosts that drive several devices or threads.  `with Handle(device): ...` binds it to the calling thread."""

    def __init__(self, device: int = 0):
        self.lib = load()
        self.h = ctypes.c_void_p()
        rc = self.lib.isx_create(int(device), ctypes.byref(self.h))
        if rc != 0:
            raise IsxError("isx_create failed (rc=%d): %s" % (rc, self.lib.isx_last_error().decode()))

    def make_current(self):
        self.lib.isx_make_current(self.h)

    def __enter__(self):
        self.make_current()
        return self

    def __exit__(self, *exc):
        self.lib.isx_make_current(ctypes.c_void_p(0))

    def destroy(self):
        if self.h:
            self.lib.isx_destroy(self.h)
            self.h = ctypes.c_void_p(0)
