"""CPU tier of several coupled problems in one NST job (nst(problem_size=g), isx_nst_eval_problems,
isx_lbfgs_tick_problems): the isx_nst_problems mirror matches the header, both entry points are exported and refuse bad
arguments on the host before any device work, and nst() / stylize_frames() refuse inconsistent layouts with ValueError."""
import ctypes
import re

import pytest
import torch

import iris_b200
from iris_b200 import _lib, engine

NEW = ("isx_nst_eval_problems", "isx_lbfgs_tick_problems")
D = ctypes.c_void_p(256)                   # never dereferenced: the checks come first


def test_problems_struct_mirror_matches_header():
    txt = re.sub(r"/\*.*?\*/", "", open(_lib.HEADER_PATH).read(), flags=re.S)
    body = [b for b in txt.split("typedef struct {")[1:] if re.match(r"[^}]*\}\s*isx_nst_problems;", b, flags=re.S)][0]
    body = body[: body.index("}")]
    fields = []
    for ctype, names in re.findall(r"\b((?:const\s+)?(?:int32_t|double)\s*\*?)\s*([^;]+);", body):
        fields += [(n.strip(), ctype.replace(" ", "")) for n in names.split(",")]
    assert [f for f, _ in fields] == [f[0] for f in engine.NstProblems._fields_]
    for (name, ctype), (_, py) in zip(fields, engine.NstProblems._fields_):
        assert (py is ctypes.c_void_p) == ctype.endswith("*"), name
    assert ctypes.sizeof(engine.NstProblems) == 4 + 4 + 8 + 8


def test_problems_entry_points_are_exported():
    lib = _lib.load()
    names = _lib.declared_symbols()
    for n in NEW:
        assert n in names and hasattr(lib, n), n


def _cfg(B):
    cfg = engine.NstConfig()
    cfg.B, cfg.H, cfg.W, cfg.xc, cfg.n_conv = B, 32, 32, 3, 2
    cfg.n_style, cfg.n_content = 1, 1
    cfg.style_conv[0], cfg.content_conv[0] = 0, 1
    cfg.style_target_b = cfg.content_target_b = B
    return cfg


def _eval(B, g, tb, cw=D, sw=D):
    cfg, bufs = _cfg(B), engine.NstBuffers()
    bufs.workspace = 256
    pr = engine.NstProblems()
    pr.images_per_problem, pr.style_target_b, pr.c_weight, pr.s_weight = g, tb, cw.value if cw else None, sw.value if sw else None
    _lib.call("isx_nst_eval_problems", ctypes.byref(cfg), ctypes.byref(bufs), ctypes.byref(pr), D, D, D, D, None)


@pytest.mark.parametrize("B,g,tb,cw,sw,msg", [
    (6, 4, 6, D, D, b"whole number of problems"),      # B % g != 0
    (4, 0, 4, D, D, b"whole number of problems"),
    (4, 5, 4, D, D, b"whole number of problems"),
    (4, 2, 3, D, D, b"style target batch"),            # not 1, P = 2 or B = 4
    (4, 2, 0, D, D, b"style target batch"),
    (8, 2, 2, D, D, b"style target batch"),            # P = 4
    (4, 2, 2, None, D, b"weight array"),
    (4, 2, 2, D, None, b"weight array"),
])
def test_eval_problems_rejects_bad_arguments(B, g, tb, cw, sw, msg):
    with pytest.raises(_lib.IsxError):
        _eval(B, g, tb, cw, sw)
    assert msg in _lib.load().isx_last_error()


def test_eval_problems_rejects_null_problems():
    cfg, bufs = _cfg(4), engine.NstBuffers()
    bufs.workspace = 256
    with pytest.raises(_lib.IsxError):
        _lib.call("isx_nst_eval_problems", ctypes.byref(cfg), ctypes.byref(bufs), None, D, D, D, D, None)
    assert b"null pointer" in _lib.load().isx_last_error()


def _tick(ipp=2, P=2, cw=D, sw=D, history=10):
    cfg = engine.LbfgsConfig(epochs=20, max_iter=20, max_eval=25, history=history, history_bf16=0, reserved_=0, lr=1.0,
                             tolerance_grad=1e-7, tolerance_change=1e-9, c_weight=1.0, s_weight=1.0)
    _lib.call("isx_lbfgs_tick_problems", D, D, D, D, D, D, D, D, D, D, ipp, P, _lib.i64(1024), ctypes.byref(cfg), cw, sw,
              D, D, 0, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(cw=None), b"weight array"),
    (dict(sw=None), b"weight array"),
    (dict(ipp=0), b"problems of"),
    (dict(P=0), b"problems of"),
    (dict(history=0), b"history"),
])
def test_lbfgs_tick_problems_rejects_bad_arguments(kw, msg):
    with pytest.raises(_lib.IsxError):
        _tick(**kw)
    assert msg in _lib.load().isx_last_error()


def _imgs(B, Bs=None, size=16):
    c = torch.rand(B, 3, size, size)
    s = torch.rand(B if Bs is None else Bs, 3, size, size)
    return c, s


@pytest.mark.parametrize("kw", [
    dict(problem_size=2, s_loss_weight=[1.0, 2.0, 3.0]),            # P = 2
    dict(problem_size=2, c_loss_weight=torch.ones(4)),
    dict(problem_size=2, c_loss_weight=[[1.0, 1.0]]),               # not 1-D
    dict(s_loss_weight=[1.0, 2.0]),                                 # default layout: P = 1
    dict(independent=True, s_loss_weight=[1.0, 2.0]),               # P = B = 4
    dict(problem_size=3),                                           # 4 % 3
    dict(problem_size=0),
    dict(problem_size=2, independent=True),
    dict(problem_size=4, streams=2),
    dict(problem_size=2, streams=2),
])
def test_nst_rejects_inconsistent_problem_layouts(kw):
    c, s = _imgs(4)
    with pytest.raises(ValueError):
        iris_b200.nst(c, s, use_tqdm=False, **kw)


@pytest.mark.parametrize("Bs", [3, 5, 8])
def test_nst_style_batch_must_be_one_problems_or_images(Bs):
    c, s = _imgs(4, Bs)
    with pytest.raises(ValueError):
        iris_b200.nst(c, s, problem_size=2, use_tqdm=False)


def test_stylize_frames_does_not_take_problem_size():
    frames = torch.rand(2, 1, 32, 32)
    with pytest.raises(ValueError):
        iris_b200.stylize_frames(frames, torch.rand(1, 16, 16), segs=torch.zeros(2, 1, 32, 32, dtype=torch.int64),
                                 problem_size=1)
