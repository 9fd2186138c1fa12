"""CPU tier of coupled problems of unequal size in one NST job (nst(problem_sizes=...), isx_nst_eval_ranges,
isx_lbfgs_tick_ranges, stylize_frames(frames_per_problem=g)): the isx_nst_problem_ranges mirror matches the header, both
entry points are exported and refuse bad arguments on the host before any device work, nst() / stylize_frames() refuse
inconsistent layouts with ValueError, and the frame grouping of stylize_frames gives the expected layouts."""
import ctypes
import re

import pytest
import torch

import iris_b200
from iris_b200 import _lib, engine, frames

NEW = ("isx_nst_eval_ranges", "isx_lbfgs_tick_ranges")
D = ctypes.c_void_p(256)                   # never dereferenced: the checks come first


def test_ranges_struct_mirror_matches_header():
    txt = re.sub(r"/\*.*?\*/", "", open(_lib.HEADER_PATH).read(), flags=re.S)
    body = [b for b in txt.split("typedef struct {")[1:] if re.match(r"[^}]*\}\s*isx_nst_problem_ranges;", b, flags=re.S)][0]
    body = body[: body.index("}")]
    fields = []
    for ctype, names in re.findall(r"\b((?:const\s+)?(?:int32_t|double)\s*\*?)\s*([^;]+);", body):
        fields += [(n.strip(), ctype.replace(" ", "")) for n in names.split(",")]
    assert [f for f, _ in fields] == [f[0] for f in engine.NstProblemRanges._fields_]
    for (name, ctype), (_, py) in zip(fields, engine.NstProblemRanges._fields_):
        assert (py is ctypes.c_void_p) == ctype.endswith("*"), name
    assert ctypes.sizeof(engine.NstProblemRanges) == 4 + 4 + 8 + 8 + 8


def test_ranges_entry_points_are_exported():
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


def _ranges(first, tb=1, cw=D, sw=D, P=None):
    offsets = (ctypes.c_int32 * max(1, len(first)))(*first)
    pr = engine.NstProblemRanges()
    pr.n_problems = len(first) - 1 if P is None else P
    pr.style_target_b = tb
    pr.first_image = ctypes.cast(offsets, ctypes.c_void_p).value if first else None
    pr.c_weight, pr.s_weight = cw.value if cw else None, sw.value if sw else None
    return pr, offsets


def _eval(B, first, **kw):
    cfg, bufs = _cfg(B), engine.NstBuffers()
    bufs.workspace = 256
    pr, keep = _ranges(first, **kw)
    _lib.call("isx_nst_eval_ranges", ctypes.byref(cfg), ctypes.byref(bufs), ctypes.byref(pr), D, D, D, D, None)


def _tick(B, first, n_img=1024, history=10, **kw):
    cfg = engine.LbfgsConfig(epochs=20, max_iter=20, max_eval=25, history=history, history_bf16=0, reserved_=0, lr=1.0,
                             tolerance_grad=1e-7, tolerance_change=1e-9, c_weight=1.0, s_weight=1.0)
    pr, keep = _ranges(first, **kw)
    _lib.call("isx_lbfgs_tick_ranges", D, D, D, D, D, D, D, D, D, D, ctypes.byref(pr), B, _lib.i64(n_img),
              ctypes.byref(cfg), D, D, 0, None)


RANGE_CASES = [
    (7, [1, 3, 7], {}, b"first_image[0] = 1 must be 0"),
    (7, [0, 3, 6], {}, b"must be the batch 7"),
    (7, [0, 3, 8], {}, b"must be the batch 7"),
    (7, [0, 3, 3, 7], {}, b"problem 1 is empty"),
    (7, [0, 5, 3, 7], {}, b"problem 1 is empty"),
    (7, [0, 7], dict(P=0), b"problem count 0"),
    (2050, list(range(0, 2051, 2)), {}, b"problem count 1025"),
    (7, [0, 3, 7], dict(cw=None), b"weight array"),
    (7, [0, 3, 7], dict(sw=None), b"weight array"),
    (7, [], {}, b"null pointer"),
]


@pytest.mark.parametrize("B,first,kw,msg", RANGE_CASES)
def test_eval_ranges_rejects_bad_ranges(B, first, kw, msg):
    with pytest.raises(_lib.IsxError):
        _eval(B, first, **kw)
    assert msg in _lib.load().isx_last_error()


@pytest.mark.parametrize("B,first,kw,msg", RANGE_CASES)
def test_lbfgs_tick_ranges_rejects_bad_ranges(B, first, kw, msg):
    with pytest.raises(_lib.IsxError):
        _tick(B, first, **kw)
    assert msg in _lib.load().isx_last_error()


@pytest.mark.parametrize("B,first,tb", [
    (7, [0, 3, 7], 3),          # not 1, P = 2 or B = 7
    (7, [0, 3, 7], 0),
    (8, [0, 1, 2, 8], 2),       # P = 3
])
def test_eval_ranges_rejects_style_target_batch(B, first, tb):
    with pytest.raises(_lib.IsxError):
        _eval(B, first, tb=tb)
    assert b"style target batch" in _lib.load().isx_last_error()


def test_eval_ranges_rejects_null_ranges():
    cfg, bufs = _cfg(4), engine.NstBuffers()
    bufs.workspace = 256
    with pytest.raises(_lib.IsxError):
        _lib.call("isx_nst_eval_ranges", ctypes.byref(cfg), ctypes.byref(bufs), None, D, D, D, D, None)
    assert b"null pointer" in _lib.load().isx_last_error()


@pytest.mark.parametrize("kw,msg", [
    (dict(n_img=0), b"elements per image"),
    (dict(history=0), b"history"),
    (dict(history=101), b"history"),
])
def test_lbfgs_tick_ranges_rejects_bad_arguments(kw, msg):
    with pytest.raises(_lib.IsxError):
        _tick(7, [0, 3, 7], **kw)
    assert msg in _lib.load().isx_last_error()


def test_the_problem_limit_itself_passes_the_range_checks():
    """1024 problems are within the limit: the checks pass and the call fails only later, on the (dummy) buffers or the
    missing device -- never with a problem-count message."""
    try:
        _tick(2048, list(range(0, 2049, 2)), history=0)
    except _lib.IsxError:
        pass
    err = _lib.load().isx_last_error()
    assert b"history" in err and b"problem count" not in err


def _imgs(B, Bs=None, size=16):
    c = torch.rand(B, 3, size, size)
    s = torch.rand(B if Bs is None else Bs, 3, size, size)
    return c, s


@pytest.mark.parametrize("kw", [
    dict(problem_sizes=[2, 3]),                                       # sum 5 != 6
    dict(problem_sizes=[2, 5]),
    dict(problem_sizes=[6, 0]),                                       # empty problem
    dict(problem_sizes=[7, -1]),
    dict(problem_sizes=[2.5, 3.5]),                                   # not integers
    dict(problem_sizes=[2.0, 4.0]),
    dict(problem_sizes=[True, 5]),
    dict(problem_sizes=[]),
    dict(problem_sizes=[2, 4], problem_size=2),
    dict(problem_sizes=[2, 4], problem_size=3),
    dict(problem_sizes=[1] * 6, independent=True),
    dict(problem_sizes=[2, 4], independent=True),
    dict(problem_sizes=[2, 4], streams=2),
    dict(problem_sizes=[1] * 6, streams=3),
    dict(problem_sizes=[2, 4], s_loss_weight=[1.0, 2.0, 3.0]),        # P = 2
    dict(problem_sizes=[2, 4], c_loss_weight=torch.ones(6)),
    dict(problem_sizes=[2, 4], c_loss_weight=[[1.0, 1.0]]),           # not 1-D
    dict(problem_sizes=[1, 2, 3], s_loss_weight=[1.0]),
])
def test_nst_rejects_bad_problem_sizes(kw):
    c, s = _imgs(6)
    with pytest.raises(ValueError):
        iris_b200.nst(c, s, use_tqdm=False, **kw)


@pytest.mark.parametrize("Bs", [2, 4, 5, 7])
def test_nst_ranged_style_batch_must_be_one_problems_or_images(Bs):
    c, s = _imgs(6, Bs)
    with pytest.raises(ValueError):
        iris_b200.nst(c, s, problem_sizes=[1, 2, 3], use_tqdm=False)


def _frames(B):
    return torch.rand(B, 1, 32, 32), torch.zeros(B, 1, 32, 32, dtype=torch.int64)


@pytest.mark.parametrize("kw", [
    dict(frames_per_problem=0),
    dict(frames_per_problem=-2),
    dict(frames_per_problem=2.5),
    dict(frames_per_problem=3, c_loss_weight=[1.0, 2.0]),            # K = 3 runs of 7 frames
    dict(frames_per_problem=3, s_loss_weight=[1.0, 2.0, 3.0, 4.0]),
    dict(frames_per_problem=3, s_loss_weight=torch.ones(7)),
    dict(frames_per_problem=3, independent=True),
    dict(frames_per_problem=3, problem_sizes=[3, 3, 1]),
    dict(problem_size=1),
])
def test_stylize_frames_rejects_bad_runs(kw):
    f, segs = _frames(7)
    with pytest.raises(ValueError):
        iris_b200.stylize_frames(f, torch.rand(1, 16, 16), segs=segs, **kw)


@pytest.mark.parametrize("Bs", [2, 4, 6, 8])
def test_stylize_frames_style_batch_must_be_one_runs_or_frames(Bs):
    f, segs = _frames(7)
    with pytest.raises(ValueError):
        iris_b200.stylize_frames(f, torch.rand(Bs, 1, 16, 16), segs=segs, frames_per_problem=3)


def test_group_frames_all_valid():
    r = frames.group_frames([True] * 8, 4)
    assert r["run_sizes"] == [4, 4] and r["kept_runs"] == [0, 1] and r["problem_sizes"] == [4, 4]
    assert r["frames"] == list(range(8)) and r["style_index"] is None


def test_group_frames_one_run_emptied_and_short_last_run():
    valid = [True] * 4 + [False] * 4 + [True, False, True]           # runs of 4: full, empty, short (2 of 3)
    r = frames.group_frames(valid, 4, style_batch=3)                  # one style per run
    assert r["run_sizes"] == [4, 0, 2]
    assert r["kept_runs"] == [0, 2] and r["problem_sizes"] == [4, 2]
    assert r["frames"] == [0, 1, 2, 3, 8, 10]
    assert r["style_index"] == [0, 2]


def test_group_frames_short_last_run_all_valid():
    r = frames.group_frames([True] * 7, 3)
    assert r["run_sizes"] == [3, 3, 1] and r["problem_sizes"] == [3, 3, 1] and r["kept_runs"] == [0, 1, 2]


def test_group_frames_per_frame_styles_with_dropped_frames():
    valid = torch.tensor([True, False, True, True, False, False, True])
    r = frames.group_frames(valid, 2, style_batch=7)                  # one style per frame
    assert r["run_sizes"] == [1, 2, 0, 1]
    assert r["kept_runs"] == [0, 1, 3] and r["problem_sizes"] == [1, 2, 1]
    assert r["frames"] == [0, 2, 3, 6] and r["style_index"] == [0, 2, 3, 6]


def test_group_frames_one_frame_per_run_maps_styles_alike():
    valid = [True, False, True]
    r = frames.group_frames(valid, 1, style_batch=3)                  # K == B: per-run and per-frame agree
    assert r["run_sizes"] == [1, 0, 1] and r["kept_runs"] == r["frames"] == r["style_index"] == [0, 2]
