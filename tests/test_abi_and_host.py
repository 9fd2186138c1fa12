"""CPU tier: the C-ABI library loads and exports every symbol include/isx.h declares (no compute calls
without a GPU), the host-side mirrors of the reference interface are consistent, and the product path
refuses to run without CUDA instead of falling back."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import iris_b200
from iris_b200 import _lib, engine, synthetic


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = _lib.declared_symbols()
    assert len(names) >= 25 and "isx_nst_eval" in names and "isx_lbfgs_tick" in names
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    assert lib.isx_version() == 100
    assert isinstance(lib.isx_last_error(), bytes)


def test_kernel_selection_options():
    """isx_set_option / isx_get_option know exactly the five kernel-selection options; the names of removed experiment
    options are refused like any unknown name."""
    lib = _lib.load()
    defaults = {b"c64": 1, b"halo2": 1, b"tail_n": 1, b"sweep64": 1, b"smem_reserve_kb": 0}
    for name, default in defaults.items():
        v = ctypes.c_int(-1)
        assert lib.isx_get_option(name, ctypes.byref(v)) == 0 and v.value == default, name
        assert lib.isx_set_option(name, default) == 0, name
    for name in (b"pool_idx", b"head_ctas", b"lm_planes", b"sweep_dbg", b"c64_slots", b"halo2_stages"):
        assert lib.isx_set_option(name, 1) != 0, name
        assert b"unknown option '%s'" % name in lib.isx_last_error()
        assert lib.isx_get_option(name, ctypes.byref(ctypes.c_int())) != 0, name


def test_header_has_no_torch_types():
    txt = open(_lib.HEADER_PATH).read()
    assert 'extern "C"' in txt
    code = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)  # declarations only, comments stripped
    assert "torch" not in code.lower() and "at::" not in code and "Tensor" not in code and "#include <stdint.h>" in code


def test_struct_mirrors_match_header():
    """ctypes mirrors vs the C structs: field order and a size the C side would compute."""
    txt = re.sub(r"/\*.*?\*/", "", open(_lib.HEADER_PATH).read(), flags=re.S)

    def c_struct_fields(name):
        body = [b for b in txt.split("typedef struct {")[1:] if re.match(r"[^}]*\}\s*%s;" % name, b, flags=re.S)][0]
        body = body[: body.index("}")]
        out = []
        for decl in re.findall(r"\b(?:int32_t|float|double)\s+([^;]+);", body):
            out += [re.sub(r"\[.*?\]", "", n).strip() for n in decl.split(",")]
        return out

    assert [f[0] for f in engine.NstConfig._fields_] == c_struct_fields("isx_nst_config")
    assert [f[0] for f in engine.LbfgsConfig._fields_] == c_struct_fields("isx_lbfgs_config")
    assert ctypes.sizeof(engine.NstConfig) == 4 * 7 + 4 * 8 * 2 + 4 + 4 * 8 * 2 + 4 * 6 + 8 * 2
    assert ctypes.sizeof(engine.LbfgsConfig) == 24 + 8 * 5
    # pure-host size queries work without a device
    assert _lib.call_i64("isx_lbfgs_mats_bytes", 2, 100) == 2 * 3 * 101 * 101 * 8
    assert _lib.call_i64("isx_lbfgs_state_bytes", 1) > 0
    assert _lib.call_i64("isx_gram_workspace_bytes", 1, 256000, 64) >= 64 * 64 * 4


def test_workspace_query_and_argument_errors():
    cfg = engine.NstConfig()
    cfg.B, cfg.H, cfg.W, cfg.xc, cfg.n_conv = 2, 64, 48, 3, 10
    cfg.n_style, cfg.n_content = 4, 1
    for t, c in enumerate([0, 2, 4, 8]):
        cfg.style_conv[t] = c
    cfg.content_conv[0] = 9
    n = _lib.call_i64("isx_nst_workspace_bytes", ctypes.byref(cfg))
    acts = 2 * 64 * 48 * 2 * (64 + 64) + 2 * 32 * 24 * 2 * (128 + 128) + 2 * 16 * 12 * 2 * 256 * 4 + 2 * 8 * 6 * 2 * 512 * 2
    assert n > acts
    cfg.style_conv[3] = 12  # tap beyond n_conv -> error, not UB
    assert _lib.call_i64("isx_nst_workspace_bytes", ctypes.byref(cfg)) == -1
    assert b"style tap" in _lib.load().isx_last_error()
    with pytest.raises(_lib.IsxError):
        _lib.call("isx_gram_fwd", None, 1, 16, 64, _lib.f32(1.0), None, None, None, 1, _lib.f64(0), None, _lib.f32(0),
                  None, None)


def test_layer_map_matches_reference_table():
    # models/vgg/vgg.py:6-10
    L = engine.VGG19_LAYERS
    assert (L["conv1_1"], L["relu1_1"], L["pool1"], L["relu2_1"], L["relu3_1"], L["relu4_1"], L["relu4_2"],
            L["relu5_1"], L["pool5"]) == (0, 1, 4, 6, 11, 20, 22, 29, 36)
    assert len(L) == 37
    conv = engine.CONV_OF_FEATURE_INDEX
    assert conv[L["relu4_2"]] == 9 and conv[L["conv4_2"]] == 9 and conv[L["relu5_1"]] == 12
    assert engine.CONV_COUT == [64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512, 512]


def test_vgg19_surface_and_no_cpu_fallback():
    from oracle import nst_oracle as O

    w = O.random_vgg19_weights(0)
    net = iris_b200.VGG19(weights=w)
    assert net.content_layers_idx == [22] and net.style_layers_idx == [1, 6, 11, 20]
    assert net.content_convs == [9] and net.style_convs == [0, 2, 4, 8]
    net5 = iris_b200.VGG19(style_layers=["conv1_1", "relu2_1", "relu3_1", "relu4_1", "relu5_1"], weights=w)
    assert net5.style_convs == [0, 2, 4, 8, 12]
    # vgg19_bn (models/vgg/vgg.py:12-17,41-44): BatchNorm folded; bn* / relu* taps map to the conv ordinals, conv* taps raise
    from iris_b200 import vgg as V

    assert V.vgg19_bn_layers["relu4_2"] == 32 and V.vgg19_bn_layers["bn1_1"] == 1 and V.vgg19_bn_layers["pool5"] == 52
    nb = iris_b200.VGG19(bn=True, weights=w, style_layers=["relu1_1", "bn2_1", "relu3_1", "relu4_1"])
    assert nb.style_layers_idx == [2, 8, 16, 29] and nb.style_convs == [0, 2, 4, 8] and nb.content_convs == [9]
    with pytest.raises(NotImplementedError):
        iris_b200.VGG19(bn=True, weights=w, style_layers=["conv1_1"])
    # pooling layers are taps too (vgg.py:6-10): tap ids 16 + k
    netp = iris_b200.VGG19(content_layers=["pool4"], style_layers=["pool1", "relu2_1"], weights=w)
    assert netp.style_convs == [16, 2] and netp.content_convs == [19] and netp.style_layers_idx == [4, 6]
    cfgp = engine.NstConfig()
    cfgp.B, cfgp.H, cfgp.W, cfgp.xc, cfgp.n_conv, cfgp.n_style, cfgp.n_content = 1, 64, 64, 3, 12, 2, 1
    cfgp.style_conv[0], cfgp.style_conv[1], cfgp.content_conv[0] = 16, 2, 19
    assert _lib.call_i64("isx_nst_workspace_bytes", ctypes.byref(cfgp)) > 0
    cfgp.n_conv = 11                      # pool4 follows conv index 11: not computed with n_conv = 11
    assert _lib.call_i64("isx_nst_workspace_bytes", ctypes.byref(cfgp)) == -1
    g = torch.Generator().manual_seed(1)
    cw, cb = torch.randn(8, 4, 3, 3, generator=g), torch.randn(8, generator=g)
    bn = torch.nn.BatchNorm2d(8).eval()
    with torch.no_grad():
        bn.weight.copy_(torch.rand(8, generator=g) + 0.5); bn.bias.copy_(torch.randn(8, generator=g))
        bn.running_mean.copy_(torch.randn(8, generator=g)); bn.running_var.copy_(torch.rand(8, generator=g) + 0.2)
        fw, fb = V.fold_batchnorm(cw, cb, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps)
        xin = torch.randn(2, 4, 9, 9, generator=g)
        ref = bn(torch.nn.functional.conv2d(xin, cw, cb, padding=1))
        assert torch.allclose(torch.nn.functional.conv2d(xin, fw, fb, padding=1), ref, atol=1e-5)
    x = torch.rand(1, 3, 32, 32)
    if not torch.cuda.is_available():
        with pytest.raises(Exception):
            net(x)
        with pytest.raises(_lib.IsxError):
            iris_b200.nst(x, x, vgg=net, use_tqdm=False, device="cpu")
        with pytest.raises(_lib.IsxError):
            iris_b200.GramMatrix(torch.rand(1, 64, 8, 8))
        with pytest.raises(_lib.IsxError):
            iris_b200.crop_image(torch.rand(8, 8))


def test_synthetic_eyes_are_deterministic_and_exercise_the_mask():
    f1, s1 = synthetic.synthetic_eye(5, 640, 400)
    f2, s2 = synthetic.synthetic_eye(5, 640, 400)
    assert np.array_equal(f1, f2) and np.array_equal(s1, s2)
    assert f1.shape == (1, 640, 400) and f1.dtype == np.float32 and s1.dtype == np.int64
    assert 0.0 <= f1.min() and f1.max() <= 1.0
    iris = s1 == 2
    frac = iris.mean()
    assert 0.04 < frac < 0.16, frac                      # 6-10 % of the frame like the shipped eye PNGs
    assert ((f1 > 0.8) & iris).sum() > 0                 # glints inside the iris: the x <= 0.8 test matters
    assert set(np.unique(s1)) == {0, 1, 2, 3}
    crops = synthetic.synthetic_iris_crops([1, 2], 64)
    assert crops.shape == (2, 3, 64, 64) and np.array_equal(crops[:, 0], crops[:, 2])


def test_landmark_and_metric_entry_points_validate_on_the_host():
    """Row f4 / the drivers' metrics: pure-host size query and the argument checks that run before any device work."""
    lib = _lib.load()
    q = lambda *a: _lib.call_i64("isx_eye_landmarks_workspace_bytes", *a)
    small, big = q(1, 400, 640, 4096), q(128, 400, 640, 16384)
    # per frame: two bit planes (400 rows x 20 words), two classes x two point buffers, results, sclera box
    assert small >= 2 * 400 * 20 * 4 + 2 * 2 * 4096 * 4 and big >= 128 * (2 * 400 * 20 * 4 + 2 * 2 * 16384 * 4)
    assert q(0, 400, 640, 4096) == -1 and q(1, 400, 640, 4) == -1          # at least five points to fit an ellipse
    dummy = ctypes.c_void_p(256)                                           # never dereferenced: the checks come first
    bad = [(None, 0, 1, 400, 640), (dummy, 3, 1, 400, 640), (dummy, 0, 1, 40000, 640), (dummy, 0, 70000, 64, 64),
           (dummy, 0, 1, 4000, 4000)]                                      # null map, dtype, 16-bit coordinates, batch, shared memory
    for seg, dt, B, H, W in bad:
        with pytest.raises(_lib.IsxError):
            _lib.call("isx_eye_landmarks", seg, dt, B, H, W, _lib.f64(1e-6), 4096, dummy, dummy, dummy, None)
    assert b"shared" in lib.isx_last_error()
    with pytest.raises(_lib.IsxError):
        _lib.call("isx_seg_iou", dummy, dummy, 1, _lib.i64(16), 9, _lib.f32(1e-6), dummy, dummy, dummy, None)
    assert b"num_class" in lib.isx_last_error()
    with pytest.raises(_lib.IsxError):
        _lib.call("isx_gaze_head_fwd", dummy, _lib.i64(8), 4, 19, 64, 3, dummy, dummy, dummy, dummy, dummy, dummy, dummy, None)   # ld_x < in_dim
    with pytest.raises(_lib.IsxError):
        _lib.call("isx_angular_distance", dummy, None, 4, 3, dummy, dummy, None)
    # the Python surface mirrors the reference's names and refuses to run without CUDA
    for name in ("extract_eye_landmarks", "extract_eye_landmarks_batch", "GazeEstimator1", "GazeEstimator2", "cal_IoUs", "angular_distance"):
        assert hasattr(iris_b200, name), name
    net = iris_b200.GazeEstimator1()
    assert sorted(net.state_dict()) == ["model.0.bias", "model.0.weight", "model.3.bias", "model.3.weight", "model.6.bias", "model.6.weight"]
    assert tuple(net.model[0].weight.shape) == (64, 19) and tuple(iris_b200.GazeEstimator2().model[0].weight.shape) == (64, 2048)
    with pytest.raises(ValueError):
        iris_b200.GazeEstimator2(extract_feature=True)
    if not torch.cuda.is_available():
        with pytest.raises(_lib.IsxError):
            net(torch.zeros(2, 19))                                        # parameters on the CPU: no fallback
