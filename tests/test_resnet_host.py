"""CPU tier of iris_b200.ResNet50 (the GazeEstimator2 feature extractor): BatchNorm folding, strict state-dict loading, the
planned stage shapes against torchvision's, the host-only workspace query, the ctypes mirror of isx_resnet50_weights, and
the precision-emulation oracle against torchvision.  No device needed."""
import ctypes
import re

import pytest
import torch
import torch.nn.functional as F

import iris_b200
from iris_b200 import _lib
from iris_b200 import resnet as R
from oracle import resnet_oracle as O


def randomise_bn(model, seed=1):
    """Non-trivial eval-mode BatchNorm statistics: with torchvision's defaults (mean 0, var 1, gamma 1, beta 0) folding would be
    nearly the identity and prove nothing."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                n = m.num_features
                m.running_mean.copy_(torch.randn(n, generator=g) * 0.2)
                m.running_var.copy_(torch.rand(n, generator=g) * 1.5 + 0.5)
                m.weight.copy_(torch.rand(n, generator=g) + 0.5)
                m.bias.copy_(torch.randn(n, generator=g) * 0.2)
    return model.eval()


@pytest.fixture(scope="module")
def model():
    return randomise_bn(R.random_resnet50(0))


def test_fold_matches_eval_module_fp64(model):
    """One Conv+BN pair (the strided 3x3 of layer2.0) folded == the eval-mode modules, all in float64."""
    idx = [s[0] for s in R.conv_specs()].index("layer2.0.conv2")
    w, b = R.fold_state_dict(model.state_dict())[idx]
    blk = model.layer2[0]
    conv, bn = blk.conv2, blk.bn2
    x = torch.randn(2, 128, 13, 11, dtype=torch.float64)
    ref = F.batch_norm(F.conv2d(x, conv.weight.double(), stride=2, padding=1), bn.running_mean.double(),
                       bn.running_var.double(), bn.weight.double(), bn.bias.double(), False, 0.0, bn.eps)
    got = F.conv2d(x, w.double(), b.double(), stride=2, padding=1)
    assert float(bn.running_var.std()) > 0.1 and float(bn.weight.detach().std()) > 0.1
    torch.testing.assert_close(got, ref, rtol=1e-6, atol=1e-6 * float(ref.abs().max()))


def test_state_dict_loading():
    net = R.random_resnet50(3)
    sd = net.state_dict()
    assert any(k.startswith("fc.") for k in sd)
    a = iris_b200.ResNet50(weights=sd)                 # fc.* ignored
    b = iris_b200.ResNet50(weights=net)                # the module itself
    c = iris_b200.ResNet50(weights="random", seed=3)   # torchvision resnet50(weights=None) under manual_seed(3)
    assert len(a.host_weights) == R.N_CONVS
    for (wa, ba), (wb, bb), (wc, bc) in zip(a.host_weights, b.host_weights, c.host_weights):
        assert torch.equal(wa, wb) and torch.equal(wa, wc) and torch.equal(ba, bb) and torch.equal(ba, bc)
    assert tuple(a.host_weights[0][0].shape) == (64, 3, 7, 7)
    missing = {k: v for k, v in sd.items() if k != "layer3.4.bn2.running_var"}
    with pytest.raises(KeyError, match="layer3.4.bn2.running_var"):
        iris_b200.ResNet50(weights=missing)
    extra = dict(sd, **{"layer1.0.conv4.weight": torch.zeros(1)})
    with pytest.raises(KeyError, match="layer1.0.conv4.weight"):
        iris_b200.ResNet50(weights=extra)
    with pytest.raises(ValueError):
        iris_b200.ResNet50(weights="imagenet")         # the library never downloads
    bad = dict(sd, **{"layer1.0.conv2.weight": torch.zeros(64, 64, 1, 1)})
    with pytest.raises(ValueError, match="layer1.0.conv2.weight"):
        iris_b200.ResNet50(weights=bad)


@pytest.mark.parametrize("H,W", [(224, 224), (400, 640), (97, 131), (32, 32)])
def test_planned_shapes_match_torchvision(model, H, W):
    with torch.no_grad():
        h = model.relu(model.bn1(model.conv1(torch.zeros(1, 3, H, W))))
        got = {"conv1": tuple(h.shape[1:])}
        h = model.maxpool(h)
        got["maxpool"] = tuple(h.shape[1:])
        for i, layer in enumerate((model.layer1, model.layer2, model.layer3, model.layer4)):
            h = layer(h)
            got["layer%d" % (i + 1)] = tuple(h.shape[1:])
    assert R.plan_shapes(H, W) == got


def test_workspace_query_without_device():
    lib = _lib.load()
    n1 = _lib.call_i64("isx_resnet50_workspace_bytes", 1, 224, 224)
    n4 = _lib.call_i64("isx_resnet50_workspace_bytes", 4, 224, 224)
    # five 256-byte aligned buffers; the largest holds 64 x 112 x 112 bf16 (the stem output)
    assert n1 >= 112 * 112 * 64 * 2 and 4 * n1 - 5 * 4 * 255 <= n4 <= 4 * n1
    assert _lib.call_i64("isx_resnet50_workspace_bytes", 3, 97, 131) > 0
    for B, H, W in ((1, 31, 64), (1, 64, 31), (0, 224, 224), (-2, 224, 224)):
        assert _lib.call_i64("isx_resnet50_workspace_bytes", B, H, W) == -1
        assert b"isx_resnet50_workspace_bytes: bad shape" in lib.isx_last_error()


def test_weights_struct_mirrors_header():
    txt = re.sub(r"/\*.*?\*/", "", open(_lib.HEADER_PATH).read(), flags=re.S)
    n = int(re.search(r"#define ISX_RESNET50_CONVS (\d+)", txt).group(1))
    body = re.search(r"typedef struct \{([^}]*)\}\s*isx_resnet50_weights;", txt).group(1)
    fields = re.findall(r"const\s+\w+\s*\*\s*(\w+)\[ISX_RESNET50_CONVS\];", body)
    assert n == R.N_CONVS == len(R.conv_specs())
    assert fields == [f[0] for f in R.ResNet50Weights._fields_] == ["w", "bias"]
    assert ctypes.sizeof(R.ResNet50Weights) == 2 * n * ctypes.sizeof(ctypes.c_void_p)


def test_conv_specs_follow_torchvision_module_order(model):
    convs = [name for name, m in model.named_modules() if isinstance(m, torch.nn.Conv2d)]
    assert convs == [s[0] for s in R.conv_specs()]
    for name, _, cin, cout, k, stride in R.conv_specs():
        m = model.get_submodule(name)
        assert (m.in_channels, m.out_channels, m.kernel_size[0], m.stride[0]) == (cin, cout, k, stride)


def test_emulation_oracle_fp32_reproduces_torchvision(model):
    x = torch.rand(2, 3, 97, 131, generator=torch.Generator().manual_seed(5))
    ref = O.torchvision_features(model, x)
    got = O.resnet50_forward(model, x, operand_dtype=torch.float32)
    torch.testing.assert_close(got, ref, rtol=1e-6, atol=1e-6 * float(ref.abs().max()))
    # and the bf16 emulation moves it by the storage precision, not more
    e16 = O.resnet50_forward(model, x, operand_dtype=torch.bfloat16)
    rel = float((e16 - ref).norm() / ref.norm())
    assert 1e-4 < rel < 3e-2


def test_host_surface_refuses_without_running():
    net = iris_b200.ResNet50(weights="random")
    net.train()
    with pytest.raises(RuntimeError):
        net(torch.zeros(1, 3, 32, 32))                 # inference only
    net.eval()
    with pytest.raises(ValueError):
        net(torch.zeros(1, 3, 31, 64))
    with pytest.raises(ValueError):
        net(torch.zeros(1, 2, 64, 64))
    with pytest.raises(ValueError, match="ResNet50"):
        iris_b200.GazeEstimator2(extract_feature=True)
