"""iris_b200.ResNet50 on the B200: the entry points one at a time against float64 references of the same bf16 operands
(strided / 1x1 / 3x3 convolutions with residual and ReLU, the 7x7 stem, the 3x3/2 max pool bit for bit, the global
average pool), then the whole trunk against fp32 torchvision with the bf16-storage emulation's own error as the yardstick,
and GazeEstimator2 frames -> unit vectors.  Weights are seeded torchvision initialisations with randomised BatchNorm
statistics (the defaults would make folding trivial)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _lib():
    from iris_b200 import _lib as L

    return L


def randomise_bn(model, seed=1):
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


def bf16_round(t):
    return t.to(torch.bfloat16).float()


def assert_within_bf16(got, ref, abssum, what):
    """|got - ref| <= one bf16 rounding of the result (2^-8 relative) + fp32 accumulation (1e-5 of the sum of |terms|)."""
    err = (got.double() - ref).abs()
    bound = 2.0 ** -8 * ref.abs() + 1e-5 * abssum + 1e-30
    worst = float((err / bound).max())
    print("%s: max |err| %.3g, worst err / bound %.3f" % (what, float(err.max()), worst))
    assert worst <= 1.0, what


CONV_CASES = [
    # k, stride, Cin, Cout, B, H, W, residual, relu
    (1, 1, 64, 256, 3, 25, 33, True, True),      # layer1 conv3 + identity
    (1, 2, 256, 512, 17, 25, 33, False, False),  # layer2 projection shortcut
    (3, 2, 128, 128, 3, 25, 33, False, True),    # layer2.0 conv2
    (3, 1, 64, 64, 1, 31, 17, True, True),
    (3, 2, 512, 512, 1, 13, 17, False, True),    # layer4.0 conv2
    (1, 1, 2048, 512, 3, 7, 9, False, True),
    (1, 1, 512, 2048, 17, 7, 9, True, True),
    (3, 1, 256, 256, 3, 13, 17, False, False),
    (1, 2, 1024, 2048, 1, 13, 17, False, False),
    (3, 2, 64, 128, 17, 9, 11, True, True),
]


@pytest.mark.parametrize("k,stride,cin,cout,B,H,W,res,relu", CONV_CASES)
def test_conv_entry_point_vs_fp64(k, stride, cin, cout, B, H, W, res, relu):
    L = _lib()
    g = torch.Generator(device=DEV).manual_seed(k * 1000 + cin + cout + B)
    x = torch.randn(B, H, W, cin, device=DEV, generator=g).to(torch.bfloat16)
    w = bf16_round(torch.randn(cout, cin, k, k, device=DEV, generator=g) / (cin * k * k) ** 0.5)
    bias = torch.randn(cout, device=DEV, generator=g) * 0.1
    Ho, Wo = (H + stride - 1) // stride, (W + stride - 1) // stride
    r = torch.randn(B, Ho, Wo, cout, device=DEV, generator=g).to(torch.bfloat16) if res else None
    s = L.stream_ptr()
    if k == 1:
        wp = torch.empty(cout, cin, device=DEV, dtype=torch.bfloat16)
        L.call("isx_pack_conv1x1_weights", w.contiguous(), cout, cin, wp, s)
    else:
        wp = torch.empty(9, cout, cin, device=DEV, dtype=torch.bfloat16)
        L.call("isx_pack_conv3x3_weights", w.contiguous(), cout, cin, wp, None, s)
    out = torch.empty(B, Ho, Wo, cout, device=DEV, dtype=torch.bfloat16)
    L.call("isx_conv_bias_act_fwd", x, wp, bias, r, out, B, H, W, cin, cout, k, stride, int(relu), s)
    torch.cuda.synchronize()
    xd = x.permute(0, 3, 1, 2).double()
    ref = F.conv2d(xd, w.double(), bias.double(), stride=stride, padding=k // 2)
    abssum = F.conv2d(xd.abs(), w.double().abs(), bias.double().abs(), stride=stride, padding=k // 2)
    if res:
        ref = ref + r.permute(0, 3, 1, 2).double()
        abssum = abssum + r.permute(0, 3, 1, 2).double().abs()
    if relu:
        ref = ref.clamp_min(0)
    assert tuple(ref.shape) == (B, cout, Ho, Wo)
    assert_within_bf16(out.permute(0, 3, 1, 2), ref, abssum, "conv k%d s%d %d->%d B%d %dx%d" % (k, stride, cin, cout, B, H, W))


def test_conv_entry_point_refuses_bad_arguments():
    L = _lib()
    t = torch.zeros(64 * 64 * 9, device=DEV, dtype=torch.bfloat16)
    for k, stride, cin in ((5, 1, 64), (3, 3, 64), (1, 1, 48)):
        with pytest.raises(L.IsxError):
            L.call("isx_conv_bias_act_fwd", t, t, None, None, t, 1, 8, 8, cin, 64, k, stride, 1, L.stream_ptr())


@pytest.mark.parametrize("B,xc,H,W", [(3, 3, 97, 131), (1, 1, 224, 224), (17, 3, 32, 33)])
def test_stem_vs_fp64(B, xc, H, W):
    L = _lib()
    g = torch.Generator(device=DEV).manual_seed(B * 7 + H)
    x = torch.rand(B, xc, H, W, device=DEV, generator=g) * 2 - 0.5
    w = torch.randn(64, 3, 7, 7, device=DEV, generator=g) / 147 ** 0.5
    bias = torch.randn(64, device=DEV, generator=g) * 0.1
    wp = torch.empty(64, 192, device=DEV, dtype=torch.bfloat16)
    s = L.stream_ptr()
    L.call("isx_pack_resnet_stem_weights", w.contiguous(), wp, s)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    out = torch.empty(B, Ho, Wo, 64, device=DEV, dtype=torch.bfloat16)
    L.call("isx_resnet_stem_fwd", x, xc, wp, bias, out, B, H, W, s)
    torch.cuda.synchronize()
    xd = bf16_round(x.repeat(1, 3 // xc, 1, 1)).double()
    wd = bf16_round(w).double()
    ref = F.conv2d(xd, wd, bias.double(), stride=2, padding=3).clamp_min(0)
    abssum = F.conv2d(xd.abs(), wd.abs(), bias.double().abs(), stride=2, padding=3)
    assert_within_bf16(out.permute(0, 3, 1, 2), ref, abssum, "stem B%d xc%d %dx%d" % (B, xc, H, W))
    if xc == 1:
        out3 = torch.empty_like(out)
        L.call("isx_resnet_stem_fwd", x.repeat(1, 3, 1, 1).contiguous(), 3, wp, bias, out3, B, H, W, s)
        torch.cuda.synchronize()
        assert torch.equal(out.view(torch.int16), out3.view(torch.int16))


@pytest.mark.parametrize("B,H,W,C", [(3, 49, 66, 64), (2, 33, 17, 256), (1, 112, 112, 64), (5, 2, 3, 8)])
def test_maxpool3x3s2_bit_exact(B, H, W, C):
    L = _lib()
    g = torch.Generator(device=DEV).manual_seed(H * W + C)
    x = torch.randn(B, H, W, C, device=DEV, generator=g)
    x = torch.where(torch.rand(B, H, W, C, device=DEV, generator=g) < 0.2, torch.zeros_like(x), x)  # ties at 0 (ReLU output)
    x = torch.where(torch.rand(B, H, W, C, device=DEV, generator=g) < 0.05, -torch.zeros_like(x), x)
    x = x.to(torch.bfloat16)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    out = torch.empty(B, Ho, Wo, C, device=DEV, dtype=torch.bfloat16)
    L.call("isx_maxpool3x3s2_fwd", x, out, B, H, W, C, L.stream_ptr())
    ref = F.max_pool2d(x.permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1)
    torch.cuda.synchronize()
    assert tuple(ref.shape) == tuple(out.shape)
    assert torch.equal(out.view(torch.int16), ref.contiguous().view(torch.int16))


@pytest.mark.parametrize("B,HW,C", [(3, 20, 2048), (5, 49, 2048), (1, 260, 64), (2, 1, 8)])
def test_global_avgpool_vs_fp64(B, HW, C):
    L = _lib()
    g = torch.Generator(device=DEV).manual_seed(HW * 3 + C)
    x = (torch.rand(B, HW, C, device=DEV, generator=g) * 4).to(torch.bfloat16)
    out = torch.empty(B, C, device=DEV, dtype=torch.float32)
    L.call("isx_global_avgpool", x, out, B, HW, C, L.stream_ptr())
    out2 = torch.empty_like(out)
    L.call("isx_global_avgpool", x, out2, B, HW, C, L.stream_ptr())
    torch.cuda.synchronize()
    torch.testing.assert_close(out.double(), x.double().mean(1), rtol=1e-6, atol=0)
    assert torch.equal(out, out2)


@pytest.fixture(scope="module")
def trunk():
    import iris_b200
    from iris_b200 import resnet as R

    model = randomise_bn(R.random_resnet50(0))
    net = iris_b200.ResNet50(weights=model)
    return model.to(DEV), net


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


TRUNK_CASES = [(224, 224, 1, 3), (224, 224, 16, 1), (400, 640, 3, 3), (400, 640, 16, 1), (97, 131, 3, 1), (97, 131, 16, 3),
               (400, 640, 1, 1), (97, 131, 1, 3), (224, 224, 3, 1)]


@pytest.mark.parametrize("H,W,B,xc", TRUNK_CASES)
def test_trunk_vs_torchvision(trunk, H, W, B, xc):
    from oracle import resnet_oracle as O

    model, net = trunk
    g = torch.Generator(device=DEV).manual_seed(H + W + B + xc)
    x = torch.rand(B, xc, H, W, device=DEV, generator=g)
    got = net(x)
    ref = O.torchvision_features(model, x)
    emu = O.resnet50_forward(model, x, operand_dtype=torch.bfloat16)
    torch.cuda.synchronize()
    e_got, e_emu = _rel(got, ref), _rel(emu, ref)
    print("%dx%d B%d xc%d: rel L2 vs fp32 torchvision %.4g (bf16 emulation %.4g)" % (H, W, B, xc, e_got, e_emu))
    assert tuple(got.shape) == (B, 2048) and got.dtype == torch.float32
    assert e_got <= 1.25 * e_emu + 0.01
    assert torch.equal(net(x), got)                                    # deterministic
    for i in sorted({0, B // 2, B - 1}):
        assert torch.equal(net(x[i:i + 1]), got[i:i + 1]), i           # independent of the batch it is in
    if xc == 1:
        assert torch.equal(net(x.repeat(1, 3, 1, 1)), got)
        assert torch.equal(net(x.cpu()), got)                          # CPU input is moved to the module's device


def test_trunk_chunks_large_batches(trunk, monkeypatch):
    from iris_b200 import resnet as R

    _, net = trunk
    x = torch.rand(5, 3, 97, 131, device=DEV, generator=torch.Generator(device=DEV).manual_seed(9))
    whole = net(x)
    per_image = _lib().call_i64("isx_resnet50_workspace_bytes", 1, 97, 131)
    monkeypatch.setattr(R, "WORKSPACE_BUDGET", 2 * per_image)
    assert net.chunk_size(5, 97, 131) == 2
    assert torch.equal(net(x), whole)


def test_gaze_estimator2_frames_to_unit_vectors(trunk):
    import iris_b200
    from oracle import resnet_oracle as O

    model, net = trunk
    torch.manual_seed(4)
    gaze = iris_b200.GazeEstimator2(extract_feature=True, resnet=net).to(DEV)
    frames = torch.rand(4, 1, 400, 640, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
    got = gaze(frames)

    def head(feats):
        y = gaze.model(feats)
        return y / y.norm(dim=1, keepdim=True)

    with torch.no_grad():
        ref = head(O.torchvision_features(model, frames))
        emu = head(O.resnet50_forward(model, frames, operand_dtype=torch.bfloat16))
    _, deg = iris_b200.angular_distance(got, ref)
    _, deg_emu = iris_b200.angular_distance(emu, ref)
    print("GazeEstimator2: max angle to fp32 torch %.4g deg (bf16 emulation %.4g deg)" % (float(deg.max()), float(deg_emu.max())))
    assert tuple(got.shape) == (4, 3)
    torch.testing.assert_close(got.norm(dim=1), torch.ones(4, device=DEV), rtol=1e-5, atol=1e-5)
    assert float(deg.max()) <= 1.25 * float(deg_emu.max()) + 0.1
    gaze.train()
    with pytest.raises(RuntimeError):
        gaze(frames)
    with pytest.raises(ValueError):
        iris_b200.GazeEstimator2(extract_feature=True)
