"""tcgen05 ConvTranspose3d kernel (csrc/convt3d.cu) against torch's fp32 conv_transpose3d (TF32 off)."""
import pytest
import torch
import torch.nn.functional as F

from genre_shapehd_b200 import ops_conv
import networks.networks as nets

from contextlib import contextmanager

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@contextmanager
def fp32_reference():
    """plain torch / cuDNN fp32 convolutions: custom kernels off, TF32 off"""
    old = ops_conv.ENABLED
    ops_conv.ENABLED = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        yield
    finally:
        ops_conv.ENABLED = old
        torch.backends.cudnn.allow_tf32 = True


def _tol():
    """max |err| / max |ref| allowed for one layer: 10-bit operand mantissa for the single-pass modes (fp32 accumulate);
    1e-4 for the 3xTF32 mode (north_star: values within 1e-4).  Measured for 3xTF32: 1e-6 .. 4e-5, growing with the number
    of MMA steps per output (3000 for Unet_3D.dec5) because the tensor core's fp32 accumulator truncates (~2^-25 of the
    partial sum per step); the operand split itself is good to 2^-21."""
    return 1e-4 if ops_conv.PRECISION in EXACT_MODES else 4e-3


EXACT_MODES = ("fp32x3", "f16x2")


@pytest.fixture(autouse=True, params=["f16", "tf32", "fp32x3", "f16x2"])
def _precision(request):
    """every test runs with the four operand modes of the tensor-core kernels: two single-pass ones (10-bit mantissa) and
    the two fp32-accurate operand splits (3xTF32 along K; fp16 hi/lo with separate accumulators)"""
    torch.backends.cudnn.allow_tf32 = True   # the custom kernels decline when reduced-mantissa convolutions are disallowed
    old, oldp = ops_conv.PRECISION, set(ops_conv.POLICY)
    ops_conv.PRECISION = request.param
    ops_conv.POLICY = set(ops_conv._all_policy)   # exercise every kernel, not only the ones routed by default
    yield
    ops_conv.PRECISION, ops_conv.POLICY = old, oldp
    torch.backends.cudnn.allow_tf32 = True


def _ref(x, m):
    torch.backends.cudnn.allow_tf32 = False
    try:
        return F.conv_transpose3d(x, m.weight, m.bias, stride=2, padding=m.padding)
    finally:
        torch.backends.cudnn.allow_tf32 = True


@pytest.mark.parametrize("k,cin,cout,b,d,h,w", [(4, 16, 4, 1, 1, 16, 16), (8, 16, 20, 1, 2, 16, 16), (8, 80, 20, 2, 4, 32, 32),
                                                 (4, 64, 32, 1, 3, 32, 32), (4, 128, 64, 2, 2, 16, 16), (8, 32, 40, 1, 2, 32, 16)])
def test_convt3d_vs_torch(k, cin, cout, b, d, h, w):
    torch.manual_seed(k * 1000 + cin + cout)
    m = nets.ConvTranspose3d(cin, cout, k, 2, k // 2 - 1).to(DEV)
    x = torch.randn(b, cin, d, h, w, device=DEV)
    with torch.no_grad():
        y = ops_conv.conv_transpose3d(x, m)
        assert y is not None, "layer should be covered by the custom kernel"
        ref = _ref(x, m)
    assert y.shape == ref.shape
    err = (y - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= _tol() * scale, "max err %g vs scale %g" % (err, scale)   # TF32 operands (10-bit mantissa)


@pytest.mark.parametrize("cin,cout,b,d,h,w", [(16, 20, 1, 2, 16, 16), (80, 20, 2, 3, 32, 32), (32, 7, 1, 1, 16, 32)])
def test_convt_k8_merged_parities_vs_separate_and_torch(cin, cout, b, d, h, w):
    """MODE 2 (four (y,x) parity classes in one N=80 MMA stream) against the per-class kernel and torch"""
    torch.manual_seed(cin + cout)
    m = nets.ConvTranspose3d(cin, cout, 8, 2, 3).to(DEV)
    x = torch.randn(b, cin, d, h, w, device=DEV)
    old = ops_conv.MERGE_PARITIES
    try:
        with torch.no_grad():
            ops_conv.MERGE_PARITIES = True
            ym = ops_conv.conv_transpose3d(x, m)
            ops_conv.MERGE_PARITIES = False
            ys = ops_conv.conv_transpose3d(x, m)
            ref = _ref(x, m)
    finally:
        ops_conv.MERGE_PARITIES = old
    assert ym is not None and ys is not None
    scale = ref.abs().max().item()
    assert (ym - ref).abs().max().item() <= _tol() * scale
    # same products, same fp32 accumulator; only the order of the K walk differs
    assert (ym - ys).abs().max().item() <= 1e-4 * scale


def test_blocked_layout_roundtrip():
    x = torch.randn(2, 24, 3, 16, 16, device=DEV)
    assert torch.equal(ops_conv.from_blocked(ops_conv.to_blocked(x), 2, 24), x)
    assert ops_conv.to_blocked(x, 8, torch.float16).shape == (6, 3, 16, 16, 8)


@pytest.mark.parametrize("group,dtype", [(4, None), (8, torch.float16)])
def test_layout_kernels_match_torch_permutes(group, dtype):
    """csrc/layout.cu against the torch permute formulation of the same layouts (bit-exact: pure moves / one rounding)"""
    torch.manual_seed(11)
    x = torch.randn(2, 16, 6, 10, 12, device=DEV)
    xc = x.cpu()
    assert torch.equal(ops_conv.to_blocked(x, group, dtype).cpu(), ops_conv.to_blocked(xc, group, dtype))
    x2 = torch.randn(3, 2, 4, 6, 8, device=DEV)
    assert torch.equal(ops_conv.space_to_depth_blocked(x2, group, dtype).cpu(),
                       ops_conv.space_to_depth_blocked(x2.cpu(), group, dtype))
    x4 = torch.randn(2, 3, 8, 4, 12, device=DEV)
    assert torch.equal(ops_conv.space_to_depth4_blocked(x4, group, dtype).cpu(),
                       ops_conv.space_to_depth4_blocked(x4.cpu(), group, dtype))
    x3 = torch.randn(2, 5, 4, 6, 8, device=DEV)           # 5 channels padded to 8 / 16 per sub-volume
    for cpad in (8, 16):
        assert torch.equal(ops_conv.space_to_depth_sources(x3, cpad, group, dtype).cpu(),
                           ops_conv.space_to_depth_sources(x3.cpu(), cpad, group, dtype))
    y = torch.randn(2 * 3, 5, 7, 9, 4, device=DEV)        # 5 groups = 20 padded channels, 18 real
    assert torch.equal(ops_conv.from_blocked(y, 2, 18).cpu(), ops_conv.from_blocked(y.cpu(), 2, 18))


def test_deconv_skip_fused_bn_leaky_vs_torch():
    torch.manual_seed(5)
    blk = nets.Deconv3d_skip(80, 20, 8, 2, 3, 0).to(DEV).eval()
    blk.net[1].running_mean.normal_(0, 0.1)
    blk.net[1].running_var.uniform_(0.5, 1.5)
    blk.net[1].weight.data.uniform_(0.5, 1.5)
    blk.net[1].bias.data.normal_(0, 0.1)
    x, s = torch.randn(1, 40, 2, 32, 32, device=DEV), torch.randn(1, 40, 2, 32, 32, device=DEV)
    with torch.no_grad():
        y = blk(x, s)
        with fp32_reference():
            ref = blk.net(torch.cat((x, s), 1))
    assert (y - ref).abs().max().item() <= _tol() * ref.abs().max().item()


def test_autograd_and_unsupported_shapes_fall_back(monkeypatch):
    m = nets.ConvTranspose3d(16, 4, 4, 2, 1).to(DEV)
    x = torch.randn(1, 16, 2, 16, 16, device=DEV, requires_grad=True)
    assert ops_conv.conv_transpose3d(x, m, None, 0.0) is None  # fused epilogues are inference-only
    monkeypatch.setattr(ops_conv, "TRAIN_FORWARD", False)
    assert ops_conv.conv_transpose3d(x, m) is None             # autograd with the training forward off: cuDNN path
    y = m(x)
    y.sum().backward()
    assert x.grad is not None
    with torch.no_grad():
        assert ops_conv.conv_transpose3d(torch.randn(1, 16, 2, 12, 12, device=DEV), m) is None   # W=12: no kernel


@pytest.mark.parametrize("cin,cout,b,d,h,w", [(2, 20, 1, 4, 32, 32), (2, 20, 2, 8, 64, 64), (4, 12, 1, 6, 32, 128),
                                                 (2, 20, 1, 4, 64, 128), (4, 7, 1, 8, 128, 64)])
def test_conv3d_k8s2_via_space_to_depth_vs_torch(cin, cout, b, d, h, w):
    torch.manual_seed(cin * 100 + cout + w)
    m = nets.Conv3d(cin, cout, 8, 2, 3).to(DEV)
    x = torch.randn(b, cin, d, h, w, device=DEV)
    with torch.no_grad():
        y = ops_conv.conv3d(x, m)
        assert y is not None
        with fp32_reference():
            ref = F.conv3d(x, m.weight, m.bias, stride=2, padding=3)
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() <= _tol() * ref.abs().max().item()


@pytest.mark.parametrize("shape", [(2, 2, 8, 64, 128), (1, 2, 16, 64, 64)], ids=["b2_d8_64x128", "b1_d16_64x64"])
def test_conv3d_k8s2_s4d_class_layout_of_each_precision(shape):
    """Unet_3D.enc1's 4x space-to-depth form: f16x2 puts the z class on blockIdx.y (MODE 2, N=80: its 2 x 160 accumulator
    columns would not fit), the other modes keep all 8 classes in N=160 (MODE 3)"""
    torch.manual_seed(13)
    m = nets.Conv3d(2, 20, 8, 2, 3).to(DEV)
    x = torch.randn(*shape, device=DEV)
    with torch.no_grad():
        y = ops_conv.conv3d(x, m)
        with fp32_reference():
            ref = F.conv3d(x, m.weight, m.bias, stride=2, padding=3)
    assert y is not None and (y - ref).abs().max().item() <= _tol() * ref.abs().max().item()


def test_conv_block_fused_bn_leaky_vs_torch():
    torch.manual_seed(11)
    blk = nets.Conv3d_block(2, 20, 8, 2, 3).to(DEV).eval()
    blk.net[1].running_mean.normal_(0, 0.1)
    blk.net[1].running_var.uniform_(0.5, 1.5)
    x = torch.rand(1, 2, 8, 64, 64, device=DEV)
    with torch.no_grad():
        y = blk(x)
        with fp32_reference():
            ref = blk.net(x)
    assert (y - ref).abs().max().item() <= _tol() * ref.abs().max().item()


def test_tf32_switch_selects_the_fp32_accurate_mode(monkeypatch):
    """torch.backends.cudnn.allow_tf32 = False asks for fp32 convolutions: the kernels answer with the 3xTF32 scheme
    (fp32-grade accuracy), or hand the layer back to cuDNN when GENRE_B200_CONV_EXACT=0"""
    torch.manual_seed(2)
    m = nets.ConvTranspose3d(32, 8, 4, 2, 1).to(DEV)
    x = torch.randn(1, 32, 2, 16, 16, device=DEV)
    with torch.no_grad():
        with fp32_reference():
            ref = F.conv_transpose3d(x, m.weight, m.bias, stride=2, padding=1)
        torch.backends.cudnn.allow_tf32 = False
        try:
            assert ops_conv._mode() == (ops_conv.PRECISION if ops_conv.PRECISION in EXACT_MODES else ops_conv.EXACT_IMPL)
            y = ops_conv.conv_transpose3d(x, m)
            monkeypatch.setattr(ops_conv, "EXACT_WHEN_TF32_OFF", False)
            assert ops_conv.conv_transpose3d(x, m) is None
        finally:
            torch.backends.cudnn.allow_tf32 = True
    assert y is not None and (y - ref).abs().max().item() <= 1e-4 * ref.abs().max().item()


@pytest.mark.parametrize("cin,b,d,h,w", [(8, 1, 3, 8, 8), (40, 2, 4, 16, 32), (32, 1, 5, 12, 20)])
def test_convt_one_output_channel_vs_torch(cin, b, d, h, w):
    ops_conv.POLICY = ops_conv.POLICY - {"convt_c1_tc"}      # this test is about the FP32-pipe kernel
    torch.manual_seed(cin + w)
    m = nets.ConvTranspose3d(cin, 1, 4, 2, 1).to(DEV)
    x = torch.randn(b, cin, d, h, w, device=DEV)
    with torch.no_grad():
        y = ops_conv.conv_transpose3d(x, m)
        assert y is not None
        with fp32_reference():
            ref = F.conv_transpose3d(x, m.weight, m.bias, stride=2, padding=1)
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() <= 1e-4 * max(1.0, ref.abs().max().item())   # plain fp32 FMAs


@pytest.mark.parametrize("chans,b,d,h,w,sigmoid", [((48,), 2, 3, 16, 32, False), ((32,), 1, 2, 32, 64, False), ((64,), 1, 2, 16, 16, True),
                                                    ((20, 20), 1, 4, 16, 16, False), ((24, 8), 2, 2, 32, 32, False)])
def test_convt_c1_tensor_core_vs_torch(chans, b, d, h, w, sigmoid):
    """MODE 4: ConvT(Cin -> 1) as 27 union taps x 8 output classes on the tensor cores; one or two (skip) sources, the
    20-channel ones arriving as blocked twins of a previous custom layer (zero-padded to the operand group size)"""
    if ops_conv.PRECISION in EXACT_MODES:
        pytest.skip("fp32 wanted: the 1-channel layer goes to the exact FP32-pipe kernel instead (test_dec6_two_source_path)")
    torch.manual_seed(sum(chans) + w)
    m = nets.ConvTranspose3d(sum(chans), 1, 4, 2, 1).to(DEV)
    xs = []
    for c in chans:
        t = torch.randn(b, c, d, h, w, device=DEV)
        if c % 8:   # give it the blocked fp32 twin a custom layer would have attached
            t = ops_conv.from_blocked(ops_conv.to_blocked(t, 4), b, c)
        xs.append(t)
    with torch.no_grad():
        y = ops_conv.convt_c1_tc(tuple(xs), m, sigmoid)
        assert y is not None
        with fp32_reference():
            ref = F.conv_transpose3d(torch.cat(xs, 1), m.weight, m.bias, stride=2, padding=1)
        if sigmoid:
            ref = torch.sigmoid(ref)
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() <= _tol() * max(1.0, ref.abs().max().item())


def test_dec6_two_source_path_vs_torch():
    ops_conv.POLICY = ops_conv.POLICY - {"convt_c1_tc"}
    torch.manual_seed(3)
    blk = nets.Deconv3d_skip(40, 1, 4, 2, 1, 0, is_activate=False).to(DEV).eval()
    x, s = torch.randn(1, 20, 4, 16, 16, device=DEV), torch.randn(1, 20, 4, 16, 16, device=DEV)
    with torch.no_grad():
        y = blk(x, s)
        with fp32_reference():
            ref = blk.net(torch.cat((x, s), 1))
    assert (y - ref).abs().max().item() <= 1e-4 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("cin,cout,b,d,h,w", [(16, 24, 1, 4, 32, 32), (64, 64, 1, 6, 64, 64), (20, 40, 2, 8, 64, 64),
                                              (40, 80, 1, 4, 32, 32), (64, 128, 1, 4, 32, 64)])
def test_conv3d_k4s2_parity_subvolumes_vs_torch(cin, cout, b, d, h, w, monkeypatch):
    monkeypatch.setattr(ops_conv, "K4S2_MIN_CIN", 8)   # exercise the kernel on small layers too
    torch.manual_seed(cin + cout + w)
    m = nets.Conv3d(cin, cout, 4, 2, 1, bias=(cout % 3 != 0)).to(DEV)
    x = torch.randn(b, cin, d, h, w, device=DEV)
    with torch.no_grad():
        y = ops_conv.conv3d(x, m)
        assert y is not None
        with fp32_reference():
            ref = F.conv3d(x, m.weight, m.bias, stride=2, padding=1)
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() <= _tol() * ref.abs().max().item()


def test_default_policy_routes():
    ops_conv.POLICY = set(ops_conv._default_policy)
    with torch.no_grad():
        assert ops_conv.conv_transpose3d(torch.randn(1, 80, 2, 32, 32, device=DEV), nets.ConvTranspose3d(80, 20, 8, 2, 3).to(DEV)) is not None
        assert ops_conv.conv3d(torch.rand(1, 2, 4, 64, 64, device=DEV), nets.Conv3d(2, 20, 8, 2, 3).to(DEV)) is not None
        assert ops_conv.conv_transpose3d(torch.randn(1, 64, 2, 32, 32, device=DEV), nets.ConvTranspose3d(64, 32, 4, 2, 1).to(DEV)) is not None
        assert ops_conv.conv3d(torch.randn(1, 64, 4, 64, 64, device=DEV), nets.Conv3d(64, 64, 4, 2, 1).to(DEV)) is not None
        assert ops_conv.conv_transpose3d(torch.randn(1, 32, 2, 16, 16, device=DEV), nets.ConvTranspose3d(32, 1, 4, 2, 1).to(DEV)) is not None
        # FP32-pipe 1-channel kernel: not beyond C1_MAX_CIN input channels (cuDNN is faster there)
        assert not ops_conv._convt_c1_supported(64, (2, 16, 16), nets.ConvTranspose3d(64, 1, 4, 2, 1).to(DEV))


def test_cached_blocked_twin_is_dropped_after_inplace_update():
    m = nets.ConvTranspose3d(16, 8, 4, 2, 1).to(DEV)
    with torch.no_grad():
        y = ops_conv.conv_transpose3d(torch.randn(1, 16, 2, 16, 16, device=DEV), m)
        assert ops_conv._has_blocked(y)
        torch.relu_(y)
        assert not ops_conv._has_blocked(y)      # the blocked copy still holds pre-activation values


@pytest.mark.parametrize("name", ["VoxelDecoder", "VoxelGenerator", "VoxelDiscriminator"])
def test_fused_sequential_matches_module_by_module(name):
    """conv -> BN -> ReLU runs as one kernel (FusedSequential) and must equal the plain nn.Sequential walk"""
    torch.manual_seed(21)
    net = getattr(nets, name)().to(DEV).eval()
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm3d):
            m.running_mean.normal_(0, 0.05)
            m.running_var.uniform_(0.8, 1.2)
    x = {"VoxelDecoder": torch.randn(1, 200, device=DEV), "VoxelGenerator": torch.randn(1, 200, 1, 1, 1, device=DEV),
         "VoxelDiscriminator": torch.rand(1, 1, 128, 128, 128, device=DEV)}[name]
    with torch.no_grad():
        y = net(x)
        with fp32_reference():
            ref = net(x)
    tol = 2e-4 if ops_conv.PRECISION in EXACT_MODES else 2e-2
    # the critic has no normalisation layers and its scalar output is a heavily cancelling sum: floor the scale
    assert (y - ref).abs().max().item() <= tol * max(1e-2, ref.abs().max().item())


@pytest.mark.parametrize("kind,cin,cout", [("convt", 1280, 320), ("convt", 200, 512)])
def test_degenerate_convolutions_as_gemm(kind, cin, cout):
    """1^3 -> 4^3 transposed convolutions routed to one cuBLAS GEMM: forward and gradients against the cuDNN module"""
    torch.manual_seed(cin)
    if kind == "convt":
        m, x = nets.ConvTranspose3d(cin, cout, 4, 1, 0).to(DEV), torch.randn(3, cin, 1, 1, 1, device=DEV, requires_grad=True)
    else:
        m, x = nets.Conv3d(cin, cout, 4, 1, 0).to(DEV), torch.randn(3, cin, 4, 4, 4, device=DEV, requires_grad=True)
    y = ops_conv.gemm_conv(x, m)
    assert y is not None
    with fp32_reference():
        ref = torch.nn.ConvTranspose3d.forward(m, x) if kind == "convt" else torch.nn.Conv3d.forward(m, x)
    assert y.shape == ref.shape and (y - ref).abs().max().item() <= 1e-4 * max(1.0, ref.abs().max().item())
    g = torch.randn_like(ref)
    gx, gw = torch.autograd.grad(y, (x, m.weight), g)
    with fp32_reference():
        rx, rw = torch.autograd.grad(ref, (x, m.weight), g)
    assert (gx - rx).abs().max().item() <= 1e-4 * max(1.0, rx.abs().max().item())
    assert (gw - rw).abs().max().item() <= 1e-4 * max(1.0, rw.abs().max().item())


@pytest.mark.parametrize("kind,cin,cout,k,shape", [("conv", 2, 20, 8, (2, 8, 64, 64)), ("conv", 24, 40, 4, (2, 8, 64, 64)),
                                                   ("convt", 80, 20, 8, (1, 2, 32, 32)), ("convt", 64, 32, 4, (2, 2, 16, 16))])
def test_training_forward_on_custom_kernel_backward_on_cudnn(kind, cin, cout, k, shape):
    """under autograd the conv-only forward runs on the custom kernel and the backward is aten::convolution_backward:
    outputs and all three gradients against the plain cuDNN module"""
    torch.manual_seed(cin + cout)
    b, d, h, w = shape
    m = (nets.Conv3d(cin, cout, k, 2, k // 2 - 1) if kind == "conv" else nets.ConvTranspose3d(cin, cout, k, 2, k // 2 - 1)).to(DEV)
    x = torch.randn(b, cin, d, h, w, device=DEV, requires_grad=True)
    y = m(x)
    assert y.grad_fn is not None and "ConvForward" in type(y.grad_fn).__name__
    g = torch.randn_like(y)
    gx, gw, gb = torch.autograd.grad(y, (x, m.weight, m.bias), g)
    with fp32_reference():
        ref = m(x)
        rx, rw, rb = torch.autograd.grad(ref, (x, m.weight, m.bias), g)
    assert (y - ref).abs().max().item() <= _tol() * ref.abs().max().item()
    for a, r in ((gx, rx), (gw, rw), (gb, rb)):     # backward itself ran on cuDNN with TF32 allowed
        assert (a - r).abs().max().item() <= 4e-3 * r.abs().max().item()


def test_training_forward_supports_double_backward():
    """WGAN-GP differentiates the critic's input gradient (wgangp.py:144-164): the wrapper's backward is built from
    differentiable aten ops"""
    torch.manual_seed(9)
    m = nets.Conv3d(64, 64, 4, 2, 1, bias=False).to(DEV)
    x = torch.randn(1, 64, 4, 32, 32, device=DEV, requires_grad=True)
    y = m(x)
    (gx,) = torch.autograd.grad(y.sum(), x, create_graph=True)
    pen = (gx.norm() - 1) ** 2
    pen.backward()
    assert m.weight.grad is not None and torch.isfinite(m.weight.grad).all() and m.weight.grad.abs().sum().item() > 0


@pytest.mark.parametrize("cin,b,d,h,w", [(40, 2, 3, 16, 64), (32, 1, 4, 8, 16), (8, 3, 2, 24, 20)])
def test_convt_one_channel_training_path_vs_cudnn(cin, b, d, h, w):
    """ConvT(Cin -> 1) under autograd: exact-fp32 forward, custom dgrad and (deterministic) wgrad against cuDNN fp32"""
    torch.manual_seed(cin + w)
    m = nets.ConvTranspose3d(cin, 1, 4, 2, 1).to(DEV)
    x = torch.randn(b, cin, d, h, w, device=DEV, requires_grad=True)
    y = m(x)
    assert "ConvTC1Train" in type(y.grad_fn).__name__
    g = torch.randn_like(y)
    gx, gw, gb = torch.autograd.grad(y, (x, m.weight, m.bias), g, retain_graph=True)
    gw2 = torch.autograd.grad(y, m.weight, g)[0]
    assert torch.equal(gw, gw2)                              # fixed-order reduction: bitwise reproducible
    with fp32_reference():
        ref = m(x)
        rx, rw, rb = torch.autograd.grad(ref, (x, m.weight, m.bias), g)
    for a, r in ((y, ref), (gx, rx), (gw, rw), (gb, rb)):
        assert a.shape == r.shape and (a - r).abs().max().item() <= 2e-5 * max(1.0, r.abs().max().item())


@pytest.mark.parametrize("cin,cout,b,d,h,w", [(2, 20, 2, 4, 32, 64), (1, 7, 1, 6, 16, 20), (2, 20, 1, 2, 64, 128)])
def test_conv_k8s2_weight_gradient_vs_cudnn(cin, cout, b, d, h, w):
    """csrc/convt_c1_wgrad.cu conv_k8s2_wgrad (Unet_3D.enc1's dW) against cuDNN fp32; bitwise reproducible"""
    torch.manual_seed(cout + w)
    x = torch.randn(b, cin, d, h, w, device=DEV)
    wt = torch.randn(cout, cin, 8, 8, 8, device=DEV, requires_grad=True)
    with fp32_reference():
        y = F.conv3d(x, wt, None, stride=2, padding=3)
        g = torch.randn_like(y)
        (ref,) = torch.autograd.grad(y, wt, g)
    from genre_shapehd_b200 import _lib
    nbytes = _lib.load().genre_b200_conv_k8s2_wgrad_workspace_bytes()
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    outs = []
    for _ in range(2):
        dw = torch.empty_like(wt)
        _lib.call("genre_b200_conv_k8s2_wgrad", x.data_ptr(), g.data_ptr(), b, cin, cout, d, h, w, dw.data_ptr(), ws.data_ptr(),
                  nbytes, _lib.stream_ptr(x))
        outs.append(dw)
    assert torch.equal(outs[0], outs[1])
    assert (outs[0] - ref).abs().max().item() <= 2e-5 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("cin,cout,b,d,h,w", [(1, 64, 2, 4, 64, 128), (2, 40, 1, 6, 32, 32), (1, 64, 1, 2, 32, 64)])
def test_conv3d_k4s2_few_input_channels_vs_torch(cin, cout, b, d, h, w):
    """VoxelDiscriminator main.0 (Conv3d 1 -> 64, k4 s2 p1 + LeakyReLU) as 3 taps over the space-to-depth input"""
    torch.manual_seed(cin + cout + w)
    m = nets.Conv3d(cin, cout, 4, 2, 1, bias=False).to(DEV)
    x = torch.rand(b, cin, d, h, w, device=DEV)
    with torch.no_grad():
        y = ops_conv.conv3d(x, m, None, 0.2)
        assert y is not None
        with fp32_reference():
            ref = F.leaky_relu(F.conv3d(x, m.weight, None, stride=2, padding=1), 0.2)
    assert y.shape == ref.shape and (y - ref).abs().max().item() <= _tol() * ref.abs().max().item()
    xg = x.clone().requires_grad_(True)                      # and under autograd (WGAN-GP feeds a leaf that needs grad)
    yg = m(xg)
    assert "ConvForward" in type(yg.grad_fn).__name__
    (gx,) = torch.autograd.grad(yg.sum(), xg)
    with fp32_reference():
        (rx,) = torch.autograd.grad(m(xg).sum(), xg)
    assert (gx - rx).abs().max().item() <= 4e-3 * rx.abs().max().item()


@pytest.mark.parametrize("cin,cout,shape", [(64, 64, (1, 4, 32, 32)), (1, 64, (2, 4, 32, 64))])
def test_gradient_penalty_double_backward_vs_cudnn(cin, cout, shape):
    """WGAN-GP's penalty (wgangp.py:144-164) through the custom forward / _ConvInputGrad nodes against plain autograd"""
    torch.manual_seed(cin + 31)
    b, d, h, w = shape
    m = nets.Conv3d(cin, cout, 4, 2, 1, bias=False).to(DEV)
    x = torch.rand(b, cin, d, h, w, device=DEV, requires_grad=True)
    proj = torch.randn(1, cout, d // 2, h // 2, w // 2, device=DEV)

    def penalty():     # a smooth nonlinearity: LeakyReLU's kink would turn rounding-level sign flips into O(1) differences
        out = (torch.tanh(m(x)) * proj).sum()
        (gx,) = torch.autograd.grad(out, x, create_graph=True)
        return ((gx.reshape(b, -1).norm(2, dim=1) - 1) ** 2).mean()
    pen = penalty()
    (gw,) = torch.autograd.grad(pen, m.weight)
    with fp32_reference():
        ref = penalty()
        (rw,) = torch.autograd.grad(ref, m.weight)
    assert abs(pen.item() - ref.item()) <= 2e-2 * max(1e-3, abs(ref.item()))
    assert (gw - rw).abs().max().item() <= 2e-2 * rw.abs().max().item()


def test_double_backward_keeps_tiny_grad_of_grads():
    """ADVICE r1: the grad-of-grad convolution of _ConvInputGrad must not run on fp16 operands: penalty gradients of 1e-5..1e-7
    are subnormal / flushed in fp16.  The double backward of sum(gx * v) with |v| ~ 1e-6 equals the forward convolution of v;
    relative error must stay at operand-rounding level whatever the magnitude."""
    torch.manual_seed(77)
    m = nets.Conv3d(64, 64, 4, 2, 1, bias=False).to(DEV)
    x = torch.rand(1, 64, 4, 32, 32, device=DEV, requires_grad=True)
    v = torch.randn_like(x) * 1e-6
    out = m(x)
    gy = torch.randn_like(out).requires_grad_(True)
    (gx,) = torch.autograd.grad(out, x, gy, create_graph=True)
    (ggy,) = torch.autograd.grad((gx * v).sum(), gy)             # = conv3d(v, W): tiny values through the custom forward kernel
    with fp32_reference():
        ref = F.conv3d(v, m.weight, None, 2, 1)
    assert ref.abs().max().item() < 1e-4
    assert (ggy - ref).abs().max().item() <= _tol() * ref.abs().max().item()


@pytest.mark.skipif(not ops_conv.TC_BACKWARD, reason="tensor-core input gradients switched off (GENRE_B200_CONV_TC_BACKWARD=0)")
@pytest.mark.parametrize("kind,cin,cout,shape", [("convt", 80, 20, (1, 2, 32, 32)), ("conv", 2, 20, (1, 4, 64, 64))])
def test_tensor_core_input_gradients_of_the_k8_layers(kind, cin, cout, shape):
    torch.manual_seed(cin)
    b, d, h, w = shape
    m = (nets.ConvTranspose3d(cin, cout, 8, 2, 3) if kind == "convt" else nets.Conv3d(cin, cout, 8, 2, 3)).to(DEV)
    x = torch.randn(b, cin, d, h, w, device=DEV, requires_grad=True)
    with fp32_reference():
        y = m(x)
        gy = torch.randn_like(y)
        (ref,) = torch.autograd.grad(y, x, gy)
    dx = (ops_conv.dgrad_convt_k8s2 if kind == "convt" else ops_conv.dgrad_conv_k8s2)(gy, m)
    assert dx is not None and dx.shape == ref.shape
    assert (dx - ref).abs().max().item() <= 4e-3 * ref.abs().max().item()


@pytest.mark.skipif(not ops_conv.BN_TRAIN, reason="fused training BatchNorm switched off (GENRE_B200_BN_TRAIN=0)")
@pytest.mark.parametrize("act", [None, "relu", "leaky"])
@pytest.mark.parametrize("shape", [(4, 20, 8, 16, 16), (2, 5, 3, 4, 4), (3, 64, 4, 8, 8)])
def test_bn_act_train_forward_backward_vs_torch(shape, act):
    torch.manual_seed(shape[1])
    bn, ref_bn = torch.nn.BatchNorm3d(shape[1]).to(DEV).train(), torch.nn.BatchNorm3d(shape[1]).to(DEV).train()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5); bn.bias.normal_(0, 0.2)
        ref_bn.load_state_dict(bn.state_dict())
    a = {None: None, "relu": torch.nn.ReLU(), "leaky": torch.nn.LeakyReLU(0.01)}[act]
    x = (torch.randn(*shape, device=DEV) * 2 + 0.7).requires_grad_(True)
    xr = x.detach().clone().requires_grad_(True)
    y = ops_conv.bn_act_train(x, bn, a)
    assert y is not None
    yr = ref_bn(xr) if a is None else a(ref_bn(xr))
    g = torch.randn_like(yr)
    y.backward(g); yr.backward(g)
    assert (y - yr).abs().max().item() <= 1e-4 * max(1.0, yr.abs().max().item())
    assert (x.grad - xr.grad).abs().max().item() <= 1e-4 * max(1.0, xr.grad.abs().max().item())
    assert (bn.weight.grad - ref_bn.weight.grad).abs().max().item() <= 1e-3 * max(1.0, ref_bn.weight.grad.abs().max().item())
    assert (bn.bias.grad - ref_bn.bias.grad).abs().max().item() <= 1e-3 * max(1.0, ref_bn.bias.grad.abs().max().item())
    assert torch.allclose(bn.running_mean, ref_bn.running_mean, atol=1e-5) and torch.allclose(bn.running_var, ref_bn.running_var, rtol=1e-4)
    assert int(bn.num_batches_tracked) == int(ref_bn.num_batches_tracked) == 1


def test_split2_f16_layout_kernel_is_the_hi_lo_decomposition():
    """csrc/layout.cu split2_f16_kernel against its definition in torch: hi = fp16(a), lo' = fp16((a - hi) * 2^11), parts stacked
    along the channel-group axis, odd group counts zero-padded; hi + lo' / 2^11 reproduces a to ~2^-22"""
    torch.manual_seed(3)
    t = torch.randn(6, 5, 16, 16, 4, device=DEV) * torch.logspace(-6, 2, 5, device=DEV).view(1, 5, 1, 1, 1)
    out = ops_conv._split2(t)
    assert out.shape == (6, 6, 16, 16, 8) and out.dtype == torch.float16
    pad = torch.cat((t, torch.zeros_like(t[:, :1])), dim=1)                           # 6 groups of 4 -> 3 groups of 8
    x8 = torch.cat((pad[:, 0::2], pad[:, 1::2]), dim=-1)
    hi = x8.half()
    lo = ((x8 - hi.float()) * 2048.0).half()
    assert torch.equal(out[:, :3], hi) and torch.equal(out[:, 3:], lo)
    rec = out[:, :3].float() + out[:, 3:].float() / 2048.0
    assert ((rec - x8).abs() <= 2.0 ** -21 * x8.abs() + 2e-11).all()


def test_f16x2_matches_fp32_much_closer_than_single_pass():
    """the point of the mode: the dominant refiner layer (ConvT 80 -> 20, k8: 1000 K steps per output) within 2e-5 of fp32
    where single-pass fp16 operands sit at ~1e-3"""
    torch.manual_seed(21)
    m = nets.ConvTranspose3d(80, 20, 8, 2, 3).to(DEV)
    x = torch.randn(2, 80, 4, 32, 32, device=DEV)
    with torch.no_grad():
        ref = _ref(x, m)
        errs = {}
        for mode in ("f16", "f16x2", "fp32x3"):
            with ops_conv.precision(mode):
                y = ops_conv.conv_transpose3d(x, m)
            assert y is not None
            errs[mode] = ((y - ref).abs().max() / ref.abs().max()).item()
    assert errs["f16x2"] <= 2e-5 and errs["f16x2"] < errs["f16"] / 20, errs


def test_direct_hi_lo_conversions_equal_convert_then_split():
    """csrc/layout.cu with group code 16 (NCDHW -> hi/lo operand in ONE pass) against the two-pass route (fp32 blocked, then
    split2_f16): bit-identical for the plain, 2x space-to-depth, parity-sub-volume and 4x space-to-depth layouts"""
    torch.manual_seed(13)
    x = torch.randn(2, 16, 6, 16, 24, device=DEV) * 3
    assert torch.equal(ops_conv.to_blocked(x, 16, torch.float16), ops_conv._split2(ops_conv.to_blocked(x, 4)))
    x2 = torch.randn(3, 2, 4, 6, 8, device=DEV)
    for cpad in (0, 32):
        assert torch.equal(ops_conv.space_to_depth_blocked(x2, 16, torch.float16, cpad),
                           ops_conv._split2(ops_conv.space_to_depth_blocked(x2, 4, None, cpad)))
    x3 = torch.randn(2, 20, 4, 6, 8, device=DEV)
    assert torch.equal(ops_conv.space_to_depth_sources(x3, 32, 16, torch.float16),
                       ops_conv._split2(ops_conv.space_to_depth_sources(x3, 32, 4, None)))
    x4 = torch.randn(2, 2, 8, 4, 12, device=DEV)
    assert torch.equal(ops_conv.space_to_depth4_blocked(x4, 16, torch.float16),
                       ops_conv._split2(ops_conv.space_to_depth4_blocked(x4, 4, None)))
