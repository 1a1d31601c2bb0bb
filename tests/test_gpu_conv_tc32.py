"""GPU parity of the fp32-parity tensor-core convolution (vps_conv2d_tc32: every operand split into two fp16 planes,
v = fp16(v) + 2^-11 fp16(2^11 (v - fp16(v))), three products per K slab) vs fp64 convolution on the CPU, over the layer
shapes of the model.  Tolerance: 2e-5 of the output scale -- fp32-class (the CUDA-core fp32 kernel is held to 1e-4 in
test_gpu_conv.py), 100x below what one bf16 pass gives (2e-3).  The elementwise error bound, the truncation bias, the
fp16 range edges, the saturation counter and the rarer epilogue paths are tested in test_gpu_tc32_numerics.py."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

TOL = 2e-5


def _nhwc(t, c_align=8):
    n, c, h, w = t.shape
    cs = (c + c_align - 1) // c_align * c_align
    buf = torch.zeros(n, h, w, cs, dtype=torch.float32)
    buf[..., :c] = t.permute(0, 2, 3, 1).float()
    return buf


@pytest.fixture()
def tc32():
    from vps_b200 import ops
    old = ops.F32_TC[0]
    ops.F32_TC[0] = True
    yield ops
    ops.F32_TC[0] = old


CASES = [
    # n, cin, cout, h, w, k, stride, pad
    (1, 64, 64, 16, 32, 3, 1, 1),
    (2, 128, 256, 24, 40, 3, 1, 1),
    (1, 256, 64, 32, 32, 1, 1, 0),
    (1, 64, 128, 33, 47, 3, 2, 1),
    (1, 128, 512, 20, 28, 1, 2, 0),
    (1, 473, 256, 16, 24, 3, 1, 1),      # ragged cin: TMA OOB zero fill on channels, partial last K chunk
    (1, 64, 2, 16, 32, 3, 1, 1),         # cout 2 -> N = 16
    (1, 128, 128, 24, 24, 5, 2, 2),      # FlowNet 5x5 s2
    (3, 256, 256, 14, 14, 3, 1, 1),      # mask-head shape (batch of RoIs)
    (1, 192, 1024, 1, 300, 1, 1, 0),     # Linear as 1x1 over a row of "pixels"
    (1, 1026, 2, 8, 16, 3, 1, 1),
    (1, 194, 2, 32, 48, 3, 1, 1),
    (1, 16, 2, 40, 56, 3, 1, 1),
    (1, 12, 64, 32, 64, 7, 2, 3),        # thin stem without s2d: flat mode, 49 taps
    (1, 48, 32, 20, 36, 3, 1, 1),
    (1, 3, 64, 30, 44, 3, 1, 1),         # cin 3: one K8 / one K16 slab
    (1, 82, 16, 40, 64, 3, 1, 1),        # FlowNetFusion conv0-like
    (1, 256, 256, 128, 256, 3, 1, 1),    # N = 256 halo layer, two tiles per CTA
    (1, 256, 256, 120, 248, 3, 1, 1),    # ragged tiles
    (1, 12, 64, 40, 72, 4, 1, 2),        # the s2d stem's 4x4 stride-1 form
]


@pytest.mark.parametrize("case", CASES)
def test_conv_tc32_vs_fp64(cuda, tc32, case):
    ops = tc32
    n, cin, cout, h, w, k, s, p = case
    g = torch.Generator().manual_seed(hash(case) % (2 ** 31))
    x = torch.randn(n, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
    b = torch.randn(cout, generator=g)
    ref = F.leaky_relu(F.conv2d(x.double(), wt.double(), b.double(), stride=s, padding=p), 0.1)
    pk = ops.PackedConv(wt.to(cuda), b.to(cuda))
    xd = _nhwc(x).to(cuda)[..., :cin]
    oh, ow = ref.shape[2:]
    y = torch.full((n, oh, ow, cout), float("nan"), dtype=torch.float32, device=cuda)
    assert ops.f32_tc_ok(xd)
    ops.conv2d(xd, pk, y, stride=s, pad=p, act=ops.ACT_LRELU, slope=0.1, use_tc=True)
    torch.cuda.synchronize()
    got = y.cpu().permute(0, 3, 1, 2).double()
    err = (got - ref).abs().max().item()
    assert err <= TOL * max(1.0, ref.abs().max().item()), "max err %g" % err


def test_conv_tc32_residual_and_slice(cuda, tc32):
    """fp32 output into a channel slice of a concat buffer, fp32 residual added before ReLU (resnet.py:236-258)."""
    ops = tc32
    g = torch.Generator().manual_seed(7)
    n, cin, cout, h, w = 1, 64, 256, 37, 53
    x = torch.randn(n, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, 1, 1, generator=g) / cin ** 0.5
    res = torch.randn(n, cout, h, w, generator=g)
    ref = F.relu(F.conv2d(x.double(), wt.double()) + res.double())
    pk = ops.PackedConv(wt.to(cuda))
    buf = torch.full((n, h, w, cout + 64), 7.0, dtype=torch.float32, device=cuda)
    ops.conv2d(_nhwc(x).to(cuda), pk, buf[..., 32:32 + cout], act=ops.ACT_RELU, res=_nhwc(res).to(cuda), use_tc=True)
    torch.cuda.synchronize()
    got = buf[..., 32:32 + cout].cpu().permute(0, 3, 1, 2).double()
    assert (buf[..., :32] == 7.0).all() and (buf[..., 32 + cout:] == 7.0).all()
    err = (got - ref).abs().max().item()
    assert err <= TOL * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("k", [4, 2])
def test_deconv_tc32_phases(cuda, tc32, k):
    """ConvTranspose2d(4,2,1) / (2,2) as four stride-phase problems sharing one tc32 launch and one packed buffer."""
    ops = tc32
    from vps_b200.layers import deconv2x2_s2, deconv4x4_s2
    g = torch.Generator().manual_seed(11 + k)
    cin, cout, h, w = 128, 64, 12, 20
    x = torch.randn(1, cin, h, w, generator=g)
    wt = torch.randn(cin, cout, k, k, generator=g) / (cin * 4) ** 0.5
    b = torch.randn(cout, generator=g)
    ref = F.leaky_relu(F.conv_transpose2d(x.double(), wt.double(), b.double(), stride=2, padding=1 if k == 4 else 0), 0.1)
    layer = (deconv4x4_s2 if k == 4 else deconv2x2_s2)(wt.to(cuda), b.to(cuda))
    y = torch.full((1, 2 * h, 2 * w, cout), float("nan"), dtype=torch.float32, device=cuda)
    layer(_nhwc(x).to(cuda), y, act=ops.ACT_LRELU)
    torch.cuda.synchronize()
    got = y.cpu().permute(0, 3, 1, 2).double()
    err = (got - ref).abs().max().item()
    assert err <= TOL * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("cin,h,w", [(3, 33, 47), (12, 32, 64), (6, 17, 30)])
def test_stem_7x7s2_tc32(cuda, tc32, cin, h, w):
    ops = tc32
    from vps_b200.layers import StemConv7x7s2
    g = torch.Generator().manual_seed(100 + cin)
    x = torch.randn(1, cin, h, w, generator=g)
    wt = torch.randn(64, cin, 7, 7, generator=g) / (cin * 49) ** 0.5
    b = torch.randn(64, generator=g)
    ref = F.relu(F.conv2d(x.double(), wt.double(), b.double(), stride=2, padding=3))
    stem = StemConv7x7s2(wt.to(cuda), b.to(cuda), act=ops.ACT_RELU)
    y = stem(_nhwc(x).to(cuda)[..., :cin])
    torch.cuda.synchronize()
    got = y.cpu().permute(0, 3, 1, 2).double()
    assert got.shape == ref.shape
    err = (got - ref).abs().max().item()
    assert err <= TOL * max(1.0, ref.abs().max().item()), err


def test_linear_tc32(cuda, tc32):
    ops = tc32
    from vps_b200.layers import Linear
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1000, 12544, generator=g)
    wt = torch.randn(1024, 12544, generator=g) / 112.0
    b = torch.randn(1024, generator=g)
    ref = F.relu(F.linear(x.double(), wt.double(), b.double()))
    fc = Linear(wt.to(cuda), b.to(cuda), act=ops.ACT_RELU)
    y = fc(x.to(cuda))
    torch.cuda.synchronize()
    err = (y.cpu().double() - ref).abs().max().item()
    assert err <= TOL * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("cin,h,w,cout", [(194, 24, 40, 2), (1026, 8, 16, 2), (16, 33, 47, 2), (64, 16, 16, 3)])
def test_thin_3x3_as_tap_major_1x1(cuda, tc32, cin, h, w, cout):
    """predict_flow layers (3x3, cout <= 3): 1x1 tensor-core convolution over tap-major output channels + vps_tap_gather3x3,
    written into a channel slice of a wider concat buffer like the FlowNet decoders do"""
    ops = tc32
    from vps_b200.layers import Conv, empty_nhwc
    g = torch.Generator().manual_seed(7 + cin)
    x = torch.randn(1, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, 3, 3, generator=g) / (cin * 9) ** 0.5
    b = torch.randn(cout, generator=g)
    ref = F.leaky_relu(F.conv2d(x.double(), wt.double(), b.double(), padding=1), 0.1) * 0.5
    layer = Conv(wt.to(cuda), b.to(cuda), stride=1, pad=1, act=ops.ACT_LRELU)
    assert layer.pk_tap is not None
    xd = empty_nhwc(1, h, w, cin, torch.float32, cuda)
    xd.copy_(x.permute(0, 2, 3, 1).to(cuda))
    cat = torch.full((1, h, w, 24), float("nan"), dtype=torch.float32, device=cuda)
    layer(xd, cat[..., 5:5 + cout], out_scale=0.5)   # first call packs the weights
    n0 = ops.launch_count()
    layer(xd, cat[..., 5:5 + cout], out_scale=0.5)
    assert ops.launch_count() - n0 == 2              # the 1x1 tensor-core GEMM + the gather
    torch.cuda.synchronize()
    got = cat[..., 5:5 + cout].cpu().permute(0, 3, 1, 2).double()
    assert torch.isnan(cat[..., :5]).all() and torch.isnan(cat[..., 5 + cout:]).all()
    err = (got - ref).abs().max().item()
    assert err <= TOL * max(1.0, ref.abs().max().item()), err
