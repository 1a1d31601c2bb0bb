"""The tc32 kernels (vps_conv2d_tc32, the fused DCN, the three-pass correlation) held to the elementwise error bound and
the bias threshold of tests/tc32_ref.py -- fixed on the CPU emulation by test_tc32_bounds_cpu.py -- where kernels go wrong:

  * bias: all-positive data and long K (truncating tensor-core accumulation; the promotion every K step must hold the mean
    signed relative error to ~1e-7, an unpromoted chain drifts by ~5e-6);
  * magnitudes: inputs from fp16 subnormals (2^-24) to the top of the fp16 range, per-channel scales 1e-4 .. 1e4, weights
    around 1e-6 folded in through PackedConv(scale=...), on the halo, flat, stride-2 and transposed-convolution paths;
  * the saturation counter: every site that increments it, 65504 itself does not, reset clears it, outputs away from a
    saturated input keep the bound;
  * epilogues and tiling: sigmoid, residual after the activation, out_scale, unaligned slices / bf16 output / bf16 and
    unaligned residuals (the scalar epilogue), odd and > 128 output widths, ragged stride-2 tiles over a batch, a stride-phase
    launch into a slice -- NaN sentinels around every output, every launch repeated and bit-identical;
  * the detector: a frame that saturates raises VpsError and leaves the detector (and a ClipRunner with prefetch) usable.

The bound has no floor on the output scale: |got - ref| <= TAU * B / 2^-21 elementwise."""
import pytest
import torch
import torch.nn.functional as F

from tests import tc32_ref as R

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture()
def ops(cuda):
    from vps_b200 import ops as _ops
    old = _ops.F32_TC[0]
    _ops.F32_TC[0] = True
    _ops.tc32_overflow(reset=True)
    yield _ops
    _ops.F32_TC[0] = old
    _ops.tc32_overflow(reset=True)


def _nhwc(t, c_align=8, off=0):
    """NCHW cpu -> NHWC device view [.., off:off + c] of a buffer with an aligned pixel stride"""
    n, c, h, w = t.shape
    cs = (off + c + c_align - 1) // c_align * c_align
    buf = torch.zeros(n, h, w, cs, dtype=torch.float32)
    buf[..., off:off + c] = t.permute(0, 2, 3, 1).float()
    return buf.to(DEV)[..., off:off + c]


def _sentinel_out(n, h, w, c, off=0, extra=5, dtype=torch.float32):
    """NaN-filled buffer with `off` channels before and >= `extra` after the output slice"""
    cs = (off + c + extra + 7) // 8 * 8
    buf = torch.full((n, h, w, cs), float("nan"), dtype=dtype, device=DEV)
    return buf, buf[..., off:off + c]


def _nchw(y):
    return y.float().cpu().permute(0, 3, 1, 2).double()


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).clone()


def _twice(launch, buf):
    """run `launch` twice into `buf` (which starts with NaN sentinels): the second result must be bit-identical"""
    launch()
    torch.cuda.synchronize()
    first = _bits(buf)
    launch()
    torch.cuda.synchronize()
    assert torch.equal(first, _bits(buf)), "repeated launch not bit-identical"


def _sentinels_intact(buf, off, c):
    assert torch.isnan(buf[..., :off].float()).all() and torch.isnan(buf[..., off + c:].float()).all(), "neighbouring channels written"


def _report(name, r, b=None):
    print("tc32 numerics %-40s max|d|/B*2^-21 %.3e%s" % (name, r, "" if b is None else "  mean bias %+.3e" % b))


# ------------------------------------------------------------------ bias: all-positive data, long K
def _pos(g, *shape):
    return torch.rand(*shape, generator=g) + 0.05


@pytest.mark.parametrize("kind", ["flat_1x1_cin4096", "halo_3x3_cin512", "dcn_cin256", "corr_c256"])
def test_bias_positive_long_k(ops, kind):
    g = torch.Generator().manual_seed(1234)
    H, W = 16, 32
    if kind.startswith("flat") or kind.startswith("halo"):
        k, cin = (1, 4096) if kind.startswith("flat") else (3, 512)
        x = _pos(g, 1, cin, H, W)
        w = _pos(g, 32, cin, k, k) / (cin * k * k)
        ref, B = R.conv_ref_bound(x, w, 1, k // 2)
        y = torch.full((1, H, W, 32), float("nan"), device=DEV)
        ops.conv2d(_nhwc(x), ops.PackedConv(w.to(DEV)), y, stride=1, pad=k // 2, use_tc=True)
    elif kind.startswith("dcn"):
        cin = 256
        x = _pos(g, 1, cin, H, W)
        off = torch.round((torch.rand(1, 18, H, W, generator=g) - 0.5) * 6 * 64) / 64     # exact bilinear weights in fp32
        w = _pos(g, 32, cin, 3, 3) / (cin * 9)
        ref, B = R.dcn_ref_bound(x, off, w)
        y = torch.full((1, H, W, 32), float("nan"), device=DEV)
        ops.deform_conv_tc32(_nhwc(x), _nhwc(off), ops.PackedConv(w.to(DEV)), y)
    else:
        C, md, s2 = 256, 20, 2
        f1, f2 = _pos(g, 1, C, 24, 40), _pos(g, 1, C, 24, 40)
        ref, B = R.corr_ref_bound(f1, f2, md, s2)
        _, y = _sentinel_out(1, 24, 40, (2 * (md // s2) + 1) ** 2, off=8)
        ops.correlation(_nhwc(f1), _nhwc(f2), y, md, md, 1, s2, impl="tc32")
    torch.cuda.synchronize()
    got = _nchw(y)
    r, b = R.bound_ratio(got, ref, B), R.mean_bias(got, ref)
    _report("bias " + kind, r, b)
    assert ops.tc32_overflow() == 0
    assert r <= R.TAU, r
    assert abs(b) <= (R.CORR_BIAS_MAX if kind.startswith("corr") else R.BIAS_MAX), b


# ------------------------------------------------------------------ magnitude sweep
SHAPES = {
    # n, cin, cout, h, w, k, stride, pad
    "halo": (1, 64, 64, 20, 36, 3, 1, 1),
    "flat": (1, 96, 48, 16, 40, 1, 1, 0),
    "stride2": (1, 64, 64, 33, 47, 3, 2, 1),
}
MAGS = [2.0 ** -24, 2.0 ** -14, 2.0 ** -6, 1.0, 2.0 ** 10, 6.0e4]


def _conv_case(ops, x, w, stride, pad, scale=None, name=""):
    """launch the tc32 conv of fp32 x / w (folded with `scale` in fp32 exactly as the packer does) and check the bound"""
    wd = w.to(DEV)
    pk = ops.PackedConv(wd, None, scale=scale.to(DEV) if scale is not None else None)
    w_eff = w if scale is None else (w.float() * scale.float().view(-1, 1, 1, 1))      # fp32 product, as pack_weights_tc32
    ref, B = R.conv_ref_bound(x, w_eff, stride, pad)
    y = torch.full((x.shape[0], ref.shape[2], ref.shape[3], w.shape[0]), float("nan"), device=DEV)
    ops.conv2d(_nhwc(x), pk, y, stride=stride, pad=pad, use_tc=True)
    torch.cuda.synchronize()
    r = R.bound_ratio(_nchw(y), ref, B)
    _report(name, r)
    assert ops.tc32_overflow() == 0, name
    assert r <= R.TAU, (name, r)


@pytest.mark.parametrize("mag", MAGS, ids=["2^-24", "2^-14", "2^-6", "1", "2^10", "6e4"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_magnitude_sweep_conv(ops, shape, mag):
    n, cin, cout, h, w, k, s, p = SHAPES[shape]
    g = torch.Generator().manual_seed(int(mag * 1e9) % 1000 + len(shape))
    x = (torch.randn(n, cin, h, w, generator=g) * mag).clamp(-65504.0, 65504.0)
    wt = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
    _conv_case(ops, x, wt, s, p, name="%s x%g" % (shape, mag))


@pytest.mark.parametrize("shape", list(SHAPES))
def test_per_channel_scales_and_folded_tiny_weights(ops, shape):
    """input channels scaled 1e-4 .. 1e4; weights ~1 folded with a per-cout scale ~1e-6 (B below the fp16 normal range)"""
    n, cin, cout, h, w, k, s, p = SHAPES[shape]
    g = torch.Generator().manual_seed(99 + len(shape))
    cscale = torch.logspace(-4, 4, cin)[torch.randperm(cin, generator=g)]
    x = torch.randn(n, cin, h, w, generator=g) * cscale.view(1, -1, 1, 1)
    wt = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
    _conv_case(ops, x, wt, s, p, name="%s channel scales" % shape)
    fold = (torch.rand(cout, generator=g) + 0.5) * 1e-6
    x1 = torch.randn(n, cin, h, w, generator=g)
    _conv_case(ops, x1, wt, s, p, scale=fold, name="%s folded 1e-6 scale" % shape)


@pytest.mark.parametrize("mag", [2.0 ** -24, 1.0, 6.0e4], ids=["2^-24", "1", "6e4"])
def test_magnitude_sweep_deconv_phases(ops, mag):
    from vps_b200.layers import deconv4x4_s2
    g = torch.Generator().manual_seed(31)
    cin, cout, h, w = 64, 32, 12, 20
    x = (torch.randn(1, cin, h, w, generator=g) * mag).clamp(-65504.0, 65504.0)
    wt = torch.randn(cin, cout, 4, 4, generator=g) / (cin * 4) ** 0.5
    ref, B = R.deconv_ref_bound(x, wt, 2, 1)
    y = torch.full((1, 2 * h, 2 * w, cout), float("nan"), device=DEV)
    deconv4x4_s2(wt.to(DEV), None)(_nhwc(x), y)
    torch.cuda.synchronize()
    r = R.bound_ratio(_nchw(y), ref, B)
    _report("deconv x%g" % mag, r)
    assert ops.tc32_overflow() == 0
    assert r <= R.TAU, r


# ------------------------------------------------------------------ the saturation counter
def test_overflow_counter_conv_activation(ops):
    """one activation of 7e4 (and one NaN) fires the converter warps' count; 65504 exactly does not; reset clears it; the
    outputs whose receptive field misses the saturated pixel keep the bound"""
    g = torch.Generator().manual_seed(5)
    cin, cout, h, w = 64, 32, 20, 36
    x = torch.randn(1, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, 3, 3, generator=g) / (cin * 9) ** 0.5
    pk = ops.PackedConv(wt.to(DEV))
    pk.tc32()
    assert ops.tc32_overflow() == 0
    y = torch.full((1, h, w, cout), float("nan"), device=DEV)

    x_edge = x.clone()
    x_edge[0, 3, 4, 5] = 65504.0
    x_edge[0, 7, 9, 9] = -65504.0
    ops.conv2d(_nhwc(x_edge), pk, y, stride=1, pad=1, use_tc=True)
    assert ops.tc32_overflow(reset=False) == 0
    ref, B = R.conv_ref_bound(x_edge, wt, 1, 1)
    assert R.bound_ratio(_nchw(y), ref, B) <= R.TAU

    for bad in (7.0e4, float("nan")):
        xb = x.clone()
        xb[0, 3, 4, 5] = bad
        ops.conv2d(_nhwc(xb), pk, y, stride=1, pad=1, use_tc=True)
        assert ops.tc32_overflow(reset=False) > 0, bad
        assert ops.tc32_overflow(reset=True) > 0
        assert ops.tc32_overflow(reset=False) == 0
        m = torch.zeros(1, 1, h, w)
        m[0, 0, 4, 5] = 1.0
        hit = F.conv2d(m, torch.ones(1, 1, 3, 3), padding=1)[0, 0] > 0       # outputs that read the saturated pixel
        xc = x.clone()
        xc[0, 3, 4, 5] = 0.0
        ref, B = R.conv_ref_bound(xc, wt, 1, 1)
        got = _nchw(y)
        keep = ~hit.view(1, 1, h, w).expand_as(got)
        assert R.bound_ratio(got[keep], ref[keep], B[keep]) <= R.TAU, bad


def test_overflow_counter_weight_packing(ops):
    g = torch.Generator().manual_seed(6)
    wt = torch.randn(32, 64, 3, 3, generator=g)
    wt[5, 7, 1, 1] = 65504.0
    ops.PackedConv(wt.to(DEV)).tc32()
    assert ops.tc32_overflow() == 0
    wt[5, 7, 1, 1] = 7.0e4
    ops.PackedConv(wt.to(DEV)).tc32()
    assert ops.tc32_overflow() > 0
    assert ops.tc32_overflow() == 0
    # a per-cout scale can push a weight over the range as well: the product is what is split
    wt[5, 7, 1, 1] = 1.0e3
    ops.PackedConv(wt.to(DEV), scale=torch.full((32,), 100.0, device=DEV)).tc32()
    assert ops.tc32_overflow() > 0


def test_overflow_counter_dcn_sample(ops):
    """the sampling warps count a bilinear sample above 65504 (integer offsets: the sample is the pixel itself)"""
    g = torch.Generator().manual_seed(7)
    cin, cout, H, W = 64, 32, 12, 20
    x = torch.randn(1, cin, H, W, generator=g)
    off = torch.zeros(1, 18, H, W)
    wt = torch.randn(cout, cin, 3, 3, generator=g) / (cin * 9) ** 0.5
    pk = ops.PackedConv(wt.to(DEV))
    pk.tc32()
    y = torch.full((1, H, W, cout), float("nan"), device=DEV)
    ops.deform_conv_tc32(_nhwc(x), _nhwc(off), pk, y)
    assert ops.tc32_overflow() == 0
    ref, B = R.dcn_ref_bound(x, off, wt)
    assert R.bound_ratio(_nchw(y), ref, B) <= R.TAU
    x[0, 9, 6, 10] = 1.0e5
    ops.deform_conv_tc32(_nhwc(x), _nhwc(off), pk, y)
    assert ops.tc32_overflow() > 0
    assert ops.tc32_overflow() == 0


def test_overflow_counter_correlation(ops):
    g = torch.Generator().manual_seed(8)
    C, md, s2, H, W = 64, 20, 2, 16, 24
    f1, f2 = torch.randn(1, C, H, W, generator=g), torch.randn(1, C, H, W, generator=g)
    _, out = _sentinel_out(1, H, W, (2 * (md // s2) + 1) ** 2, off=8)
    ops.correlation(_nhwc(f1), _nhwc(f2), out, md, md, 1, s2, impl="tc32")
    assert ops.tc32_overflow() == 0
    ref, B = R.corr_ref_bound(f1, f2, md, s2)
    torch.cuda.synchronize()
    assert R.bound_ratio(_nchw(out), ref, B) <= R.TAU
    for t in (f1, f2):
        t[0, 3, 5, 6] = 1.0e5
        ops.correlation(_nhwc(f1), _nhwc(f2), out, md, md, 1, s2, impl="tc32")
        assert ops.tc32_overflow() > 0
        t[0, 3, 5, 6] = 0.0


# ------------------------------------------------------------------ epilogues and tiling
def _epi_case(ops, *, n=1, cin=64, cout=64, h=20, w=36, k=3, s=1, p=1, act=None, res=None, res_after_act=False,
              out_scale=1.0, off=0, out_dtype=torch.float32, res_dtype=torch.float32, res_off=0, bias=True, seed=0):
    act = ops.ACT_NONE if act is None else act
    g = torch.Generator().manual_seed(seed + cout)
    x = torch.randn(n, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
    b = torch.randn(cout, generator=g) if bias else None
    conv, B = R.conv_ref_bound(x, wt, s, p)
    oh, ow = conv.shape[2:]
    pre = conv + (b.double().view(1, -1, 1, 1) if bias else 0)
    r_t = None
    rd = None
    if res:
        r_t = torch.randn(n, cout, oh, ow, generator=g).to(res_dtype).float()
        rd = _nhwc(r_t, off=res_off).to(res_dtype) if res_dtype == torch.float32 else _nhwc(r_t).to(res_dtype)
        if res_dtype != torch.float32:
            rd = rd[..., :cout]
    z = pre + (r_t.double() if res and not res_after_act else 0)
    lip = 1.0
    if act == ops.ACT_RELU:
        z = z.clamp_min(0)
    elif act == ops.ACT_LRELU:
        z = F.leaky_relu(z, 0.1)
    elif act == ops.ACT_SIGMOID:
        z, lip = torch.sigmoid(z), 0.25
    ref = z * out_scale + (r_t.double() if res and res_after_act else 0)
    # accumulation bound through the 1-Lipschitz (sigmoid: 1/4) activation and the scale, plus the fp32 roundings of the
    # epilogue's bias / residual / scale operations, __expf, and the bf16 rounding of a bf16 output
    tol = R.TAU / R.U * B * lip * abs(out_scale) + 4 * R.OUT_ROUND * (ref.abs() + pre.abs() * abs(out_scale) +
                                                                          (r_t.double().abs() if res else 0))
    if act == ops.ACT_SIGMOID:
        tol = tol + 2.0 ** -20
    if out_dtype == torch.bfloat16:
        tol = tol + 2.0 ** -8 * ref.abs()
    buf, y = _sentinel_out(n, oh, ow, cout, off=off, dtype=out_dtype)
    pk = ops.PackedConv(wt.to(DEV), b.to(DEV) if bias else None)
    xd = _nhwc(x)
    _twice(lambda: ops.conv2d(xd, pk, y, stride=s, pad=p, act=act, slope=0.1, res=rd, res_after_act=res_after_act,
                              out_scale=out_scale, use_tc=True), buf)
    _sentinels_intact(buf, off, cout)
    got = _nchw(y)
    assert not torch.isnan(got).any()
    ratio = float(((got - ref).abs() / tol).max())
    assert ratio <= 1.0, ratio
    assert ops.tc32_overflow() == 0


EPI_CASES = {
    "sigmoid": dict(act="SIGMOID"),
    "relu_res_after_act_scale": dict(act="RELU", res=True, res_after_act=True, out_scale=0.5),
    "lrelu_res_scale": dict(act="LRELU", res=True, out_scale=-2.0),
    "slice_off2_scalar": dict(act="LRELU", off=2),
    "slice_off4_tma": dict(act="LRELU", off=4, cout=60),
    "bf16_out": dict(act="RELU", out_dtype=torch.bfloat16),
    "bf16_res": dict(act="RELU", res=True, res_dtype=torch.bfloat16),
    "res_misaligned_fp32": dict(act="RELU", res=True, res_off=1),
    "sigmoid_scalar_slice": dict(act="SIGMOID", off=3, out_scale=0.25),
}


@pytest.mark.parametrize("case", list(EPI_CASES))
def test_epilogue_paths(ops, case):
    kw = dict(EPI_CASES[case])
    kw["act"] = getattr(ops, "ACT_" + kw["act"])
    _epi_case(ops, **kw)


@pytest.mark.parametrize("cout", [15, 19, 45, 96, 144, 160, 208, 384])
@pytest.mark.parametrize("k", [1, 3])
def test_output_widths(ops, cout, k):
    """odd widths (partial 32-channel boxes), > 128 channels (several N tiles), cout_pad / 16 odd above 128 (144, 208: no N
    tile the TMA-store epilogue can write)"""
    _epi_case(ops, cout=cout, cin=96, h=12, w=40, k=k, p=k // 2, act=ops.ACT_LRELU, seed=k)


def test_batch_ragged_stride2(ops):
    _epi_case(ops, n=3, cin=64, cout=96, h=37, w=53, k=3, s=2, p=1, act=ops.ACT_RELU)
    _epi_case(ops, n=3, cin=40, cout=48, h=29, w=61, k=1, s=2, p=0, act=ops.ACT_NONE, seed=2)


@pytest.mark.parametrize("off", [4, 2])
def test_deconv_phases_bias_scale_into_slice(ops, off):
    """one four-phase launch (strided output views) with bias and out_scale into a channel slice of a concat buffer"""
    from vps_b200.layers import deconv4x4_s2
    g = torch.Generator().manual_seed(40 + off)
    cin, cout, h, w = 64, 36, 11, 19
    x = torch.randn(1, cin, h, w, generator=g)
    wt = torch.randn(cin, cout, 4, 4, generator=g) / (cin * 4) ** 0.5
    b = torch.randn(cout, generator=g)
    conv, B = R.deconv_ref_bound(x, wt, 2, 1)
    pre = conv + b.double().view(1, -1, 1, 1)
    ref = F.leaky_relu(pre, 0.1) * 0.5
    tol = R.TAU / R.U * B * 0.5 + 4 * R.OUT_ROUND * (ref.abs() + pre.abs())
    layer = deconv4x4_s2(wt.to(DEV), b.to(DEV))
    buf, y = _sentinel_out(1, 2 * h, 2 * w, cout, off=off)
    xd = _nhwc(x)
    _twice(lambda: layer(xd, y, act=ops.ACT_LRELU, out_scale=0.5), buf)
    _sentinels_intact(buf, off, cout)
    got = _nchw(y)
    assert float(((got - ref).abs() / tol).max()) <= 1.0
    assert ops.tc32_overflow() == 0


# ------------------------------------------------------------------ detector: a saturating frame
def test_detector_overflow_raises_and_recovers(ops):
    """simple_test raises VpsError for a frame whose normalised values exceed 65504; afterwards the same detector, called
    directly and through ClipRunner with prefetch, gives a fresh detector's results"""
    from tests.e2e_util import build_models, make_pair, meta
    from vps_b200.runner import ClipRunner
    _, det = build_models("C", 0, "tc32", DEV)
    _, fresh = build_models("C", 0, "tc32", DEV)
    H, W = 64, 128
    img, ref = make_pair(H, W)
    bad = img.clone()
    bad[..., 20:24, 40:44] = 1.0e6
    img, ref, bad = img.to(DEV), ref.to(DEV), bad.to(DEV)

    def labels(r):
        return (r[2]["panoptic_outputs"].cpu().clone(), r[2]["fcn_outputs"].cpu().clone(),
                r[2]["panoptic_det_obj_ids"].cpu().clone())

    fresh.reset_tracker()
    want = labels(fresh.simple_test(img, [meta(10001, H, W)], ref_img=[ref]))
    det.reset_tracker()
    with pytest.raises(ops.VpsError):
        det.simple_test(bad, [meta(10001, H, W)], ref_img=[ref])
    assert ops.tc32_overflow(reset=False) == 0
    got = labels(det.simple_test(img, [meta(10001, H, W)], ref_img=[ref]))
    assert all(torch.equal(a, b) for a, b in zip(got, want))

    # prefetch: the next pair's static part is enqueued before the saturating pair raises
    with pytest.raises(ops.VpsError):
        for _ in ClipRunner(det, DEV).run([(bad, ref), (img, ref)], [meta(10001, H, W), meta(10002, H, W)], resident=True):
            pass
    assert not det._pf_queue
    res = [labels(r) for r in ClipRunner(det, DEV).run([(img, ref)], [meta(10001, H, W)], resident=True)]
    assert len(res) == 1 and all(torch.equal(a, b) for a, b in zip(res[0], want))
    assert ops.tc32_overflow() == 0
