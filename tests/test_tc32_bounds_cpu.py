"""The error bound and bias thresholds of the tc32 precision, fixed on the CPU emulation of the kernel's arithmetic
(tests/tc32_ref.py) before the GPU tests (test_gpu_tc32_numerics.py) hold the kernels to them.

For every GEMM shape and magnitude class the GPU tests use, the emulated correct scheme (promotion every K step) must meet
tc32_ref.TAU on max |d| / B and tc32_ref.BIAS_MAX on the mean signed relative error, and the stand-ins for broken kernels
must miss them by >= 3x: a main product that is never promoted (tcgen05.mma truncates every addition: a bias that grows
with K) fails the bias check, a missing correction product (an 11-bit operand) fails the bound.  The split itself is
checked over the whole fp16 range, subnormals to 65504, and at its saturation edge."""
import numpy as np
import pytest

from tests import tc32_ref as R

SEP = 3.0      # every threshold must separate correct from broken by this factor


def _pos(rng, shape):
    return rng.random(shape, dtype=np.float32) + np.float32(0.05)


# (label, K, emulation of the correct kernel): the K of the bias cases of the GPU tests, all-positive data
BIAS_CASES = [
    ("flat 1x1 cin 4096", 4096, dict(group=1)),
    ("halo 3x3 cin 512", 4608, dict(group=1, corr_bufs=2)),     # four issuers: two correction accumulators
    ("dcn cin 256", 2304, dict(group=1)),
]


@pytest.mark.parametrize("label,K,kw", BIAS_CASES, ids=[c[0] for c in BIAS_CASES])
def test_emulated_scheme_meets_bound_and_bias(label, K, kw):
    rng = np.random.default_rng(K)
    x, w = _pos(rng, (256, K)), _pos(rng, (K, 32))
    ref, B = R.gemm_ref_bound(x, w)
    good = R.emulate_tc32(x, w, **kw)
    r, b = R.bound_ratio(good, ref, B), R.mean_bias(good, ref)
    assert r * SEP <= R.TAU, (label, r)
    assert abs(b) * SEP <= R.BIAS_MAX, (label, b)
    # never promoted: the truncation bias compounds over the K steps
    nopromo = R.emulate_tc32(x, w, **dict(kw, group=None))
    assert abs(R.mean_bias(nopromo, ref)) >= SEP * R.BIAS_MAX, label
    # one correction product missing: ~11 significant bits in one operand
    for drop in ("a2b", "ab2"):
        bad = R.emulate_tc32(x, w, **dict(kw, drop=drop))
        assert R.bound_ratio(bad, ref, B) >= SEP * R.TAU, (label, drop)


def test_emulated_correlation_chain_meets_bound_and_bias():
    """the tc32 correlation never promotes: one truncating chain over K = C = 256 (16 MMAs) stays inside the bound and the
    correlation's bias threshold (which is set from the B200 measurement: the hardware drifts ~3.5x more than this model)"""
    rng = np.random.default_rng(256)
    x, w = _pos(rng, (256, 256)), _pos(rng, (256, 32))
    ref, B = R.gemm_ref_bound(x, w)
    got = R.emulate_tc32(x, w, group=None)
    assert R.bound_ratio(got, ref, B) * SEP <= R.TAU
    assert abs(R.mean_bias(got, ref)) * SEP <= R.CORR_BIAS_MAX
    for drop in ("a2b", "ab2"):
        assert R.bound_ratio(R.emulate_tc32(x, w, group=None, drop=drop), ref, B) >= SEP * R.TAU


MAGNITUDES = [2.0 ** -24, 2.0 ** -14, 2.0 ** -6, 1.0, 2.0 ** 10, 6.0e4]


@pytest.mark.parametrize("mag", MAGNITUDES)
def test_emulated_scheme_meets_bound_across_magnitudes(mag):
    """inputs from fp16 subnormals to the top of the fp16 range, unit weights; zero-mean data (cancellation)"""
    rng = np.random.default_rng(int(np.log2(mag) + 100))
    K = 576
    x = (rng.standard_normal((128, K)) * mag).astype(np.float32)
    x = np.clip(x, -R.F16_MAX, R.F16_MAX)
    w = (rng.standard_normal((K, 32)) / np.sqrt(K)).astype(np.float32)
    ref, B = R.gemm_ref_bound(x, w)
    r = R.bound_ratio(R.emulate_tc32(x, w), ref, B)
    assert r * SEP <= R.TAU, r
    if mag >= 2.0 ** -6:       # the correction products carry the accuracy wherever the operands are normal fp16 numbers
        assert R.bound_ratio(R.emulate_tc32(x, w, drop="a2b"), ref, B) >= SEP * R.TAU


def test_emulated_scheme_meets_bound_with_mixed_scales():
    """per-channel input scales 1e-4 .. 1e4 and weights around 1e-6 (below the fp16 normal range: carried by B2 alone)"""
    rng = np.random.default_rng(7)
    K = 576
    scale = np.logspace(-4, 4, K).astype(np.float32)
    rng.shuffle(scale)
    x = (rng.standard_normal((128, K)) * scale).astype(np.float32)
    for wmag in (1.0, 1e-6):
        w = (rng.standard_normal((K, 48)) * wmag / np.sqrt(K)).astype(np.float32)
        ref, B = R.gemm_ref_bound(x, w)
        assert R.bound_ratio(R.emulate_tc32(x, w), ref, B) * SEP <= R.TAU, wmag


# ------------------------------------------------------------------ the operand split over the fp16 range
def test_split_from_subnormals_to_fp16_max():
    """v = A + 2^-11 A2 to 2^-22 |v| + 2^-36 for every |v| <= 65504: ~22 bits for normal values, an absolute 2^-36 below
    2^-14 (A2 is then an fp16 subnormal), no saturation of A2 anywhere (|v - A| is at most half an fp16 ulp of v)"""
    rng = np.random.default_rng(3)
    mag = np.exp2(rng.uniform(-40, np.log2(65504.0), 1 << 17))
    v = (mag * rng.choice([-1.0, 1.0], mag.size)).astype(np.float32)
    edges = np.array([0.0, 2.0 ** -36, 2.0 ** -25, 2.0 ** -24, 3 * 2.0 ** -24, 2.0 ** -14 - 2.0 ** -24, 2.0 ** -14,
                      np.nextafter(np.float32(2.0 ** -14), np.float32(1)), 1.0 / 3, 2048.0 + 1.0, 32767.9,
                      65503.0, 65504.0], np.float32)
    v = np.concatenate([v, edges, -edges])
    v = v[np.abs(v) <= 65504.0]
    hi, lo = R.split16(v)
    assert np.all(np.isfinite(hi)) and np.all(np.abs(lo) <= 2.0 ** 15)
    err = np.abs(hi.astype(np.float64) + lo.astype(np.float64) / 2048.0 - v.astype(np.float64))
    lim = 2.0 ** -22 * np.abs(v.astype(np.float64)) + 2.0 ** -36
    assert np.all(err <= lim), float((err / lim).max())
    # the absolute term is needed: below 2^-14 the relative error grows
    small = (np.abs(v) < 2.0 ** -20) & (v != 0)
    assert float((err[small] / np.abs(v[small])).max()) > 2.0 ** -21
    hi, lo = R.split16(np.array([65504.0, -65504.0], np.float32))
    assert list(hi) == [65504.0, -65504.0] and list(lo) == [0.0, 0.0]


def test_split_saturates_above_fp16_max():
    """what the kernels flag (|v| > 65504 or NaN): the main plane saturates to +-65504 and the value is lost"""
    v = np.array([65505.0, 65519.0, 7.0e4, -7.0e4, 1e7], np.float32)
    hi, lo = R.split16(v)
    assert np.all(np.abs(hi) == 65504.0) and np.all(np.isfinite(lo))
    rec = hi.astype(np.float64) + lo.astype(np.float64) / 2048.0
    assert abs(rec[2] - 7.0e4) > 1000.0 and abs(rec[4] - 1e7) > 1e6
    assert not np.any(np.abs(v) <= 65504.0)          # the kernels' test: !(|v| <= 65504) -- also true for NaN
