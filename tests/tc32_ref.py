"""Reference arithmetic of the tc32 precision (conv_tc32.cu, the fused DCN and the three-pass correlation of corr_tc.cu),
shared by test_tc32_bounds_cpu.py and test_gpu_tc32_numerics.py.

* fp64 references and the elementwise error bound the kernels are held to:

      B = 2^-21 * op(|x|, |w|)  +  2^-36 * (op(|x|, 1) + op(1, |w|))  +  2^-23 * |ref|

  The first term is the split's ~22 significant bits per operand (and the truncating tensor-core accumulation of the
  promoted scheme), the middle one the absolute error 2^-36 of an operand below 2^-14 (its A2 plane is an fp16 subnormal),
  the last one the fp32 rounding of the output.  A result passes with |got - ref| <= tau * B / 2^-21, i.e.
  bound_ratio() <= tau: no floor on the output scale, so small outputs are checked as tightly as large ones.

* emulate_tc32(): a numpy model of the kernel's arithmetic -- saturating fp16 split, K16 MMAs that add their exact sum
  into an fp32 accumulator with round-toward-zero, main-product chains of 2 * group MMAs promoted to a round-to-nearest
  fp32 sum, the correction products truncation-accumulated over the whole tile and added once times 2^-11.  group=None
  (never promote) and drop="a2b" / "ab2" (one correction product missing) are the broken kernels the thresholds of the
  tests must reject.
"""
import numpy as np
import torch
import torch.nn.functional as F

U = 2.0 ** -21            # relative error per product of the split scheme
ABS_SUB = 2.0 ** -36      # absolute error of an operand below 2^-14
OUT_ROUND = 2.0 ** -23    # fp32 rounding of the output
F16_MAX = 65504.0
LO_SCALE = 2048.0

# Thresholds of the tests (test_tc32_bounds_cpu.py checks that they separate the emulated correct scheme from the broken
# ones by >= 3x at the shapes and data test_gpu_tc32_numerics.py runs).
TAU = 2e-6                # max(|got - ref| / B) * 2^-21
BIAS_MAX = 1e-6           # |mean signed relative error| on all-positive data, long K
# The correlation never promotes (one truncating chain over K = C <= 256).  On a B200 its drift at C = 256 is -1.2e-6,
# ~3.5x what the emulation gives (-3.5e-7): the threshold is the measured value with some margin, not an emulated one.
CORR_BIAS_MAX = 2e-6


# ------------------------------------------------------------------ metrics
def bound_ratio(got, ref, bound):
    """max |got - ref| / bound * 2^-21 (comparable with TAU); NaN anywhere in got gives inf"""
    got, ref, bound = (torch.as_tensor(t).double() for t in (got, ref, bound))
    if torch.isnan(got).any():
        return float("inf")
    d = (got - ref).abs()
    return float((d / bound.clamp_min(1e-300)).max()) * U


def mean_bias(got, ref):
    """mean signed relative error (got - ref) / |ref| over the nonzero references"""
    got, ref = torch.as_tensor(got).double(), torch.as_tensor(ref).double()
    m = ref != 0
    return float(((got - ref)[m] / ref[m].abs()).mean())


def _bound(s_abs, s_x, s_w, ref):
    return U * s_abs + ABS_SUB * (s_x + s_w) + OUT_ROUND * ref.abs()


# ------------------------------------------------------------------ fp64 references + bounds
def conv_ref_bound(x, w, stride=1, padding=0):
    """x NCHW, w OIHW (fp32 values): fp64 conv2d and its bound B"""
    x, w = x.double(), w.double()
    ref = F.conv2d(x, w, None, stride, padding)
    s_abs = F.conv2d(x.abs(), w.abs(), None, stride, padding)
    s_x = F.conv2d(x.abs(), torch.ones_like(w), None, stride, padding)
    s_w = F.conv2d(torch.ones_like(x), w.abs(), None, stride, padding)
    return ref, _bound(s_abs, s_x, s_w, ref)


def deconv_ref_bound(x, w, stride, padding):
    """x NCHW, w IOHW: fp64 conv_transpose2d and its bound B"""
    x, w = x.double(), w.double()
    ref = F.conv_transpose2d(x, w, None, stride, padding)
    s_abs = F.conv_transpose2d(x.abs(), w.abs(), None, stride, padding)
    s_x = F.conv_transpose2d(x.abs(), torch.ones_like(w), None, stride, padding)
    s_w = F.conv_transpose2d(torch.ones_like(x), w.abs(), None, stride, padding)
    return ref, _bound(s_abs, s_x, s_w, ref)


def deform_cols64(x, offset):
    """fp64 DCNv1 columns [B, C, 9, H, W] of a 3x3 / stride 1 / pad 1 kernel (deform_conv_cuda_kernel.cu:189-242 in fp64:
    corner taps outside the image contribute 0, samples outside (-1, H) x (-1, W) are 0)"""
    x, offset = x.double(), offset.double()
    B, C, H, W = x.shape
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    cols = torch.zeros(B, C, 9, H, W, dtype=torch.float64)
    for k in range(9):
        h = ys[None] - 1 + k // 3 + offset[:, 2 * k]
        w = xs[None] - 1 + k % 3 + offset[:, 2 * k + 1]
        inside = (h > -1) & (w > -1) & (h < H) & (w < W)
        hl, wl = torch.floor(h), torch.floor(w)
        lh, lw = h - hl, w - wl
        hl, wl = hl.long(), wl.long()
        for b in range(B):
            acc = torch.zeros(C, H, W, dtype=torch.float64)
            for hi, wi, wt in ((hl[b], wl[b], (1 - lh[b]) * (1 - lw[b])), (hl[b], wl[b] + 1, (1 - lh[b]) * lw[b]),
                               (hl[b] + 1, wl[b], lh[b] * (1 - lw[b])), (hl[b] + 1, wl[b] + 1, lh[b] * lw[b])):
                ok = inside[b] & (hi >= 0) & (hi <= H - 1) & (wi >= 0) & (wi <= W - 1)
                v = x[b][:, hi.clamp(0, H - 1), wi.clamp(0, W - 1)]
                acc += v * (wt * ok)
            cols[b, :, k] = acc
    return cols


def dcn_ref_bound(x, offset, w):
    """fp64 deformable convolution (3x3, pad 1) and its bound over the fp64 samples of |x| (>= |samples|)"""
    cols = deform_cols64(x, offset)
    cabs = deform_cols64(x.abs(), offset)
    B, C, _, H, W = cols.shape
    wm = w.double().reshape(w.shape[0], C * 9)
    mm = lambda m, c: torch.einsum("ok,bkp->bop", m, c.reshape(B, C * 9, H * W)).reshape(B, -1, H, W)
    ref = mm(wm, cols)
    ones = deform_cols64(torch.ones_like(x[:, :1]), offset).expand(B, C, 9, H, W)
    return ref, _bound(mm(wm.abs(), cabs), mm(torch.ones_like(wm), cabs), mm(wm.abs(), ones), ref)


def corr_ref_bound(f1, f2, max_disp, stride2):
    """fp64 FlowNet correlation (kernel 1, stride1 1, pad = max_disp) [B, D*D, H, W] and its bound"""
    f1, f2 = f1.double(), f2.double()
    B, C, H, W = f1.shape
    R = max_disp // stride2
    D = 2 * R + 1
    p2 = F.pad(f2, (max_disp,) * 4)
    p2a = F.pad(f2.abs(), (max_disp,) * 4)
    p2o = F.pad(torch.ones_like(f2), (max_disp,) * 4)
    outs = [torch.zeros(B, D * D, H, W, dtype=torch.float64) for _ in range(4)]
    for tj in range(-R, R + 1):
        for ti in range(-R, R + 1):
            y0, x0 = max_disp + tj * stride2, max_disp + ti * stride2
            k = (tj + R) * D + (ti + R)
            sl = (slice(None), slice(None), slice(y0, y0 + H), slice(x0, x0 + W))
            outs[0][:, k] = (f1 * p2[sl]).sum(1) / C
            outs[1][:, k] = (f1.abs() * p2a[sl]).sum(1) / C
            outs[2][:, k] = (f1.abs() * p2o[sl]).sum(1) / C
            outs[3][:, k] = p2a[sl].sum(1) / C
    ref = outs[0]
    return ref, _bound(outs[1], outs[2], outs[3], ref)


# ------------------------------------------------------------------ emulation of the kernel's arithmetic
def split16(v):
    """the saturating operand split: (A, A2) as fp32 arrays of fp16 values, v = A + 2^-11 A2"""
    v = np.asarray(v, np.float32)
    hi = np.clip(v, -F16_MAX, F16_MAX).astype(np.float16).astype(np.float32)
    lo = np.clip((v - hi) * np.float32(LO_SCALE), -F16_MAX, F16_MAX).astype(np.float16).astype(np.float32)
    return hi, lo


def rz32(v):
    """fp64 -> fp32 rounded toward zero"""
    f = v.astype(np.float32)
    over = np.abs(f.astype(np.float64)) > np.abs(v)
    f[over] = np.nextafter(f[over], np.float32(0))
    return f


def emulate_tc32(x, w, group=1, drop=None, corr_bufs=1):
    """x [P, K], w [K, N] fp32 -> the tc32 GEMM [P, N] as the kernel computes it.

    K is consumed in steps of 32 channels = 2 K16 MMAs per product.  group: K steps per main-product chain (None = one
    chain over the whole K, i.e. never promoted); drop: "a2b" / "ab2" leaves out one correction product; corr_bufs: 2 =
    the even / odd K steps' corrections in separate accumulators (the four-issuer halo mode), each added at the end."""
    x = np.asarray(x, np.float32)
    w = np.asarray(w, np.float32)
    P, K = x.shape
    Kp = (K + 31) // 32 * 32
    xp = np.zeros((P, Kp), np.float32)
    xp[:, :K] = x
    wp = np.zeros((Kp, w.shape[1]), np.float32)
    wp[:K] = w
    ah, al = (t.astype(np.float64) for t in split16(xp))
    bh, bl = (t.astype(np.float64) for t in split16(wp))
    zero = np.zeros((P, w.shape[1]), np.float32)
    total, acc, in_group = None, zero.copy(), 0
    corr = [zero.copy() for _ in range(corr_bufs)]
    for s in range(Kp // 32):
        c = corr[s % corr_bufs]
        for h in (0, 1):
            k = slice(32 * s + 16 * h, 32 * s + 16 * h + 16)
            acc = rz32(acc + ah[:, k] @ bh[k])
        for prod in ("a2b", "ab2"):
            if prod == drop:
                continue
            for h in (0, 1):
                k = slice(32 * s + 16 * h, 32 * s + 16 * h + 16)
                c = rz32(c + (al[:, k] @ bh[k] if prod == "a2b" else ah[:, k] @ bl[k]))
        corr[s % corr_bufs] = c
        in_group += 1
        if group is not None and in_group == group:
            total = acc if total is None else (total.astype(np.float64) + acc).astype(np.float32)
            acc, in_group = zero.copy(), 0
    if total is None or in_group:
        total = acc if total is None else (total.astype(np.float64) + acc).astype(np.float32)
    for c in corr:                     # fmaf(c, 2^-11, sum)
        total = (c.astype(np.float64) / LO_SCALE + total).astype(np.float32)
    return total


def gemm_ref_bound(x, w):
    """fp64 x @ w and its bound, x [P, K], w [K, N]"""
    x, w = np.asarray(x, np.float64), np.asarray(w, np.float64)
    ref = x @ w
    s_abs = np.abs(x) @ np.abs(w)
    s_x = np.abs(x) @ np.ones_like(w)
    s_w = np.ones_like(x) @ np.abs(w)
    return ref, U * s_abs + ABS_SUB * (s_x + s_w) + OUT_ROUND * np.abs(ref)
