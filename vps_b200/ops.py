"""Python-side wrappers of the C-ABI kernels.

Tensors handed to these functions are torch CUDA tensors used purely as device-memory handles
(pointer + shape); all arithmetic happens in libvps_b200.so.  Activations are NHWC: a tensor of shape
[N, H, W, C] whose last dim is contiguous; a channel slice `buf[..., a:b]` of a wider buffer is a
valid view (pixel stride = buf.shape[-1]).
"""
import ctypes as C
import os

import torch

from . import _lib
from ._lib import (ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, VPS_BF16, VPS_F32, VpsConvArgs, VpsError,
                   VpsTensor, check, lib)

_DT = {torch.float32: VPS_F32, torch.bfloat16: VPS_BF16}

# ---- optional per-call device timing (bench.py / profiling only; off on the normal path) -----------------
PROFILE = None        # set to a list to collect [c_function, start_event, end_event, flops, tag] per C-ABI call
_NOTE = {"flops": 0, "tag": ""}
SCOPE = [""]          # pipeline stage label attached to profiled calls (set by the detector)
_real_lib = lib


class _ProfLib(object):
    def __getattr__(self, name):
        f = getattr(_real_lib(), name)
        if PROFILE is None or not name.startswith("vps_") or name in ("vps_last_error", "vps_launch_count", "vps_packed_tc_bytes"):
            return f

        def w(*a):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = f(*a)
            e.record()
            PROFILE.append([name, s, e, _NOTE["flops"], _NOTE["tag"], SCOPE[0]])
            _NOTE["flops"], _NOTE["tag"] = 0, ""
            return r
        return w


_plib = _ProfLib()


def lib():  # noqa: F811  (shadows the import: every wrapper below goes through the profiling proxy)
    return _plib


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Branch:
    """Run an independent part of the frame-pair graph on a side stream (fork at __enter__, `join()` makes the current
    stream wait for it).  Inside a CUDA-graph capture this records parallel branches, so kernels whose grids do not fill
    the GPU (coarse pyramid levels, tails) overlap with the other branch.  VPS_BRANCHES=0 runs everything in line."""
    _streams = {}
    max_level = int(os.environ.get("VPS_BRANCHES", "1"))     # 0: everything in line, 1: whole sub-networks as branches

    def __init__(self, name, level=1):
        self.name = name
        self.main = torch.cuda.current_stream()
        if level <= Branch.max_level and PROFILE is None:
            key = (name, self.main.device.index, self.main.cuda_stream)     # one side stream per (branch, parent stream)
            if key not in Branch._streams:
                Branch._streams[key] = torch.cuda.Stream(self.main.device)
            self.side = Branch._streams[key]
        else:
            self.side = None
        self._ctx = None

    def __enter__(self):
        if self.side is not None:
            self.side.wait_stream(self.main)
            self._ctx = torch.cuda.stream(self.side)
            self._ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self._ctx is not None:
            self._ctx.__exit__(*exc)
            self._ctx = None
        return False

    def join(self, *tensors):
        """the current stream waits for the branch; `tensors` produced on the branch are marked as used by it"""
        if self.side is not None:
            cur = torch.cuda.current_stream()
            cur.wait_stream(self.side)
            for t in tensors:
                if t is not None:
                    t.record_stream(cur)


def vt(t):
    """torch NHWC tensor (possibly a channel-slice view) -> VpsTensor."""
    if t is None:
        return VpsTensor(None, 0, 0, 0, 0, 0, 0)
    assert t.is_cuda and t.dim() == 4, "expected a CUDA NHWC tensor, got %s" % (tuple(t.shape),)
    n, h, w, c = t.shape
    assert t.stride(3) == 1 or c == 1
    if w > 1:
        cs = t.stride(2)
    elif h > 1:
        cs = t.stride(1)
    elif n > 1:
        cs = t.stride(0)
    else:
        cs = max(c, 1)
    if h > 1:
        assert t.stride(1) == w * cs, "rows must be dense: %s %s" % (t.shape, t.stride())
    if n > 1:
        assert t.stride(0) == h * w * cs, "images must be dense: %s %s" % (t.shape, t.stride())
    return VpsTensor(t.data_ptr(), n, h, w, c, cs, _DT[t.dtype])


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def launch_count():
    return int(lib().vps_launch_count())


# ------------------------------------------------------------------ weights
class PackedConv:
    """Packed weights of one convolution for both kernels' layouts (built lazily per precision)."""

    def __init__(self, weight, bias=None, scale=None, transposed=False):
        # weight: OIHW fp32 CUDA tensor (IOHW if transposed); scale: per-cout multiplier folded in
        self.transposed = transposed
        if transposed:
            self.cin, self.cout, self.kh, self.kw = weight.shape
        else:
            self.cout, self.cin, self.kh, self.kw = weight.shape
        self.weight = weight.contiguous().float()
        self.scale = scale.contiguous().float() if scale is not None else None
        self.bias = bias.contiguous().float() if bias is not None else None
        self._tc = {}
        self._tc32 = None
        self._simt = None

    def gran(self):
        """channel granularity of the tensor-core K step (16 or 64)."""
        return 16 if self.cin <= 16 else 64     # thin stems only: bk=16 multiplies the number of (tiny) K steps

    def tc(self, gran=None):
        gran = gran or self.gran()
        if gran not in self._tc:
            nbytes = lib().vps_packed_tc_bytes(self.cout, self.cin, self.kh, self.kw, gran)
            buf = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=self.weight.device)
            check(lib().vps_pack_weights_tc(_ptr(self.weight), _ptr(self.scale), _ptr(buf), self.cout, self.cin,
                                            self.kh, self.kw, int(self.transposed), gran, stream()), "pack_weights_tc")
            torch.cuda.current_stream().synchronize()   # one-time: the packed buffer may next be read from ANY stream / branch
            self._tc[gran] = buf
        return self._tc[gran]

    def tc32(self):
        """[B | B2] fp16 planes of the fp32-parity tensor-core kernel (vps_conv2d_tc32): B = fp16(w * scale),
        B2 = fp16(2^11 (w * scale - B)), the scale folded in fp32."""
        if self._tc32 is None:
            self._tc32 = pack_tc32([self])
        return self._tc32

    def simt(self):
        if self._simt is None:
            buf = torch.empty(self.kh * self.kw * self.cin * self.cout, dtype=torch.float32,
                              device=self.weight.device)
            check(lib().vps_pack_weights_simt(_ptr(self.weight), _ptr(self.scale), _ptr(buf), self.cout, self.cin,
                                              self.kh, self.kw, int(self.transposed), stream()),
                  "pack_weights_simt")
            torch.cuda.current_stream().synchronize()   # one-time: see tc()
            self._simt = buf
        return self._simt


def pack_tc32(pws):
    """one packed tc32 weight buffer for len(pws) problems of identical geometry (the stride phases of a transposed
    convolution share a launch and therefore a buffer)."""
    p0 = pws[0]
    n = len(pws)
    nbytes = lib().vps_packed_tc32_bytes(p0.cout, p0.cin, p0.kh, p0.kw, n)
    buf = torch.empty(nbytes, dtype=torch.uint8, device=p0.weight.device)
    for i, pw in enumerate(pws):
        assert (pw.cout, pw.cin, pw.kh, pw.kw) == (p0.cout, p0.cin, p0.kh, p0.kw)
        check(lib().vps_pack_weights_tc32(_ptr(pw.weight), _ptr(pw.scale), _ptr(buf), pw.cout, pw.cin, pw.kh, pw.kw,
                                          int(pw.transposed), i, n, stream()), "pack_weights_tc32")
    torch.cuda.current_stream().synchronize()   # one-time: the packed buffer may next be read from ANY stream / branch
    return buf


# fp32 activations: True = tensor cores with split operands (vps_conv2d_tc32, the "tc32" parity precision),
# False = CUDA-core fp32 FMA (vps_conv2d_simt, the debugging reference of the parity mode)
F32_TC = [False]


def tc32_overflow(reset=True):
    """threads of the tc32 kernels that met |value| > 65504 (the fp16 range of the main product) since the last reset"""
    return int(lib().vps_tc32_overflow(int(reset)))


def f32_tc_ok(x):
    """fp32 activations the tc32 kernel can read through TMA: 16-byte aligned base and pixel stride"""
    return F32_TC[0] and x.dtype == torch.float32 and vt(x).cs % 4 == 0 and x.data_ptr() % 16 == 0


def _conv_args(x, pw, y, stride, pad, act, slope, res, res_after_act, out_scale, oh, ow, omap, pad_hw):
    a = VpsConvArgs()
    a.x, a.y, a.res = vt(x), vt(y), vt(res)
    kh, kw = pw.kh, pw.kw
    sh, sw = (stride, stride) if isinstance(stride, int) else stride
    ph, pw_ = pad_hw if pad_hw is not None else ((pad, pad) if isinstance(pad, int) else pad)
    a.kh, a.kw, a.sh, a.sw, a.ph, a.pw = kh, kw, sh, sw, ph, pw_
    if oh is None:
        oh = (x.shape[1] + 2 * ph - kh) // sh + 1
        ow = (x.shape[2] + 2 * pw_ - kw) // sw + 1
    a.oh, a.ow = oh, ow
    a.oy_mul, a.oy_off, a.ox_mul, a.ox_off = omap
    a.cin, a.cout = pw.cin, pw.cout
    a.act, a.slope, a.res_after_act, a.out_scale = act, slope, int(res_after_act), out_scale
    a.bias = pw.bias.data_ptr() if pw.bias is not None else None
    return a


def conv2d(x, pw, y, stride=1, pad=0, act=ACT_NONE, slope=0.1, res=None, res_after_act=False, out_scale=1.0,
           oh=None, ow=None, omap=(1, 0, 1, 0), pad_hw=None, use_tc=None):
    """y <- conv(x) with fused bias/activation/residual.  `omap` = (oy_mul, oy_off, ox_mul, ox_off)."""
    a = _conv_args(x, pw, y, stride, pad, act, slope, res, res_after_act, out_scale, oh, ow, omap, pad_hw)
    if use_tc is None:
        use_tc = x.dtype == torch.bfloat16
    if PROFILE is not None:
        # algorithmic FLOPs of the layer (SURVEY 8d): a caller that runs a re-shaped form (the 7x7/s2 stems as 4x4/s1 over
        # space-to-depth input) passes the original layer's count in _NOTE["flops_alg"]
        _NOTE["flops"] = _NOTE.pop("flops_alg", None) or 2 * x.shape[0] * a.oh * a.ow * pw.cout * pw.cin * a.kh * a.kw
        _NOTE["tag"] = "%dx%d s%d %d->%d @%dx%d" % (a.kh, a.kw, a.sh, pw.cin, pw.cout, a.oh, a.ow)
    if use_tc and x.dtype == torch.float32:
        a.w = pw.tc32().data_ptr()
        check(lib().vps_conv2d_tc32(C.byref(a), stream()), "conv2d_tc32")
    elif use_tc:
        a.cin_gran = pw.gran()
        a.w = pw.tc().data_ptr()
        check(lib().vps_conv2d_tc(C.byref(a), stream()), "conv2d_tc")
    else:
        a.w = pw.simt().data_ptr()
        check(lib().vps_conv2d_simt(C.byref(a), stream()), "conv2d_simt")
    return y


def conv2d_tc_multi(x, pws, y, pads, omaps, act=ACT_NONE, slope=0.1, out_scale=1.0, oh=None, ow=None, shared32=None):
    """Up to 4 sub-convolutions (same input / output tensors, stride 1) in one persistent tensor-core launch:
    the stride phases of a transposed convolution.  fp32 x: `shared32` = pack_tc32(pws)."""
    n = len(pws)
    arr = (VpsConvArgs * n)()
    gran = pws[0].gran()
    f32 = x.dtype == torch.float32
    for i in range(n):
        a = _conv_args(x, pws[i], y, 1, 0, act, slope, None, False, out_scale, oh, ow, omaps[i], pads[i])
        a.cin_gran = gran
        a.w = shared32.data_ptr() if f32 else pws[i].tc(gran).data_ptr()
        arr[i] = a
    if PROFILE is not None:
        _NOTE["flops"] = 2 * x.shape[0] * arr[0].oh * arr[0].ow * pws[0].cout * pws[0].cin * arr[0].kh * arr[0].kw * n
        _NOTE["tag"] = "%dx%d x%d phases %d->%d @%dx%d" % (arr[0].kh, arr[0].kw, n, pws[0].cin, pws[0].cout, arr[0].oh, arr[0].ow)
    if f32:
        check(lib().vps_conv2d_tc32_multi(arr, n, stream()), "conv2d_tc32_multi")
    else:
        check(lib().vps_conv2d_tc_multi(arr, n, stream()), "conv2d_tc_multi")
    return y


# ------------------------------------------------------------------ FlowNet2 native ops
def correlation(f1, f2, out, pad, max_disp, stride1, stride2, act=ACT_NONE, slope=0.1, impl=None):
    """impl: None = dispatch (tensor cores for bf16 features, and for fp32 features in the tc32 precision), "tc" / "tc32" /
    "simt" force one implementation."""
    fn = {None: "vps_correlation", "tc": "vps_correlation_tc", "simt": "vps_correlation_simt", "tc32": "vps_correlation_tc32"}[impl]
    if PROFILE is not None:
        d = 2 * (max_disp // stride2) + 1
        _NOTE["flops"] = 2 * f1.shape[0] * f1.shape[1] * f1.shape[2] * f1.shape[3] * d * d
        _NOTE["tag"] = "corr d%d s%d C%d @%dx%d" % (max_disp, stride2, f1.shape[3], f1.shape[1], f1.shape[2])
    if impl is None and F32_TC[0] and f1.dtype == torch.float32 and f2.dtype == torch.float32 and out.dtype == torch.float32:
        c = f1.shape[3]
        # (the d4 / stride2 1 site runs 1.39 ms this way against 0.97 ms on the CUDA cores: its band is 9 of 32 columns wide)
        if (c % 64 == 0 and c <= 256 and stride1 == 1 and pad == max_disp and (max_disp, stride2) == (20, 2)
                and vt(f1).cs % 4 == 0 and vt(f2).cs % 4 == 0 and f1.data_ptr() % 16 == 0 and f2.data_ptr() % 16 == 0):
            fn = "vps_correlation_tc32"
    if fn == "vps_correlation_tc32":
        ws = torch.empty(int(lib().vps_correlation_tc32_ws_bytes(C.byref(vt(f1)))), dtype=torch.uint8, device=f1.device)
        off = (-ws.data_ptr()) % 256
        check(lib().vps_correlation_tc32(C.byref(vt(f1)), C.byref(vt(f2)), C.byref(vt(out)), pad, max_disp, stride1, stride2,
                                         act, C.c_float(slope), C.c_void_p(ws.data_ptr() + off), stream()), "correlation_tc32")
        return out
    check(getattr(lib(), fn)(C.byref(vt(f1)), C.byref(vt(f2)), C.byref(vt(out)), pad, max_disp, stride1,
                                stride2, act, C.c_float(slope), stream()), "correlation")
    return out


def resample2d(src, flow, out):
    check(lib().vps_resample2d(C.byref(vt(src)), C.byref(vt(flow)), C.byref(vt(out)), stream()), "resample2d")
    return out


def channelnorm(a, out, b=None):
    bb = C.byref(vt(b)) if b is not None else None
    check(lib().vps_channelnorm(C.byref(vt(a)), bb, C.byref(vt(out)), stream()), "channelnorm")
    return out


# ------------------------------------------------------------------ layout / pointwise / resampling
def _bt(t):
    return C.byref(vt(t))


def nchw_to_nhwc(src_nchw, dst):
    assert src_nchw.dtype == torch.float32 and src_nchw.is_contiguous()
    check(lib().vps_nchw_to_nhwc(_ptr(src_nchw), _bt(dst), stream()), "nchw_to_nhwc")
    return dst


def nhwc_to_nchw(src, dst_nchw):
    assert dst_nchw.dtype == torch.float32 and dst_nchw.is_contiguous()
    check(lib().vps_nhwc_to_nchw(_bt(src), _ptr(dst_nchw), stream()), "nhwc_to_nchw")
    return dst_nchw


def axpby(a, out, alpha=1.0, b=None, beta=0.0):
    check(lib().vps_axpby(_bt(a), _bt(b) if b is not None else None, _bt(out), C.c_float(alpha), C.c_float(beta),
                          stream()), "axpby")
    return out


def copy_scale(src, dst, alpha=1.0):
    return axpby(src, dst, alpha)


def resize_bilinear(src, out, mul=1.0):
    check(lib().vps_resize_bilinear(_bt(src), _bt(out), C.c_float(mul), stream()), "resize_bilinear")
    return out


def resize_nearest(src, out, mul=1.0, accumulate=False):
    check(lib().vps_resize_nearest(_bt(src), _bt(out), C.c_float(mul), int(accumulate), stream()), "resize_nearest")
    return out


def pool2d(src, out, k, s, p, avg=False):
    check(lib().vps_pool2d(_bt(src), _bt(out), k, s, p, int(avg), stream()), "pool2d")
    return out


def groupnorm(x, y, gamma, beta, groups, eps=1e-5, relu=False):
    check(lib().vps_groupnorm(_bt(x), _bt(y), _ptr(gamma), _ptr(beta), groups, C.c_float(eps), int(relu), stream()),
          "groupnorm")
    return y


def im2col(x, cols, kh, kw, sh, sw, ph, pw):
    check(lib().vps_im2col(_bt(x), _bt(cols), kh, kw, sh, sw, ph, pw, stream()), "im2col")
    return cols


def flownet_input(img_nchw, ref_nchw, std3, mean3, rgb_max, sums_ws, x):
    h, w = img_nchw.shape[-2:]
    s = (C.c_float * 3)(*std3)
    m = (C.c_float * 3)(*mean3)
    check(lib().vps_flownet_input(_ptr(img_nchw), _ptr(ref_nchw), h, w, s, m, C.c_float(rgb_max), _ptr(sums_ws), _bt(x),
                                  stream()), "flownet_input")
    return x


def flownet_stage(x6, flow_lo, mul, inv, cat):
    check(lib().vps_flownet_stage(_bt(x6), _bt(flow_lo), C.c_float(mul), C.c_float(inv), _bt(cat), stream()), "flownet_stage")
    return cat


def flownet_cat3(x6, s2_flow_lo, sd_flow_lo, mul_s2, mul_sd, cat):
    check(lib().vps_flownet_cat3(_bt(x6), _bt(s2_flow_lo), _bt(sd_flow_lo), C.c_float(mul_s2), C.c_float(mul_sd), _bt(cat), stream()),
          "flownet_cat3")
    return cat


# ------------------------------------------------------------------ BFPTcea / DCN
def bfp_gather(levels, out):
    arr = (VpsTensor * len(levels))(*[vt(l) for l in levels])
    check(lib().vps_bfp_gather(arr, len(levels), _bt(out), stream()), "bfp_gather")
    return out


def bfp_scatter(bsf, inp, out):
    check(lib().vps_bfp_scatter(_bt(bsf), _bt(inp), _bt(out), stream()), "bfp_scatter")
    return out


def flow_warp(src, flow, out):
    check(lib().vps_flow_warp(_bt(src), _bt(flow), _bt(out), stream()), "flow_warp")
    return out


def tcea_temporal(fea0, fea1, emb0, emb1, emb_ref, out):
    check(lib().vps_tcea_temporal(_bt(fea0), _bt(fea1), _bt(emb0), _bt(emb1), _bt(emb_ref), _bt(out), stream()),
          "tcea_temporal")
    return out


def tcea_combine(fea, att, att_add, out):
    check(lib().vps_tcea_combine(_bt(fea), _bt(att), _bt(att_add), _bt(out), stream()), "tcea_combine")
    return out


def deform_im2col(x, offset, cols):
    check(lib().vps_deform_im2col(_bt(x), _bt(offset), _bt(cols), stream()), "deform_im2col")
    return cols


def deform_conv_tc(x, offset, pw, y):
    """fused DCNv1 3x3: x bf16 NHWC, offset f32 NHWC [..,18], pw = PackedConv of the OIHW kernel, y NHWC [.., cout]"""
    if PROFILE is not None:
        _NOTE["flops"] = 2 * x.shape[0] * x.shape[1] * x.shape[2] * pw.cout * pw.cin * 9
        _NOTE["tag"] = "dcn3x3 %d->%d @%dx%d" % (pw.cin, pw.cout, x.shape[1], x.shape[2])
    check(lib().vps_deform_conv_tc(_bt(x), _bt(offset), C.c_void_p(pw.tc().data_ptr()), pw.cout, _bt(y), stream()), "deform_conv_tc")
    return y


def deform_conv_tc32(x, offset, pw, y):
    """fused DCNv1 3x3 in the tc32 precision: x fp32 NHWC, offset f32 NHWC [..,18], pw = PackedConv of the OIHW kernel"""
    if PROFILE is not None:
        _NOTE["flops"] = 2 * x.shape[0] * x.shape[1] * x.shape[2] * pw.cout * pw.cin * 9
        _NOTE["tag"] = "dcn3x3 %d->%d @%dx%d" % (pw.cin, pw.cout, x.shape[1], x.shape[2])
    check(lib().vps_deform_conv_tc32(_bt(x), _bt(offset), C.c_void_p(pw.tc32().data_ptr()), pw.cout, _bt(y), stream()),
          "deform_conv_tc32")
    return y


# ------------------------------------------------------------------ detection
def roi_align(feats, strides, rois, nroi, out, sample_num=2, nroi_dev=None):
    arr = (VpsTensor * len(feats))(*[vt(f) for f in feats])
    st = (C.c_int * len(strides))(*strides)
    check(lib().vps_roi_align(arr, st, len(feats), _ptr(rois), nroi, _ptr(nroi_dev), _bt(out), sample_num, stream()),
          "roi_align")
    return out


def sort_ws_bytes(n):
    return n * 24 + (1 << 16)


def sort_desc(keys, keys_out, idx_out, n, ws):
    check(lib().vps_sort_desc(_ptr(keys), _ptr(keys_out), _ptr(idx_out), n, _ptr(ws), C.c_int64(ws.numel() * ws.element_size()),
                              stream()), "sort_desc")


def sigmoid_flat(src, dst):
    check(lib().vps_sigmoid_flat(_bt(src), _ptr(dst), stream()), "sigmoid_flat")
    return dst


def rpn_decode(scores_sorted, idx_sorted, k, deltas, stride, base_anchors, img_h, img_w, dets):
    check(lib().vps_rpn_decode(_ptr(scores_sorted), _ptr(idx_sorted), k, _bt(deltas), deltas.shape[1], deltas.shape[2],
                               stride, _ptr(base_anchors), base_anchors.shape[0], C.c_float(img_h), C.c_float(img_w),
                               _ptr(dets), stream()), "rpn_decode")
    return dets


def nms_ws_bytes(n):
    return n * ((n + 63) // 64) * 8


def nms(dets, n, thr, keep_idx, nkeep, ws, n_dev=None):
    check(lib().vps_nms(_ptr(dets), n, _ptr(n_dev), C.c_float(thr), _ptr(keep_idx), _ptr(nkeep), _ptr(ws),
                        C.c_int64(ws.numel() * ws.element_size()), stream()), "nms")


def nms_batch(dets, ns, seg, thr, keep_idx, nkeep, ws, n_dev=None):
    """len(ns) problems in one launch pair; problem b = rows [b*seg, b*seg+ns[b]) of dets."""
    arr = (C.c_int * len(ns))(*ns)
    check(lib().vps_nms_batch(_ptr(dets), len(ns), seg, arr, _ptr(n_dev), C.c_float(thr), _ptr(keep_idx), _ptr(nkeep), _ptr(ws),
                              C.c_int64(ws.numel() * ws.element_size()), stream()), "nms_batch")


def gather_rows(src, idx, n, width, dst, n_dev=None):
    check(lib().vps_gather_rows(_ptr(src), _ptr(idx), n, _ptr(n_dev), width, _ptr(dst), stream()), "gather_rows")
    return dst


def maskroi_candidates(rois, cls_score, bbox_pred, nroi, num_classes, thr, img_h, img_w, cand, cand_cls, cand_prob,
                       ncand, nroi_dev=None):
    assert cls_score.stride(0) == bbox_pred.stride(0) and cls_score.stride(1) == 1 and bbox_pred.stride(1) == 1
    check(lib().vps_maskroi_candidates(_ptr(rois), _ptr(cls_score), _ptr(bbox_pred), cls_score.stride(0), nroi,
                                       _ptr(nroi_dev), num_classes,
                                       C.c_float(thr), C.c_float(img_h), C.c_float(img_w), _ptr(cand), _ptr(cand_cls),
                                       _ptr(cand_prob), _ptr(ncand), stream()), "maskroi_candidates")


def track_assign(emb, ref_emb, k, m, dim, det_boxes, ref_boxes, det_labels, ref_labels, cls_prob, coeff, cap,
                 det_obj_ids, match_ids, comp, mem_src, new_m, ws):
    check(lib().vps_track_assign(_ptr(emb), _ptr(ref_emb), k, m, dim, _ptr(det_boxes), _ptr(ref_boxes), _ptr(det_labels),
                                 _ptr(ref_labels), _ptr(cls_prob), C.c_float(coeff[0]), C.c_float(coeff[1]),
                                 C.c_float(coeff[2]), cap, _ptr(det_obj_ids), _ptr(match_ids), _ptr(comp), _ptr(mem_src),
                                 _ptr(new_m), _ptr(ws), C.c_int64(ws.numel() * ws.element_size()), stream()),
          "track_assign")


# ------------------------------------------------------------------ panoptic fusion
def mask_removal(boxes, order, k, mask_logit, msize, cls_idx, H, W, frac_thr, occ, num_things, counters, keep_flag,
                 keep_sorted, nkeep, k_dev=None):
    check(lib().vps_mask_removal(_ptr(boxes), _ptr(order), k, _ptr(k_dev), _ptr(mask_logit), msize, _ptr(cls_idx), H, W,
                                 C.c_float(frac_thr), _ptr(occ), num_things, _ptr(counters), _ptr(keep_flag),
                                 _ptr(keep_sorted), _ptr(nkeep), stream()), "mask_removal")


def panoptic_fuse(fcn_score, boxes, cls_idx, mask_logit, msize, keep_sorted, nkeep_dev, kcap, num_stuff, dummy, H, W,
                  pano_out, sem_out):
    check(lib().vps_panoptic_fuse(_bt(fcn_score), _ptr(boxes), _ptr(cls_idx), _ptr(mask_logit), msize, _ptr(keep_sorted),
                                  _ptr(nkeep_dev), kcap, num_stuff, int(dummy), H, W, _ptr(pano_out), _ptr(sem_out),
                                  pano_out.element_size(), stream()), "panoptic_fuse")


def rpn_finalize(dets_cat, counts, nlev, seg, cap, scores_ws, scores_sorted_ws, idx_sorted_ws, sort_ws, proposals, rois,
                 total):
    check(lib().vps_rpn_finalize(_ptr(dets_cat), _ptr(counts), nlev, seg, cap, _ptr(scores_ws), _ptr(scores_sorted_ws),
                                 _ptr(idx_sorted_ws), _ptr(sort_ws), C.c_int64(sort_ws.numel() * sort_ws.element_size()),
                                 _ptr(proposals), _ptr(rois), _ptr(total), stream()), "rpn_finalize")


def maskroi_finalize(cand_sorted, slot_sorted, cand_cls, keep, nkeep, max_det, cap, det_rois, cls_idx, cls_prob, kout):
    check(lib().vps_maskroi_finalize(_ptr(cand_sorted), _ptr(slot_sorted), _ptr(cand_cls), _ptr(keep), _ptr(nkeep), max_det,
                                     cap, _ptr(det_rois), _ptr(cls_idx), _ptr(cls_prob), _ptr(kout), stream()),
          "maskroi_finalize")


def select_class(logits, cls_idx, k, out):
    check(lib().vps_select_class(_bt(logits), _ptr(cls_idx), k, _ptr(out), stream()), "select_class")
    return out


def track_update(mem_feats, det_feats, feat_len, mem_boxes, det_boxes, mem_labels, det_labels, mem_src, old_m, cap,
                 new_m_dev):
    check(lib().vps_track_update(_ptr(mem_feats), _ptr(det_feats), _DT[mem_feats.dtype], C.c_int64(feat_len),
                                 _ptr(mem_boxes), _ptr(det_boxes), _ptr(mem_labels), _ptr(det_labels), _ptr(mem_src), old_m,
                                 cap, _ptr(new_m_dev), stream()), "track_update")


def det_split(det_rois, cls_idx, cap, boxes, labels):
    check(lib().vps_det_split(_ptr(det_rois), _ptr(cls_idx), cap, _ptr(boxes), _ptr(labels), stream()), "det_split")


def flow_deconv(x, w_host, b_host, y):
    """x [n,h,w,2] -> y [n,2h,2w,2]; w_host: 64 python floats (IOHW), b_host: 2 floats or None."""
    w = (C.c_float * 64)(*w_host)
    b = (C.c_float * 2)(*b_host) if b_host is not None else None
    check(lib().vps_flow_deconv(_bt(x), w, b, _bt(y), stream()), "flow_deconv")
    return y


def space_to_depth2(x, y):
    check(lib().vps_space_to_depth2(_bt(x), _bt(y), stream()), "space_to_depth2")
    return y


def tap_gather3x3(z, out, bias, act=ACT_NONE, slope=0.1, out_scale=1.0):
    """out = act(bias + sum over the 9 taps of the tap-major 1x1 result z) * out_scale (see vps_tap_gather3x3)"""
    check(lib().vps_tap_gather3x3(_bt(z), _bt(out), _ptr(bias), act, C.c_float(slope), C.c_float(out_scale), stream()),
          "tap_gather3x3")
    return out
