"""Generate tests/golden/ref_kernels.npz: outputs of the REFERENCE's own CUDA kernels (resample2d, channelnorm, correlation,
ROIAlign, nms, deformable_im2col) on seeded inputs.

The kernels are the library oracle/ref_kernels/build.py compiles from the reference's sources
(oracle/_ref/libvps_ref_kernels.so); building it needs the reference tree, running this script needs a GPU:

  python tests/golden/make_ref_kernels_golden.py [OUT.npz]

tests/test_gpu_ref_kernels.py regenerates the same inputs with the functions below and compares the oracle's restatements
(oracle/ops.py) with the stored outputs.  Large outputs are stored as a fixed sample of their flat indices (`sample_idx`).
"""
import ctypes
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_kernels.npz")
LIB = os.path.join(ROOT, "oracle", "_ref", "libvps_ref_kernels.so")

CORRELATION = [(20, 20, 2, 64), (4, 4, 1, 96)]     # (pad, max displacement, stride2, C): FlowNetC and LiteFlowNetCorr
ROI_SIZES = [(7, 0.25), (14, 0.25)]
NMS_SIZES = (5, 64, 65, 700)
NMS_THR = 0.5
SAMPLE = 4096
_PRIME = 1000003


def sample_idx(size):
    """min(size, SAMPLE) distinct flat indices spread over the whole array (a fixed stride modulo the size)"""
    if size <= SAMPLE:
        return np.arange(size)
    assert size % _PRIME != 0
    return (np.arange(SAMPLE, dtype=np.int64) * _PRIME) % size


def resample_inputs():
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 5, 19, 27, generator=g)
    flow = (torch.rand(2, 2, 19, 27, generator=g) - 0.5) * 14
    return x, flow


def correlation_inputs(C):
    g = torch.Generator().manual_seed(2)
    B, H, W = 1, 24, 32
    return torch.randn(B, C, H, W, generator=g), torch.randn(B, C, H, W, generator=g)


def roi_inputs():
    g = torch.Generator().manual_seed(3)
    feat = torch.randn(1, 16, 40, 56, generator=g)
    n = 37
    xy = torch.rand(n, 2, generator=g) * torch.tensor([200.0, 140.0])
    wh = torch.rand(n, 2, generator=g) * 90 + 1
    rois = torch.cat([torch.zeros(n, 1), xy, xy + wh], 1)
    rois[0, 1:] = torch.tensor([-20.0, -10.0, 5.0, 3.0])             # partly outside
    return feat, rois


def nms_inputs():
    """one [n, 5] box set per size in NMS_SIZES (x1, y1, x2, y2, score)"""
    g = torch.Generator().manual_seed(4)
    out = []
    for n in NMS_SIZES:
        xy = torch.rand(n, 2, generator=g) * 300
        wh = torch.rand(n, 2, generator=g) * 80 + 2
        out.append(torch.cat([xy, xy + wh, torch.rand(n, 1, generator=g)], 1))
    return out


def nms_order(dets):
    return torch.sort(dets[:, 4], descending=True, stable=True)[1]


def deform_inputs():
    g = torch.Generator().manual_seed(5)
    B, C, H, W = 2, 12, 13, 17
    x = torch.randn(B, C, H, W, generator=g)
    off = torch.randn(B, 18, H, W, generator=g) * 2.5
    off[:, :, 0] -= 4.0
    return x, off


def inputs_digest():
    """sha256 over every input above: the stored outputs belong to exactly these inputs"""
    ts = list(resample_inputs()) + [t for c in CORRELATION for t in correlation_inputs(c[3])] + list(roi_inputs()) + \
        nms_inputs() + list(deform_inputs())
    h = hashlib.sha256()
    for t in ts:
        h.update(t.contiguous().numpy().tobytes())
    return h.hexdigest()


def _sampled(t):
    flat = t.cpu().reshape(-1).numpy()
    return flat[sample_idx(flat.size)].astype(np.float32)


def main(out_path):
    ref = ctypes.CDLL(LIB)

    def P(t):
        return ctypes.c_void_p(t.data_ptr())

    out = {"inputs_sha256": np.array(inputs_digest())}
    # every device input is bound to a name: a temporary `P(x.cuda())` is freed as soon as P returns, and the next
    # allocation may reuse its memory before the kernel reads it
    x, flow = (t.cuda() for t in resample_inputs())
    o = torch.empty(2, 5, 19, 27, device="cuda")
    assert ref.ref_resample2d(P(x), P(flow), P(o), 2, 5, 19, 27, 19, 27) == 0
    out["resample2d"] = o.cpu().numpy()
    o2 = torch.empty(2, 1, 19, 27, device="cuda")
    assert ref.ref_channelnorm(P(x), P(o2), 2, 5, 19, 27) == 0
    out["channelnorm"] = o2.cpu().numpy()

    for pad, md, s2, C in CORRELATION:
        f1, f2 = (t.cuda() for t in correlation_inputs(C))
        B, _, H, W = f1.shape
        D = 2 * (md // s2) + 1
        oh, ow = H + 2 * pad - 2 * md, W + 2 * pad - 2 * md          # kernel size 1, stride1 1
        rb1 = torch.empty(B, H + 2 * pad, W + 2 * pad, C, device="cuda")
        rb2 = torch.empty_like(rb1)
        o = torch.empty(B, D * D, oh, ow, device="cuda")
        assert ref.ref_correlation(P(f1), P(f2), P(rb1), P(rb2), P(o), B, C, H, W, D * D, oh, ow,
                                   pad, 1, md, 1, s2) == 0
        out["correlation_%d_%d_%d_%d_shape" % (pad, md, s2, C)] = np.array(o.shape)
        out["correlation_%d_%d_%d_%d" % (pad, md, s2, C)] = _sampled(o)

    feat, rois = (t.cuda() for t in roi_inputs())
    n = rois.shape[0]
    for S, scale in ROI_SIZES:
        o = torch.empty(n, 16, S, S, device="cuda")
        assert ref.ref_roi_align(P(feat), P(rois), n, ctypes.c_float(scale), 2, 16, 40, 56, S, S, P(o)) == 0
        out["roi_align_%d" % S] = _sampled(o)

    for dets in nms_inputs():
        n = dets.shape[0]
        bs = dets[nms_order(dets)].contiguous().cuda()
        mask = torch.zeros(n * ((n + 63) // 64), dtype=torch.int64, device="cuda")
        assert ref.ref_nms_mask(P(bs), n, ctypes.c_float(NMS_THR), P(mask)) == 0
        out["nms_mask_%d" % n] = mask.cpu().numpy().view(np.uint64)

    x, off = (t.cuda() for t in deform_inputs())
    B, C, H, W = x.shape
    col = torch.empty(C * 9, B, H, W, device="cuda")
    assert ref.ref_deform_im2col(P(x), P(off), B, C, H, W, 3, 1, 1, 1, 1, P(col)) == 0
    out["deform_im2col"] = _sampled(col)

    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    np.savez_compressed(out_path, **out)
    print("wrote", out_path, os.path.getsize(out_path) // 1024, "KiB")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else OUT)
