"""The oracle's native-op restatements (oracle/ops.py) against the REFERENCE's OWN CUDA kernels: the extracted `__global__`
bodies of resample2d / channelnorm / correlation / ROIAlign / nms / deformable_im2col, compiled for sm_100a with the launch
geometry of the reference's launchers (oracle/ref_kernels/build.py) and run on a B200 on seeded inputs.  Their outputs are
stored in tests/golden/ref_kernels.npz (tests/golden/make_ref_kernels_golden.py); the oracle runs here on the same inputs.
This pins the oracle to the reference's actual kernels rather than to transcriptions.  No GPU is needed."""
import os

import numpy as np
import pytest
import torch

from tests.golden import make_ref_kernels_golden as K

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels.npz")


@pytest.fixture(scope="module")
def ref():
    g = np.load(GOLD)
    assert str(g["inputs_sha256"]) == K.inputs_digest(), \
        "seeded inputs differ from the ones the golden file was generated with (torch RNG drift?)"
    return g


def sampled(t):
    flat = t.reshape(-1)
    return flat[torch.from_numpy(K.sample_idx(flat.numel()))]


def test_resample2d_and_channelnorm(ref):
    from oracle import ops as O
    x, flow = K.resample_inputs()
    out = torch.from_numpy(ref["resample2d"])
    assert float((out - O.resample2d(x, flow)).abs().max()) <= 2e-6 * float(x.abs().max())
    o2 = torch.from_numpy(ref["channelnorm"])
    assert float((o2 - O.channelnorm(x)).abs().max()) <= 1e-6 * float(O.channelnorm(x).max())


@pytest.mark.parametrize("pad,md,s2,C", K.CORRELATION)
def test_correlation(ref, pad, md, s2, C):
    """both call sites of the path: FlowNetC (pad 20, d 20, s2 2) and LiteFlowNetCorr (pad 4, d 4, s2 1)"""
    from oracle import ops as O
    f1, f2 = K.correlation_inputs(C)
    want = O.correlation(f1, f2, pad, 1, md, 1, s2)
    key = "correlation_%d_%d_%d_%d" % (pad, md, s2, C)
    assert tuple(ref[key + "_shape"]) == tuple(want.shape)
    out = torch.from_numpy(ref[key])
    assert float((out - sampled(want)).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))


def test_roi_align(ref):
    from oracle import ops as O
    feat, rois = K.roi_inputs()
    for S, scale in K.ROI_SIZES:
        out = torch.from_numpy(ref["roi_align_%d" % S])
        want = O.roi_align(feat, rois, S, scale, 2)
        assert float((out - sampled(want)).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))


def test_nms(ref):
    """nms_kernel's bit mask + the host reduction of nms_cuda (nms_kernel.cu:99-121) == oracle.ops.nms, exactly"""
    from oracle import ops as O
    for dets in K.nms_inputs():
        n = dets.shape[0]
        order = K.nms_order(dets)
        cb = (n + 63) // 64
        m = ref["nms_mask_%d" % n].reshape(n, cb)
        remv = np.zeros(cb, np.uint64)
        keep = []
        for i in range(n):                                            # the reference's host loop
            if not (int(remv[i // 64]) >> (i % 64)) & 1:
                keep.append(i)
                remv |= m[i]
        got = torch.sort(order[torch.tensor(keep, dtype=torch.long)])[0]
        _, want = O.nms(dets, K.NMS_THR)
        assert torch.equal(got, want.sort()[0]), n


def test_deformable_im2col(ref):
    from oracle import ops as O
    x, off = K.deform_inputs()
    B, C, H, W = x.shape
    want = O.deform_im2col(x, off)                                     # [B, C*9, H*W] (c-major, tap-minor)
    want_col = want.reshape(B, C * 9, H, W).permute(1, 0, 2, 3)       # the kernel's [C*9, B, H, W] layout
    got = torch.from_numpy(ref["deform_im2col"])
    assert float((got - sampled(want_col.contiguous())).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))
