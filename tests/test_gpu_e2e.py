"""GPU parity, end to end: the CUDA FuseTrack path vs (a) the oracle on the same seeded clip and
(b) the golden vectors generated from the reference's own python code (tests/golden/make_golden.py).

fp32 parity mode: panoptic / semantic label maps, class ids and track ids bit-exact; logits within 1e-3
(north_star tolerance).  bf16 tensor-core mode: same clip, tolerance = bf16 storage of ~60 stacked layers
(relative 5e-2 on continuous tensors; label maps compared by agreement fraction)."""
import os

import numpy as np
import pytest
import torch

from tests.e2e_util import build_models, compare_frame, make_pair, meta
from tests.golden.make_golden import keep

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fusetrack_clip_128x256.npz")


@pytest.fixture(scope="module")
def models(cuda):
    return build_models("C", 0, "fp32", "cuda:0")


@pytest.mark.parametrize("precision", ["tc32", "fp32"])
def test_fp32_clip_matches_oracle(models, precision):
    """tc32 = the tensor-core parity precision (the benchmarked headline mode); fp32 = its CUDA-core debugging twin."""
    oracle, prod = models
    prod.precision = precision
    prod.reset_tracker()
    oracle.prev_bboxes = None
    H, W = 128, 256
    img, ref = make_pair(H, W)
    for iid, (a, b) in ((10001, (img, ref)), (10002, (ref, img)), (10003, (img, ref))):
        rep, _, _ = compare_frame(oracle, prod, a, b, iid)
        assert rep["flow_full"] <= 1e-4 and rep["flow_fine"] <= 1e-3, rep
        assert max(rep["fused%d" % i] for i in range(5)) <= 1e-4, rep
        assert rep["fcn_score_abs"] <= 1e-3 and rep["fcn_output_abs"] <= 1e-3, rep          # fp32 logits within 1e-3
        assert max(rep["rpn_cls%d" % l] for l in range(5)) <= 1e-3, rep
        assert rep["n_proposals"][0] == rep["n_proposals"][1], rep
        assert rep["proposals_abs"] <= 5e-3 and rep["cls_score_abs"] <= 1e-3 and rep["bbox_pred_abs"] <= 1e-3, rep
        assert rep["n_det"][0] == rep["n_det"][1] and rep["cls_idx_equal"], rep
        assert rep["det_rois_abs"] <= 5e-3 and rep["mask_logit_abs"] <= 1e-3, rep
        assert rep["obj_ids_equal"] and rep["keep_equal"] and rep["ids_kept_equal"], rep        # track ids bit-exact
        assert rep["pano_agree"] == 1.0 and rep["sem_agree"] == 1.0, rep                        # label maps bit-exact


@pytest.mark.parametrize("precision", ["tc32", "fp32"])
def test_fp32_clip_matches_reference_golden(models, precision):
    _, prod = models
    prod.precision = precision
    prod.reset_tracker()
    g = np.load(GOLD)
    H, W = int(g["H"]), int(g["W"])
    img, ref = make_pair(H, W)
    for f, (iid, a, b) in enumerate(((10001, img, ref), (10002, ref, img))):
        taps = {}
        r = prod.simple_test(a.cuda(), [meta(iid, H, W)], ref_img=[b.cuda()], taps=taps)
        p = r[2]
        assert np.array_equal(p["panoptic_outputs"].cpu().numpy().astype(np.uint8), g["f%d_pano" % f])
        assert np.array_equal(p["fcn_outputs"].cpu().numpy().astype(np.uint8), g["f%d_sem" % f])
        assert np.array_equal(p["panoptic_cls_inds"].cpu().numpy(), g["f%d_cls_inds" % f])
        assert np.array_equal(p["panoptic_det_obj_ids"].cpu().numpy(), g["f%d_obj_ids" % f])
        assert np.array_equal(p["panoptic_det_labels"].cpu().numpy(), g["f%d_det_labels" % f])
        assert np.abs(p["panoptic_cls_prob"].cpu().numpy() - g["f%d_cls_prob" % f]).max() <= 1e-4
        ids = sorted(r[0].keys())
        assert ids == g["f%d_bbox_ids" % f].tolist()
        assert np.abs(np.stack([r[0][i]["bbox"] for i in ids]) - g["f%d_bbox" % f]).max() <= 5e-3
        fs = keep("fcn_score", taps["fcn_score"].float().permute(0, 3, 1, 2).cpu().numpy())
        assert np.abs(fs - g["f%d_fcn_score" % f]).max() <= 1e-3
        fl = keep("flow_full", taps["flow_full"].permute(0, 3, 1, 2).cpu().numpy())
        assert np.abs(fl - g["f%d_flow_full" % f]).max() <= 1e-3


def test_bf16_clip_close_to_oracle(models):
    oracle, prod = models
    prod.precision = "bf16"
    prod.reset_tracker()
    oracle.prev_bboxes = None
    H, W = 128, 256
    img, ref = make_pair(H, W)
    rep, _, _ = compare_frame(oracle, prod, img, ref, 10001)
    prod.precision = "fp32"
    assert rep["flow_full"] <= 5e-2 and rep["flow"] <= 5e-2, rep
    assert max(rep["fpn%d" % i] for i in range(5)) <= 5e-2 and max(rep["fused%d" % i] for i in range(5)) <= 5e-2, rep
    assert rep["fcn_score"] <= 5e-2, rep
    assert rep["sem_agree"] >= 0.95, rep
    assert abs(rep["n_proposals"][0] - rep["n_proposals"][1]) <= 30, rep


def test_dummy_detection_path(models):
    """weight set A (reference init): no RoI passes 0.6 -> MaskROI dummy result (mask_roi.py:136-142)."""
    from oracle.weights import make_model
    oracle, prod = models
    oa = make_model("A", 0, calibrated=False)
    sd_c = {k: v.clone() for k, v in prod.state_dict().items()}
    prod.load_state_dict(oa.state_dict(), strict=True)
    prod.prepare(force=True)
    prod.precision = "fp32"
    prod.reset_tracker()
    try:
        H, W = 64, 128
        img, ref = make_pair(H, W, seed=5)
        rep, (o_res, _), (p_res, _) = compare_frame(oa, prod, img, ref, 10001)
        assert rep["n_det"] == (1, 1) and rep["pano_agree"] == 1.0 and rep["sem_agree"] == 1.0, rep
        assert p_res[2]["panoptic_cls_inds"].tolist() == [0] == o_res[2]["panoptic_cls_inds"].tolist()
    finally:
        prod.load_state_dict(sd_c, strict=True)
        prod.prepare(force=True)


@pytest.mark.parametrize("precision", ["tc32", "fp32"])
def test_cuda_graph_replay_equals_eager(models, precision):
    """The static part replayed as a CUDA graph gives bit-identical results to eager launches, across frames with
    different inputs (static buffers are refreshed) and with the tracker state carried in the eager tail."""
    _, prod = models
    prod.precision = precision
    H, W = 128, 256
    frames = [make_pair(H, W, seed=s) for s in (1, 2, 3, 4)]
    outs = {}
    for mode in (False, True):
        prod.use_cuda_graph = mode
        prod.reset_tracker()
        res = []
        for f, (a, b) in enumerate(frames):
            r = prod.simple_test(a.cuda(), [meta(10001 + f, H, W)], ref_img=[b.cuda()])
            res.append((r[2]["panoptic_outputs"].cpu().clone(), r[2]["fcn_outputs"].cpu().clone(),
                        r[2]["panoptic_det_obj_ids"].cpu().clone(), r[2]["panoptic_cls_inds"].cpu().clone()))
        outs[mode] = res
    prod.use_cuda_graph = True
    assert len(prod._graphs) >= 1 and any(isinstance(v, tuple) for v in prod._graphs.values()), "graph was not captured"
    for e, g in zip(outs[False], outs[True]):
        for x, y in zip(e, g):
            assert torch.equal(x, y)


def test_clip_runner_equals_direct_calls(models):
    """ClipRunner (prefetching clip loop, uint8 label maps downloaded on a copy stream) returns exactly what direct
    simple_test calls return for the same clip (int64 maps), including the tracker ids carried across frames."""
    from vps_b200.runner import ClipRunner
    _, prod = models
    prod.precision = "tc32"
    H, W = 128, 256
    frames = [make_pair(H, W, seed=s) for s in (5, 6, 7, 8, 9, 10, 11, 12)]
    metas = [meta(10001 + f, H, W) for f in range(len(frames))]
    prod.label_dtype = torch.int64
    prod.reset_tracker()
    direct = []
    for (a, b), m in zip(frames, metas):
        r = prod.simple_test(a.cuda(), [m], ref_img=[b.cuda()])
        direct.append((r[2]["panoptic_outputs"].cpu().clone(), r[2]["fcn_outputs"].cpu().clone(),
                       r[2]["panoptic_det_obj_ids"].cpu().clone(), r[2]["panoptic_cls_inds"].cpu().clone()))
    try:
        prod.label_dtype = torch.uint8
        prod.reset_tracker()
        pinned = [(a.pin_memory(), b.pin_memory()) for a, b in frames]
        got = []
        for r in ClipRunner(prod, "cuda:0").run(pinned, metas):
            assert r[2]["panoptic_outputs"].dtype == torch.uint8 and not r[2]["panoptic_outputs"].is_cuda
            got.append((r[2]["panoptic_outputs"].clone(), r[2]["fcn_outputs"].clone(),
                        r[2]["panoptic_det_obj_ids"].cpu().clone(), r[2]["panoptic_cls_inds"].cpu().clone()))
    finally:
        prod.label_dtype = torch.int64
    assert len(got) == len(direct)
    for d, g in zip(direct, got):
        assert torch.equal(d[0], g[0].long()) and torch.equal(d[1], g[1].long())
        assert torch.equal(d[2], g[2]) and torch.equal(d[3], g[3])


@pytest.mark.parametrize("precision", ["tc32", "bf16"])
def test_streaming_ref_feature_cache_is_bit_exact(models, precision):
    """In a clip the reference frame of frame t is frame t - 1 (tools/dataset/cityscapes_vps.py:137-142).
    ClipRunner(streaming=True) reuses the previous pair's FPN features as the reference features (one ResNet-50-FPN pass
    per pair instead of two): label maps, class ids and track ids must equal the uncached run bit for bit, with and
    without the prefetching graph pipeline, across a clip boundary."""
    from vps_b200.runner import ClipRunner
    _, prod = models
    H, W = 128, 256
    g = torch.Generator().manual_seed(77)
    imgs = [torch.randn(1, 3, H, W, generator=g) for _ in range(7)]
    # two clips: frames 0-3 (iid 10001..10004) and 4-6 (iid 20001..20003); the first frame of a clip references itself
    pairs, metas = [], []
    for t in range(7):
        first = t in (0, 4)
        pairs.append((imgs[t], imgs[t] if first else imgs[t - 1]))
        metas.append(meta((10001 + t) if t < 4 else (20001 + t - 4), H, W))
    pinned = [(a.pin_memory(), b.pin_memory()) for a, b in pairs]
    outs = {}
    try:
        prod.precision = precision
        prod.label_dtype = torch.uint8
        for mode in ("plain", "stream", "stream_noprefetch"):
            prod.reset_tracker()
            res = []
            runner = ClipRunner(prod, "cuda:0", streaming=mode != "plain")
            for r in runner.run(pinned, metas, prefetch=mode != "stream_noprefetch"):
                res.append((r[2]["panoptic_outputs"].clone(), r[2]["fcn_outputs"].clone(),
                            r[2]["panoptic_det_obj_ids"].cpu().clone(), r[2]["panoptic_cls_inds"].cpu().clone()))
            outs[mode] = res
    finally:
        prod.label_dtype = torch.int64
        prod.precision = "fp32"
    for mode in ("stream", "stream_noprefetch"):
        assert len(outs[mode]) == len(outs["plain"]) == 7
        for a, b in zip(outs["plain"], outs[mode]):
            for x, y in zip(a, b):
                assert torch.equal(x, y), mode


def test_clip_runner_unified_pan_result(models):
    """ClipRunner(unify=True): the uint8 [H,W,3] image produced on the GPU right after each pair equals the oracle of the
    reference's get_unified_pan_result applied, after the clip, to the collected maps / class ids / track ids."""
    import numpy as np
    from oracle import unify as U
    from vps_b200.runner import ClipRunner
    _, prod = models
    prod.precision = "fp32"
    H, W = 128, 256
    frames = [make_pair(H, W, seed=s) for s in (21, 22, 23, 24)]
    metas = [meta(10001 + f, H, W) for f in range(len(frames))]
    try:
        prod.label_dtype = torch.uint8
        prod.reset_tracker()
        pinned = [(a.pin_memory(), b.pin_memory()) for a, b in frames]
        segs, pans, clss, objs, got = [], [], [], [], []
        for r in ClipRunner(prod, "cuda:0", unify=True).run(pinned, metas):
            segs.append(r[2]["fcn_outputs"][0].numpy().copy())
            pans.append(r[2]["panoptic_outputs"][0].numpy().copy())
            clss.append(r[2]["panoptic_cls_inds"].cpu().numpy())
            objs.append(r[2]["panoptic_det_obj_ids"].cpu().numpy())
            got.append(r[2]["pan_2ch"].numpy().copy())
    finally:
        prod.label_dtype = torch.int64
    ref = U.get_unified_pan_result(segs, pans, clss, objs)
    for g, e in zip(got, ref):
        assert np.array_equal(g, e)


@pytest.mark.parametrize("precision", ["tc32", "fp32"])
def test_viper_aspect_fp32_matches_oracle(models, precision):
    """BASELINE config 4 shape family (1088x1920 = 17x30 blocks of 64): a small frame of the same odd block counts
    (192x320 = 3x5 blocks) through the fp32 path: detections, class ids, kept set and track ids equal the oracle's, label
    maps agree up to argmax near-ties."""
    oracle, prod = models
    prod.precision = precision
    prod.reset_tracker()
    oracle.prev_bboxes = None
    H, W = 192, 320
    img, ref = make_pair(H, W, seed=31)
    for iid, (a, b) in ((10001, (img, ref)), (10002, (ref, img))):
        rep, _, _ = compare_frame(oracle, prod, a, b, iid)
        assert rep["fcn_score_abs"] <= 1e-3 and rep["flow_full"] <= 1e-4, rep
        assert rep["n_det"][0] == rep["n_det"][1] and rep["cls_idx_equal"], rep
        assert rep["obj_ids_equal"] and rep["keep_equal"] and rep["ids_kept_equal"], rep
        # label maps: identical except where two class logits are closer than the fp32 path's 2.5e-5 logit error
        # (measured here: one pixel of 61440 in the second frame)
        assert rep["pano_agree"] >= 1.0 - 1e-4 and rep["sem_agree"] >= 1.0 - 1e-4, rep


def test_viper_full_size_clip_properties(models):
    """BASELINE config 4 at full size (1080 padded to 1088 x 1920, bf16): the oracle is too slow for this size, so check the
    size-independent properties -- the pipelined clip loop (prefetch, second graph instance, copy stream) returns exactly
    what one-call-at-a-time inference returns, label values stay in range, every kept instance id is unique per frame and
    the unified-pan-result channels are consistent with the maps."""
    from vps_b200.runner import ClipRunner
    _, prod = models
    H, W = 1088, 1920
    frames = [make_pair(H, W, seed=s) for s in (41, 42, 43, 44, 45)]
    metas = [meta(10001 + f, H, W) for f in range(len(frames))]
    try:
        prod.precision = "bf16"
        prod.label_dtype = torch.uint8
        prod.reset_tracker()
        direct = []
        for (a, b), m in zip(frames, metas):
            r = prod.simple_test(a.cuda(), [m], ref_img=[b.cuda()])
            direct.append((r[2]["panoptic_outputs"].cpu().clone(), r[2]["fcn_outputs"].cpu().clone(),
                           r[2]["panoptic_det_obj_ids"].cpu().clone(), r[2]["panoptic_cls_inds"].cpu().clone()))
        prod.reset_tracker()
        pinned = [(a.pin_memory(), b.pin_memory()) for a, b in frames]
        n = 0
        for r, d in zip(ClipRunner(prod, "cuda:0", unify=True).run(pinned, metas), direct):
            pano, sem = r[2]["panoptic_outputs"], r[2]["fcn_outputs"]
            assert torch.equal(pano, d[0]) and torch.equal(sem, d[1])
            assert torch.equal(r[2]["panoptic_det_obj_ids"].cpu(), d[2]) and torch.equal(r[2]["panoptic_cls_inds"].cpu(), d[3])
            k = d[3].numel()
            assert pano.shape == (1, H, W) and int(sem.max()) <= 18 and int(pano.max()) <= 10 + k
            ids = d[2].tolist()
            assert len(set(ids)) == len(ids)                      # the tracker never hands one id to two kept instances
            p2 = r[2]["pan_2ch"]
            assert p2.shape == (H, W, 3)
            stuff = pano[0] <= 10
            assert bool((p2[..., 1][stuff] == 0).all())           # stuff pixels carry no instance rank
            n += 1
        assert n == len(frames)
    finally:
        prod.precision = "fp32"
        prod.label_dtype = torch.int64
