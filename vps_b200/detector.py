"""PanopticFuseTrack on B200 -- the detector class the reference registers in DETECTORS
(mmdet/models/detectors/panoptic_fusetrack.py:24-606), inference path.

Construction follows TwoStageDetector.__init__ (two_stage.py:15-69): sub-modules are built from the
config dicts through the registries, in the reference's order and under the reference's attribute
names, so `state_dict()` keys match a reference checkpoint.  Differences by design:
  * FlowNet2 weights are NOT read from a hard-coded work_dirs/ path at construction
    (panoptic_fusetrack.py:100-106); they are part of the detector's state_dict (as in latest.pth).
  * simple_test keeps everything on the device: the five host round-trips of the reference
    (NMS mask download, MaskROI numpy, MaskRemoval numpy/cv2, SegTerm numpy, tracker loops) are kernels.
    Two 4-byte counters (number of detections, tracker memory size) are read back per frame to size the
    data-dependent launches.
  * `precision`: "tc32" (fp32 activations, tcgen05 tensor cores with split operands: two fp16 planes per
    operand, v = fp16(v) + 2^-11 fp16(2^11 (v - fp16(v))), three products per K slab -- the parity mode, label maps / ids bit-exact vs the oracle), "bf16" (bf16 activations, one
    tensor-core pass: fastest, ~1e-2 relative on features) or "fp32" (CUDA-core fp32 FMA: debugging reference).
"""
import numpy as np
import torch
import torch.nn as nn

from . import ops
from .flownet2 import FlowNet2
from .layers import empty_nhwc
from .registry import (DETECTORS, build_backbone, build_extra_neck, build_head, build_neck, build_panoptic,
                       build_roi_extractor)

MAX_DET_CAP = 128      # detections kept per frame (config.test.max_det = 100, ties may exceed it)
TRACK_CAP = 4096       # tracker memory slots


def bbox2result_with_id(bboxes, labels, obj_ids):
    """mmdet/core/bbox/transforms.py:159-180."""
    results = {}
    if bboxes.shape[0] == 0:
        return results
    for bbox, label, obj_id in zip(bboxes, labels, obj_ids):
        if obj_id >= 0:
            results[int(obj_id)] = {'bbox': bbox, 'label': label}
    return results


@DETECTORS.register_module
class PanopticFuseTrack(nn.Module):
    mean = [123.675, 116.28, 103.53]      # panoptic_fusetrack.py:92-93
    std = [58.395, 57.12, 57.375]
    # UPSNet globals read by MaskROI (tools/config/config.py:47,169) and ctor constants (:83-87)
    score_thresh, nms_thresh, max_det, fraction_threshold = 0.6, 0.5, 100, 0.3

    def __init__(self, backbone, rpn_head, bbox_roi_extractor, bbox_head, mask_roi_extractor, mask_head, train_cfg,
                 test_cfg, neck=None, extra_neck=None, panoptic=None, track_head=None, shared_head=None,
                 pretrained=None, precision="tc32"):
        super().__init__()
        assert shared_head is None
        self.backbone = build_backbone(backbone)
        self.neck = build_neck(neck)
        self.extra_neck = build_extra_neck(extra_neck)
        self.panopticFPN = build_panoptic(panoptic)
        self.rpn_head = build_head(rpn_head)
        self.bbox_roi_extractor = build_roi_extractor(bbox_roi_extractor)
        self.bbox_head = build_head(bbox_head)
        self.track_head = build_head(track_head)
        self.mask_roi_extractor = build_roi_extractor(mask_roi_extractor)
        self.mask_head = build_head(mask_head)
        self.train_cfg, self.test_cfg = train_cfg, test_cfg
        cfg = train_cfg if (train_cfg is not None and 'class_mapping' in train_cfg) else test_cfg
        self.class_mapping = dict(cfg['class_mapping']) if cfg is not None and 'class_mapping' in cfg else None
        num_stuff = self.panopticFPN.num_stuff_classes
        assert self.class_mapping == {i: num_stuff - 1 + i for i in range(1, self.panopticFPN.num_things_classes + 1)}, \
            "the fused kernel assumes the Cityscapes thing->semantic mapping of fusetrack.py:148"
        has_flow = (train_cfg is not None and 'flownet2' in train_cfg) or (test_cfg is not None and 'flownet2' in test_cfg)
        assert has_flow, "Feature flow must be implemented."          # panoptic_fusetrack.py:513
        self.flownet2 = FlowNet2(rgb_max=255.0)
        self.precision = precision
        self.use_cuda_graph = True
        self.label_dtype = torch.int64        # dtype of the label maps: int64 as torch.max returns in the reference, or torch.uint8
        self._graphs = {}
        self._pf_stream, self._pf_queue, self._pf_next, self._tail_done = None, [], 0, [None, None]
        self.reset_tracker()
        self.eval()

    # ------------------------------------------------------------------ housekeeping
    @property
    def act_dtype(self):
        return torch.bfloat16 if self.precision == "bf16" else torch.float32

    def prepare(self, force=False):
        if force:
            self._graphs.clear()          # captured graphs reference the old packed weights
            self._pf_queue, self._tail_done = [], [None, None]
        for m in (self.backbone, self.neck, self.extra_neck, self.panopticFPN, self.rpn_head, self.bbox_head,
                  self.track_head, self.mask_head, self.flownet2):
            m.prepare(force)
        return self

    def reset_tracker(self):
        self.prev_n = 0
        self.prev_roi_feats = self.prev_bboxes = self.prev_det_labels = None

    def extract_feat(self, x_nhwc):
        return self.neck(self.backbone(x_nhwc))

    # ------------------------------------------------------------------ flow
    def compute_flow(self, img, ref_img, scale_factor=0.25, taps=None):
        """panoptic_fusetrack.py:117-143: FlowNet2 on the de-normalised pair, bilinear x0.25 and x0.25 scale.
        img, ref_img: NCHW fp32 CUDA.  Returns NHWC fp32 [1,H/4,W/4,2]."""
        n, _, H, W = img.shape
        assert n == 1 and H % 64 == 0 and W % 64 == 0, "Flownet input must be divisible by 64."
        dev = img.device
        x6 = empty_nhwc(1, H, W, 6, self.act_dtype, dev)
        ops.flownet_input(img, ref_img, self.std, self.mean, 255.0, torch.empty(3, dtype=torch.float64, device=dev), x6)
        flow = self.flownet2(x6, taps)
        out = torch.empty(1, int(H * scale_factor), int(W * scale_factor), 2, dtype=torch.float32, device=dev)
        ops.resize_bilinear(flow, out, mul=scale_factor)
        if taps is not None:
            taps['flow_full'] = flow
        return out

    # ------------------------------------------------------------------ detection + tracking
    def _mask_roi(self, rois, cls_score, bbox_pred, nroi, nroi_dev, img_h, img_w):
        """MaskROI.forward (mask_roi.py:37-147) on device. Returns det_rois [cap,5], cls_idx, cls_prob, kout."""
        dev = rois.device
        nc = self.bbox_head.num_classes
        m = nroi * (nc - 1)
        cand = torch.empty(m, 5, device=dev)
        cand_cls = torch.empty(m, dtype=torch.int32, device=dev)
        cand_prob = torch.empty(m, device=dev)
        ncand = torch.zeros(1, dtype=torch.int32, device=dev)
        ops.maskroi_candidates(rois, cls_score, bbox_pred, nroi, nc, self.score_thresh, img_h, img_w, cand, cand_cls,
                               cand_prob, ncand, nroi_dev)
        p_sorted = torch.empty(m, device=dev)
        slot_sorted = torch.empty(m, dtype=torch.int32, device=dev)
        ops.sort_desc(cand_prob, p_sorted, slot_sorted, m, torch.empty(ops.sort_ws_bytes(m), dtype=torch.uint8, device=dev))
        cand_sorted = torch.empty(m, 5, device=dev)
        ops.gather_rows(cand, slot_sorted, m, 5, cand_sorted)
        keep = torch.empty(m, dtype=torch.int32, device=dev)
        nkeep = torch.zeros(1, dtype=torch.int32, device=dev)
        ops.nms(cand_sorted, m, self.nms_thresh, keep, nkeep, torch.empty(max(ops.nms_ws_bytes(m), 8), dtype=torch.uint8, device=dev),
                n_dev=ncand)
        det_rois = torch.empty(MAX_DET_CAP, 5, device=dev)
        cls_idx = torch.empty(MAX_DET_CAP, dtype=torch.int32, device=dev)
        cls_prob = torch.empty(MAX_DET_CAP, device=dev)
        kout = torch.zeros(2, dtype=torch.int32, device=dev)
        ops.maskroi_finalize(cand_sorted, slot_sorted, cand_cls, keep, nkeep, self.max_det, MAX_DET_CAP, det_rois, cls_idx,
                             cls_prob, kout)
        return det_rois, cls_idx, cls_prob, kout

    def _track(self, det_roi_feats, det_boxes, det_labels, cls_prob, k, is_first, taps=None):
        """panoptic_fusetrack.py:399-469 on device; returns det_obj_ids int32 [k] (device)."""
        dev = det_boxes.device
        feat_len = det_roi_feats[0].numel()
        if self.prev_roi_feats is None or self.prev_roi_feats.dtype != det_roi_feats.dtype:
            self.prev_roi_feats = torch.zeros((TRACK_CAP,) + tuple(det_roi_feats.shape[1:]), dtype=det_roi_feats.dtype, device=dev)
            self.prev_bboxes = torch.zeros(TRACK_CAP, 4, device=dev)
            self.prev_det_labels = torch.zeros(TRACK_CAP, dtype=torch.int32, device=dev)
            self.prev_n = 0
        ids = torch.empty(k, dtype=torch.int32, device=dev)
        new_m = torch.zeros(1, dtype=torch.int32, device=dev)
        if is_first or self.prev_n == 0:
            # ids = arange(k); memory := detections  (:400-406)
            mem_src = torch.arange(TRACK_CAP, dtype=torch.int32, device=dev)      # host-built constant table
            mem_src[k:] = -1
            ids.copy_(mem_src[:k])
            new_m.fill_(k)
            ops.track_update(self.prev_roi_feats, det_roi_feats, feat_len, self.prev_bboxes, det_boxes, self.prev_det_labels,
                             det_labels, mem_src, 0, TRACK_CAP, new_m)
            self.prev_n = k
            return ids
        m = self.prev_n
        emb = self.track_head.embed(det_roi_feats[:k])
        ref_emb = self.track_head.embed(self.prev_roi_feats[:m])
        match_ids = torch.empty(k, dtype=torch.int32, device=dev)
        comp = torch.empty(k, m + 1, device=dev)
        mem_src = torch.empty(TRACK_CAP, dtype=torch.int32, device=dev)
        ws = torch.empty((k * m + k + 2 * TRACK_CAP) * 4, dtype=torch.uint8, device=dev)
        assert emb.is_contiguous() or emb.stride(0) == emb.shape[1]
        ops.track_assign(emb, ref_emb, k, m, emb.shape[1], det_boxes, self.prev_bboxes, det_labels, self.prev_det_labels,
                         cls_prob, self.track_head.match_coeff, TRACK_CAP, ids, match_ids, comp, mem_src, new_m, ws)
        ops.track_update(self.prev_roi_feats, det_roi_feats, feat_len, self.prev_bboxes, det_boxes, self.prev_det_labels,
                         det_labels, mem_src, m, TRACK_CAP, new_m)
        self.prev_n = int(new_m.item())                     # 4-byte read-back: tracker memory size
        if taps is not None:
            taps.update(comp_scores=comp, match_ids=match_ids)
        return ids

    # ------------------------------------------------------------------ static part + CUDA graph
    def _static_eager(self, img, ref_img, img_shape, taps=None, ref_feats=None):
        """ref_feats: FPN features (tuple of 5 NHWC maps) of the reference frame from an earlier call -- in a clip the
        reference frame of frame t IS frame t - 1 (tools/dataset/cityscapes_vps.py:137-142), so its features were already
        computed as `x` of the previous pair; only the current frame then goes through ResNet-50-FPN."""
        dev = img.device
        _, _, H, W = img.shape
        dt = self.act_dtype
        # ResNet-50-FPN does not depend on the flow: it runs as a parallel branch (side stream / parallel graph branch), so
        # the many launches that cannot fill 148 SMs on either side overlap with the other side's kernels
        br = ops.Branch("r50fpn")
        if br.side is None:
            ops.SCOPE[0] = 'flownet2'
            flow = self.compute_flow(img, ref_img, 0.25, taps)
        ops.SCOPE[0] = 'r50fpn'
        br.__enter__()
        # both frames go through ResNet-50-FPN as ONE batch of 2 (the reference runs extract_feat twice,
        # panoptic_fusetrack.py:516-517; frozen BN makes the batched pass identical per image): half the launches, twice
        # the tiles per launch for the small-spatial stages, weights fetched once
        nb = 1 if ref_feats is not None else 2
        xr_in = empty_nhwc(nb, H, W, 3, dt, dev)
        ops.nchw_to_nhwc(img, xr_in[0:1])
        if ref_feats is None:
            ops.nchw_to_nhwc(ref_img, xr_in[1:2])
        feats = self.extract_feat(xr_in)
        br.__exit__(None, None, None)
        if br.side is not None:
            ops.SCOPE[0] = 'flownet2'
            flow = self.compute_flow(img, ref_img, 0.25, taps)
            br.join(*feats)
        x = tuple(f[0:1] for f in feats)
        ref_x = tuple(f[1:2] for f in feats) if ref_feats is None else tuple(ref_feats)
        ops.SCOPE[0] = 'bfp_tcea'
        xf = self.extra_neck(x, ref_x, flow, taps)
        ops.SCOPE[0] = 'upsnet_fpn'
        nl = self.panopticFPN.num_levels
        # the semantic head and the RPN -> bbox head -> MaskROI chain both start from xf and meet only in the fusion tail
        br2 = ops.Branch("upsnet_fpn")
        with br2:
            fcn_output, fcn_score = self.panopticFPN(xf[0:nl], want_full=taps is not None)
        ops.SCOPE[0] = 'rpn'
        # RPN (test_mixins.py:13-17, rpn_head.py:55-104)
        heads = self.rpn_head(xf)
        proposals_t, rois, nprop = self.rpn_head.get_bboxes(heads, img_shape, self.test_cfg['rpn'], taps)
        nroi = proposals_t.shape[0]
        # bbox head + MaskROI (:367-389)
        ops.SCOPE[0] = 'bbox_head'
        roi_feats = self.bbox_roi_extractor(xf, rois, nroi, nprop)
        cls_score, bbox_pred, _ = self.bbox_head(roi_feats)
        det_rois, cls_idx, cls_prob, kout = self._mask_roi(rois, cls_score, bbox_pred, nroi, nprop, float(H), float(W))
        br2.join(fcn_score, fcn_output)
        return dict(flow=flow, x=x, ref_x=ref_x, xf=xf, fcn_output=fcn_output, fcn_score=fcn_score, heads=heads,
                    proposals=proposals_t, rois=rois, nprop=nprop, roi_feats=roi_feats, cls_score=cls_score,
                    bbox_pred=bbox_pred, det_rois=det_rois, cls_idx=cls_idx, cls_prob=cls_prob, kout=kout)

    def _static_part(self, img, ref_img, img_shape, use_graph, taps=None, slot=0, ref_feats=None):
        if not use_graph:
            return self._static_eager(img, ref_img, img_shape, taps, ref_feats)
        cached = ref_feats is not None
        key = (tuple(img.shape), img_shape, self.precision, img.device.index, slot, cached)   # slot: ping-pong graph instance
        ent = self._graphs.get(key)
        if ent is None:
            # first call for this key runs eagerly (lazy weight packing, function attributes, scratch allocations
            # must happen outside a capture); the second call captures
            self._graphs[key] = "warm"
            return self._static_eager(img, ref_img, img_shape, None, ref_feats)
        if ent == "warm":
            g_img, g_ref = torch.empty_like(img), torch.empty_like(ref_img)
            g_img.copy_(img); g_ref.copy_(ref_img)
            g_feats = None
            if cached:          # the graph reads the cached features from its own static buffers
                g_feats = tuple(torch.empty_like(f) for f in ref_feats)
                for d_, s_ in zip(g_feats, ref_feats):
                    d_.copy_(s_)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            n0 = ops.launch_count()
            with torch.cuda.graph(graph):
                outs = self._static_eager(g_img, g_ref, img_shape, None, g_feats)
            ent = self._graphs[key] = (graph, g_img, g_ref, outs, ops.launch_count() - n0, g_feats)
            ops.lib().vps_add_launch_count(-ent[4])        # capture itself launched nothing
        graph, g_img, g_ref, outs, nlaunch, g_feats = ent
        g_img.copy_(img, non_blocking=True)
        g_ref.copy_(ref_img, non_blocking=True)
        if cached:
            for d_, s_ in zip(g_feats, ref_feats):
                d_.copy_(s_, non_blocking=True)
        graph.replay()
        ops.lib().vps_add_launch_count(nlaunch)            # kernels of ours re-launched by the replay
        return outs

    @torch.no_grad()
    def prefetch(self, img, img_meta, ref_img=None, ref_feats=None):
        """Enqueue the static part (flow, backbones, necks, semantic head, RPN, bbox head, MaskROI -- everything that does
        not depend on the tracker) of a FUTURE `simple_test(img, ...)` call on a side stream.  Two graph instances
        ping-pong, so frame i+1's static part overlaps frame i's data-dependent tail and its host round-trips.  The
        matching simple_test call (same `img` object, in call order) picks the result up; results are identical."""
        if isinstance(ref_img, (list, tuple)):
            ref_img = ref_img[0]
        meta = img_meta[0] if isinstance(img_meta, (list, tuple)) else img_meta
        if not (self.use_cuda_graph and ops.PROFILE is None):
            return
        self.prepare()
        ops.F32_TC[0] = self.precision == "tc32"
        cur = torch.cuda.current_stream(img.device)
        if self._pf_stream is None:
            self._pf_stream = torch.cuda.Stream(img.device)
        st = self._pf_stream
        slot = self._pf_next
        self._pf_next ^= 1
        st.wait_stream(cur)                                     # inputs are ready on the caller's stream
        if self._tail_done[slot] is not None:
            st.wait_event(self._tail_done[slot])                # the tail that last read this slot's outputs is done
        with torch.cuda.stream(st):
            a = img.contiguous().float()
            b = ref_img.contiguous().float()
            outs = self._static_part(a, b, tuple(meta['img_shape'][:2]), True, None, slot, ref_feats)
            ev = torch.cuda.Event()
            ev.record(st)
        img.record_stream(st)
        ref_img.record_stream(st)
        self._pf_queue.append((img, slot, outs, ev))

    # ------------------------------------------------------------------ the hot path
    @torch.no_grad()
    def simple_test(self, img, img_meta, proposals=None, rescale=False, ref_img=None, taps=None, ref_feats=None):
        """panoptic_fusetrack.py:502-606.  img / ref_img: NCHW fp32 CUDA tensors [1,3,H,W] (ref_img may be the
        one-element list the reference's collate produces).  Returns (bbox_results, segm_results, pano_results).
        ref_feats: optional cached FPN features of ref_img (pano_results['fpn_feats'] of the call that had ref_img as its
        current frame): skips the reference frame's ResNet-50-FPN pass, results are bit-identical."""
        assert proposals is None
        if isinstance(ref_img, (list, tuple)):
            ref_img = ref_img[0]
        meta = img_meta[0] if isinstance(img_meta, (list, tuple)) else img_meta
        assert 'city' in meta['filename'] and 'iid' in meta            # :375
        self.prepare()
        assert self.precision in ("tc32", "bf16", "fp32"), self.precision
        ops.F32_TC[0] = self.precision == "tc32"
        dev = img.device
        n, _, H, W = img.shape
        assert n == 1
        img_arg = img
        img = img.contiguous().float()
        ref_img = ref_img.contiguous().float()
        # ---- static part (flow, backbones, fuse neck, semantic head, RPN, bbox head, MaskROI): fixed shapes, no host
        # decisions -> replayed as ONE CUDA graph after the first eager call for this (shape, precision)
        use_graph = self.use_cuda_graph and taps is None and ops.PROFILE is None
        pf_slot = None
        if self._pf_queue and self._pf_queue[0][0] is img_arg and taps is None:
            _, pf_slot, st, ev = self._pf_queue.pop(0)           # static part was enqueued by prefetch()
            cur = torch.cuda.current_stream(dev)
            cur.wait_event(ev)
            for v in st.values():
                for t in (v if isinstance(v, (tuple, list)) else (v,)):
                    if torch.is_tensor(t):
                        t.record_stream(cur)
        else:
            assert not self._pf_queue, "prefetch() / simple_test() calls out of order"
            st = self._static_part(img, ref_img, tuple(meta['img_shape'][:2]), use_graph, taps, 0, ref_feats)
        flow, x, ref_x, xf, fcn_output, fcn_score = st['flow'], st['x'], st['ref_x'], st['xf'], st['fcn_output'], st['fcn_score']
        heads, proposals_t, rois, nprop = st['heads'], st['proposals'], st['rois'], st['nprop']
        roi_feats, cls_score, bbox_pred = st['roi_feats'], st['cls_score'], st['bbox_pred']
        det_rois, cls_idx, cls_prob, kout = st['det_rois'], st['cls_idx'], st['cls_prob'], st['kout']
        ops.SCOPE[0] = 'track_mask_fuse'
        k, dummy = [int(v) for v in kout.tolist()]            # 8-byte read-back: number of detections
        if self.precision == "tc32" and ops.tc32_overflow():
            # leave the detector usable (e.g. for the fp32 rerun suggested below): drop the static parts prefetch() enqueued
            # for later frames, and clear the counts their kernels may still add once they finish
            self._pf_queue.clear()
            torch.cuda.synchronize(dev)
            ops.tc32_overflow(reset=True)
            raise ops.VpsError("tc32: an activation or weight exceeded the fp16 range (65504) of the main tensor-core "
                               "product; use precision='fp32' for this input")
        iid = meta['iid']
        is_first = (iid % 10000) == 1
        det_roi_feats = self.bbox_roi_extractor(xf, det_rois, k)
        det_boxes_c = torch.empty(MAX_DET_CAP, 4, device=dev)
        det_labels = torch.empty(MAX_DET_CAP, dtype=torch.int32, device=dev)
        ops.det_split(det_rois, cls_idx, MAX_DET_CAP, det_boxes_c, det_labels)
        cls_idx_h = cls_idx[:k].cpu().numpy()
        det_obj_ids = self._track(det_roi_feats, det_boxes_c, det_labels, cls_prob, k, is_first, taps)

        # ---- mask head on the detections (:561-568)
        mask_feats = self.mask_roi_extractor(xf, det_rois, k)
        mask_pred = self.mask_head(mask_feats)
        ms = mask_pred.shape[1]
        mask_logit = torch.empty(k, ms, ms, device=dev)
        ops.select_class(mask_pred, cls_idx, k, mask_logit)

        # ---- MaskRemoval + fused panoptic argmax (:572-597)
        order = torch.empty(k, dtype=torch.int32, device=dev)
        ops.sort_desc(cls_prob, torch.empty(k, device=dev), order, k, torch.empty(ops.sort_ws_bytes(k), dtype=torch.uint8, device=dev))
        nthings = self.panopticFPN.num_things_classes
        keep_sorted = torch.zeros(MAX_DET_CAP, dtype=torch.int32, device=dev)
        nkeep = torch.zeros(1, dtype=torch.int32, device=dev)
        if not dummy:
            ops.mask_removal(det_boxes_c, order, k, mask_logit, ms, cls_idx, H, W, self.fraction_threshold,
                             torch.empty(nthings, H, W, dtype=torch.uint8, device=dev), nthings,
                             torch.empty(2 * k, dtype=torch.int32, device=dev), torch.empty(k, dtype=torch.int32, device=dev),
                             keep_sorted, nkeep)
        pano = torch.empty(H, W, dtype=self.label_dtype, device=dev)
        sem = torch.empty(H, W, dtype=self.label_dtype, device=dev)
        num_stuff = self.panopticFPN.num_stuff_classes
        ops.panoptic_fuse(fcn_score, det_boxes_c, cls_idx, mask_logit, ms, keep_sorted, nkeep, MAX_DET_CAP, num_stuff,
                          dummy, H, W, pano, sem)

        # ---- results (:545-546, 598-606); small per-detection arrays are assembled on the host
        nk = int(nkeep.item()) if not dummy else 0
        keep_h = keep_sorted[:nk].cpu().numpy().astype(np.int64)
        if dummy or nk == 0:
            keep_h = np.array([0], dtype=np.int64)           # mask_removal.py:52-54,89-91
        det_rois_h = det_rois[:k].cpu().numpy()
        cls_prob_h = cls_prob[:k].cpu().numpy()
        ids_h = det_obj_ids[:k].cpu().numpy()
        labels_h = cls_idx_h - 1
        h0, w0 = meta['img_shape'][:2]
        pano_results = {
            'fcn_outputs': sem[None, :h0, :w0],
            'panoptic_cls_inds': torch.from_numpy(cls_idx_h[keep_h].astype(np.int64)).to(dev),
            'panoptic_cls_prob': torch.from_numpy(cls_prob_h[keep_h]).to(dev),
            'panoptic_det_labels': torch.from_numpy(labels_h[keep_h].astype(np.int64)).to(dev),
            'panoptic_det_obj_ids': torch.from_numpy(ids_h[keep_h]).to(dev),
            'panoptic_outputs': pano[None, :h0, :w0],
            # host copies of the two small per-instance arrays (already on the host here): the post-processing that follows
            # the path (vps_b200.postproc.PanUnifier) needs them there
            'host': dict(panoptic_cls_inds=cls_idx_h[keep_h].astype(np.int64), panoptic_det_obj_ids=ids_h[keep_h]),
            # FPN features of the current frame: a streaming caller hands them back as `ref_feats` of the next pair
            'fpn_feats': x,
        }
        bbox_results = bbox2result_with_id(det_rois_h[:, 1:], labels_h, ids_h)
        segm_results = [[] for _ in range(self.mask_head.num_classes - 1)]     # :484-485 (`or True`)
        if taps is not None:
            taps.update(flow=flow, fpn=x, ref_fpn=ref_x, fused=xf, fcn_score=fcn_score, fcn_output=fcn_output,
                        rpn_heads=heads, proposals=proposals_t, nprop=nprop, roi_feats=roi_feats, cls_score=cls_score,
                        bbox_pred=bbox_pred, det_rois=det_rois[:k], cls_idx=cls_idx[:k], cls_prob=cls_prob[:k],
                        det_roi_feats=det_roi_feats, mask_logit=mask_logit, keep_inds=keep_h, det_obj_ids_all=ids_h,
                        order=order)
        if pf_slot is not None:                                   # this slot's graph may be replayed once the tail is done
            done = torch.cuda.Event()
            done.record(torch.cuda.current_stream(dev))
            self._tail_done[pf_slot] = done
        return bbox_results, segm_results, pano_results

    # reference-compatible entry (base.py:79-104)
    def forward_test(self, imgs, img_metas, **kwargs):
        for var, name in [(imgs, 'imgs'), (img_metas, 'img_metas')]:
            if not isinstance(var, list):
                raise TypeError('{} must be a list, but got {}'.format(name, type(var)))
        if len(imgs) != len(img_metas):
            raise ValueError('num of augmentations ({}) != num of image meta ({})'.format(len(imgs), len(img_metas)))
        assert imgs[0].size(0) == 1 and len(imgs) == 1
        return self.simple_test(imgs[0], img_metas[0], **kwargs)

    def forward(self, img, img_meta, return_loss=True, **kwargs):
        if return_loss:
            raise NotImplementedError("forward_train: training path is a later scope row (SURVEY 8f rank 3)")
        return self.forward_test(img, img_meta, **kwargs)
