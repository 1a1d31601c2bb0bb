"""Generate tests/golden/fusetrack_clip_128x256.npz from the REFERENCE's own python code.

The reference (mcahny/vps, /root/reference) is imported through tests/golden/ref_import.py (mmcv / compiled
extensions stubbed, see that file), its PanopticFuseTrack is built from its unmodified
configs/cityscapes/fusetrack.py, loaded with the synthetic weight set "C" (oracle/weights.py, seed 0) and run
on a seeded 2-frame clip.  Outputs (label maps, class ids, track ids, probabilities, boxes) and a few
intermediate tensors captured with forward hooks are stored; tests compare the oracle (CPU) and the CUDA path
(GPU) against them.  Run here (needs /root/reference):  python tests/golden/make_golden.py
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.weights import calibrate, make_model  # noqa: E402
from tests.e2e_util import make_pair, meta  # noqa: E402
from tests.golden.run_reference import build_reference_detector  # noqa: E402

H, W = 128, 256
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fusetrack_clip_128x256.npz")
# host threads of the golden run: the summation order of the CPU kernels, hence the last bits of every float, depends on
# it; tests/test_golden_cpu.py runs the oracle with as many
THREADS = 8


def keep(name, a):
    """the part of an intermediate tensor ([N, C, H, W] maps, [rows, C] cls_score) the golden file stores, which keeps the
    file small: every 4th pixel each way of the maps (and every 16th channel of fused0), every 2nd row of cls_score"""
    if name == "cls_score":
        return a[::2]
    if name == "fused0":
        a = a[:, ::16]
    return a[..., ::4, ::4]


def weights_digest(sd):
    h = hashlib.sha256()
    for k in sorted(sd.keys()):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def main():
    torch.set_num_threads(THREADS)
    oracle = make_model("C", 0, calibrated=False)
    scales = calibrate(oracle)
    sd = oracle.state_dict()
    det = build_reference_detector(sd)
    cap = {}
    det.flownet2.register_forward_hook(lambda m, i, o: cap.__setitem__("flow_full", o.detach().clone()))
    det.panopticFPN.register_forward_hook(lambda m, i, o: cap.__setitem__("fcn_score", o[1].detach().clone()))
    def _first_cls(m, i, o):
        if "cls_score" not in cap:          # first call of the frame = the 1000-proposal pass
            cap["cls_score"] = o[0].detach().clone()
    det.bbox_head.register_forward_hook(_first_cls)
    det.extra_neck.register_forward_hook(lambda m, i, o: cap.__setitem__("fused0", o[0].detach().clone()))
    img, ref = make_pair(H, W)
    out = {"weights_sha256": np.array(weights_digest(sd)), "calib_scales": np.array(scales, np.float64), "H": H, "W": W}
    with torch.no_grad():
        for f, (iid, a, b) in enumerate(((10001, img, ref), (10002, ref, img))):
            cap.clear()
            r = det.simple_test(a, [meta(iid, H, W)], ref_img=[b])
            p = r[2]
            out["f%d_pano" % f] = p["panoptic_outputs"].numpy().astype(np.uint8)
            out["f%d_sem" % f] = p["fcn_outputs"].numpy().astype(np.uint8)
            out["f%d_cls_inds" % f] = p["panoptic_cls_inds"].numpy().astype(np.int32)
            out["f%d_cls_prob" % f] = p["panoptic_cls_prob"].numpy().astype(np.float32)
            out["f%d_obj_ids" % f] = p["panoptic_det_obj_ids"].numpy().astype(np.int32)
            out["f%d_det_labels" % f] = p["panoptic_det_labels"].numpy().astype(np.int32)
            ids = sorted(r[0].keys())
            out["f%d_bbox_ids" % f] = np.array(ids, np.int32)
            out["f%d_bbox" % f] = np.stack([r[0][i]["bbox"] for i in ids]).astype(np.float32)
            for name in ("flow_full", "fcn_score", "cls_score", "fused0"):
                out["f%d_%s" % (f, name)] = keep(name, cap[name].numpy()).astype(np.float32)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT) // 1024, "KiB")


if __name__ == "__main__":
    main()
