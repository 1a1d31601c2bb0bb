"""CPU: the oracle restatement reproduces the golden vectors generated from the REFERENCE's own python code
(tests/golden/make_golden.py) on the seeded 2-frame clip: integer outputs bit-exact, floats to 1e-5."""
import os

import numpy as np
import torch

from tests.e2e_util import make_pair
from tests.golden.make_golden import THREADS, keep, weights_digest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fusetrack_clip_128x256.npz")


def test_oracle_reproduces_reference_golden_clip():
    from oracle.weights import make_model
    g = np.load(GOLD)
    H, W = int(g["H"]), int(g["W"])
    oracle = make_model("C", 0, scales=g["calib_scales"])       # the golden run's calibration, whatever this host measures
    assert weights_digest(oracle.state_dict()) == str(g["weights_sha256"]), \
        "synthetic weights differ from the ones the golden file was generated with (torch RNG drift?)"
    img, ref = make_pair(H, W)
    threads = torch.get_num_threads()
    torch.set_num_threads(THREADS)
    try:
        check_clip(g, oracle, img, ref, H, W)
    finally:
        torch.set_num_threads(threads)


def check_clip(g, oracle, img, ref, H, W):
    for f, (iid, a, b) in enumerate(((10001, img, ref), (10002, ref, img))):
        taps = {}
        r = oracle.simple_test(a, dict(iid=iid, img_shape=(H, W, 3)), b, taps)
        p = r[2]
        assert np.array_equal(p["panoptic_outputs"].numpy().astype(np.uint8), g["f%d_pano" % f])
        assert np.array_equal(p["fcn_outputs"].numpy().astype(np.uint8), g["f%d_sem" % f])
        assert np.array_equal(p["panoptic_cls_inds"].numpy(), g["f%d_cls_inds" % f])
        assert np.array_equal(p["panoptic_det_obj_ids"].numpy(), g["f%d_obj_ids" % f])
        assert np.array_equal(p["panoptic_det_labels"].numpy(), g["f%d_det_labels" % f])
        assert np.abs(p["panoptic_cls_prob"].numpy() - g["f%d_cls_prob" % f]).max() <= 1e-6
        ids = sorted(r[0].keys())
        assert ids == g["f%d_bbox_ids" % f].tolist()
        assert np.abs(np.stack([r[0][i]["bbox"] for i in ids]) - g["f%d_bbox" % f]).max() <= 1e-4
        assert np.abs(keep("flow_full", taps["flow_full"].numpy()) - g["f%d_flow_full" % f]).max() <= 1e-5
        assert np.abs(keep("fcn_score", taps["fcn_score"].numpy()) - g["f%d_fcn_score" % f]).max() <= 1e-5
        assert np.abs(keep("cls_score", taps["cls_score"].numpy()) - g["f%d_cls_score" % f]).max() <= 1e-5
        assert np.abs(keep("fused0", taps["fused"][0].numpy()) - g["f%d_fused0" % f]).max() <= 1e-5
