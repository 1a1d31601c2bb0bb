"""CPU: the drop-in boundary -- registries, config loader, state_dict layout, C-ABI exports, no-fallback rule."""
import ast
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the `model` / `test_cfg` entries of the reference's configs/cityscapes/fusetrack.py (tests/golden/make_config_golden.py)
REF_CFG = os.path.join(ROOT, "tests", "golden", "fusetrack_config.txt")


def reference_config(tmp_path):
    """the stored reference config, written back as a python config file and loaded like one"""
    path = tmp_path / "fusetrack.py"
    path.write_text("".join("%s = %r\n" % kv for kv in ast.literal_eval(open(REF_CFG).read()).items()))
    from vps_b200 import Config
    return Config.fromfile(str(path))


def test_registry_semantics_match_reference():
    from vps_b200.registry import Registry, build_from_cfg
    r = Registry("thing")

    @r.register_module
    class A(object):
        def __init__(self, x, y=2):
            self.x, self.y = x, y
    with pytest.raises(KeyError):          # duplicate name (mmdet/utils/registry.py:40-43)
        r.register_module(A)
    with pytest.raises(TypeError):
        r.register_module(3)
    obj = build_from_cfg(dict(type="A", x=1), r, default_args=dict(y=5, x=9))
    assert (obj.x, obj.y) == (1, 5)        # cfg wins over default_args (setdefault)
    with pytest.raises(KeyError):
        build_from_cfg(dict(type="Nope"), r)
    assert r.get("A") is A and r.get("B") is None and "A" in r.module_dict


def test_all_reference_names_are_registered():
    import vps_b200 as V
    assert V.DETECTORS.get("PanopticFuseTrack") is not None
    for reg, names in ((V.BACKBONES, ["ResNet"]), (V.NECKS, ["FPN"]), (V.EXTRA_NECKS, ["BFPTcea"]),
                       (V.PANOPTIC, ["UPSNetFPN"]), (V.ROI_EXTRACTORS, ["SingleRoIExtractor"]),
                       (V.HEADS, ["RPNHead", "SharedFCBBoxHead", "TrackHead", "FCNMaskHead"]),
                       (V.LOSSES, ["CrossEntropyLoss", "SmoothL1Loss"])):
        for n in names:
            assert reg.get(n) is not None, n


def test_reference_config_loads_unmodified_and_builds(tmp_path):
    from vps_b200 import build_detector, fusetrack_cfg
    cfg = reference_config(tmp_path)
    assert hasattr(cfg.test_cfg, "flownet2") and not hasattr(cfg.test_cfg, "nope")
    assert cfg.test_cfg.rpn.nms_thr == 0.7 and cfg.model.bbox_head.num_classes == 9
    det = build_detector(cfg.model, train_cfg=None, test_cfg=cfg.test_cfg)
    mine = fusetrack_cfg()
    ref_model = {k: v for k, v in cfg.model.items()}
    ref_model["pretrained"] = None
    assert _plain(ref_model) == _plain(mine["model"])
    assert _plain(cfg.test_cfg) == _plain(mine["test_cfg"])
    assert det.class_mapping == {i: 10 + i for i in range(1, 9)}


def test_b200_classes_install_into_mmdet_style_registries(tmp_path):
    """SURVEY 8b, second route: install_into_reference() overwrites the entries of the reference's registries
    (mmdet.models.registry.*.module_dict[name]) with the B200 classes, after which a build through those registries from the
    reference config yields the B200 detector.  The registry module is a stand-in with the reference's nine registry
    names, each holding a placeholder class under every name the B200 side registers (the Registry contract is pinned by
    test_registry_semantics_match_reference)."""
    import types
    from vps_b200.registry import REGISTRIES, Registry, build_from_cfg, install_into_reference
    RR = types.SimpleNamespace()
    for attr, mine in REGISTRIES.items():
        theirs = Registry(mine.name)
        for name in mine.module_dict:
            theirs.register_module(type(name, (), {"__module__": "mmdet.models.placeholder"}))
        setattr(RR, attr, theirs)
    done = install_into_reference(RR)
    assert ("DETECTORS", "PanopticFuseTrack") in done and ("BACKBONES", "ResNet") in done and len(done) >= 12
    assert all(getattr(RR, a).get(n).__module__.startswith("vps_b200.") for a, n in done)
    cfg = reference_config(tmp_path)
    cfg.model["pretrained"] = None
    det = build_from_cfg(cfg.model, RR.DETECTORS, dict(train_cfg=None, test_cfg=cfg.test_cfg))
    assert type(det).__module__ == "vps_b200.detector", type(det)
    for name in ("backbone", "neck", "extra_neck", "panopticFPN", "rpn_head", "bbox_head", "track_head", "mask_head"):
        assert type(getattr(det, name)).__module__.startswith("vps_b200."), name
    assert len(det.state_dict()) == 629


def _plain(x):
    if isinstance(x, dict):
        return {k: _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    return x


def test_state_dict_layout_matches_oracle_and_reference_names():
    from oracle.model import PanopticFuseTrack as Oracle
    from vps_b200 import ConfigDict, build_detector, fusetrack_cfg
    c = fusetrack_cfg()
    det = build_detector(ConfigDict(c["model"]), train_cfg=None, test_cfg=ConfigDict(c["test_cfg"]))
    o = Oracle()
    a, b = det.state_dict(), o.state_dict()
    assert set(a) == set(b)
    assert all(a[k].shape == b[k].shape for k in a)
    det.load_state_dict(b, strict=True)
    for k in ("backbone.layer1.0.downsample.0.weight", "neck.lateral_convs.3.conv.bias",
              "extra_neck.liteflownet.flow_estimator.convs.2.0.weight", "extra_neck.tcea_fusion.sAtt_add_2.bias",
              "extra_neck.refine.conv.weight", "panopticFPN.deform_convs.0.3.conv_offset.weight",
              "panopticFPN.deform_convs.0.6.conv.weight", "panopticFPN.deform_convs.0.7.bias",
              "panopticFPN.conv_pred.conv.weight", "rpn_head.rpn_reg.bias", "bbox_head.shared_fcs.1.weight",
              "track_head.fcs.0.weight", "mask_head.convs.3.conv.weight", "mask_head.upsample.weight",
              "flownet2.flownetc.conv_redir.0.weight", "flownet2.flownets_2.upsampled_flow6_to_5.weight",
              "flownet2.flownets_d.inter_conv3.0.bias", "flownet2.flownetfusion.predict_flow0.weight"):
        assert k in a, k


def test_cabi_library_exports_every_declared_symbol():
    from vps_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "vps_b200.h")).read()
    declared = set(re.findall(r"^\s*(?:const char\*|int64_t|int|void)\s+(vps_[a-z0-9_]+)\s*\(", hdr, re.M))
    assert len(declared) >= 40
    assert declared == set(_lib.EXPORTS), (declared ^ set(_lib.EXPORTS))
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in declared:
        assert hasattr(lib, s), s
    assert lib.vps_version() >= 100


def test_no_cpu_fallback():
    """The product path must fail loudly without CUDA: no oracle / torch fallback."""
    from vps_b200 import ConfigDict, build_detector, fusetrack_cfg
    c = fusetrack_cfg()
    det = build_detector(ConfigDict(c["model"]), train_cfg=None, test_cfg=ConfigDict(c["test_cfg"]))
    img = torch.zeros(1, 3, 64, 64)
    with pytest.raises(Exception):
        det.simple_test(img, [dict(filename="city", iid=1, img_shape=(64, 64, 3))], ref_img=[img])
    src = "".join(open(os.path.join(ROOT, "vps_b200", f)).read() for f in os.listdir(os.path.join(ROOT, "vps_b200"))
                  if f.endswith(".py"))
    assert "import oracle" not in src and "from oracle" not in src


def test_synth_table_matches_oracle_calibration():
    """vps_b200.synth.make_weights (table-driven) reproduces oracle.weights.make_model (measured calibration)."""
    from oracle.weights import make_model
    from vps_b200 import ConfigDict, build_detector, fusetrack_cfg
    from vps_b200.synth import make_weights
    c = fusetrack_cfg()
    det = build_detector(ConfigDict(c["model"]), train_cfg=None, test_cfg=ConfigDict(c["test_cfg"]))
    make_weights(det, "C", 0)
    a, b = det.state_dict(), make_model("C", 0).state_dict()
    for k in a:
        tol = 2e-5 * max(1.0, float(b[k].abs().max()))
        assert float((a[k].float() - b[k].float()).abs().max()) <= tol, k
