"""Generate tests/golden/fusetrack_config.txt: the `model` and `test_cfg` entries of the reference's unmodified
configs/cityscapes/fusetrack.py as vps_b200.Config parses them, as one python literal (ast.literal_eval reads it back with
its tuples and integer keys).  tests/test_boundary.py builds the detector from them and compares them with
vps_b200.fusetrack_cfg().  Needs the reference tree (VPS_REFERENCE, see
tests/golden/ref_import.py):  python tests/golden/make_config_golden.py
"""
import os
import pprint
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests.golden.ref_import import REF  # noqa: E402
from vps_b200.config import Config  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fusetrack_config.txt")


def main():
    cfg = Config.fromfile(os.path.join(REF, "configs", "cityscapes", "fusetrack.py"))
    with open(OUT, "w") as f:
        f.write(pprint.pformat({"model": dict(cfg.model), "test_cfg": dict(cfg.test_cfg)}, sort_dicts=False) + "\n")
    print("wrote", OUT)


if __name__ == "__main__":
    main()
