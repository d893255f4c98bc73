"""TEST INFRASTRUCTURE ONLY -- regenerates tests/golden/model_configs.json: the reference's Hydra model configs
(`configs/model/*.yaml` of a reference checkout), parsed, for tests/test_boundary_cpu.py.

    python -m oracle.make_golden_configs
"""
from __future__ import annotations

import json
import os

import yaml

from . import ref_import

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "model_configs.json")
CONFIGS = ("model/large.yaml", "model/ae_net/dinov2_l.yaml", "model/ist_net/resnet.yaml")


def main():
    out = {}
    for rel in CONFIGS:
        with open(os.path.join(ref_import.REF_ROOT, "configs", rel)) as f:
            out[rel] = yaml.safe_load(f)
    with open(GOLDEN, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(GOLDEN, sorted(out))


if __name__ == "__main__":
    main()
