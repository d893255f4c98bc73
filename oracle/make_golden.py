"""TEST INFRASTRUCTURE ONLY -- regenerates tests/golden/*.npz by running the UNMODIFIED reference modules
(imported from /root/reference, build container only) on seeded synthetic inputs.

    python -m oracle.make_golden

Inputs are not stored (they are re-derived from the seed by gigapose_b200.synth / the seeded port
weights); each fixture carries float64 checksums of its inputs so RNG drift is detected, plus every output of
the reference retrieval sequence (gigaPose.py:497-604).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

from gigapose_b200 import synth
from . import port, ref_import, ref_run

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
# intra-op threads the fixtures are recorded with: how torch splits fp32 reductions across threads changes their last
# bits, so tests/test_oracle_golden.py runs the port with the same count
GOLDEN_THREADS = 8

RETRIEVAL_CASES = {
    # BASELINE.json configs[0]: single query vs 16 templates, 1 object
    "retrieval_c1": dict(B=1, O=1, T=16, seed=11, sub_batch=None),
    # reduced LM-O shape: several objects, sub-batching as in test.yaml:21 (max_num_dets_per_forward=4)
    "retrieval_small": dict(B=6, O=3, T=24, seed=12, sub_batch=4),
}


def checksum(t: torch.Tensor) -> float:
    return float(t.double().sum())


def input_checksums(case):
    return dict(ck_bank_feat=checksum(case.bank_feat), ck_q_feat=checksum(case.q_feat),
                ck_bank_ist=checksum(case.bank_ist), ck_q_ist=checksum(case.q_ist),
                ck_bank_mask=checksum(case.bank_mask16), ck_q_mask=checksum(case.q_mask16))


def write_reference_init_case(B=3, O=2, T=12, seed=5):
    """The retrieval sequence with the reference's own seeded IST initialisation (`ref_run.build_ist`), not the port's
    weights: the regressor is rebuilt from the seed by the test, checked by `ck_regressor`."""
    case = synth.make_feature_case(B=B, O=O, T=T, seed=seed)
    ist = ref_run.build_ist()
    out = ref_run.retrieval(synth.to_reference_layout(case), ist)
    arrays = {k: v.numpy() for k, v in out.items()}
    arrays.update({k: np.float64(v) for k, v in input_checksums(case).items()})
    arrays["ck_regressor"] = np.float64(sum(checksum(v) for v in ist.regressor.state_dict().values()))
    arrays["cfg"] = np.array([B, O, T, seed, 0])
    np.savez_compressed(os.path.join(GOLDEN_DIR, "retrieval_reference_init.npz"), **arrays)
    print("retrieval_reference_init", {k: v.shape for k, v in arrays.items() if v.ndim})


def reference_ist_with_port_weights():
    ist = ref_run.build_ist()
    ist.regressor.load_state_dict(port.RegressorPort().state_dict())
    ist.backbone.load_state_dict(port.ISTBackbonePort().state_dict())
    return ist.eval()


def main():
    torch.set_num_threads(GOLDEN_THREADS)
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    ist = reference_ist_with_port_weights()
    for name, cfg in RETRIEVAL_CASES.items():
        case = synth.make_feature_case(B=cfg["B"], O=cfg["O"], T=cfg["T"], seed=cfg["seed"])
        out = ref_run.retrieval(synth.to_reference_layout(case), ist, sub_batch=cfg["sub_batch"])
        arrays = {k: v.numpy() for k, v in out.items()}
        arrays.update({k: np.float64(v) for k, v in input_checksums(case).items()})
        arrays["cfg"] = np.array([cfg["B"], cfg["O"], cfg["T"], cfg["seed"], cfg["sub_batch"] or 0])
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **arrays)
        print(name, {k: v.shape for k, v in arrays.items() if hasattr(v, "shape") and v.ndim})
    write_reference_init_case()

    # a1: reference AENet (ae_net.py:55-69) wrapping the seeded ViT restatement; a6: reference ResNet
    ns = ref_import.load()
    rgb, _ = synth.make_crops(2, seed=31)
    vit = port.DinoV2Port()
    ae = ns.AENet("dinov2_vitl14", dinov2_model=vit, descriptor_size=1024, max_batch_size=64)
    with torch.no_grad():
        feat = ae(rgb)                                             # [2,1024,16,16]
        ist_feat = ist.forward_by_chunk(rgb)                       # [2,256,16,16]
    np.savez_compressed(os.path.join(GOLDEN_DIR, "backbones.npz"),
                        ck_rgb=np.float64(checksum(rgb)),
                        ae_feat_sub=feat[:, ::8].numpy(), ist_feat_sub=ist_feat[:, ::2].numpy(),
                        ae_feat_sum=np.float64(checksum(feat)), ist_feat_sum=np.float64(checksum(ist_feat)))
    print("backbones", feat.shape, ist_feat.shape)


if __name__ == "__main__":
    sys.exit(main())
