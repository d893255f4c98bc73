#!/usr/bin/env python
"""Similarity kernel at the per-GPU shard of BASELINE.json configs[4] (stress: 256 objects x 576 templates over 8 GPUs
= 72 local templates per object, batch 256, ONE query per object -> no template reuse, B_o = 1): reports the achieved
HBM GB/s and TFLOP/s of `sim_search_pair_kernel` in both precisions.  Feature-level synthetic data generated on the device.

    python scripts/stress_sim.py [--objects 256] [--templates 72] [--out gpurun_out/stress_sim.json]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gigapose_b200 import synth  # noqa: E402
from gigapose_b200.engine import Engine  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--objects", type=int, default=256)
    ap.add_argument("--templates", type=int, default=72)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "stress_sim.json"))
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    O, T = a.objects, a.templates
    B = O
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    res = {"workload": f"per-GPU shard of c5: {O} objects x {T} local templates, batch {B}, one query per object",
           "bank_GB": O * T * 256 * 1024 * 4 / 1e9}
    labels = torch.arange(1, O + 1)
    for prec in ("fp32_split", "bf16"):
        eng = Engine(O, T, B, device=dev, precision=prec)
        # generate + load the bank object-chunk by object-chunk (keeps the fp32 staging copy small)
        q_feat = None
        for o0 in range(0, O, 16):
            n = min(16, O - o0)
            case = synth.make_feature_case(B=n, O=n, T=T, seed=1000 + o0, device=dev, labels=torch.arange(1, n + 1))
            for i in range(n):
                eng.bank_write(o0 + i, 0, case.bank_feat[i], case.bank_mask16[i].reshape(-1, 16, 16), norm_passes=1)
            q = case.q_feat
            q_feat = q if q_feat is None else torch.cat([q_feat, q], 0)
            q_mask = case.q_mask16 if o0 == 0 else torch.cat([q_mask, case.q_mask16], 0)
            del case
        eng.set_queries(q_feat, q_mask.reshape(-1, 16, 16), labels - 1, norm_passes=1)
        m = eng.sim_topk()
        torch.cuda.synchronize()
        ms = eng.time_sim_kernel(iters=a.iters)
        passes = 3 if prec == "fp32_split" else 1
        plane_bytes = 4 if passes == 3 else 2                      # bf16 mode streams the hi planes only
        alg_bytes = O * T * 256 * 1024 * plane_bytes + B * 256 * 1024 * plane_bytes + B * T * (256 * 6 + 4)
        flops = 2.0 * B * T * 256 * 256 * 1024
        res[prec] = {"ms_per_launch": ms, "kernel": "sim_search_pair_kernel (2-CTA cluster)", "algorithmic_GB": alg_bytes / 1e9, "achieved_GBps": alg_bytes / (ms / 1e3) / 1e9,
                     "hbm_peak_GBps": peaks.get("hbm_gbs"), "hbm_frac": alg_bytes / (ms / 1e3) / 1e9 / peaks.get("hbm_gbs", 6650.0),
                     "algorithmic_TFLOPs": flops / (ms / 1e3) / 1e12, "executed_TFLOPs": passes * flops / (ms / 1e3) / 1e12,
                     "bf16_peak_TFLOPs": peaks.get("bf16_tflops"), "detections_per_s_sim_only": B / (ms / 1e3),
                     "id_src_checksum": int(m["id_src"].sum()), "src_pts_checksum": int(m["src_pts"].sum())}
        del eng
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
