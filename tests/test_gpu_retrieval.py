"""-m gpu parity tests: the CUDA path (through the C ABI) against the CPU oracle and the reference-generated
golden fixtures.  Bars: integer / index tensors bit-exact; floats within the tolerance written in each test."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gigapose_b200 import synth
from oracle import port

from helpers import FLOAT_KEYS, INT_KEYS, cpu, engine_from_case, reference_slice, run_engine, write_report

pytestmark = pytest.mark.gpu


def _ref_tiles(case, dtype=torch.float64):
    """[T, B(sorted by object), 256 t, 256 s] similarity of the matching-time-normalised descriptors."""
    order = torch.argsort(case.q_label, stable=True)
    q = F.normalize(case.q_feat.to(dtype), dim=-1)[order]
    bank = F.normalize(case.bank_feat.to(dtype), dim=-1)[case.q_label[order] - 1]       # [B,T,256,C]
    return torch.einsum("btc,bnsc->nbts", q, bank)


@pytest.mark.parametrize("precision,tol,B,O,T,seed", [
    pytest.param("fp32_split", 1e-5, 3, 2, 6, 3, id="fp32_split-1e-05"),
    pytest.param("bf16", 2e-2, 3, 2, 6, 3, id="bf16-0.02"),
    pytest.param("fp32_split", 1e-5, 5, 2, 10, 82, id="fp32_split-1e-05-5x2x10"),
    pytest.param("fp32_split", 1e-5, 3, 3, 5, 80, id="fp32_split-1e-05-3x3x5"),
])
def test_similarity_tiles_against_fp64(precision, tol, B, O, T, seed):
    """The TMA + tcgen05 main loop alone: raw fp32 tiles vs an fp64 einsum on the same descriptors.
    fp32_split measures ~4e-6 (the tensor core adds into its fp32 accumulator with truncation, 192 adds per
    element); the reference's own fp32 einsum sits at ~1e-7, plain bf16 at ~5e-3."""
    case = synth.make_feature_case(B=B, O=O, T=T, seed=seed)
    eng = engine_from_case(case, precision=precision)
    eng.set_queries(case.q_feat, case.q_mask16.reshape(-1, 16, 16), case.q_label - 1)
    tiles = eng.debug_sim_tiles().cpu().double()
    ref = _ref_tiles(case)
    err = (tiles - ref).abs().max().item()
    assert err < tol, f"{precision}: max |sim - fp64| = {err:.3e}"


def _compare(out, ref, pose_tol=1e-3):
    bad = {}
    for k in INT_KEYS:
        a, b = out[k], ref[k]
        a = a.bool() if b.dtype == torch.bool else a
        if not torch.equal(a, b.to(a.dtype)):
            bad[k] = int((a != b.to(a.dtype)).sum())
    for k in FLOAT_KEYS:
        # M: the regressor's hidden layers run on tensor cores (fp16 hi/lo pairs, ~2e-5 on sigma: accumulation in the
        # tensor core truncates), everything else is fp32 SIMT
        tol = pose_tol if k == "pred_poses" else (5e-5 if k in ("M", "relScale", "relInplane") else 2e-5)
        scale = 1.0
        if k == "pred_poses":                       # translations are in mm (~400): relative 1e-3 on t, abs on R
            d = (out[k] - ref[k]).abs()
            d[..., :3, 3] = d[..., :3, 3] / ref[k][..., :3, 3].abs().clamp(min=1.0)
            err = d.max().item()
        elif k == "M":                              # 2x2 block (sigma R): 2e-5 relative; translation column in pixels (up to
            d = (out[k] - ref[k]).abs() / ref[k].abs().clamp(min=1.0)   # 1e3): 2e-5 relative with a floor of 2e-3 px
            d[..., :2, 2] = (out[k] - ref[k]).abs()[..., :2, 2] / (ref[k][..., :2, 2].abs() + 100.0)   # (t = 14 tar - sigma R 14 src:
            err = d.max().item()                    # 1e-5 on sigma from the tensor-core regressor times |14 src| ~ 200 px)
        else:
            err = ((out[k] - ref[k]).abs() / ref[k].abs().clamp(min=1.0)).max().item()
        if not err < tol:
            bad[k] = err
    return bad


@pytest.mark.parametrize("name", ["retrieval_c1", "retrieval_small"])
def test_retrieval_matches_reference_golden(golden_dir, name):
    """Whole a3-a9 chain on the GPU vs the outputs of the UNMODIFIED reference recorded in tests/golden."""
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    B, O, T, seed, _ = [int(x) for x in g["cfg"]]
    case = synth.make_feature_case(B=B, O=O, T=T, seed=seed)
    eng = engine_from_case(case, regressor=port.RegressorPort())
    out = cpu(run_engine(eng, case))
    ref = {k: torch.from_numpy(g[k]) for k in INT_KEYS + FLOAT_KEYS}
    bad = _compare(out, ref)
    assert not bad, f"mismatches vs reference golden: {bad}"


def test_retrieval_matches_oracle_live():
    """A second seed/shape, compared with the CPU oracle run on the spot (uneven object population)."""
    labels = torch.tensor([1, 1, 1, 3, 3, 2, 1, 3, 3])
    case = synth.make_feature_case(B=9, O=3, T=20, seed=21, labels=labels)
    reg = port.RegressorPort(seed=4)
    ref = port.retrieval(synth.to_reference_layout(case), reg)
    eng = engine_from_case(case, regressor=reg)
    out = cpu(run_engine(eng, case))
    bad = _compare(out, ref)
    assert not bad, f"mismatches vs CPU oracle: {bad}"


def test_stagewise_against_oracle():
    """Each stage fed with the ORACLE's inputs, so a failure names the stage."""
    case = synth.make_feature_case(B=5, O=2, T=12, seed=33)
    reg = port.RegressorPort(seed=6)
    ri = synth.to_reference_layout(case)
    sim = port.similarity_search(ri["src_feats"], ri["tar_feat"], ri["src_masks"], ri["tar_mask"])
    eng = engine_from_case(case, regressor=reg)
    eng.set_queries(case.q_feat, case.q_mask16.reshape(-1, 16, 16), case.q_label - 1)
    # a4
    m = eng.sim_topk()
    for k in ("id_src", "tar_pts", "src_pts"):
        assert torch.equal(m[k].cpu(), sim[k]), k
    assert torch.allclose(m["score_src"].cpu(), sim["score_src"], atol=2e-6)
    assert torch.allclose(m["score_pts"].cpu(), sim["score_pts"], atol=2e-6)
    # a5 on the oracle's matches
    dev = eng.device
    m_ref = {k: v.to(dev) for k, v in sim.items()}
    rs, ri_ = eng.ist_mlp(case.q_ist, m_ref)
    B, K = sim["id_src"].shape
    rs_ref = torch.zeros(B, K, 256)
    ri_ref = torch.zeros(B, K, 256, 2)
    bi = torch.arange(B)
    for kk in range(K):
        rs_ref[:, kk], ri_ref[:, kk] = port.ist_mlp(reg, ri["src_ist"][bi, sim["id_src"][:, kk]], ri["tar_ist"],
                                                   sim["src_pts"][:, kk], sim["tar_pts"][:, kk])
    assert torch.allclose(rs.cpu(), rs_ref, atol=1e-4, rtol=1e-5)
    assert torch.allclose(ri_.cpu(), ri_ref, atol=1e-4, rtol=1e-5)
    # a7 on the oracle's MLP outputs
    r = eng.ransac(m_ref, rs_ref.to(dev), ri_ref.to(dev))
    M, failed, in_src, in_tar, in_sc = port.ransac(sim["src_pts"], sim["tar_pts"], rs_ref, ri_ref)
    assert torch.equal(r["idx_failed"].cpu().bool(), failed)
    assert torch.equal(r["ransac_scores"].cpu(), in_sc)
    assert torch.equal(r["ransac_src_pts"].cpu(), in_src)
    assert torch.equal(r["ransac_tar_pts"].cpu(), in_tar)
    assert torch.allclose(r["M"].cpu(), M, atol=1e-5, rtol=1e-5)
    assert torch.equal(r["inlier_count"].cpu().long(), in_sc.sum(-1))


def test_empty_and_degenerate_queries():
    """Edge cases: an all-zero query mask (no valid patch anywhere) and a single-template-valid query."""
    case = synth.make_feature_case(B=3, O=1, T=8, seed=44)
    case.q_mask16[1] = 0
    reg = port.RegressorPort(seed=6)
    ref = port.retrieval(synth.to_reference_layout(case), reg)
    eng = engine_from_case(case, regressor=reg)
    out = cpu(run_engine(eng, case))
    # the masked query has no valid correspondence at all: identity M, not failed, zero scores
    assert (out["src_pts"][1] == -1).all() and (out["tar_pts"][1] == -1).all()
    assert torch.equal(out["M"][1], torch.eye(3).expand(5, 3, 3))
    assert not out["idx_failed"][1].any()
    assert (out["scores"][1] == 0).all()
    for k in ("tar_pts", "src_pts", "ransac_scores", "idx_failed"):
        assert torch.equal(out[k][[0, 2]].to(ref[k].dtype), ref[k][[0, 2]]), k


@pytest.mark.parametrize("B,O,T", [(5, 2, 10), (3, 3, 5), (32, 8, 162)])
def test_pair_kernel_against_oracle(B, O, T):
    """Row a4 (`sim_search_pair_kernel`: 2-CTA clusters, tcgen05 cta_group::2, column maxima exchanged through
    distributed shared memory) against the CPU oracle for every detection: template ids and correspondences bit-exact,
    scores within 2e-6.  The oracle is fed a few detections at a time (the full c2 reference layout is ~5 GB)."""
    case = synth.make_feature_case(B=B, O=O, T=T, seed=77 + B)
    eng = engine_from_case(case)
    eng.set_queries(case.q_feat, case.q_mask16.reshape(-1, 16, 16), case.q_label - 1)
    m = cpu(eng.sim_topk())
    for b0 in range(0, B, 4):
        sel = torch.arange(b0, min(B, b0 + 4))
        ri = reference_slice(case, sel)
        sim = port.similarity_search(ri["src_feats"], ri["tar_feat"], ri["src_masks"], ri["tar_mask"])
        for k in ("id_src", "tar_pts", "src_pts"):
            assert torch.equal(m[k][sel], sim[k]), (k, b0)
        assert torch.allclose(m["score_src"][sel], sim["score_src"], atol=2e-6), b0
        assert torch.allclose(m["score_pts"][sel], sim["score_pts"], atol=2e-6), b0


def test_tensor_core_mlp_against_oracle():
    """Row a5 on tcgen05 (fp16 hi/lo x3 hidden layers through vit_gemm_kernel, fp32 heads) against the fp32 oracle on
    the c2-sized planted case and the engine's own matches: the -1000 pattern is identical, regressor outputs agree to
    5e-5, and RANSAC + sort + pose on the GPU give the same integer outputs and scores with either set of outputs."""
    case = synth.make_feature_case(B=32, O=8, T=162, seed=42)
    reg = port.RegressorPort(seed=9)
    eng = engine_from_case(case, regressor=reg)
    eng.set_queries(case.q_feat, case.q_mask16.reshape(-1, 16, 16), case.q_label - 1)
    m = eng.sim_topk()
    rs, ri = eng.ist_mlp(case.q_ist, m)
    mc = cpu(m)
    src_ist = case.bank_ist[(case.q_label - 1)[:, None], mc["id_src"]]          # [B,k,...] template IST features
    rs_ref, ri_ref = torch.zeros(rs.shape), torch.zeros(ri.shape)
    for kk in range(mc["id_src"].shape[1]):
        rs_ref[:, kk], ri_ref[:, kk] = port.ist_mlp(reg, src_ist[:, kk], case.q_ist, mc["src_pts"][:, kk], mc["tar_pts"][:, kk])
    rs_gpu, ri_gpu = rs.cpu(), ri.cpu()
    valid = mc["src_pts"][..., 0] != -1
    assert torch.equal(rs_gpu == -1000, rs_ref == -1000)
    assert torch.equal(ri_gpu == -1000, ri_ref == -1000)
    d = max(float((rs_gpu - rs_ref)[valid].abs().max()), float((ri_gpu - ri_ref)[valid].abs().max()))
    dev = eng.device
    a = cpu(eng.sort_and_pose(case.q_K, case.q_M, m, rs, ri, eng.ransac(m, rs, ri)))
    rs_ref, ri_ref = rs_ref.to(dev), ri_ref.to(dev)
    b = cpu(eng.sort_and_pose(case.q_K, case.q_M, m, rs_ref, ri_ref, eng.ransac(m, rs_ref, ri_ref)))
    perr = (a["pred_poses"] - b["pred_poses"]).abs()
    perr[..., :3, 3] /= b["pred_poses"][..., :3, 3].abs().clamp(min=1.0)
    write_report("mlp_tc_vs_oracle.json", {"case": "c2 planted features (32 detections, 8 x 162 templates)", "hypotheses": 160,
                                           "valid_correspondences": int(valid.sum()), "regressor_output_max_abs_diff": d,
                                           "pose_max_diff": float(perr.max()),
                                           "integer_outputs_changed": int(sum((a[k] != b[k]).sum() for k in INT_KEYS))})
    assert d < 5e-5, d
    assert float(perr.max()) < 1e-3
    for k in INT_KEYS:
        assert torch.equal(a[k], b[k]), k
    assert torch.equal(a["scores"], b["scores"])
