"""The CPU oracle (oracle/port.py) must reproduce the outputs of the UNMODIFIED reference modules that
oracle/make_golden.py recorded in tests/golden/ (the reference has no tests of its own, SURVEY.md §4)."""
import os
import types

import numpy as np
import pytest
import torch

from gigapose_b200 import synth
from oracle import port, ref_run
from oracle.make_golden import GOLDEN_THREADS

INT_KEYS = ["id_src", "tar_pts", "src_pts", "idx_failed", "ransac_scores", "ransac_src_pts", "ransac_tar_pts"]
FLOAT_KEYS = ["score_src", "score_pts", "relScale", "relInplane", "M", "scores", "pred_poses"]


@pytest.fixture(autouse=True)
def golden_threads():
    """The port with the thread count the fixtures were recorded with: split differently, its fp32 reductions round
    differently in the last bits, and translations of ~200 px in M carry that past the 1e-6 compared here."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def _case_from_golden(g):
    B, O, T, seed, sub = [int(x) for x in g["cfg"]]
    case = synth.make_feature_case(B=B, O=O, T=T, seed=seed)
    # the inputs are re-derived from the seed: make sure the RNG streams did not drift
    assert float(case.bank_feat.double().sum()) == pytest.approx(float(g["ck_bank_feat"]), abs=1e-6)
    assert float(case.q_feat.double().sum()) == pytest.approx(float(g["ck_q_feat"]), abs=1e-6)
    assert float(case.bank_ist.double().sum()) == pytest.approx(float(g["ck_bank_ist"]), abs=1e-6)
    return case, (sub or None)


@pytest.mark.parametrize("name", ["retrieval_c1", "retrieval_small"])
def test_port_reproduces_reference_golden(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    case, sub = _case_from_golden(g)
    out = port.retrieval(synth.to_reference_layout(case), port.RegressorPort(), sub_batch=sub)
    for k in INT_KEYS:
        assert np.array_equal(out[k].numpy(), g[k]), k
    for k in FLOAT_KEYS:
        np.testing.assert_allclose(out[k].numpy(), g[k], rtol=0, atol=1e-6, err_msg=k)


def test_port_backbones_reproduce_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "backbones.npz"))
    rgb, _ = synth.make_crops(2, seed=31)
    assert float(rgb.double().sum()) == pytest.approx(float(g["ck_rgb"]), abs=1e-6)
    ist_feat = port.ISTBackbonePort()(rgb)
    np.testing.assert_allclose(ist_feat[:, ::2].numpy(), g["ist_feat_sub"], rtol=0, atol=2e-5)
    feat = port.ae_features(port.DinoV2Port(), rgb)
    np.testing.assert_allclose(feat[:, ::8].numpy(), g["ae_feat_sub"], rtol=0, atol=1e-6)
    assert torch.allclose(feat.norm(dim=1), torch.ones(2, 16, 16), atol=1e-5)


def test_port_matches_reference_initialised_weights(golden_dir):
    """The reference's retrieval with its own seeded IST initialisation (`ref_run.build_ist`), recorded by
    oracle/make_golden.py; the regressor is rebuilt from the same seed with this repository's drop-in classes."""
    from src.models.network.ist_net import ISTNet, Regressor
    from src.models.network.resnet import ResNet
    g = np.load(os.path.join(golden_dir, "retrieval_reference_init.npz"))
    case, _ = _case_from_golden(g)
    ist = ref_run.build_ist(classes=types.SimpleNamespace(ResNet=ResNet, Regressor=Regressor, ISTNet=ISTNet))
    weights = ist.regressor.state_dict()
    assert sum(float(v.double().sum()) for v in weights.values()) == pytest.approx(float(g["ck_regressor"]), abs=1e-6)
    reg = port.RegressorPort(seed=None)
    reg.load_state_dict(weights)
    mine = port.retrieval(synth.to_reference_layout(case), reg)
    keys = [k for k in g.files if k != "cfg" and not k.startswith("ck_")]
    assert set(keys) <= set(mine) and "pred_poses" in keys
    for k in keys:
        v = torch.from_numpy(g[k])
        if v.dtype in (torch.int64, torch.bool):
            assert torch.equal(v, mine[k]), k
        else:
            assert torch.allclose(v, mine[k], rtol=0, atol=1e-6), k


def test_vit_port_matches_hf_dinov2_architecture():
    """Cross-check of the restated architecture against transformers' Dinov2 (same maths, different code),
    on a 2-block, 64-dim toy so it runs in a second."""
    tr = pytest.importorskip("transformers")
    cfg = tr.Dinov2Config(hidden_size=64, num_hidden_layers=2, num_attention_heads=4, mlp_ratio=4, image_size=518,
                          patch_size=14, layerscale_value=1.0, hidden_act="gelu", qkv_bias=True,
                          attn_implementation="eager")
    hf = tr.Dinov2Model(cfg).eval()
    mine = port.DinoV2Port(dim=64, depth=2, heads=4, seed=3)
    sd = hf.state_dict()
    with torch.no_grad():
        sd["embeddings.cls_token"].copy_(mine.cls_token)
        sd["embeddings.position_embeddings"].copy_(mine.pos_embed)
        sd["embeddings.patch_embeddings.projection.weight"].copy_(mine.patch_embed.proj.weight)
        sd["embeddings.patch_embeddings.projection.bias"].copy_(mine.patch_embed.proj.bias)
        for i, blk in enumerate(mine.blocks):
            p = f"encoder.layer.{i}."
            q, k, v = blk.attn.qkv.weight.chunk(3, 0)
            qb, kb, vb = blk.attn.qkv.bias.chunk(3, 0)
            for nm, w, b in (("query", q, qb), ("key", k, kb), ("value", v, vb)):
                sd[p + f"attention.attention.{nm}.weight"].copy_(w)
                sd[p + f"attention.attention.{nm}.bias"].copy_(b)
            sd[p + "attention.output.dense.weight"].copy_(blk.attn.proj.weight)
            sd[p + "attention.output.dense.bias"].copy_(blk.attn.proj.bias)
            sd[p + "norm1.weight"].copy_(blk.norm1.weight); sd[p + "norm1.bias"].copy_(blk.norm1.bias)
            sd[p + "norm2.weight"].copy_(blk.norm2.weight); sd[p + "norm2.bias"].copy_(blk.norm2.bias)
            sd[p + "layer_scale1.lambda1"].copy_(blk.ls1.gamma); sd[p + "layer_scale2.lambda1"].copy_(blk.ls2.gamma)
            sd[p + "mlp.fc1.weight"].copy_(blk.mlp.fc1.weight); sd[p + "mlp.fc1.bias"].copy_(blk.mlp.fc1.bias)
            sd[p + "mlp.fc2.weight"].copy_(blk.mlp.fc2.weight); sd[p + "mlp.fc2.bias"].copy_(blk.mlp.fc2.bias)
    # full-resolution input (37x37 grid): no positional interpolation in either implementation
    x = torch.randn(1, 3, 518, 518, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        ref = hf(pixel_values=x, output_hidden_states=True).hidden_states[-1]
        got = mine.forward_features(x)["x_prenorm"]
    assert torch.allclose(ref, got, atol=2e-4), float((ref - got).abs().max())
