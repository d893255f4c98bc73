"""TEST INFRASTRUCTURE ONLY -- drives the *unmodified reference modules* (oracle/ref_import.py) through the
same sequence as GigaPose.eval_retrieval (gigaPose.py:497-604).  `retrieval` needs the reference tree."""
from __future__ import annotations

import pandas as pd
import torch

from . import ref_import

IST_CFG = dict(n_heads=0, input_dim=3, input_size=256, initial_dim=128, block_dims=[128, 192, 256, 512],
               descriptor_size=256)


def build_ist(seed=8, classes=None):
    """Seeded ISTNet of the reference's classes, or of `classes` (a namespace with ResNet, Regressor, ISTNet): this
    repository's drop-in classes create and initialise their parameters in the reference's order, so the same seed
    gives the same weights without a reference tree."""
    ns = classes or ref_import.load()
    torch.manual_seed(seed)
    backbone = ns.ResNet(dict(IST_CFG))
    regressor = ns.Regressor(descriptor_size=256, hidden_dim=256, use_tanh_act=True, normalize_output=True)
    ist = ns.ISTNet("resnet", backbone, regressor, max_batch_size=64)
    # give the (zero-initialised) biases and BN statistics non-trivial seeded values
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for n, p in ist.named_parameters():
            if n.endswith("bias"):
                p.copy_(0.05 * torch.randn(p.shape, generator=g))
        for n, b in ist.named_buffers():
            if n.endswith("running_mean"):
                b.copy_(0.1 * torch.randn(b.shape, generator=g))
            elif n.endswith("running_var"):
                b.copy_(1.0 + 0.2 * torch.rand(b.shape, generator=g))
    return ist.eval()


@torch.no_grad()
def retrieval(ref_inputs, ist, k=5, sim_threshold=0.5, patch_threshold=3, sub_batch=None):
    ns = ref_import.load()
    metric = ns.LocalSimilarity(k=k, sim_threshold=sim_threshold, patch_threshold=patch_threshold)
    B = ref_inputs["tar_feat"].shape[0]
    sub = sub_batch or B
    predictions = None
    for b0 in range(0, B, sub):
        sl = slice(b0, b0 + sub)
        p = metric.test(src_feats=ref_inputs["src_feats"][sl], tar_feat=ref_inputs["tar_feat"][sl],
                        src_masks=ref_inputs["src_masks"][sl], tar_mask=ref_inputs["tar_mask"][sl],
                        max_batch_size=None)
        predictions = p if predictions is None else predictions.cat_df(p)
    predictions.infos = pd.DataFrame(dict(label=[str(int(l)) for l in ref_inputs["tar_label"]]))
    P = predictions.src_pts.shape[2]
    rel_scale = torch.zeros(B, k, P)
    rel_inpl = torch.zeros(B, k, P, 2)
    bi = torch.arange(B)
    for kk in range(k):
        src_ist = ref_inputs["src_ist"][bi, predictions.id_src[:, kk]]
        rel_scale[:, kk], rel_inpl[:, kk] = ist.inference(src_feat=src_ist, tar_feat=ref_inputs["tar_ist"],
                                                          src_pts=predictions.src_pts[:, kk],
                                                          tar_pts=predictions.tar_pts[:, kk])
    predictions.register_tensor("relScale", rel_scale)
    predictions.register_tensor("relInplane", rel_inpl)
    recovery = ns.ObjectPoseRecovery(template_K=ref_inputs["template_K"], template_Ms=ref_inputs["template_Ms"],
                                     template_poses=ref_inputs["template_poses"])
    predictions = recovery.forward_ransac(predictions=predictions)
    score = torch.sum(predictions.ransac_scores, dim=2) / P
    predictions.register_tensor("scores", score)
    order = torch.argsort(score, dim=1, descending=True)
    for name, v in list(predictions._tensors.items()):
        predictions.register_tensor(name, v[bi[:, None], order])
    poses = recovery.forward_recovery(tar_label=ref_inputs["tar_label"], tar_K=ref_inputs["tar_K"],
                                      tar_M=ref_inputs["tar_M"], pred_src_views=predictions.id_src,
                                      pred_M=predictions.M.clone())
    predictions.register_tensor("pred_poses", poses)
    return {n: v for n, v in predictions._tensors.items()}
