#!/usr/bin/env python
"""Benchmark of the GigaPose inference hot path (BASELINE.json metric: detections/sec on 224x224 crops against a
162-template bank; similarity-GEMM fraction of roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic query crops:
  a1 ViT-L/14 patch tokens -> a3/a4 similarity search + top-k against the resident bank -> a6 IST backbone ->
  a5 per-correspondence MLP -> a7 RANSAC -> a8 re-sort -> a9 pose lifting.
`value` times it with the crops already resident in HBM; `e2e` times the plugin call (`GigaPose.retrieve`) on
pinned HOST tensors with the H2D copy of the crops and the D2H read of poses + scores inside the timed region.
Prints ONE JSON line (rank 0).  `--dump-outputs DIR` also writes the outputs of the last timed step as DIR/<name>.npy:
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (which may be read-only)

import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402
import torch  # noqa: E402

_REAL_STDOUT = None


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


WORKLOADS = {
    # name: (objects, templates, batch)  -- BASELINE.json configs[1..4]
    "c1": dict(O=1, T=16, B=1, desc="single query vs 16 templates (CPU-runnable plumbing case)"),
    "c2": dict(O=8, T=162, B=32, desc="LM-O-shaped: 8 objects x 162 templates, batch 32"),
    "c3": dict(O=30, T=162, B=64, desc="T-LESS-shaped: 30 objects x 162 templates, batch 64"),
    "c4": dict(O=21, T=162, B=128, desc="YCB-V-shaped: 21 objects x 162 templates, batch 128"),
    # BASELINE.json configs[4]: 8 GPUs only (154.6 GB of descriptors); one query per object = no template reuse (B_o = 1)
    "c5": dict(O=256, T=576, B=256, desc="stress: 256 objects x 576 templates (HANDAL-scale), batch 256, one query per object",
               one_query_per_object=True),
}
DTYPE = ("f32 (a1, a4, a6: bf16 hi/lo split x3 on tensor cores with fp32 accumulate = fp32-faithful; "
         "a5, a7-a9: fp32)")
METRIC = "detections/sec (224x224 crops, 162-template bank)"
UNIT = "detections/s"


# ----------------------------------------------------------------------------------------------------------------
# synthetic world: template crops per object, queries = noisy copies of planted templates
# ----------------------------------------------------------------------------------------------------------------
def rows_config():
    """Which SURVEY §8 rows run on this library's kernels (all of them) and which on a vendor library (none)."""
    from gigapose_b200 import vit_engine, ist_trunk
    return dict(native_rows=[f"a1 ViT-L/14 ({vit_engine.BACKEND})", "a2", "a3", "a4", "a5",
                             f"a6 IST ResNet ({ist_trunk.BACKEND})", "a7", "a8", "a9"], library_rows=[])


def build_models(device, seed_vit=7, seed_ist=8):
    from gigapose_b200.vit import DinoVisionTransformer
    from src.models.gigaPose import GigaPose
    from src.models.matching import LocalSimilarity
    from src.models.network.ae_net import AENet
    from src.models.network.ist_net import ISTNet, Regressor
    from src.models.network.resnet import ResNet

    vit = DinoVisionTransformer(init_seed=seed_vit)
    ae = AENet("dinov2_vitl14", dinov2_model=vit, descriptor_size=1024, max_batch_size=64)
    torch.manual_seed(seed_ist)
    backbone = ResNet(dict(n_heads=0, input_dim=3, input_size=256, initial_dim=128, block_dims=[128, 192, 256, 512],
                           descriptor_size=256))
    reg = Regressor(descriptor_size=256, hidden_dim=256, use_tanh_act=True, normalize_output=True)
    ist = ISTNet("resnet", backbone, reg, max_batch_size=64)
    g = torch.Generator().manual_seed(seed_ist + 1)
    with torch.no_grad():
        for n, p in ist.named_parameters():
            if n.endswith("bias"):
                p.copy_(0.05 * torch.randn(p.shape, generator=g))
    metric = LocalSimilarity(k=5, sim_threshold=0.5, patch_threshold=3)
    # GigaPose creates <log_dir>/predictions; the benchmark saves no predictions, so it gets a directory removed at exit
    log_dir = tempfile.mkdtemp(prefix="gigapose-bench-")
    atexit.register(shutil.rmtree, log_dir, True)
    model = GigaPose("large", ae, ist, training_loss=None, testing_metric=metric, optim_config=None, log_interval=1000,
                     log_dir=log_dir, max_num_dets_per_forward=None)
    return model.to(device).eval()


class SyntheticTemplates:
    """Stands in for `TemplateSet` (dataloader/template.py:55-81): item o -> collection(K, rgb, mask, M, poses)."""

    def __init__(self, O, T, device):
        from gigapose_b200 import synth
        self.O, self.T, self.device, self.synth = O, T, device, synth
        gc = torch.Generator().manual_seed(99)
        s = torch.empty(O * T).uniform_(0.6, 1.8, generator=gc)
        M = torch.zeros(O * T, 3, 3)
        M[:, 0, 0] = s
        M[:, 1, 1] = s
        M[:, 0, 2] = 112.0 - s * torch.empty(O * T).uniform_(150, 490, generator=gc)
        M[:, 1, 2] = 112.0 - s * torch.empty(O * T).uniform_(120, 360, generator=gc)
        M[:, 2, 2] = 1
        self.M = M.reshape(O, T, 3, 3)
        self.poses = synth.fibonacci_view_poses(T)
        self.K = torch.tensor(synth.LM_K)

    def __len__(self):
        return self.O

    def crops(self, o):
        return self.synth.make_crops(self.T, seed=3000 + o, device=self.device)

    def __getitem__(self, o):
        import src.megapose.utils.tensor_collection as tc
        rgb, mask = self.crops(o)
        return tc.PandasTensorCollection(infos=pd.DataFrame(), K=self.K, rgb=rgb, mask=mask, M=self.M[o], poses=self.poses)


def make_queries(templates: SyntheticTemplates, B, seed=42, one_per_object=False):
    """B query crops = planted template crops + noise; host-pinned tensors (what the DataLoader hands over)."""
    import src.megapose.utils.tensor_collection as tc
    gc = torch.Generator().manual_seed(seed)
    labels = torch.randint(1, templates.O + 1, (B,), generator=gc)
    if one_per_object:
        labels = (torch.arange(B) % templates.O) + 1
    views = torch.randint(0, templates.T, (B,), generator=gc)
    imgs, masks = [], []
    for b in range(B):
        rgb, mask = templates.crops(int(labels[b]) - 1)
        imgs.append(rgb[views[b]].cpu())
        masks.append(mask[views[b]].cpu())
    img = torch.stack(imgs) + 0.05 * torch.randn(B, 3, 224, 224, generator=gc)
    s = torch.empty(B).uniform_(0.6, 1.8, generator=gc)
    M = torch.zeros(B, 3, 3)
    M[:, 0, 0] = s
    M[:, 1, 1] = s
    M[:, 0, 2] = 112.0 - s * torch.empty(B).uniform_(150, 490, generator=gc)
    M[:, 1, 2] = 112.0 - s * torch.empty(B).uniform_(120, 360, generator=gc)
    M[:, 2, 2] = 1
    K = templates.K.repeat(B, 1, 1)
    infos = pd.DataFrame(dict(label=[str(int(l)) for l in labels], scene_id=[0] * B, view_id=list(range(B))))
    pin = (lambda t: t.pin_memory()) if torch.cuda.is_available() else (lambda t: t)
    batch = tc.PandasTensorCollection(infos=infos, tar_img=pin(img), tar_mask=pin(torch.stack(masks)), tar_K=pin(K),
                                      tar_M=pin(M))
    return batch, labels, views


# ----------------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock + throttle reasons DURING the timed region through NVML (in-process: a polling `nvidia-smi`
    subprocess was measured to slow the launching thread by 50 %).  Falls back to one `nvidia-smi` query before and
    after the region when pynvml is unavailable."""

    def __init__(self, index=0):
        self.index, self.samples, self.reasons = index, [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        self._nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[index])
            except Exception:
                return index
        return index

    def _sample_nvml(self):
        nv = self._nv
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        flags = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        for n, bit in flags.items():
            if r & bit:
                self.reasons.add(n)

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                 capture_output=True, text=True, timeout=5).stdout.strip()
            f = [x.strip() for x in out.split(",")]
            self.samples.append(float(f[0]))
            self.max_mhz = float(f[1])
            for n, v in zip(names, f[2:]):
                if v.lower().startswith("active"):
                    self.reasons.add(n)
        except Exception:
            pass

    def _run(self):
        while not self._stop.is_set():
            try:
                self._sample_nvml()
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self._nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        else:
            self._sample_smi()
        return self

    def __exit__(self, *a):
        if self._t is not None:
            self._stop.set()
            self._t.join(timeout=2)
        else:
            self._sample_smi()

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "source": "nvml" if self._nv is not None else "nvidia-smi"}


# ----------------------------------------------------------------------------------------------------------------
# CPU reference arm: the oracle port (the reference modules cannot travel to the GPU box) on all host threads
# ----------------------------------------------------------------------------------------------------------------
class CpuReference:
    """The reference's PyTorch path restated on the CPU (oracle/port.py: pinned against the unmodified reference by
    tests/golden), sequenced exactly like `GigaPose.eval_retrieval` (gigaPose.py:497-604), on the box's host cores.

    World: `n_det` detections over `n_obj` objects x T templates (for c2 that IS the full batch: 32 detections, 8 objects;
    for the larger configurations a bounded sample of the same shape).  Template descriptors / IST features / masks are
    the planted synthetic bank in the reference's own layout ([O,T,1024,16,16] f32 etc.); query crops go through the
    ViT-L/14 and IST backbones (their outputs are timed, the downstream stages run on the planted query features of the
    same shapes so that the matching stage has real structure to work on).

    Variants (BASELINE.md section 3):  "as_written" = the reference as it stands: per-detection bank gathers
    `ae_features[label-1]`, `mask[label-1]` (gigaPose.py:520-521) and, inside the k loop, `ist_features[label-1]` plus a
    fresh IST backbone pass over all crops for each of the k hypotheses (gigaPose.py:552-553);  "fair" = the same
    arithmetic with the backbone run once and the IST bank gathered once."""

    def __init__(self, T, n_det=32, n_obj=8, k=5, device="cpu"):
        from gigapose_b200 import synth
        from oracle import port
        self.port, self.k, self.T = port, k, T
        self.device = torch.device(device)
        gc = torch.Generator().manual_seed(4242)
        labels = torch.randint(1, n_obj + 1, (n_det,), generator=gc)
        case = synth.make_feature_case(B=n_det, O=n_obj, T=T, seed=77, labels=labels, obj_chunk=1)
        O = n_obj
        # the reference's template_data tensors (gigaPose.py:383-390)
        self.ae_features = case.bank_feat.permute(0, 1, 3, 2).reshape(O, T, 1024, 16, 16).contiguous()
        self.masks = synth.mask16_to_224(case.bank_mask16).contiguous()                     # [O,T,224,224]
        self.ist_features = case.bank_ist
        self.tar_feat = case.q_feat.permute(0, 2, 1).reshape(n_det, 1024, 16, 16).contiguous()
        self.tar_mask = synth.mask16_to_224(case.q_mask16)
        self.tar_ist = case.q_ist
        self.case = case
        self.rgb = synth.make_crops(n_det, seed=78)[0]
        self.vit, self.backbone, self.reg = port.DinoV2Port(), port.ISTBackbonePort(), port.RegressorPort()
        self.n_det, self.n_obj = n_det, n_obj
        if self.device.type != "cpu":          # --gpu-eager-baseline: the same eager torch code on the B200 (cuBLAS / cuDNN)
            for name in ("ae_features", "masks", "ist_features", "tar_feat", "tar_mask", "tar_ist", "rgb"):
                setattr(self, name, getattr(self, name).to(self.device))
            self.case = case.to(self.device)
            for m in (self.vit, self.backbone, self.reg):
                m.to(self.device)

    @torch.no_grad()
    def run(self, variant="fair", n=None):
        """One pass over the first `n` detections; returns (seconds, per-stage seconds)."""
        port, k = self.port, self.k
        n = n or self.n_det
        c = self.case
        st = {}
        on_gpu = self.device.type != "cpu"
        if on_gpu:
            torch.cuda.synchronize()
        t_all = time.perf_counter()

        def tic(name, t0):
            if on_gpu:
                torch.cuda.synchronize()
            st[name] = st.get(name, 0.0) + time.perf_counter() - t0

        t0 = time.perf_counter(); _ = port.ae_features(self.vit, self.rgb[:n]); tic("a1_vit", t0)
        lab = c.q_label[:n] - 1
        t0 = time.perf_counter()
        src_feats = self.ae_features[lab]                                        # gigaPose.py:520 (170 MB per detection)
        src_masks = self.masks[lab]                                              # gigaPose.py:521
        tic("a3_bank_gather", t0)
        t0 = time.perf_counter()
        pred = port.similarity_search(src_feats, self.tar_feat[:n], src_masks, self.tar_mask[:n], k=k)
        tic("a4_similarity_topk", t0)
        del src_feats, src_masks
        rel_scale = torch.zeros(n, k, 256, device=self.device)
        rel_inpl = torch.zeros(n, k, 256, 2, device=self.device)
        bi = torch.arange(n, device=self.device)
        src_ist = None
        for kk in range(k):                                                      # gigaPose.py:545-575
            if variant == "as_written" or kk == 0:
                t0 = time.perf_counter(); src_ist = self.ist_features[lab]; tic("a3_bank_gather", t0)   # :552
                t0 = time.perf_counter(); _ = self.backbone(self.rgb[:n]); tic("a6_ist_backbone", t0)   # :553
            t0 = time.perf_counter()
            rel_scale[:, kk], rel_inpl[:, kk] = port.ist_mlp(self.reg, src_ist[bi, pred["id_src"][:, kk]], self.tar_ist[:n],
                                                             pred["src_pts"][:, kk], pred["tar_pts"][:, kk])
            tic("a5_ist_mlp", t0)
        t0 = time.perf_counter()
        M, failed, in_src, in_tar, in_sc = port.ransac(pred["src_pts"], pred["tar_pts"], rel_scale, rel_inpl)
        tic("a7_ransac", t0)
        t0 = time.perf_counter()
        scores = torch.sum(in_sc, dim=2) / 256
        order = torch.argsort(scores, dim=1, descending=True)
        ids = pred["id_src"][bi[:, None], order]
        Ms = M[bi[:, None], order]
        _ = port.pose_recovery(c.q_label[:n], c.q_K[:n], c.q_M[:n], ids, Ms.clone(), c.bank_K, c.bank_M, c.bank_poses)
        tic("a8_a9_sort_pose", t0)
        return time.perf_counter() - t_all, st

    def run_on_device(self, variant="fair"):
        """`run` with torch's factory functions defaulting to this reference's device (the port creates index tensors
        with bare torch.arange / torch.zeros, exactly like the reference)."""
        with torch.device(self.device):
            return self.run(variant)

    def sweep_threads(self, cands, n):
        """Fastest thread count for the whole chain on the first `n` detections (more threads are not always faster for
        the reference's many small ops: 128 threads were measured 20x slower than 8 on the RANSAC python loops)."""
        best, best_t, seen = cands[0], float("inf"), {}
        for cnum in cands:
            torch.set_num_threads(cnum)
            self.run("fair", n=min(2, n))                       # warm the thread pool
            t, _ = self.run("fair", n=n)
            seen[cnum] = round(t, 3)
            if t < best_t:
                best, best_t = cnum, t
        torch.set_num_threads(best)
        return best, seen


def cpu_thread_candidates():
    """Thread counts worth trying, ascending.  All logical CPUs of a big host is NOT one of them: on the 128-thread B200
    hosts the reference's many small ops ran 12 - 40x slower at 128 threads than at 16 (measured: 4 detections in 56 s
    instead of 1.4 s), which would turn the sweep itself into minutes."""
    ncpu = os.cpu_count() or 1
    return sorted({c for c in (8, 16, 32, 64) if c <= ncpu}) or [ncpu]


def sample_shape(cfg):
    """Detections / objects of the CPU sample for a workload: the full batch for c1 / c2, a c2-sized slice otherwise."""
    return min(cfg["B"], 32), min(cfg["O"], 8)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(outputs, out_dir, limit=DUMP_LIMIT_BYTES, seed=0):
    """Writes every tensor of `outputs` (leading dimension = detection) as out_dir/<name>.npy: floating point as float32
    (float64 stays float64), integers and booleans as float64, which holds them exactly.  When the arrays exceed `limit`
    bytes in all, the same seeded sample of detections is kept of every array and its indices go to sample_rows.npy."""
    arrays = {}
    for name, t in outputs.items():
        t = t.detach().cpu()
        wide = t.dtype == torch.float64 or not t.is_floating_point()
        arrays[name] = t.to(torch.float64 if wide else torch.float32).numpy()
    n = {a.shape[0] for a in arrays.values()}
    assert len(n) == 1, f"outputs disagree on the number of detections: {n}"
    n = n.pop()
    row_bytes = sum(a.nbytes for a in arrays.values()) // n
    if n * row_bytes > limit:
        keep = max(1, limit // (row_bytes + 8))                       # + the row's index in sample_rows.npy
        rows = np.sort(np.random.default_rng(seed).choice(n, size=keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["sample_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sorted(arrays)


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cuda-graph", action="store_true", help="launch the per-batch kernel sequence eagerly")
    ap.add_argument("--gpu-eager-baseline", action="store_true",
                    help="also time the reference's eager PyTorch code (oracle port) on the SAME GPU (cuBLAS / cuDNN fp32): context "
                         "for the hand-written kernels, SURVEY section 2")
    ap.add_argument("--profile-range", action="store_true",
                    help="wrap ONE extra resident step in cudaProfilerStart/Stop (ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs writes the single-GPU path's outputs: it needs --impl ours --gpus 1")

    # stdout carries exactly ONE JSON line: libraries (NCCL's version banner, cuDNN logs) write to fd 1 too, so the
    # real stdout is kept aside and fd 1 points at stderr until the line is printed
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl_name = args.workload or {1: "c2", 2: "c2", 4: "c3", 8: "c4"}.get(args.gpus, "c2")
    cfg = WORKLOADS[wl_name]
    if wl_name == "c5" and args.gpus < 8 and args.impl != "reference":
        raise SystemExit("workload c5 (154.6 GB of template descriptors) needs --gpus 8")
    config = {"workload": f"{wl_name}: {cfg['desc']}", "objects": cfg["O"], "templates": cfg["T"], "batch": cfg["B"],
              "k": 5, "l2": "inputs larger than L2 (template bank 1.36 GB at c2 vs 126 MB L2); no explicit flush"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        n_det, n_obj = sample_shape(cfg)
        ref = CpuReference(cfg["T"], n_det=n_det, n_obj=n_obj)
        # warm-up steps double as the thread sweep on the FULL sample (one candidate per warm-up step, at least one)
        cands = cpu_thread_candidates()
        cands = cands[1:1 + max(1, min(len(cands) - 1, args.warmup))] if len(cands) > 1 else cands      # 16, 32, 64 for W >= 3
        threads, sweep = ref.sweep_threads(cands, n=n_det)
        vals, stages = [], {}
        for i in range(args.steps):
            t, st = ref.run("fair")
            vals.append(n_det / t)
            for kname, v in st.items():
                stages[kname] = stages.get(kname, 0.0) + v / args.steps
        t_aw, st_aw = ref.run("as_written")
        value = statistics.mean(vals)
        sample = (f"{n_det} detections over {n_obj} objects x {cfg['T']} templates per step"
                  + (" (the full batch)" if n_det == cfg["B"] and n_obj == cfg["O"] else f" (bounded sample of B={cfg['B']}, O={cfg['O']})")
                  + f", fp32 torch on the host CPU, {threads} of {os.cpu_count()} threads (fastest of {sweep} s per step), "
                    "'fair' variant: ViT-L/14 + bank gathers + similarity / top-k + IST backbone once + MLP + RANSAC + pose")
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_det / value, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": dict(value=value, unit=UNIT, cores=threads, kind="port", sample=sample,
                                     stage_s={kk: round(v, 4) for kk, v in stages.items()},
                                     as_written=dict(value=n_det / t_aw, unit=UNIT,
                                                     stage_s={kk: round(v, 4) for kk, v in st_aw.items()},
                                                     note="IST backbone and IST bank gather repeated for each of the k=5 "
                                                          "hypotheses (gigaPose.py:552-553), one pass")),
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return 0

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        from datetime import timedelta
        dist.init_process_group("nccl", device_id=device, timeout=timedelta(seconds=180))   # a stuck rank fails, not hangs
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    if world > 1:
        from gigapose_b200.multigpu import run_sharded_bench
        return run_sharded_bench(args, cfg, config, wl_name, rank, world, device, METRIC, UNIT, ClockSampler, emit)

    from gigapose_b200 import vit_engine
    model = build_models(device)
    model.use_cuda_graph = not args.no_cuda_graph and not args.profile_range
    templates = SyntheticTemplates(cfg["O"], cfg["T"], device)
    model.template_datasets = {"synthetic": templates}
    model.test_dataset_name = "synthetic"
    model.set_template_data("synthetic")
    eng = model.engines["synthetic"]
    batch_host, labels, views = make_queries(templates, cfg["B"])
    batch_dev = batch_host.clone().to(device)
    torch.cuda.synchronize()

    def step_resident():
        return model.retrieve(batch_dev, "synthetic")

    def step_e2e():
        pred = model.retrieve(batch_host, "synthetic")          # H2D of crops/masks/K/M happens inside
        return pred.pred_poses.cpu(), pred.scores.cpu()           # D2H of the step's result

    # kernel launches of THIS library per step, counted on one eager step (a graph replay re-issues the same kernels
    # without going through the C entry points that keep the counter)
    graph_flag, model.use_cuda_graph = model.use_cuda_graph, False
    l0 = eng.launch_count()
    step_resident()
    launches = eng.launch_count() - l0
    model.use_cuda_graph = graph_flag
    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            pred = step_resident()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    value = cfg["B"] / (ms / 1e3)
    if args.dump_outputs:
        dump_outputs(pred.tensors, args.dump_outputs)

    # per-stage CUDA-event times of one extra resident step (diagnostic, outside the timed region)
    model.profile_stages = True
    step_resident()                      # first eager step after the graph capture re-plans some library kernels
    step_resident()
    model.profile_stages = False
    stage_ms = {k: round(v, 3) for k, v in model.stage_ms.items()}

    if args.profile_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()

    # end to end through the plugin calls, host buffers: every step uploads its own inputs from pinned memory
    # (`stage`: copy stream, overlapping the previous step's kernels), runs, and copies its own poses + scores back to
    # pinned host memory (`fetch_async`); a step's results are read on the host while the next step's kernels run.
    # All `steps` uploads and read-backs are inside the timed region; the first upload has nothing to overlap with and
    # the last read-back is waited for before the clock stops.
    def e2e_pipeline(steps):
        staged = model.stage(batch_host, "synthetic")
        pending, res = None, None
        for i in range(steps):
            cur = staged
            if i + 1 < steps:
                staged = model.stage(batch_host, "synthetic")
            handle = model.fetch_async(model.retrieve(cur, "synthetic"))
            if pending is not None:
                res = pending.result()
            pending = handle
        res = pending.result()
        torch.cuda.synchronize()
        return res

    # warm-up through the SAME pipelined path: the pinned ring buffers of `stage` (4 slots) and `fetch_async` (3 slots) are
    # allocated on first use, and a cudaHostAlloc inside the timed region stalls the launching thread for milliseconds
    # (this is what made earlier e2e numbers swing between 0.5x and 0.98x of `value` from box to box)
    step_e2e()
    e2e_pipeline(6)
    t0 = time.perf_counter()
    poses, scores = e2e_pipeline(args.steps)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    h2d = sum(batch_host._tensors[k].numel() * batch_host._tensors[k].element_size() for k in ("tar_img", "tar_mask", "tar_K", "tar_M"))
    d2h = poses.numel() * 4 + scores.numel() * 4

    # correctness gate of the measured step: every query is a noisy copy of template `views[b]` of its object, and that
    # view must be among the k retrieved (a bench line for a path that retrieves the wrong templates is worthless)
    id0 = pred.id_src.cpu()
    hit = float((id0 == views[:, None]).any(dim=1).float().mean())
    assert hit == 1.0, f"planted view missing from the top-k of {1 - hit:.1%} of the queries"

    # roofline of the dominant kernel (similarity search): algorithmic FLOPs / CUDA-event time of the kernel alone
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops", 1590.0)
    sim_ms = eng.time_sim_kernel(iters=20)
    flops = eng.sim_flops(cfg["B"])
    achieved = flops / (sim_ms / 1e3) / 1e12
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed `ncu --set full` capture
        tr = json.load(open(os.path.join(ROOT, "profiles", "sim_search_traffic.json")))
        if tr.get("workload") == wl_name:
            traffic = tr["dram_bytes_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "sim_search_kernel", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved / peak_tf, "traffic": traffic, "ms_per_launch": sim_ms,
                "executed_tflops": 3 * achieved, "executed_frac_of_peak": 3 * achieved / peak_tf,
                "algorithmic_bytes_per_launch": cfg["O"] * cfg["T"] * 256 * 1024 * 4 + cfg["B"] * 256 * 1024 * 4,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if peaks else "fallback 1590 (B200_PROFILING.md)",
                "note": "algorithmic FLOPs = 2*T*P^2*C per detection; the fp32-faithful mode executes 3 bf16 tensor passes "
                        "per algorithmic FLOP, so frac <= 1/3 by construction"}

    # the kernel that dominates the step (60 % of it): the 96 linear layers of the ViT, timed alone back to back
    # (96 x iters launches = a long run: the sustained peak is the denominator)
    roofline_vit = None
    vit_entry = getattr(model.ae_net.dinov2_model, "_gp_vit_engine", None)
    if vit_entry is not None:
        vit_ms = vit_entry[1].time_linears(cfg["B"], iters=5)
        depth = vit_entry[1].depth
        vit_flops = cfg["B"] * depth * 2.0 * 257 * 1024 * (3072 + 1024 + 4096 + 4096)
        peak_sus = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0))
        ach = vit_flops / (vit_ms / 1e3) / 1e12
        roofline_vit = {"bound": "tensor", "kernel": "vit_gemm_kernel<swap=0,pair=1> (qkv, proj, fc1, fc2 of 24 blocks)",
                        "achieved": ach, "peak": peak_sus, "unit": "TFLOP/s", "frac": ach / peak_sus, "traffic": None,
                        "launches": 4 * depth, "ms_per_forward": vit_ms, "ms_per_launch": vit_ms / (4 * depth),
                        "executed_tflops": 3 * ach, "executed_frac_of_peak": 3 * ach / peak_sus,
                        "share_of_step": vit_ms / ms,
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernels timed in a long back-to-back run)",
                        "note": "algorithmic FLOPs = 2*M*N*K of the 4 linears x depth (155.2 GFLOP per crop); 3 tensor passes "
                                "per algorithmic FLOP (fp32-faithful split)"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE,
            "data": "synthetic", "config": dict(config, **rows_config(),
                                                planted_view_in_topk=hit),
            "clocks": clocks.summary(),
            "e2e": {"value": cfg["B"] / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms},
            "gpu_launches": int(launches), "roofline": roofline, "roofline_dominant": roofline_vit, "stage_ms": stage_ms}
    line["config"]["cuda_graph"] = bool(model.use_cuda_graph)
    # row f2: batched onboarding (both encoders over all O x T template crops in 64-crop chunks + bank writes), CUDA events
    line["onboarding"] = {"s_per_object": round(getattr(model, "onboarding_s_per_object", float("nan")), 4),
                          "templates_per_object": cfg["T"], "objects": cfg["O"],
                          "note": "synthetic template crops already on the device; ViT-L/14 + IST trunk + bank write"}
    if args.gpu_eager_baseline:
        torch.backends.cuda.matmul.allow_tf32 = False          # the reference's fp32 (trainer.precision: 32)
        torch.backends.cudnn.allow_tf32 = False
        n_det, n_obj = sample_shape(cfg)
        del model, eng
        torch.cuda.empty_cache()
        ref_gpu = CpuReference(cfg["T"], n_det=n_det, n_obj=n_obj, device=device)
        ref_gpu.run_on_device("fair")
        runs = [ref_gpu.run_on_device("fair") for _ in range(3)]
        t_best, st_best = min(runs, key=lambda r: r[0])
        t_aw, st_aw = ref_gpu.run_on_device("as_written")
        line["gpu_eager_baseline"] = dict(value=n_det / t_best, unit=UNIT, device=torch.cuda.get_device_name(device),
                                          what="the reference's eager PyTorch code path (oracle port) on this GPU, fp32 (TF32 off), "
                                               f"{n_det} detections, 'fair' variant, best of 3",
                                          stage_s={kk: round(v, 5) for kk, v in st_best.items()},
                                          as_written=dict(value=n_det / t_aw, stage_s={kk: round(v, 5) for kk, v in st_aw.items()}))
        del ref_gpu
        torch.cuda.empty_cache()
    if not args.no_cpu_baseline:
        # the CPU restatement of the reference on this box's host cores: thread count from a sweep on 4 detections, then
        # ONE pass over the bounded sample (the full c2 batch) with per-stage times
        n_det, n_obj = sample_shape(cfg)
        ref = CpuReference(cfg["T"], n_det=n_det, n_obj=n_obj)
        threads, sweep = ref.sweep_threads(cpu_thread_candidates(), n=min(4, n_det))
        t, st = ref.run("fair")
        line["cpu_baseline"] = dict(value=n_det / t, unit=UNIT, cores=threads, kind="port",
                                    sample=f"{n_det} detections over {n_obj} objects x {cfg['T']} templates, one pass of the "
                                           f"'fair' variant (IST backbone once), fp32 torch, {threads} of {os.cpu_count()} host "
                                           f"threads (fastest of a 4-detection sweep: {sweep} s)",
                                    stage_s={kk: round(v, 4) for kk, v in st.items()})
    emit(line)
    return 0


if __name__ == "__main__":
    sys.exit(main())
