"""CPU test of the drop-in boundary (SURVEY §8b, VERDICT r1 item 5): with this repository BEFORE a reference checkout on
sys.path -- INTEGRATION.md's recipe -- every Hydra `_target_` of the reference's own model configs resolves to this
repository's classes and instantiates with the YAML's own kwargs, while the modules outside the hot path that `test.py`
needs (`src.dataloader.template`, `src.utils.bbox`, ...) still import from the checkout.  The model configs are the
reference's own, recorded in tests/golden/model_configs.json (`python -m oracle.make_golden_configs`); the checkout is a
stand-in written by the test whose modules import the way the reference's do (see `_CHECKOUT`)."""
import importlib
import json
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONFIGS = os.path.join(ROOT, "tests", "golden", "model_configs.json")

# Modules outside the hot path, laid out like a reference checkout (`src` and its sub-packages without __init__.py).
# Their imports follow src/dataloader/template.py and src/custom_megapose/template_dataset.py of the reference: names from
# files this repository also has (`src.utils.dataset`, `src.utils.logging`, `src.megapose.utils.tensor_collection`), a
# name only the checkout's copy of such a file has (`src.utils.inout.combine`), modules only the checkout has inside
# packages both have (`src.lib3d.numpy`, `src.utils.pil`) and packages only the checkout has.
_CHECKOUT = {
    "src/dataloader/template.py": """
        import src.megapose.utils.tensor_collection as tc
        from src.custom_megapose.template_dataset import NearestTemplateFinder, TemplateDataset
        from src.utils.dataset import LMO_index_to_ID

        class TemplateSet:
            pass
        """,
    "src/custom_megapose/template_dataset.py": """
        from src.custom_megapose.transform import Transform
        from src.lib3d.numpy import R_opencv2R_opengl
        from src.megapose.utils.tensor_collection import PandasTensorCollection
        from src.utils.inout import combine
        from src.utils.logging import get_logger
        from src.utils.pil import open_image

        class TemplateDataset:
            pass

        class NearestTemplateFinder:
            pass
        """,
    "src/custom_megapose/transform.py": "class Transform:\n    pass\n",
    "src/lib3d/numpy.py": "def R_opencv2R_opengl(R):\n    return R\n",
    "src/utils/pil.py": "def open_image(path):\n    return path\n",
    "src/utils/bbox.py": "def xyxy_to_xywh(box):\n    return box\n",
    "src/utils/inout.py": "def combine(a, b):\n    return a + b\n",
}


def _write_checkout(root):
    for rel, text in _CHECKOUT.items():
        path = os.path.join(root, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            f.write(textwrap.dedent(text).lstrip())
    return os.path.realpath(root)


def _targets(node, out):
    if isinstance(node, dict):
        if "_target_" in node:
            out.append(node["_target_"])
        for v in node.values():
            _targets(v, out)
    return out


def test_every_model_target_resolves_here():
    names = []
    with open(CONFIGS) as f:
        configs = json.load(f)
    for rel in ("model/large.yaml", "model/ae_net/dinov2_l.yaml", "model/ist_net/resnet.yaml"):
        names += _targets(configs[rel], [])
    assert "src.models.gigaPose.GigaPose" in names and "src.models.network.resnet.ResNet" in names
    for t in names:
        if t.startswith("torch."):
            continue                        # torch.hub.load: the un-vendored DINOv2 dependency (needs the network)
        mod, cls = t.rsplit(".", 1)
        m = importlib.import_module(mod)
        assert os.path.realpath(m.__file__).startswith(os.path.realpath(ROOT) + os.sep), (t, m.__file__)
        assert hasattr(m, cls), t


_SCRIPT = r"""
import json, os, sys
ROOT, REF = sys.argv[1], sys.argv[2]
sys.path[:0] = [ROOT, REF, os.path.join(REF, "src")]     # INTEGRATION.md recipe (+ src/ for `import megapose...`)
import importlib, torch
import src
assert any(p.startswith(REF) for p in src.__path__), src.__path__

def instantiate(node, **extra):
    # what hydra.utils.instantiate does for these files: recursive, `_target_` = dotted path, other keys = kwargs
    if isinstance(node, dict) and "_target_" in node:
        kwargs = {k: instantiate(v) for k, v in node.items() if k != "_target_"}
        kwargs.update(extra)
        mod, cls = node["_target_"].rsplit(".", 1)
        return getattr(importlib.import_module(mod), cls)(**kwargs)
    if isinstance(node, dict):
        return {k: instantiate(v) for k, v in node.items()}
    return node

CONFIGS = json.load(open(sys.argv[4]))

def load(rel):
    return CONFIGS[rel]

ae_cfg, ist_cfg, model_cfg = load("model/ae_net/dinov2_l.yaml"), load("model/ist_net/resnet.yaml"), load("model/large.yaml")
ist_cfg["backbone"]["config"]["descriptor_size"] = ist_cfg["descriptor_size"]        # ${model.ist_net.descriptor_size}
ist_cfg["regressor"]["descriptor_size"] = ist_cfg["descriptor_size"]
from gigapose_b200.vit import DinoVisionTransformer
ae_cfg["dinov2_model"] = None                                                         # torch.hub.load needs the network
ae = instantiate(ae_cfg, dinov2_model=DinoVisionTransformer(depth=1))
ist = instantiate(ist_cfg)
model_cfg.pop("defaults"); model_cfg["log_dir"] = sys.argv[3]; model_cfg["optim_config"]["nets_to_train"] = "all"
model_cfg["checkpoint_path"] = None
model = instantiate(model_cfg, ae_net=ae, ist_net=ist, refiner=None, test_setting="localization")
for obj, name in ((model, "src.models.gigaPose"), (ae, "src.models.network.ae_net"), (ist, "src.models.network.ist_net"),
                  (ist.backbone, "src.models.network.resnet"), (model.testing_metric, "src.models.matching")):
    f = sys.modules[type(obj).__module__].__file__
    assert type(obj).__module__ == name and os.path.realpath(f).startswith(ROOT), (name, f)
assert model.testing_metric.k == 5 and model.testing_metric.sim_threshold == 0.5
# strict state-dict surface of the checkpoint (SURVEY 8b)
keys = set(model.state_dict().keys())
for k in ("ae_net.dinov2_model.cls_token", "ae_net.dinov2_model.blocks.0.attn.qkv.weight", "ist_net.backbone.layer4_outconv.weight",
          "ist_net.backbone.layer2.0.downsample.1.running_var", "ist_net.regressor.scale_predictor.4.bias",
          "ist_net.regressor.inplane_predictor.0.weight"):
    assert k in keys, k
# modules OUTSIDE the hot path come from the checkout, unmodified (test.py:54,64)
tmpl = importlib.import_module("src.dataloader.template")
assert os.path.realpath(tmpl.__file__).startswith(REF) and hasattr(tmpl, "TemplateSet")
bbox = importlib.import_module("src.utils.bbox")
assert os.path.realpath(bbox.__file__).startswith(REF)
tds = importlib.import_module("src.custom_megapose.template_dataset")
assert os.path.realpath(tds.__file__).startswith(REF)
# ... and what they import from files that exist on both sides is served: ours first, the checkout's for the rest
import src.utils.inout as io
assert os.path.realpath(io.__file__).startswith(ROOT) and callable(io.save_bop_results) and callable(io.combine)
print("BOUNDARY_OK")
"""


def test_reference_configs_instantiate_and_dataloaders_import(tmp_path):
    ref = _write_checkout(tmp_path / "checkout")
    r = subprocess.run([sys.executable, "-c", textwrap.dedent(_SCRIPT), ROOT, ref, str(tmp_path), CONFIGS],
                       capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0 and "BOUNDARY_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
