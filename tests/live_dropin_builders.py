"""The drop-in at the REAL configuration, against vectors the reference's own code produced.

``python tests/live_dropin_builders.py`` (needs the reference checkout, EMER_REFERENCE_ROOT) writes two fixtures:

  builders.npz  the reference's unmodified ``builders.py`` builds the model and the proposal estimator from its
                ``configs/default_config.yaml`` with every branch switched on (dynamic, flow, shadow, feature head; real
                table sizes, 203 MB of grids) and the reference's classes (oracle stand-ins for tiny-cuda-nn / nerfacc);
                stored: the state-dict's names and shapes, the parameter count and a sample of the rendered outputs
  raygen.npz    the reference's ``get_rays`` (datasets/base/pixel_source.py, executed from its source file) on seeded
                pixels and poses, every element

tests/test_live_reference_variants.py builds the same model with ``emernerf_b200.configs`` (same seed, hence the same
weights) and compares.  Only ``omegaconf`` (annotation only) and ``datasets.base`` (annotation only; its real import
chain needs timm) are stubbed while the reference builds.
"""
from __future__ import annotations

import os
import re
import sys
import types
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("EMER_REFERENCE_ROOT", "/root/reference")
for p in (ROOT, HERE, os.path.join(HERE, "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)
warnings.filterwarnings("ignore")

N_RAYS, T = 40, 12
AABB = [-25.0, -35.0, -2.0, 90.0, 45.0, 25.0]      # the dataset's aabb, which builders.py gives the model


class Cfg(dict):
    """attribute-style access like OmegaConf's DictConfig (what builders.py / render_rays do with cfg)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


def to_cfg(o):
    if isinstance(o, dict):
        return Cfg({k: to_cfg(v) for k, v in o.items()})
    if isinstance(o, list):
        return [to_cfg(v) for v in o]
    if isinstance(o, str) and re.fullmatch(r"[+-]?\d+(\.\d*)?[eE][+-]?\d+", o):
        return float(o)                     # "1e-5": a float to OmegaConf (YAML 1.2), a string to PyYAML (YAML 1.1)
    return o


def load_cfg():
    import yaml

    with open(os.path.join(REF, "configs", "default_config.yaml")) as f:
        cfg = to_cfg(yaml.safe_load(f))
    head = cfg.nerf.model.head
    head.enable_dynamic_branch = True
    head.enable_flow_branch = True
    head.enable_shadow_head = True
    head.enable_feature_head = True
    # what train_emernerf.py:130-133 copies into the model section before calling the builders
    cfg.nerf.model.num_cams = cfg.data.pixel_source.num_cams
    cfg.nerf.model.unbounded = cfg.nerf.unbounded
    cfg.nerf.model.resume_from = cfg.resume_from
    return cfg


def dataset_stub():
    px = types.SimpleNamespace(features=None)
    return types.SimpleNamespace(num_train_timesteps=T, test_pixel_set=None, num_img_timesteps=T,
                                 unique_normalized_training_timestamps=torch.linspace(0, 1, T),
                                 aabb=torch.tensor(AABB), pixel_source=px)


def stub_annotation_only_modules():
    if "omegaconf" not in sys.modules:
        m = types.ModuleType("omegaconf")
        m.OmegaConf = type("OmegaConf", (), {})
        sys.modules["omegaconf"] = m
    ds = types.ModuleType("datasets")
    ds.__path__ = []
    base = types.ModuleType("datasets.base")
    base.SceneDataset = type("SceneDataset", (), {})
    sys.modules["datasets"], sys.modules["datasets.base"] = ds, base


def make_batch():
    import cases

    b = cases.make_batch("flow_feat", seed=3, n_rays=N_RAYS)
    b["img_idx"] = torch.randint(0, T * 3, (N_RAYS,), generator=torch.Generator().manual_seed(8))
    return b


def build_with_reference_builders(cfg):
    """builders.py, verbatim: whatever ``radiance_fields`` / ``third_party`` resolve to builds the model."""
    import builders

    ds = dataset_stub()
    model = builders.build_model_from_cfg(cfg.nerf.model, ds, torch.device("cpu"))
    est, props = builders.build_estimator_and_propnet_from_cfg(cfg.nerf, cfg.optim, ds, torch.device("cpu"))
    return model, est, props


def render(model, est, props, batch, cfg):
    from radiance_fields.render_utils import render_rays          # the name train_emernerf.py imports

    for m in (model, est, *props):
        m.eval()
    with torch.no_grad():
        return render_rays(radiance_field=model, proposal_estimator=est, proposal_networks=props, data_dict=batch,
                           cfg=cfg, proposal_requires_grad=False, return_decomposition=True)


def flatten(d, prefix=""):
    out = {}
    for k, v in d.items():
        if isinstance(v, dict):
            out.update(flatten(v, prefix + k + "/"))
        else:
            out[prefix + k] = v
    return out


def randomise_tables(model, props):
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():                       # give the scene structure (tcnn's own init is ~1e-4)
        for m in [model] + props:
            for k, v in m.named_parameters():
                if k.endswith("tcnn_encoding.params"):
                    v.copy_(torch.randn(v.shape, generator=g) * 0.5)


def build_ours():
    """The same model and networks from this package: default_config's values (emernerf_b200.configs, every branch on),
    the same seed as the reference's build."""
    from emernerf_b200 import configs

    cfg = configs.make_cfg("flow_feat", num_timesteps=T)
    model, props, est, _ = configs.build_hot_path(cfg, "cpu")
    for m in [model] + props:
        m.set_aabb(AABB)
    randomise_tables(model, props)
    return model, est, props, cfg


def render_ours():
    """(model, parameter count, flat outputs) of the drop-in on the fixture's rays."""
    from emernerf_b200.radiance_fields.render_utils import render_rays

    model, est, props, cfg = build_ours()
    for m in (model, est, *props):
        m.eval()
    with torch.no_grad():
        out = render_rays(radiance_field=model, proposal_estimator=est, proposal_networks=props,
                          data_dict=make_batch(), cfg=cfg, proposal_requires_grad=False, return_decomposition=True)
    return model, sum(p.numel() for p in model.parameters()), flatten(out)


RAYGEN_RAYS = 777
RAYGEN_ALL = 3 * RAYGEN_RAYS          # sample size that keeps every element of every get_rays output


def raygen_inputs():
    g = torch.Generator().manual_seed(0)
    R = RAYGEN_RAYS
    x, y = torch.randint(0, 960, (R,), generator=g).float(), torch.randint(0, 640, (R,), generator=g).float()
    c2w = torch.eye(4).repeat(R, 1, 1) + torch.randn(R, 4, 4, generator=g) * 0.3
    K = torch.tensor([[1030.0, 0, 480], [0, 1030, 320], [0, 0, 1]]).repeat(R, 1, 1)
    return x, y, c2w, K


def raygen_outputs(get_rays):
    """get_rays on per-ray poses and on one shared pose: {"batched/<i>", "shared/<i>"} for each returned tensor."""
    x, y, c2w, K = raygen_inputs()
    res = {f"batched/{i}": t for i, t in enumerate(get_rays(x, y, c2w, K))}
    res.update({f"shared/{i}": t for i, t in enumerate(get_rays(x, y, c2w[0], K[0]))})
    return res


def write_golden():
    from helpers import GOLDEN_DIR, pack_sampled
    from oracle import ref_shims

    cfg = load_cfg()
    stub_annotation_only_modules()
    sys.path.insert(0, REF)
    ref_shims.install()
    torch.manual_seed(0)
    model, est, props = build_with_reference_builders(cfg)
    randomise_tables(model, props)
    assert type(model).__module__ == "radiance_fields.radiance_field", type(model).__module__
    out = flatten(render(model, est, props, make_batch(), cfg))
    sd = model.state_dict()
    store = {f"out/{k}": v for k, v in pack_sampled(out).items()}
    store["state_dict"] = np.array(repr({k: list(v.shape) for k, v in sd.items()}))
    store["n_params"] = np.array(sum(p.numel() for p in model.parameters()))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "builders.npz"), **store)

    src = open(os.path.join(REF, "datasets", "base", "pixel_source.py")).read()
    body = src[src.index("def get_rays("):src.index("class ScenePixelSource")]
    ns = {}
    exec("import torch\nfrom torch import Tensor\nfrom typing import Tuple\n" + body, ns)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "raygen.npz"), **pack_sampled(raygen_outputs(ns["get_rays"]), k=RAYGEN_ALL))


if __name__ == "__main__":
    write_golden()
