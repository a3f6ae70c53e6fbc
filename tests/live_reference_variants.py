"""Option variants of the field / estimator beyond the four golden cases (constructor options and data-dict shapes of
SURVEY.md section 8b that the shipped configs do not exercise).

``run_variant(name, side)`` builds one variant from ``side``'s classes (the reference's or the drop-in's: both draw the
same weights from the same seeds), renders the same rays and returns every output, plus, in training mode, the
proposal loss and the parameter gradients.  tests/test_live_reference_variants.py runs the drop-in (C ABI answered by
tests/cabi_emulator.py) against ``tests/golden/variants.npz``, which this script writes from the reference's own
classes (with the oracle stand-ins for tiny-cuda-nn / nerfacc, oracle/ref_shims.py):

    python tests/live_reference_variants.py        # needs the reference checkout (EMER_REFERENCE_ROOT)
"""
from __future__ import annotations

import os
import sys
import types
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(HERE, "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)
warnings.filterwarnings("ignore")

import cases  # noqa: E402

GOLDEN = os.path.join(HERE, "golden", "variants.npz")


def ours():
    """The drop-in's classes (the C ABI must be answered: a GPU, or tests/cabi_emulator.py)."""
    from emernerf_b200.radiance_fields import RadianceField, build_density_field
    from emernerf_b200.radiance_fields.encodings import HashEncoder
    from emernerf_b200.radiance_fields.render_utils import render_rays
    from emernerf_b200.third_party.nerfacc_prop_net import PropNetEstimator

    return types.SimpleNamespace(HashEncoder=HashEncoder, RadianceField=RadianceField,
                                 build_density_field=build_density_field, render_rays=render_rays,
                                 PropNetEstimator=PropNetEstimator)


def reference():
    """The reference's own classes, unmodified, with the oracle stand-ins for tiny-cuda-nn / nerfacc."""
    from oracle import ref_shims

    assert ref_shims.reference_available(), "needs the reference checkout (EMER_REFERENCE_ROOT)"
    ref_shims.install()
    from radiance_fields import RadianceField, build_density_field
    from radiance_fields.encodings import HashEncoder
    from radiance_fields.render_utils import render_rays
    from third_party.nerfacc_prop_net import PropNetEstimator

    return types.SimpleNamespace(HashEncoder=HashEncoder, RadianceField=RadianceField,
                                 build_density_field=build_density_field, render_rays=render_rays,
                                 PropNetEstimator=PropNetEstimator)


BASE = dict(geometry_feature_dim=64, base_mlp_layer_width=64, head_mlp_layer_width=64, enable_cam_embedding=False,
            enable_img_embedding=True, num_cams=cases.N_CAMS, appearance_embedding_dim=16, semantic_feature_dim=64,
            feature_mlp_layer_width=64, feature_embedding_dim=64, enable_sky_head=True, enable_shadow_head=False,
            enable_feature_head=False, num_train_timesteps=cases.N_TIMESTEPS, interpolate_xyz_encoding=True,
            enable_learnable_pe=True, enable_temporal_interpolation=False, unbounded=True)

# name -> (field kwargs, dynamic grid?, flow grid?, batch edits, render cfg edits, estimator kwargs, mode)
VARIANTS = {
    "cam_embedding": (dict(enable_cam_embedding=True, enable_img_embedding=False), False, False, "cam_idx", {}, {}, "eval"),
    "no_embedding": (dict(enable_img_embedding=False), False, False, None, {}, {}, "eval"),
    "mean_embedding": ({}, False, False, "drop_idx", {}, {}, "eval"),          # novel view: no img_idx in the batch
    "bounded_aabb": (dict(unbounded=False), False, False, None, {}, {}, "eval"),
    "no_sky_head": (dict(enable_sky_head=False), False, False, None, {}, {}, "eval"),
    "narrow_widths": (dict(geometry_feature_dim=32, base_mlp_layer_width=32, head_mlp_layer_width=32,
                           appearance_embedding_dim=8), False, False, None, {}, {}, "eval"),
    "odd_geometry_width": (dict(geometry_feature_dim=15), False, False, None, {}, {}, "eval"),   # the class default
    "dynamic_no_shadow": ({}, True, False, None, {}, {}, "eval"),
    "feature_head_no_pe": (dict(enable_feature_head=True, enable_learnable_pe=False), True, True, "features", {}, {},
                           "eval"),
    "wide_embedding": (dict(appearance_embedding_dim=48), False, False, None, {}, {}, "train"),   # > 32: generic tail
    "wide_heads": (dict(head_mlp_layer_width=256, base_mlp_layer_width=256, geometry_feature_dim=128), True, False,
                   None, {}, {}, "train"),                 # layers the tensor-core kernels cannot hold -> CUDA-core path
    "wide_feature_head": (dict(enable_feature_head=True, feature_mlp_layer_width=256, feature_embedding_dim=384,
                               semantic_feature_dim=32), True, True, "features384", {}, {}, "train"),
    "dynamic_model_no_time": ({}, True, False, "drop_time", {}, {}, "eval"),      # no timestamps: static branch only
    "one_proposal": ({}, False, False, None, dict(num_samples_per_prop=[24], n_props=1), {}, "train"),
    "three_proposals": ({}, False, False, None, dict(num_samples_per_prop=[40, 24, 16], n_props=3), {}, "eval"),
    "many_samples": ({}, False, False, None, dict(num_samples_per_prop=[300, 280], num_samples=270), {}, "eval"),
    "sampling_lindisp": ({}, False, False, None, dict(sampling_type="lindisp"), {}, "eval"),
    "sampling_uniform": ({}, False, False, None, dict(sampling_type="uniform", far_plane=120.0), {}, "eval"),
    "train_stratified": ({}, True, False, None, {}, {}, "train"),
    "train_plain_pdf_loss": ({}, False, False, None, {}, dict(enable_anti_aliasing_loss=False), "train"),
}


def build(ns, kwargs, dynamic, flow, seed=0):
    torch.manual_seed(seed)
    enc = ns.HashEncoder(verbose=False, **cases.ENC_STATIC)
    dyn = ns.HashEncoder(verbose=False, **cases.ENC_DYN) if dynamic else None
    flw = ns.HashEncoder(verbose=False, **cases.ENC_FLOW) if flow else None
    kw = dict(BASE)
    kw.update(kwargs)
    field = ns.RadianceField(xyz_encoder=enc, dynamic_xyz_encoder=dyn, flow_xyz_encoder=flw, aabb=cases.AABB, **kw)
    field.register_normalized_training_timesteps(torch.linspace(0, 1, cases.N_TIMESTEPS),
                                                 time_diff=1.0 / cases.N_TIMESTEPS)
    props = []
    for e in cases.ENC_PROP:
        p = ns.build_density_field(n_input_dims=3, n_levels=e["n_levels"], max_resolution=e["max_resolution"],
                                   log2_hashmap_size=e["log2_hashmap_size"],
                                   n_features_per_level=e["n_features_per_level"], unbounded=kw["unbounded"])
        p.set_aabb(cases.AABB)
        props.append(p)
    return field, props


def randomise(field, props, seed=1):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in [field] + props:
            for k, v in m.named_parameters():
                if k.endswith("tcnn_encoding.params"):
                    v.copy_(torch.randn(v.shape, generator=g) * 0.5)


def flatten(d, prefix=""):
    out = {}
    for k, v in d.items():
        if isinstance(v, dict):
            out.update(flatten(v, prefix + k + "/"))
        else:
            out[prefix + k] = v
    return out


def run_variant(name, side):
    """Every output of variant ``name`` rendered with ``side``'s classes, flat: ``out/<key>``, and in training mode
    ``prop_loss`` and ``grad/<parameter>`` / ``grad/prop<i>/<parameter>`` for every parameter that receives a gradient.
    A refusal (the same on both sides is parity too) is returned as ``{"raises": "<type>: <message>"}``."""
    kwargs, dynamic, flow, edit, cfg_edit, est_kw, mode = VARIANTS[name]
    field, props = build(side, kwargs, dynamic, flow)
    randomise(field, props)
    case = "flow_feat" if edit in ("features", "features384") else "static"
    batch = cases.make_batch(case)
    if edit == "features384":
        batch["features"] = torch.rand(batch["origins"].shape[0], 384, generator=torch.Generator().manual_seed(5))
    if edit == "cam_idx":
        batch["cam_idx"] = batch.pop("img_idx") % cases.N_CAMS
    elif edit == "drop_idx":
        batch.pop("img_idx")
    elif edit == "drop_time":
        batch.pop("normed_timestamps")
    cfg = cases.render_cfg()
    cfg_edit = dict(cfg_edit)
    n_props = cfg_edit.pop("n_props", None)
    if "num_samples" in cfg_edit:
        cfg.nerf.sampling.num_samples = cfg_edit.pop("num_samples")
    for k, v in cfg_edit.items():
        setattr(cfg.nerf.propnet, k, v)
    if n_props is not None:
        # drop one network, or append a third built like the second
        props = props[:n_props]
        while len(props) < n_props:
            e = cases.ENC_PROP[-1]
            torch.manual_seed(9)
            p = side.build_density_field(n_input_dims=3, n_levels=e["n_levels"], max_resolution=e["max_resolution"],
                                         log2_hashmap_size=e["log2_hashmap_size"],
                                         n_features_per_level=e["n_features_per_level"], unbounded=True)
            p.set_aabb(cases.AABB)
            randomise(p, [], seed=3)
            props.append(p)
    train = mode == "train"
    est = side.PropNetEstimator(torch.optim.Adam([q for p in props for q in p.parameters()], lr=0.01), None, **est_kw)
    for m in (field, est, *props):
        m.train(train)
    with torch.set_grad_enabled(train):
        torch.manual_seed(77)
        try:
            out = side.render_rays(field, est, props, dict(batch), cfg, proposal_requires_grad=train,
                                   return_decomposition=not train)
        except (AssertionError, ValueError, KeyError) as e:
            return {"raises": f"{type(e).__name__}: {e}"}
    res = flatten(out, "out/")
    if train:
        ploss = est.compute_loss(out["extras"]["trans"], 1024.0)
        res["prop_loss"] = ploss
        loss = (out["rgb"] - batch["pixels"]).square().mean() + out["depth"].mean() * 1e-2
        (loss + ploss).backward()
        res.update({"grad/" + k: v.grad for k, v in field.named_parameters() if v.grad is not None})
        for i, p in enumerate(props):
            res.update({f"grad/prop{i}/" + k: v.grad for k, v in p.named_parameters() if v.grad is not None})
    return {k: v if isinstance(v, str) else v.detach() for k, v in res.items()}


if __name__ == "__main__":
    from helpers import pack_sampled

    ref = reference()
    store = {}
    for name in VARIANTS:
        res = run_variant(name, ref)
        if "raises" in res:
            store[f"{name}/raises"] = np.array(res["raises"])
        else:
            store.update({f"{name}/{k}": v for k, v in pack_sampled(res).items()})
    np.savez_compressed(GOLDEN, **store)
    print(GOLDEN, os.path.getsize(GOLDEN), "bytes")
