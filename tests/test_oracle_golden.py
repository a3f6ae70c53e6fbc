"""The functional oracle against the committed golden vectors (generated from the reference's
own Python by tests/golden/make_golden.py)."""
import pytest
import torch

import cases
from helpers import Golden, assert_close_dict, rel_err
from oracle import adapters, hotpath

CASES = list(cases.CASES)


def _specs(case):
    c = cases.CASES[case]
    f = hotpath.FieldSpec(
        xyz=hotpath.hash_encoder_config(*[cases.ENC_STATIC[k] for k in
                                          ("n_levels", "base_resolution", "max_resolution", "log2_hashmap_size", "n_features_per_level")]),
        dynamic=hotpath.hash_encoder_config(*[cases.ENC_DYN[k] for k in
                                              ("n_levels", "base_resolution", "max_resolution", "log2_hashmap_size", "n_features_per_level")]) if c["dynamic"] else None,
        flow=hotpath.hash_encoder_config(*[cases.ENC_FLOW[k] for k in
                                           ("n_levels", "base_resolution", "max_resolution", "log2_hashmap_size", "n_features_per_level")]) if c["flow"] else None,
        unbounded=True, geometry_feature_dim=64, semantic_feature_dim=64 if c["feature"] else 0,
        enable_img_embedding=True, appearance_embedding_dim=16, enable_sky_head=True,
        enable_shadow_head=c["shadow"], enable_feature_head=c["feature"], enable_learnable_pe=True,
        time_diff=1.0 / cases.N_TIMESTEPS)
    props = [hotpath.FieldSpec(xyz=hotpath.hash_encoder_config(e["n_levels"], e["base_resolution"], e["max_resolution"],
                                                               e["log2_hashmap_size"], e["n_features_per_level"]),
                               unbounded=True, density_only=True) for e in cases.ENC_PROP]
    return f, props


def _render(g: Golden, case, mode, grads=False):
    fs, ps = _specs(case)
    fsd = g.tensors("sd/field")
    psd = [g.tensors(f"sd/prop{i}") for i in range(2)]
    if grads:
        for sd in [fsd] + psd:
            for k, v in sd.items():
                if v.dtype.is_floating_point and (k.endswith(".weight") or k.endswith(".bias") or k.endswith("params")
                                                 or k == "learnable_pe_map"):
                    v.requires_grad_(True)
    lidar = mode == "lidar"
    batch = g.tensors("in/lidar" if lidar else "in/pixel")
    training = mode != "eval"
    with torch.set_grad_enabled(grads):
        out, cache = hotpath.render_rays(
            fsd, fs, psd, ps, batch, num_samples=cases.NUM_SAMPLES, prop_samples=cases.PROP_SAMPLES,
            near_plane=cases.NEAR, far_plane=cases.FAR, training=training,
            proposal_requires_grad=(mode == "train"), return_decomposition=(mode == "eval"),
            prefix="lidar_" if lidar else "", jitters=g.jitters(mode) if training else None,
            noise=g.noise(mode) if training else None)
    return out, cache, fsd, psd


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("mode", ["train", "eval", "lidar"])
def test_oracle_matches_golden_outputs(case, mode):
    g = Golden(case)
    out, _, _, _ = _render(g, case, mode)
    assert_close_dict(out, g.nested(f"{mode}/out"), 5e-6)


@pytest.mark.parametrize("case", CASES)
def test_oracle_matches_golden_gradients(case):
    g = Golden(case)
    out, cache, fsd, psd = _render(g, case, "train", grads=True)
    ploss = hotpath.proposal_loss(cache, out["extras"]["trans"], (0.03, 0.003), 1024.0)
    assert abs(ploss.item() - g.scalar("train/prop_loss")) <= 1e-5 * max(1.0, abs(g.scalar("train/prop_loss")))
    loss = adapters.parity_loss(out)
    assert abs(loss.item() - g.scalar("train/loss")) <= 1e-5
    want = g.tensors("train/grad/field")
    keys = sorted(want)
    got = torch.autograd.grad(loss, [fsd[k] for k in keys], allow_unused=True)
    for k, gr in zip(keys, got):
        assert gr is not None, k
        assert rel_err(gr, want[k]) < 1e-4, k
    # propnet gradients: only the LAST proposal network is ever evaluated (Q21, late-binding lambda)
    assert len(g.tensors("train/grad/prop0")) == 0
    wantp = g.tensors("train/grad/prop1")
    gotp = torch.autograd.grad(ploss, [psd[1][k] for k in sorted(wantp)])
    for k, gr in zip(sorted(wantp), gotp):
        assert rel_err(gr, wantp[k]) < 1e-4, k

