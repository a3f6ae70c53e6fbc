"""Constructor options and data-dict shapes beyond the four golden cases: the drop-in (host side on CPU through
tests/cabi_emulator.py) against what the REFERENCE's own classes rendered (tests/golden/variants.npz, written by
tests/live_reference_variants.py), plus the drop-in at the real configuration and its ray generation against the
reference's vectors (tests/golden/builders.npz, tests/golden/raygen.npz, written by tests/live_dropin_builders.py)."""
import numpy as np

from helpers import GOLDEN_DIR, sampled_errors


def test_option_variants_match_the_live_reference(monkeypatch):
    import cabi_emulator
    import live_reference_variants as lv

    cabi_emulator.install(monkeypatch)
    z = np.load(lv.GOLDEN)
    side = lv.ours()
    assert len(lv.VARIANTS) >= 20
    calls = {}
    for name in lv.VARIANTS:
        del cabi_emulator.CALLS[:]
        res = lv.run_variant(name, side)
        calls[name] = set(cabi_emulator.CALLS)
        if f"{name}/raises" in z.files or "raises" in res:
            # the same refusal on both sides is parity too
            assert res.get("raises") == (str(z[f"{name}/raises"]) if f"{name}/raises" in z.files else None), name
            continue
        for key, err in sampled_errors(res, z, f"{name}/").items():
            # rendered outputs and per-sample extras: same arithmetic on the same host -> rounding level;
            # gradients: summation order of the scatter / weight-gradient reductions
            tol = 2e-5 if key.startswith("grad/") or key == "prop_loss" else 2e-6
            assert err <= tol, (name, key, err)
    # the fused tail must step aside where the kernel cannot take the layout ...
    for name in ("mean_embedding", "odd_geometry_width", "wide_embedding"):
        assert "emer_field_tail_fwd" not in calls[name], name
    # ... and be the path everywhere else
    for name in ("cam_embedding", "no_embedding", "bounded_aabb", "narrow_widths", "wide_heads"):
        assert "emer_field_tail_fwd" in calls[name], name
    assert "emer_linear_fwd" in calls["wide_heads"] and "emer_linear_bwd_weight" in calls["wide_heads"]


def test_reference_builders_and_default_config_build_the_dropin(monkeypatch):
    """INTEGRATION.md section 1: the reference's ``builders.py`` + ``configs/default_config.yaml`` (every branch switched
    on, real table sizes) built the model from the reference's classes; this package builds the same model (same
    state-dict names and shapes, same weights from the same seed) and renders the same rays to the same outputs."""
    import cabi_emulator
    import live_dropin_builders as lb

    cabi_emulator.install(monkeypatch)
    z = np.load(f"{GOLDEN_DIR}/builders.npz")
    del cabi_emulator.CALLS[:]
    model, n_params, out = lb.render_ours()
    assert n_params == int(z["n_params"]) > 50_000_000
    assert repr({k: list(v.shape) for k, v in model.state_dict().items()}) == str(z["state_dict"])
    assert "dino_feat" in out and "forward_flow" in out
    errs = sampled_errors(out, z, "out/")
    assert len(errs) >= 30
    for k, e in errs.items():
        assert e <= 2e-6, (k, e)
    assert {"emer_field_tail_fwd", "emer_prop_level", "emer_grid_fwd", "emer_composite_fwd"} <= set(cabi_emulator.CALLS)


def test_raygen_module_matches_the_reference_get_rays(monkeypatch):
    """emernerf_b200.raygen.get_rays (host side through the emulator) against what the reference's own function
    (datasets/base/pixel_source.py:39-76) returned for the same pixels and poses."""
    import cabi_emulator
    import live_dropin_builders as lb
    from emernerf_b200 import raygen

    cabi_emulator.install(monkeypatch)
    z = np.load(f"{GOLDEN_DIR}/raygen.npz")
    got = lb.raygen_outputs(raygen.get_rays)
    assert max(v.numel() for v in got.values()) <= lb.RAYGEN_ALL      # the fixture holds every element
    for k, e in sampled_errors(got, z, "", k=lb.RAYGEN_ALL).items():
        assert e == 0.0, (k, e)
