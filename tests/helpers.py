"""Shared test helpers: golden loading and tensor comparison."""
from __future__ import annotations

import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class Golden:
    def __init__(self, case: str):
        self.case = case
        self.z = np.load(os.path.join(GOLDEN_DIR, f"{case}.npz"))

    def tensors(self, prefix: str, device="cpu"):
        out = {}
        pre = prefix.rstrip("/") + "/"
        for k in self.z.files:
            if k.startswith(pre):
                out[k[len(pre):]] = torch.from_numpy(self.z[k]).to(device)
        return out

    def nested(self, prefix: str, device="cpu"):
        """'train/out' -> {'rgb':..., 'extras': {...}}"""
        flat = self.tensors(prefix, device)
        out = {}
        for k, v in flat.items():
            if "/" in k:
                a, b = k.split("/", 1)
                out.setdefault(a, {})[b] = v
            else:
                out[k] = v
        return out

    def scalar(self, key):
        return float(self.z[key])

    def jitters(self, mode, device="cpu"):
        js, i = [], 0
        while f"{mode}/jitter{i}" in self.z.files:
            js.append(torch.from_numpy(self.z[f"{mode}/jitter{i}"]).to(device))
            i += 1
        return js or None

    def noise(self, mode, device="cpu"):
        k = f"{mode}/noise"
        return torch.from_numpy(self.z[k]).to(device) if k in self.z.files else None


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def assert_close_dict(got, want, tol, path="", skip=()):
    assert set(got) == set(want), f"{path}: keys differ {set(got) ^ set(want)}"
    for k in want:
        if k in skip:
            continue
        if isinstance(want[k], dict):
            assert_close_dict(got[k], want[k], tol, path + k + "/", skip)
            continue
        assert tuple(got[k].shape) == tuple(want[k].shape), f"{path}{k}: {got[k].shape} vs {want[k].shape}"
        t = tol[k] if isinstance(tol, dict) and k in tol else (tol["*"] if isinstance(tol, dict) else tol)
        e = rel_err(got[k], want[k])
        assert e <= t, f"{path}{k}: rel err {e:.3e} > {t:.1e}"


# ---- sampled fixtures: a fixed, seeded sample of every array, so that a whole set of outputs stays a few kB
SAMPLE = 128


def sample_positions(n: int, k: int = SAMPLE) -> torch.Tensor:
    """Flat positions compared in an array of ``n`` elements: all of them, or ``k`` drawn with seed 0 (sorted)."""
    if n <= k:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values


def pack_sampled(arrays, k: int = SAMPLE):
    """{name: tensor} -> the npz entries of one sampled set: ``meta`` (JSON: name -> shape, in order), ``values`` (the
    sampled elements, concatenated, float32) and ``maxabs`` (each array's full max |x|, the comparison's scale)."""
    import json

    names = sorted(arrays)
    vals, scale = [], []
    for n in names:
        a = arrays[n].detach().double().cpu().reshape(-1)
        vals.append(a[sample_positions(a.numel(), k)])
        scale.append(a.abs().max().item() if a.numel() else 0.0)
    meta = json.dumps({n: list(arrays[n].shape) for n in names})
    return {"meta": np.array(meta), "values": (torch.cat(vals) if vals else torch.zeros(0)).float().numpy(),
            "maxabs": np.array(scale, dtype=np.float64)}


def sampled_errors(got, z, prefix: str, k: int = SAMPLE):
    """Max relative error of each array of ``got`` against the sampled set ``prefix`` of the npz ``z``: the names
    and shapes must agree; the error is max |got - want| over the sampled positions over the full max |want|."""
    import json

    meta = json.loads(str(z[prefix + "meta"]))
    assert sorted(got) == list(meta), (prefix, sorted(set(got) ^ set(meta)))
    values, maxabs = torch.from_numpy(z[prefix + "values"]).double(), z[prefix + "maxabs"]
    errs, off = {}, 0
    for i, n in enumerate(meta):
        a = got[n].detach().double().cpu()
        assert list(a.shape) == meta[n], (prefix + n, list(a.shape), meta[n])
        pos = sample_positions(a.numel(), k)
        want = values[off:off + len(pos)]
        off += len(pos)
        errs[n] = ((a.reshape(-1)[pos] - want).abs().max().item() / max(maxabs[i], 1e-12)) if len(pos) else 0.0
    return errs
