"""Shared helpers for the parity tests."""
from __future__ import annotations

import os
import re

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(case: str) -> dict:
    return dict(np.load(os.path.join(GOLDEN_DIR, f"{case}.npz")))


def reference_state_dict(name: str, cfg: dict) -> list:
    """[(key, shape)] in order of the reference policy's state dict, recorded by tests/golden/make_state_dict_golden.py."""
    import json

    with open(os.path.join(GOLDEN_DIR, "reference_state_dicts.json")) as fh:
        entry = json.load(fh)[name]
    assert entry["cfg"] == dict(cfg), (name, entry["cfg"], cfg)  # the recording is of this configuration
    return [(k, tuple(shape)) for k, shape in entry["state_dict"]]


def golden_pick(g: dict, name: str, actual: torch.Tensor):
    """Returns (expected, actual) numpy arrays laid out alike; undoes the strided storage of large tensors."""
    a = actual.detach().cpu()
    if a.dtype == torch.bool:
        a = a.to(torch.uint8)
    a = a.numpy()
    if name in g:
        assert tuple(g[name].shape) == tuple(a.shape), (name, g[name].shape, a.shape)
        return g[name], a
    for k in g:
        m = re.fullmatch(re.escape(name) + r"__stride(\d+)", k)
        if m:
            assert tuple(g[name + "__shape"]) == tuple(a.shape), (name, g[name + "__shape"], a.shape)
            return g[k], a.reshape(-1)[:: int(m.group(1))]
    raise KeyError(name)


def rel_l2(expected, actual) -> float:
    e = np.asarray(expected, dtype=np.float64)
    a = np.asarray(actual, dtype=np.float64)
    return float(np.linalg.norm(a - e) / max(np.linalg.norm(e), 1e-30))


def max_rel(expected, actual, floor=1e-3) -> float:
    e = np.asarray(expected, dtype=np.float64)
    a = np.asarray(actual, dtype=np.float64)
    return float(np.max(np.abs(a - e) / np.maximum(np.abs(e), floor * max(np.abs(e).max(), 1e-30))))


def allclose_ratio(expected, actual, rtol=1e-3, atol_frac=1e-4) -> float:
    """max |a - e| / (atol + rtol*|e|) with atol = atol_frac * max|e|: <= 1 means numpy.allclose(a, e, rtol, atol) holds."""
    e = np.asarray(expected, dtype=np.float64)
    a = np.asarray(actual, dtype=np.float64)
    atol = atol_frac * max(np.abs(e).max(), 1e-30)
    return float(np.max(np.abs(a - e) / (atol + rtol * np.abs(e))))


def assert_close(name, expected, actual, tol):
    r = rel_l2(expected, actual)
    assert np.isfinite(np.asarray(actual, dtype=np.float64)).all(), f"{name}: non-finite values"
    assert r <= tol, f"{name}: rel-L2 {r:.3e} > {tol:.1e}"
    return r


def argmax_safe_mask(logits: np.ndarray, dims, margin: float):
    """Per head: True where the top-2 gap of the expected logits exceeds `margin` (so an index flip is a bug,
    not a tie)."""
    out, off = [], 0
    for n in dims:
        s = np.sort(logits[..., off:off + n], axis=-1)
        out.append((s[..., -1] - s[..., -2]) > margin)
        off += n
    return np.stack(out, axis=-1)
