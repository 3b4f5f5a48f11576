"""ORACLE (test infrastructure): compact pins of reference results for tests/golden/.

Some results of the reference are too large to store whole (its streaming state is megabytes, its
weights 8 MB).  They are pinned by a fixed sample of their elements plus the norm of the whole tensor
(``pin`` / ``pin_error``), and a state_dict by per-key sums and a fixed sample of each tensor
(``fingerprint`` / ``fingerprint_mismatches``).  tests/golden/make_golden.py records these from the
reference; the tests recompute them from this project's code and compare.
"""
import numpy as np
import torch


def _flat(t):
    if isinstance(t, torch.Tensor):
        t = t.detach().cpu().numpy()
    return np.asarray(t).ravel()


def pin(name, t, n=256, seed=0):
    """npz entries pinning tensor `t` under `name`: its shape, its L2 norm and `n` sampled elements,
    half of them drawn from the non-zero ones (ring buffers are mostly zeros after a short stream)."""
    a = _flat(t).astype(np.float32)
    rng = np.random.default_rng(seed)
    idx = rng.choice(a.size, size=min(n // 2, a.size), replace=False)
    nz = np.flatnonzero(a)
    if nz.size:
        idx = np.concatenate([idx, rng.choice(nz, size=min(n - n // 2, nz.size), replace=False)])
    idx = np.unique(idx)
    return {f"{name}.shape": np.array(np.shape(t), dtype=np.int64), f"{name}.idx": idx.astype(np.int32),
            f"{name}.val": a[idx], f"{name}.norm": np.float64(np.linalg.norm(a.astype(np.float64)))}


def pin_error(g, name, t):
    """Relative error of `t` against the pin `name` in the loaded npz `g`: the larger of the rel-L2 error
    over the sampled elements and the relative error of the norm.  A shape mismatch is an error of 1."""
    if tuple(np.shape(t)) != tuple(g[f"{name}.shape"]):
        return 1.0
    a = _flat(t).astype(np.float64)
    ref = g[f"{name}.val"].astype(np.float64)
    norm = float(g[f"{name}.norm"])
    e_sample = np.linalg.norm(a[g[f"{name}.idx"]] - ref) / max(np.linalg.norm(ref), 1e-30)
    e_norm = abs(np.linalg.norm(a) - norm) / max(norm, 1e-30)
    return float(max(e_sample, e_norm))


def _spots(size, n):
    return np.linspace(0, size - 1, n).round().astype(np.int64)


def fingerprint(prefix, sd, n=8):
    """npz entries fingerprinting state_dict `sd` under `prefix`: its keys, per key the sum and the sum of
    squares (fp64) and `n` elements at evenly spaced positions."""
    keys = sorted(sd)
    stats, val = [], []
    for k in keys:
        a = _flat(sd[k]).astype(np.float64)
        stats.append([a.sum(), (a * a).sum()])
        val.append(a[_spots(a.size, n)])
    return {f"{prefix}.keys": np.array(keys), f"{prefix}.stats": np.array(stats),
            f"{prefix}.val": np.array(val, dtype=np.float32)}


def fingerprint_mismatches(g, prefix, sd, atol=1e-7):
    """Keys of `sd` that differ from the fingerprint `prefix` in the loaded npz `g` (sampled elements beyond
    `atol`, sums beyond rounding); a key present on one side only counts as a mismatch."""
    keys = [str(k) for k in g[f"{prefix}.keys"]]
    bad = sorted(set(keys) ^ set(sd))
    for j, k in enumerate(keys):
        if k not in sd:
            continue
        a = _flat(sd[k]).astype(np.float64)
        s = np.array([a.sum(), (a * a).sum()])
        ref = g[f"{prefix}.val"][j]
        if (not np.allclose(a[_spots(a.size, ref.size)], ref, atol=atol, rtol=0)
                or not np.allclose(s, g[f"{prefix}.stats"][j], rtol=1e-9, atol=atol * np.sqrt(a.size))):
            bad.append(k)
    return bad
