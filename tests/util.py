"""Shared input generators for the tests (numpy side and torch side), and access to the golden files
that hold the reference implementation's results (tests/golden/make_golden.py writes them)."""
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FULL = 2048           # a tensor compared within a tolerance is kept whole up to this many elements,
SAMPLE = 1024         # else at (at least) this many positions, every index of every axis among them


def golden_json(name):
    with open(os.path.join(GOLD, name)) as fh:
        return json.load(fh)


def golden_values(name):
    """A golden file of tolerance records as {key: values at sample_positions, key + "/scale": max |t|}.  The
    file packs every record into one array (keys, offsets, values, scales): see pack_golden_values."""
    z = np.load(os.path.join(GOLD, name))
    out = {}
    for k, lo, hi, s in zip(z["keys"], z["offsets"][:-1], z["offsets"][1:], z["scales"]):
        out[str(k)] = z["values"][lo:hi]
        out[str(k) + "/scale"] = float(s)
    return out


def pack_golden_values(path, records):
    """Write {key: (values, scale)} in the layout golden_values reads."""
    keys = sorted(records)
    vals = [np.asarray(records[k][0], np.float32).reshape(-1) for k in keys]
    np.savez_compressed(path, keys=np.array(keys), offsets=np.cumsum([0] + [v.size for v in vals]),
                        values=np.concatenate(vals), scales=np.array([records[k][1] for k in keys], np.float64))


def case_id(shape):
    return "x".join(map(str, shape))


def digest(a, dtype=np.float32):
    """SHA-256 of an array's values as `dtype`, C order: how a golden file pins a result that must match bit
    for bit without storing it.  Takes numpy arrays and torch tensors (copied to the host)."""
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return hashlib.sha256(np.ascontiguousarray(np.asarray(a).astype(dtype, copy=False)).tobytes()).hexdigest()


def sample_positions(shape):
    """Fixed flat positions at which a golden file keeps a tensor of this shape: all of them up to FULL
    elements, else max(SAMPLE, largest dimension) seeded positions whose coordinates along every axis run
    through every index of that axis (each about equally often), so that an error confined to one slice --
    the last depth plane, say -- is among the positions."""
    shape = tuple(int(d) for d in shape)
    n = int(np.prod(shape))
    if n <= FULL:
        return np.arange(n)
    k = max(SAMPLE, max(shape))
    rng = np.random.default_rng(n)
    coords = [rng.permutation(np.resize(np.arange(d), k)) for d in shape]
    return np.unique(np.ravel_multi_index(coords, shape))


def sampled(t):
    """(values at sample_positions, max |t|) of a numpy array or torch tensor; a device tensor is gathered on
    the device, so only the sample is copied."""
    if hasattr(t, "detach"):
        import torch
        flat = t.detach().reshape(-1)
        pos = torch.from_numpy(sample_positions(t.shape)).to(flat.device)
        return (flat.index_select(0, pos).float().cpu().numpy(),
                float(flat.abs().max()) if flat.numel() else 0.0)
    t = np.asarray(t, np.float32)
    flat = t.reshape(-1)
    return flat[sample_positions(t.shape)], float(np.abs(flat).max()) if flat.size else 0.0


def assert_close_to_golden(a, gold, key, rtol=1e-4, atol=None, what=""):
    """assert_close against a reference tensor of which the golden file `gold` keeps the values at
    sample_positions (`key`) and the largest magnitude (`key/scale`): the per-tensor relative error and the
    element-wise allclose on the kept positions, and the largest magnitudes within the same bound.
    atol defaults to rtol * scale, as in assert_close."""
    vals, amax = sampled(a)
    ref, scale = gold[key], float(gold[key + "/scale"])
    what = what or key
    assert vals.shape == ref.shape, (what, vals.shape, ref.shape)
    s = max(scale, 1e-30)
    assert abs(amax - scale) <= rtol * s, "%s: max |a| %.9g vs the reference's %.9g" % (what, amax, scale)
    err = float(np.abs(vals.astype(np.float64) - ref).max()) / s if vals.size else 0.0
    assert err <= rtol, "%s: relative error %.3g > %.1g" % (what, err, rtol)
    assert np.allclose(vals, ref, rtol=rtol, atol=rtol * s if atol is None else atol * s), what


def l1norm(a, axis):
    return (a / np.abs(a).sum(axis=axis, keepdims=True)).astype(np.float32)


def sga_inputs(shape, seed=0, positive=False):
    """x, [g0..g3] L1-normalised over dim 2 (what SGABlock feeds, models/GANet_deep.py:265),
    grad_out -- all float32 numpy."""
    rng = np.random.default_rng(seed)
    N, C, D, H, W = shape
    x = rng.standard_normal(shape).astype(np.float32)
    g = [rng.standard_normal((N, C, 5, H, W)) for _ in range(4)]
    if positive:      # x in [1, 1.1), weights > 0: every aggregate stays in [1, 1.1)
        x = (1.0 + 0.1 * rng.random(shape)).astype(np.float32)
        g = [np.abs(a) + 0.05 for a in g]
    g = [l1norm(a, 2) for a in g]
    go = rng.standard_normal(shape).astype(np.float32)
    return x, g, go


def lga_inputs(shape, seed=0, radius=2):
    rng = np.random.default_rng(seed)
    F = 3 * (2 * radius + 1) ** 2
    x = rng.standard_normal(shape).astype(np.float32)
    fs = tuple(shape[:-3]) + (F,) + tuple(shape[-2:])
    f = l1norm(rng.standard_normal(fs), len(fs) - 3)
    go = rng.standard_normal(shape).astype(np.float32)
    return x, f, go


def rel_err(a, b):
    """max|a-b| / max(max|b|, tiny) -- the per-tensor relative error of SURVEY.md 8c"""
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def assert_close(a, b, rtol=1e-4, what=""):
    """north_star tolerance: 1e-4 relative fp32.  Per-tensor relative error plus an
    element-wise allclose whose atol is scaled to the tensor's magnitude."""
    a = np.asarray(a); b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    scale = max(float(np.abs(b).max()), 1e-30)
    err = rel_err(a, b)
    assert err <= rtol, "%s: relative error %.3g > %.1g" % (what, err, rtol)
    assert np.allclose(a, b, rtol=rtol, atol=rtol * scale), what
