"""Deterministic parameter filling and the compact golden-array format, shared by the golden-vector script and the tests.
TEST INFRASTRUCTURE (see oracle/__init__.py)."""
from __future__ import annotations

import contextlib
import hashlib
import zlib

import numpy as np
import torch


def fill_module(module: torch.nn.Module, seed: int = 666, running_stats: bool = True):
    """Fill every parameter / BN buffer of `module` from one numpy Generator, visiting names in sorted
    order, so the reference model, the oracle model and the CUDA model (same state_dict keys) get
    bit-identical values without storing a checkpoint."""
    rng = np.random.default_rng(seed)
    sd = module.state_dict()
    with torch.no_grad():
        for name in sorted(sd.keys()):
            t = sd[name]
            if name.endswith('num_batches_tracked'):
                t.zero_()
            elif name.endswith('running_var'):
                v = rng.uniform(0.5, 1.5, size=tuple(t.shape)) if running_stats else np.ones(tuple(t.shape))
                t.copy_(torch.from_numpy(v.astype(np.float32)))
            elif name.endswith('running_mean'):
                v = rng.normal(0, 0.1, size=tuple(t.shape)) if running_stats else np.zeros(tuple(t.shape))
                t.copy_(torch.from_numpy(v.astype(np.float32)))
            elif t.dim() == 1 and name.endswith('.weight'):      # BN gamma
                t.copy_(torch.from_numpy(rng.uniform(0.5, 1.5, size=tuple(t.shape)).astype(np.float32)))
            elif t.dim() == 1:                                   # BN beta / bias
                t.copy_(torch.from_numpy(rng.normal(0, 0.1, size=tuple(t.shape)).astype(np.float32)))
            else:                                                # conv weight (C_out, *k, C_in)
                fan_in = int(np.prod(t.shape[1:]))
                v = rng.normal(0, (2.0 / fan_in) ** 0.5, size=tuple(t.shape))
                t.copy_(torch.from_numpy(v.astype(np.float32)))
    return module


def rel_err(got, want):
    """max|got-want| / max|want| — the tolerance form BASELINE.json's north_star states (1e-4)."""
    got = torch.as_tensor(got).double()
    want = torch.as_tensor(want).double()
    return float((got - want).abs().max() / want.abs().max().clamp_min(1e-30))


# Train-mode BatchNorm on the CPU sums its batch statistics in per-thread partial sums, so the last bits of its output
# follow torch's intra-op thread count; the bit-exact fixtures of tests/golden/ are made and checked with this many threads.
GOLDEN_THREADS = 8


@contextlib.contextmanager
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def sha256_bytes(a) -> str:
    """SHA-256 of an array's (or tensor's) bytes in C order."""
    return hashlib.sha256(np.ascontiguousarray(torch.as_tensor(a).detach().cpu().numpy()).tobytes()).hexdigest()


def sha256_f32(a) -> str:
    """SHA-256 of an array as float32 bytes, -0.0 folded into +0.0 (np.array_equal's notion of equal, NaN aside)."""
    return sha256_bytes(np.asarray(torch.as_tensor(a).detach().cpu().numpy(), dtype=np.float32) + np.float32(0))


def sampled_rows(key, a):
    """A golden float array stored compactly: a seeded quarter of its rows (`key`, row numbers in `key.rows`) plus what a
    comparison of the whole array needs — its digest (`key.sha256`) and its largest magnitude (`key.absmax`)."""
    a = np.asarray(a, dtype=np.float32)
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    rows = np.sort(rng.choice(a.shape[0], -(-a.shape[0] // 4), replace=False)).astype(np.int32)
    return {key: a[rows], key + '.rows': rows, key + '.sha256': np.array(sha256_f32(a)),
            key + '.absmax': np.float32(np.abs(a).max() if a.size else 0)}


def check_sampled_rows(got, g, key, tol=None):
    """`got` against an array stored by sampled_rows in the npz `g`.  tol None: bit-exact — the sampled rows, then the
    digest of the whole array.  Otherwise rel_err on the sampled rows, relative to the whole golden array's max |x|."""
    got = torch.as_tensor(got).detach().cpu()
    rows = torch.from_numpy(g[key + '.rows']).long()
    if tol is None:
        assert np.array_equal(got[rows].numpy(), g[key]), key
        assert sha256_f32(got) == str(g[key + '.sha256']), key
    else:
        err = float((got[rows].double() - torch.from_numpy(g[key]).double()).abs().max()) if len(rows) else 0.0
        assert err / max(float(g[key + '.absmax']), 1e-30) < tol, (key, err)


def join_by_coords(idx_a, feat_a, idx_b, feat_b):
    """Align two sparse tensors by coordinate (row order may differ); returns (feat_a, feat_b[perm])."""
    a = np.asarray(idx_a).astype(np.int64)
    b = np.asarray(idx_b).astype(np.int64)
    assert a.shape == b.shape, (a.shape, b.shape)
    mx = np.maximum(a.max(0), b.max(0)) + 1
    ka = np.ravel_multi_index(a.T, mx)
    kb = np.ravel_multi_index(b.T, mx)
    oa, ob = np.argsort(ka, kind='stable'), np.argsort(kb, kind='stable')
    assert np.array_equal(ka[oa], kb[ob]), 'coordinate sets differ'
    perm = np.empty_like(oa)
    perm[oa] = ob
    return feat_a, torch.as_tensor(feat_b)[torch.from_numpy(perm)]
