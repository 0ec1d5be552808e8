"""Stored outputs of the reference's own operators (its CPU sources and its CUDA kernels built for sm_100a),
written by tests/golden/make_golden_ops.py, so that the tests comparing against them need neither the
reference sources nor its builds.

  golden/ops_digests.json  SHA-256 of every output that is compared bit for bit (integers, gathers, the
                           CPU SpMM whose summation order the oracle reproduces exactly)
  golden/ops_samples.npz   outputs compared within a tolerance, on a fixed sample of rows / edges
                           (sample_positions) to keep the file small
"""
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DIGESTS = "ops_digests.json"
SAMPLES = "ops_samples.npz"


def digest(a, dtype):
    """dtype, shape and SHA-256 of the bytes of `a` as a C-contiguous `dtype` array."""
    a = np.ascontiguousarray(np.asarray(a), dtype=dtype)
    return f"{a.dtype.str}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()}"


def expected_digest(key):
    with open(os.path.join(GOLD, DIGESTS)) as f:
        return json.load(f)[key]


def samples():
    return np.load(os.path.join(GOLD, SAMPLES))


def merged_digests(new):
    path = os.path.join(GOLD, DIGESTS)
    old = json.load(open(path)) if os.path.exists(path) else {}
    return dict(sorted({**old, **new}.items()))


def merged_samples(new):
    path = os.path.join(GOLD, SAMPLES)
    old = dict(np.load(path)) if os.path.exists(path) else {}
    return {**old, **new}


# ---- inputs of the comparisons (the generator and the tests build them from here)
def spmm_cpu_inputs(name):
    from tests.graphs import case

    rp, ci, n_cols = case(name)
    rng = np.random.default_rng(0)
    X = rng.standard_normal((n_cols, 48)).astype(np.float32)
    val = rng.random(ci.shape[0]).astype(np.float32)
    return rp, ci, val, X


SAMPLER_SHAPES = ((500, 12), (3000, 40), (40, 3))


def sampler_inputs(rng, n, hi):
    deg = rng.integers(0, hi, n)
    indptr = np.zeros(n + 1, np.int64)
    indptr[1:] = np.cumsum(deg)
    indices = rng.integers(0, n, int(indptr[-1])).astype(np.int64)
    batch = rng.permutation(n)[: max(1, n // 6)].astype(np.int64)
    return indptr, indices, batch


def cuda_spmm_inputs(F):
    """two_hubs graph: (rowptr, colind, n_cols, val, X, G)."""
    from tests.graphs import case

    rp, ci, n_cols = case("two_hubs")
    rng = np.random.default_rng(3)
    val = rng.random(ci.shape[0]).astype(np.float32)
    X = rng.standard_normal((n_cols, F)).astype(np.float32)
    G = rng.standard_normal((n_cols, F)).astype(np.float32)
    return rp, ci, n_cols, val, X, G


def cuda_gat_inputs(H, F):
    """two_hubs graph: (rowptr, colind, n_cols, logits, grad of att, feat, grad of out, edge permutation)."""
    from tests.graphs import case

    rp, ci, n_cols = case("two_hubs")
    rng = np.random.default_rng(4)
    e = np.clip(rng.standard_normal((ci.shape[0], H)) * 3, -10, 10).astype(np.float32)
    g = rng.standard_normal((ci.shape[0], H)).astype(np.float32)
    feat = rng.standard_normal((n_cols, H, F)).astype(np.float32)
    grad = rng.standard_normal((n_cols, H, F)).astype(np.float32)
    perm = rng.permutation(ci.shape[0]).astype(np.int32)
    return rp, ci, n_cols, e, g, feat, grad, perm


def scatter_max_inputs():
    from tests.graphs import case

    rp, ci, n_cols = case("hub")
    X = (np.random.default_rng(5).random((n_cols, 64)) + 0.01).astype(np.float32)
    return rp, ci, n_cols, X


def sample_positions(rowptr, n_rows=16, n_edges=384, seed=0):
    """(rows, edges): `n_rows` seeded rows plus the heaviest row, and at most `n_edges` seeded positions
    among those rows' edges, both ascending."""
    rowptr = np.asarray(rowptr, np.int64)
    deg = np.diff(rowptr)
    rng = np.random.default_rng(seed)
    rows = np.union1d(rng.choice(deg.shape[0], n_rows, replace=False), [int(deg.argmax())])
    edges = np.concatenate([np.arange(rowptr[r], rowptr[r + 1]) for r in rows])
    if edges.shape[0] > n_edges:
        edges = np.sort(rng.choice(edges, n_edges, replace=False))
    return rows, edges
