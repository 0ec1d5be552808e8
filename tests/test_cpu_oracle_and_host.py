"""CPU-side tests (run with -m "not gpu"): the oracle against the reference's golden vectors and
against the reference's own compiled sources, the C-ABI library's symbol table, and host logic.
No compute call into libcogdl_b200 happens here (there is no GPU)."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch

import oracle
from tests import refgold
from tests.graphs import CASES, case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def gold(name):
    return np.load(os.path.join(GOLD, name))


# ------------------------------------------------------------------ oracle vs golden (reference package outputs)
def test_oracle_spmm_bit_exact_vs_reference_spmm_on_cora_shape():
    g = gold("spmm_cora.npz")
    for x, y in ((g["x16"], g["y16"]), (g["x7"], g["y7"])):
        out = oracle.spmm_csr(g["row_ptr"], g["col_indices"], g["weight"], x)
        assert np.array_equal(out, y)  # same order, same rounding as cogdl.utils.spmm on CPU


def test_oracle_spmm_with_in_norm_matches_reference_row_norm_path():
    g = gold("spmm_rownorm.npz")
    assert not bool(g["has_out_norm"])
    out = oracle.spmm_csr(g["row_ptr"], g["col_indices"], None, g["x"])
    assert np.array_equal(g["in_norm"] * out, g["y"])  # in_norm applied around the kernel, spmm_utils.py:118-119


def test_oracle_edge_softmax_vs_reference_cpu_fallback():
    g = gold("edge_softmax.npz")
    out = oracle.edge_softmax_fwd(g["row_ptr"], g["logits"])
    # the reference fallback computes exp(x)/sum exp(x) in fp32 without max subtraction: tolerance
    assert np.allclose(out, g["att"], rtol=2e-5, atol=1e-8)


def test_oracle_mhspmm_bit_exact_vs_reference_cpu_fallback():
    g = gold("mh_spmm.npz")
    H, F = g["h"].shape[1:]
    out = oracle.mhspmm(g["row_ptr"], g["col_indices"], g["att"], g["h"]).reshape(-1, H * F)
    assert np.array_equal(out, g["out"])  # per-head spmm_cpu order


def test_oracle_coo2csr_index_bit_exact_vs_reference_sampler():
    g = gold("coo2csr.npz")
    rp, re_ = oracle.coo2csr_index(g["row"], int(g["num_nodes"]))
    assert np.array_equal(rp, g["row_ptr"]) and np.array_equal(re_, g["reindex"])


def test_oracle_gat_forward_vs_reference_gat_layer():
    g = gold("gat_layer.npz")
    x, W, a_l, a_r = g["x"], g["W"], g["a_l"], g["a_r"]
    H, F = a_l.shape[1:]
    h = (x @ W).reshape(-1, H, F).astype(np.float32)
    h_l, h_r = (a_l * h).sum(-1), (a_r * h).sum(-1)
    out = oracle.gat_fwd(g["row_ptr"], g["col_indices"], h_l, h_r, h, 0.2).reshape(h.shape[0], -1)
    assert np.abs(out - g["y"]).max() <= 1e-5 * max(1.0, np.abs(g["y"]).max())


# ------------------------------------------------------------------ oracle vs the reference's own compiled C++
# (its outputs stored as digests in tests/golden/ops_digests.json by tests/golden/make_golden_ops.py)
@pytest.mark.parametrize("variant", ["asis", "o3"])
@pytest.mark.parametrize("name", [k for k in CASES if k != "rect"])
def test_oracle_spmm_bit_exact_vs_compiled_reference(variant, name):
    rp, ci, val, X = refgold.spmm_cpu_inputs(name)
    got = refgold.digest(oracle.spmm_csr(rp, ci, val, X), np.float32)
    assert got == refgold.expected_digest(f"spmm_cpu/{variant}/{name}")


def test_oracle_csr2csc_is_stable_transpose():
    import scipy.sparse as sp

    for name in CASES:
        rp, ci, n_cols = case(name)
        n = rp.shape[0] - 1
        colptr, rowind, perm = oracle.csr2csc(rp, ci, n_cols)
        assert colptr[-1] == ci.shape[0]
        # entries of each column keep CSR order (ascending CSR position)
        for c in range(n_cols):
            seg = perm[colptr[c]:colptr[c + 1]]
            assert np.all(np.diff(seg) > 0)
            assert np.all(ci[seg] == c)
        rows = np.repeat(np.arange(n), np.diff(rp))
        assert np.array_equal(rowind, rows[perm])
        if ci.shape[0]:
            m = sp.csr_matrix((np.ones(ci.shape[0]), ci, rp), shape=(n, n_cols)).tocsc()
            assert np.array_equal(m.indptr, colptr)


def test_oracle_scatter_max_matches_numpy_and_reference_semantics():
    rp, ci, n_cols = case("ragged")
    X = np.random.default_rng(1).standard_normal((n_cols, 5)).astype(np.float32)
    out, arg = oracle.scatter_max_fwd(rp, ci, X)
    for i in range(rp.shape[0] - 1):
        cols = ci[rp[i]:rp[i + 1]]
        if len(cols) == 0:
            assert np.all(out[i] == 0) and np.all(arg[i] == -1)
        else:
            assert np.array_equal(out[i], X[cols].max(0))
            assert np.array_equal(arg[i], cols[X[cols].argmax(0)])  # numpy argmax = first max
    # reference semantics (FLT_MIN seed) agree on strictly positive features
    Xp = np.abs(X) + 0.1
    a, ia = oracle.scatter_max_fwd(rp, ci, Xp)
    b, ib = oracle.scatter_max_fwd(rp, ci, Xp, reference_semantics=True)
    has = np.diff(rp) > 0
    assert np.array_equal(a[has], b[has]) and np.array_equal(ia[has], ib[has])
    # ...and differ exactly where the reference's bug shows: all-negative neighbourhoods
    c, _ = oracle.scatter_max_fwd(rp, ci, -Xp, reference_semantics=True)
    assert np.all(c[has] == np.finfo(np.float32).tiny)


def test_oracle_edge_softmax_backward_matches_autograd():
    rp, ci, _ = case("ragged")
    rng = np.random.default_rng(2)
    e = rng.standard_normal((ci.shape[0], 4)).astype(np.float32)
    g = rng.standard_normal((ci.shape[0], 4)).astype(np.float32)
    y = oracle.edge_softmax_fwd(rp, e)
    gin = oracle.edge_softmax_bwd(rp, y, g)
    et = torch.tensor(e, dtype=torch.float64, requires_grad=True)
    outs = []
    for i in range(rp.shape[0] - 1):
        if rp[i + 1] > rp[i]:
            outs.append(torch.softmax(et[rp[i]:rp[i + 1]], 0))
    yt = torch.cat(outs)
    yt.backward(torch.tensor(g, dtype=torch.float64))
    assert np.allclose(y, yt.detach().numpy(), atol=1e-6)
    assert np.allclose(gin, et.grad.numpy(), atol=1e-5)


# ------------------------------------------------------------------ C-ABI library: loads, exports every declared symbol
def declared_symbols():
    with open(os.path.join(ROOT, "include", "cogdl_b200.h")) as f:
        text = f.read()
    return sorted(set(re.findall(r"COGDL_B200_API[^;(]*?\b(cogdl_b200_[a-z0-9_]+)\s*\(", text)))


def test_cabi_library_exports_every_header_symbol():
    lib_path = os.path.join(ROOT, "cogdl_b200", "lib", "libcogdl_b200.so")
    assert os.path.exists(lib_path), "build() must produce the C-ABI library"
    lib = ctypes.CDLL(lib_path)
    names = declared_symbols()
    assert len(names) >= 24
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/cogdl_b200.h but not exported"
    lib.cogdl_b200_abi_version.restype = ctypes.c_int
    assert lib.cogdl_b200_abi_version() == 5


def test_python_binding_lists_exactly_the_header_symbols():
    from cogdl_b200 import _cabi

    assert sorted(_cabi.SIGNATURES) == declared_symbols()
    _cabi.load()


def test_library_is_sm100a_only_and_has_no_torch_dependency():
    import subprocess

    lib_path = os.path.join(ROOT, "cogdl_b200", "lib", "libcogdl_b200.so")
    out = subprocess.run(["cuobjdump", "-lelf", lib_path], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs
    ldd = subprocess.run(["ldd", lib_path], capture_output=True, text=True).stdout
    assert "torch" not in ldd and "c10" not in ldd


# ------------------------------------------------------------------ host logic
def test_no_cpu_fallback():
    import cogdl_b200

    g = cogdl_b200.Graph(x=torch.randn(4, 3), edge_index=(torch.tensor([0, 1, 2]), torch.tensor([1, 2, 3])))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cogdl_b200.spmm(g, g.x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cogdl_b200.edge_softmax(g, torch.randn(3, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cogdl_b200.csrspmm(torch.tensor([0, 1], dtype=torch.int32), torch.tensor([0], dtype=torch.int32), torch.randn(1, 4), None)


def test_graph_semantics_match_reference_graph():
    import cogdl_b200

    g = gold("graph_semantics.npz")
    row, col = torch.from_numpy(g["row"]), torch.from_numpy(g["col"])
    n = 50
    ga = cogdl_b200.Graph(x=torch.zeros(n, 1), edge_index=(row, col))
    ga.add_remaining_self_loops()
    assert np.array_equal(ga.row_indptr.numpy(), g["row_ptr"]) and np.array_equal(ga.col_indices.numpy(), g["col_indices"])
    assert np.array_equal(ga.edge_weight.numpy(), g["w0"])
    ga.sym_norm()
    assert np.allclose(ga.edge_weight.numpy(), g["w_sym"], rtol=1e-6, atol=0) and ga.is_symmetric() == bool(g["sym_flag"])
    gb = cogdl_b200.Graph(x=torch.zeros(n, 1), edge_index=(row, col))
    gb.add_remaining_self_loops()
    gb.row_norm()
    assert np.allclose(gb.edge_weight.numpy(), g["w_row"], rtol=1e-6, atol=0) and gb.is_symmetric() == bool(g["row_flag"])
    gc = cogdl_b200.Graph(x=torch.zeros(n, 1), edge_index=(row, col))
    gc.add_remaining_self_loops()
    gc.edge_weight = torch.arange(gc.num_edges).float()
    assert gc.is_symmetric() == bool(g["set_flag"])
    with gc.local_graph():
        gc.edge_weight = torch.ones(gc.num_edges)
        assert float(gc.edge_weight.sum()) == gc.num_edges
    assert float(gc.edge_weight[-1]) == gc.num_edges - 1  # restored


def test_host_coo2csr_index_matches_reference():
    from cogdl_b200.data import coo2csr_index

    g = gold("coo2csr.npz")
    rp, re_ = coo2csr_index(torch.from_numpy(g["row"]), int(g["num_nodes"]))
    assert np.array_equal(rp.numpy(), g["row_ptr"]) and np.array_equal(re_.numpy(), g["reindex"])


def test_synthetic_generator_is_deterministic_and_power_law():
    from cogdl_b200 import synth

    a = synth.powerlaw_csr(5000, 40000, seed=3)
    b = synth.powerlaw_csr(5000, 40000, seed=3)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    rp, col = a
    deg = (rp[1:] - rp[:-1])
    assert int(rp[-1]) == 45000 and int(deg.min()) >= 1           # + one self loop per row
    assert int(deg.max()) > 30 * float(deg.float().median())      # heavy tail
    last = col[rp[1:] - 1]
    assert torch.equal(last, torch.arange(5000))                  # the self loop closes each row


def test_install_registers_backend_in_reference_package():
    """Drop-in mechanics against the real cogdl package (only where /root/reference exists)."""
    if not os.path.isdir("/root/reference/cogdl"):
        pytest.skip("reference package not present on this box")
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden

    make_golden.import_reference()
    import cogdl.utils.spmm_utils as ref_su
    import cogdl.layers.gcn_layer as ref_gcn
    import cogdl_b200

    patched = cogdl_b200.install()
    assert ref_su.CONFIGS["fast_spmm"] is cogdl_b200.csrspmm
    assert ref_su.CONFIGS["csr_edge_softmax"] is cogdl_b200.csr_edge_softmax
    assert ref_su.CONFIGS["csrmhspmm"] is cogdl_b200.csrmhspmm
    assert ref_su.CONFIGS["spmm_flag"] and ref_su.CONFIGS["mh_spmm_flag"]
    assert ref_gcn.spmm is cogdl_b200.spmm, "layer modules must be rebound to the cached-structure dispatch"
    assert any(p.endswith("gcn_layer.spmm") for p in patched)
    import cogdl.operators.scatter_max as ref_sm

    assert ref_sm.scatter_max is cogdl_b200.scatter_max


def test_oracle_sampler_is_pinned_to_the_reference_sample_cpp():
    """No-randomness paths of sample.cpp (sample_adj with num_neighbors = -1, subgraph) compiled from the
    reference's own source vs the oracle restatement: every output array identical (the reference's outputs
    stored as digests in tests/golden/ops_digests.json)."""
    rng = np.random.default_rng(0)
    for n, hi in refgold.SAMPLER_SHAPES:
        indptr, indices, batch = refgold.sampler_inputs(rng, n, hi)
        got = oracle.sample_adj(indptr, indices, batch, -1, False)
        assert len(got) == 4
        for k, a in enumerate(got):
            assert refgold.digest(a, np.int64) == refgold.expected_digest(f"sample_adj/{n}/{k}"), (n, k)
        got = oracle.subgraph(indptr, indices, batch)
        for k, a in ((0, got[0]), (1, got[1]), (2, np.arange(batch.shape[0])), (3, got[2])):
            assert refgold.digest(a, np.int64) == refgold.expected_digest(f"subgraph/{n}/{k}"), (n, k)
        # random paths: the row sizes and the first-appearance numbering obey the reference's rules
        for size, replace in ((4, True), (4, False)):
            oi, oc, on, oe = oracle.sample_adj(indptr, indices, batch, size, replace, seed=7)
            d = indptr[batch + 1] - indptr[batch]
            want = np.where(d > 0, size, 0) if replace else np.minimum(d, size)
            assert np.array_equal(np.diff(oi), want)
            assert np.array_equal(on[: batch.shape[0]], batch) and np.array_equal(on[oc], indices[oe])
            first = {}
            for q, s_ in enumerate(indices[oe]):
                first.setdefault(int(s_), q)
            new = [s_ for s_ in sorted(first, key=first.get) if s_ not in set(batch.tolist())]
            assert on[batch.shape[0]:].tolist() == new


def test_sampler_generator_matches_between_library_and_oracle():
    import cogdl_b200

    lib = cogdl_b200._cabi.load()
    for seed, slot, k in ((0, 0, 0), (1, 2, 3), (2**63 + 5, 10**9, 77), (2**64 - 1, 2**40, 2**33)):
        assert int(lib.cogdl_b200_sample_draw(seed, slot, k)) == oracle.sample_draw(seed, slot, k)


def test_bf16x3_split_gemm_numerics_emulated():
    """The fused GCN layer (cogdl_b200/csrc/fused_gcn.cu) multiplies fp32 operands on the bf16 tensor cores by
    splitting each into three bf16 terms and adding the six products of order <= 2^-16.  Emulated here in
    numpy (bf16 rounding through torch): the error against fp64 must be at the 1e-7 level, i.e. well inside
    the 1e-5 bar, while plain bf16 and the 3-term shortcut are not."""
    rng = np.random.default_rng(0)

    def bf16(x):
        return torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()

    def split3(x):
        a1 = bf16(x)
        r1 = (x - a1).astype(np.float32)
        a2 = bf16(r1)
        a3 = bf16((r1 - a2).astype(np.float32))
        assert np.abs(x.astype(np.float64) - (a1.astype(np.float64) + a2 + a3)).max() <= 2.0 ** -22 * np.abs(x).max()
        return a1, a2, a3

    A = (rng.standard_normal((256, 128)) * rng.random((256, 1)) * 30).astype(np.float32)
    W = (rng.standard_normal((128, 128)) / 11.3).astype(np.float32)
    ref = A.astype(np.float64) @ W.T.astype(np.float64)
    scale = np.maximum(np.abs(ref), np.abs(ref).max(1, keepdims=True))
    As, Ws = split3(A), split3(W)
    acc = np.zeros_like(ref, dtype=np.float32)
    for i, j in [(2, 0), (1, 1), (0, 2), (1, 0), (0, 1), (0, 0)]:
        acc = (acc + (As[i].astype(np.float64) @ Ws[j].T.astype(np.float64)).astype(np.float32)).astype(np.float32)
    assert (np.abs(acc - ref) / scale).max() <= 5e-7
    plain = bf16(A).astype(np.float64) @ bf16(W).T.astype(np.float64)
    assert (np.abs(plain - ref) / scale).max() > 1e-4


def test_tuning_knobs_follow_the_environment_after_reload():
    """Experiment knobs (COGDL_B200_*) are cached by the library; cogdl_b200_reload_tuning() drops the cache so a sweep
    (tools/ab_stream.py) or a test can change them inside one process and restore the defaults afterwards."""
    import os

    from cogdl_b200 import _cabi

    lib = _cabi.load()
    name = b"COGDL_B200_STREAM_BLOCK"
    old = os.environ.pop(name.decode(), None)
    try:
        lib.cogdl_b200_reload_tuning()
        assert lib.cogdl_b200_tuning_value(name, 128) == 128          # unset -> the caller's default
        os.environ[name.decode()] = "64"
        assert lib.cogdl_b200_tuning_value(name, 128) == 64
        os.environ.pop(name.decode())
        lib.cogdl_b200_reload_tuning()
        assert lib.cogdl_b200_tuning_value(name, 128) == 128
        assert lib.cogdl_b200_tuning_value(None, 7) == 7
    finally:
        if old is not None:
            os.environ[name.decode()] = old
        lib.cogdl_b200_reload_tuning()
