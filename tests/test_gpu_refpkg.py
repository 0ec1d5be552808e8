"""The drop-in, executed: the UNMODIFIED reference package's own models on a B200 through
cogdl_b200.install(), against the same models on the reference's CPU path.

  reference `GCN`        cogdl/models/nn/gcn.py:45-77        (GCNLayer -> cogdl.utils.spmm)
  reference `GAT`        cogdl/models/nn/gat.py:54-103       (GATLayer -> edge_softmax + mh_spmm, 8 heads + 1)
  reference `Graphsage`  cogdl/models/nn/graphsage.py:35-119 (SAGELayer aggr="mean" -> spmm after row_norm;
                                                              aggr="max" -> cogdl.operators.scatter_max)

Order matters and is the one INTEGRATION.md prescribes: the CPU run happens BEFORE install() (install
rebinds the dispatch functions inside every imported cogdl module to the sm_100a versions, which refuse
CPU tensors), then install(), then a NEW model with the same state_dict on CUDA.  Logits and every
parameter gradient must agree within 1e-4 (relative to the tensor's scale: cuBLAS fp32 GEMMs sit
upstream of the sparse ops, and the reference's CPU edge-softmax is a different algorithm).
GAT gradients are the exception: the reference's CPU edge-softmax fallback computes its denominator with
the non-differentiable CPU SpMM extension (spmm_utils.py:149-169: `node_sum = spmm(graph, ones)`), so its
CPU backward silently drops the -y*sum(y*g) term -- 70 % off in W, see the assertion below.  The yardstick
for GAT gradients is therefore a plain-torch fp64 restatement of GATLayer (gat_layer.py:59-86) with exact
autograd; the reference CPU run still pins the logits.
aggr="max" has NO CPU implementation in the reference (scatter_max is CUDA-only), so that model is
compared with a plain-torch restatement of SAGELayer's arithmetic using the model's own weights.
"""
import copy

import numpy as np
import pytest
import torch

from tests.refpkg import import_reference, reference_dir

pytestmark = pytest.mark.gpu

TOL = 1e-4


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def gat_exact_grads(state, graph, target, nhead=8, slope=0.2):
    """2-layer reference GAT (gat.py:54-103, GATLayer gat_layer.py:59-86, dropout 0) restated with dense torch
    ops in fp64: logits and exact parameter gradients of the cross-entropy."""
    row, col = graph.edge_index
    n = graph.num_nodes
    p = {k: v.detach().double().clone().requires_grad_(True) for k, v in state.items()}

    def layer(x, W, al, ar, H):
        h = (x @ W).view(n, H, -1)
        hl, hr = (al * h).sum(-1), (ar * h).sum(-1)
        e = torch.nn.functional.leaky_relu(hl[row] + hr[col], slope)
        m = torch.full((n, H), -1e300, dtype=torch.float64).scatter_reduce(0, row[:, None].expand(-1, H), e, "amax")
        ex = torch.exp(e - m[row])
        a = ex / torch.zeros(n, H, dtype=torch.float64).index_add(0, row, ex)[row]
        return torch.zeros_like(h).index_add(0, row, a[:, :, None] * h[col]).view(n, -1)

    x = graph.x.double()
    x = torch.nn.functional.elu(layer(x, p["attentions.0.W"], p["attentions.0.a_l"], p["attentions.0.a_r"], nhead))
    out = layer(x, p["attentions.1.W"], p["attentions.1.a_l"], p["attentions.1.a_r"], 1)
    torch.nn.functional.cross_entropy(out, target).backward()
    return out.detach(), {k: v.grad for k, v in p.items()}


def cora_shaped_graph(Graph, n=2708, e=5278, feats=64, seed=0):
    """Cora-sized symmetric graph (2 708 nodes, 10 556 directed edges) + one planted 600-edge hub so the
    hub plan's chunking is on the path; features are small so 1e-4 is meaningful."""
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, n, (e,), generator=g)
    dst = torch.randint(0, n, (e,), generator=g)
    hub = torch.randint(0, n, (300,), generator=g)
    src = torch.cat([src, torch.full((300,), 7)])
    dst = torch.cat([dst, hub])
    keep = src != dst
    src, dst = src[keep], dst[keep]
    ei = torch.stack([torch.cat([src, dst]), torch.cat([dst, src])])
    ei = torch.unique(ei, dim=1)
    x = torch.randn(n, feats, generator=g)
    graph = Graph(x=x, edge_index=ei)
    graph.add_remaining_self_loops()
    return graph


@pytest.fixture(scope="module")
def ref():
    if reference_dir() is None:
        # the reference's own Python code runs here, and the repository does not carry it: build() installs it
        # into baseline/_ref only where a checkout of the reference is present
        pytest.skip("the reference CogDL package is not installed (baseline/_ref)")
    assert torch.cuda.is_available()
    cogdl = import_reference()
    from cogdl.data import Graph
    from cogdl.models.nn.gcn import GCN
    from cogdl.models.nn.gat import GAT
    from cogdl.models.nn.graphsage import Graphsage

    torch.manual_seed(0)
    runs = {}
    # ---------------- phase 1: reference models on the reference CPU path (before install)
    g_cpu = cora_shaped_graph(Graph)
    n = g_cpu.num_nodes
    target = torch.randint(0, 7, (n,), generator=torch.Generator().manual_seed(1))

    def run(model, graph, fwd):
        model.zero_grad(set_to_none=True)
        out = fwd(model, graph)
        loss = torch.nn.functional.cross_entropy(out, target.to(out.device))
        loss.backward()
        return out.detach(), {k: p.grad.detach().clone() for k, p in model.named_parameters()}

    fwd_full = lambda m, gr: m(gr)
    fwd_sage = lambda m, gr: m(gr.x, [(None, gr, (gr.num_nodes, gr.num_nodes))] * m.num_layers)
    specs = {
        "gcn": (lambda: GCN(64, 16, 7, 2, 0.0), fwd_full),
        "gat": (lambda: GAT(64, 8, 7, 2, 0.0, 0.0, 0.2, 8, False, 1), fwd_full),
        "sage_mean": (lambda: Graphsage(64, 7, [32], 2, [10, 10], 0.0, "mean"), fwd_sage),
    }
    for name, (make, fwd) in specs.items():
        model = make()
        model.train()
        out, grads = run(model, copy.deepcopy(g_cpu), fwd)
        runs[name] = {"state": copy.deepcopy(model.state_dict()), "out": out, "grads": grads, "make": make, "fwd": fwd}
    # GAT: exact gradients (see the module docstring) + the evidence that the reference CPU backward is not exact
    ex_out, ex_grads = gat_exact_grads(runs["gat"]["state"], g_cpu, target)
    assert rel(runs["gat"]["out"], ex_out) <= 1e-5
    assert rel(runs["gat"]["grads"]["attentions.0.W"], ex_grads["attentions.0.W"]) > 0.1, \
        "the reference CPU GAT backward was expected to be inexact (detached softmax denominator)"
    runs["gat"]["grads"] = ex_grads
    # ---------------- phase 2: install the sm_100a backend into the reference package
    import cogdl_b200

    patched = cogdl_b200.install()
    return {"cogdl": cogdl, "Graph": Graph, "graph_cpu": g_cpu, "runs": runs, "run": run, "patched": patched,
            "Graphsage": Graphsage, "target": target}


def test_install_rebinds_the_reference_dispatch(ref):
    import cogdl.layers.gcn_layer as gl
    import cogdl.layers.gat_layer as gal
    import cogdl.utils.spmm_utils as su
    import cogdl_b200

    assert gl.spmm is cogdl_b200.spmm and su.CONFIGS["fast_spmm"] is cogdl_b200.csrspmm
    assert su.CONFIGS["csr_edge_softmax"] is cogdl_b200.csr_edge_softmax and su.CONFIGS["csrmhspmm"] is cogdl_b200.csrmhspmm
    assert any("gat_layer" in p for p in ref["patched"]) or gal.edge_softmax is cogdl_b200.edge_softmax


@pytest.mark.parametrize("name", ["gcn", "gat", "sage_mean"])
def test_reference_model_on_b200_matches_reference_cpu(ref, name):
    import cogdl_b200
    from cogdl_b200 import _cabi

    r = ref["runs"][name]
    dev = torch.device("cuda:0")
    model = r["make"]()
    model.load_state_dict(r["state"])
    model = model.to(dev).train()
    graph = copy.deepcopy(ref["graph_cpu"]).to(dev)
    assert type(graph).__module__.startswith("cogdl.data"), "this must be the reference's own Graph class"
    l0 = _cabi.launch_count()
    out, grads = ref["run"](model, graph, r["fwd"])
    torch.cuda.synchronize()
    assert _cabi.launch_count() - l0 >= 4, "forward + backward must have gone through libcogdl_b200 kernels"
    assert rel(out, r["out"]) <= TOL, f"{name}: logits differ from the reference CPU run"
    for k, gref in r["grads"].items():
        assert rel(grads[k], gref) <= TOL, f"{name}: grad of {k} differs from the reference CPU run"
    # second step on the same graph object: structure cache hit, same numbers (deterministic kernels)
    hits0 = dict(cogdl_b200.structure.cache_stats)
    out2, _ = ref["run"](model, graph, r["fwd"])
    assert torch.equal(out2, out)
    assert cogdl_b200.structure.cache_stats["miss"] == hits0["miss"], "no CSR/plan rebuild on the second step"


def test_reference_graphsage_max_on_b200(ref):
    """aggr='max': reference MaxAggregator -> cogdl.operators.scatter_max.scatter_max (seeded by install)
    with fresh `.int()` tensors per call (sage_layer.py:27) -- the content-matched structure cache path."""
    import cogdl_b200

    dev = torch.device("cuda:0")
    Graphsage = ref["Graphsage"]
    torch.manual_seed(3)
    model = Graphsage(64, 7, [32], 2, [10, 10], 0.0, "max").to(dev).train()
    assert model.convs[0].aggr.scatter_max is cogdl_b200.scatter_max
    graph = copy.deepcopy(ref["graph_cpu"]).to(dev)
    n = graph.num_nodes
    stats0 = dict(cogdl_b200.structure.cache_stats)
    out = model(graph.x, [(None, graph, (n, n))] * 2)
    loss = torch.nn.functional.cross_entropy(out, ref["target"].to(dev))
    loss.backward()
    stats1 = cogdl_b200.structure.cache_stats
    assert stats1["miss"] - stats0["miss"] <= 1, "fresh .int() tensors per call must hit the cache by content"
    assert stats1["content_hit"] - stats0["content_hit"] >= 1
    # plain-torch restatement of SAGELayer (sage_layer.py:69-87) with scatter_max as a segment amax
    rp, ci = graph.row_indptr.cpu(), graph.col_indices.cpu()
    lens = rp[1:] - rp[:-1]

    def seg_max(x):
        return torch.segment_reduce(x[ci], "max", lengths=lens, unsafe=True)

    ms = copy.deepcopy(model).cpu().double()
    x = graph.x.cpu().double().requires_grad_(False)
    h = x
    for i, conv in enumerate(ms.convs):
        h = conv.fc(torch.cat([h, seg_max(h)], dim=-1))
        if i != 1:
            h = torch.relu(h)
    loss_ref = torch.nn.functional.cross_entropy(h, ref["target"])
    loss_ref.backward()
    assert rel(out, h) <= TOL
    for (k, p), (_, q) in zip(model.named_parameters(), ms.named_parameters()):
        assert rel(p.grad, q.grad) <= TOL, k


def test_reference_spmm_captured_before_install_still_hits_the_cache(ref):
    """A module that did `from cogdl.utils import spmm` BEFORE install() keeps the reference function,
    which calls CONFIGS['fast_spmm'](row_indptr.int(), col_indices.int(), ...) with fresh tensors on
    every call (spmm_utils.py:106).  That path must not rebuild the plan per call."""
    import cogdl_b200
    from cogdl_b200.operators import csrspmm

    dev = torch.device("cuda:0")
    graph = copy.deepcopy(ref["graph_cpu"]).to(dev)
    graph.sym_norm()
    x = torch.randn(graph.num_nodes, 32, device=dev)
    outs = []
    s0 = dict(cogdl_b200.structure.cache_stats)
    for _ in range(4):
        outs.append(csrspmm(graph.row_indptr.int(), graph.col_indices.int(), x, graph.raw_edge_weight, graph.is_symmetric()))
    s1 = cogdl_b200.structure.cache_stats
    assert s1["miss"] - s0["miss"] <= 1 and s1["content_hit"] - s0["content_hit"] >= 3
    assert all(torch.equal(o, outs[0]) for o in outs)
    y = cogdl_b200.spmm(graph, x)
    assert torch.equal(y, outs[0])
