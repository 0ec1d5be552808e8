#!/usr/bin/env python
"""Store the outputs of the reference's OWN operators that the tests compare against (tests/refgold.py):
its CPU SpMM and sampler (sample.cpp) and its CUDA kernels, as built by oracle/build_ref.py into
oracle/_ref/ from a checkout of the reference.

  python tests/golden/make_golden_ops.py cpu  [--out DIR]     where oracle/_ref/{asis,o3} is built
  python tests/golden/make_golden_ops.py cuda [--out DIR]     on a B200, where oracle/_ref/cuda is built

Each part replaces its own keys in tests/golden/ops_digests.json and ops_samples.npz and writes the merged
files to DIR (default tests/golden).
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import oracle  # noqa: E402
from tests import refgold  # noqa: E402
from tests.graphs import CASES  # noqa: E402


def cpu_part():
    digests = {}
    for variant in ("asis", "o3"):
        fn = oracle.ref_module("spmm_cpu", variant).csr_spmm_cpu
        for name in CASES:
            if name == "rect":
                continue
            rp, ci, val, X = refgold.spmm_cpu_inputs(name)
            y = fn(torch.from_numpy(rp), torch.from_numpy(ci), torch.from_numpy(val), torch.from_numpy(X)).numpy()
            digests[f"spmm_cpu/{variant}/{name}"] = refgold.digest(y, np.float32)
    smp = oracle.ref_module("sampler", "asis")
    rng = np.random.default_rng(0)
    for n, hi in refgold.SAMPLER_SHAPES:
        t = [torch.from_numpy(a) for a in refgold.sampler_inputs(rng, n, hi)]
        for k, a in enumerate(smp.sample_adj(t[0], t[1], t[2], -1, False)):
            digests[f"sample_adj/{n}/{k}"] = refgold.digest(a.numpy(), np.int64)
        for k, a in enumerate(smp.subgraph(t[0], t[1], t[2])):
            digests[f"subgraph/{n}/{k}"] = refgold.digest(a.numpy(), np.int64)
    return digests, {}


def cuda_part():
    dev = torch.device("cuda:0")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    host = lambda t: t.cpu().numpy()
    digests, samples = {}, {}
    spmm, sddmm = oracle.ref_module("spmm", "cuda"), oracle.ref_module("sddmm", "cuda")
    for F in (128, 40, 16):
        rp, ci, n_cols, val, X, G = refgold.cuda_spmm_inputs(F)
        rows, edges = refgold.sample_positions(rp)
        rpd, cid = T(rp), T(ci)
        samples[f"spmm_F{F}"] = host(spmm.csr_spmm(rpd, cid, T(val), T(X)))[rows]
        samples[f"spmm_no_value_F{F}"] = host(spmm.csr_spmm_no_edge_value(rpd, cid, T(X)))[rows]
        samples[f"sddmm_F{F}"] = host(sddmm.csr_sddmm(rpd, cid, T(G), T(X)))[edges]

    from tests.graphs import case

    rp, ci, n_cols = case("ragged")
    ids = torch.arange(ci.shape[0], device=dev, dtype=torch.float32)     # the reference's fp32-encoded permutation
    colptr, rowind, permf = spmm.csr2csc(T(rp), T(ci), ids)
    for key, a in (("colptr", colptr), ("rowind", rowind), ("perm", permf.int())):
        digests[f"csr2csc/{key}"] = refgold.digest(host(a), np.int32)

    es, mh = oracle.ref_module("edge_softmax", "cuda"), oracle.ref_module("mhspmm", "cuda")
    mhsd, mht = oracle.ref_module("mhsddmm", "cuda"), oracle.ref_module("mhtranspose", "cuda")
    for H, F in ((8, 16), (8, 128), (4, 32)):
        rp, ci, n_cols, e, g, feat, grad, perm = refgold.cuda_gat_inputs(H, F)
        rows, edges = refgold.sample_positions(rp)
        rpd, cid = T(rp), T(ci)
        att = T(oracle.edge_softmax_fwd(rp, e))
        tag = f"H{H}_F{F}"
        samples[f"edge_softmax_{tag}"] = host(es.edge_softmax(rpd, T(e)))[edges]
        samples[f"edge_softmax_bwd_{tag}"] = host(es.edge_softmax_backward(rpd, att, T(g)))[edges]
        samples[f"mhspmm_{tag}"] = host(mh.mhspmm(rpd, cid, att, T(feat)))[rows]
        samples[f"mhsddmm_{tag}"] = host(mhsd.mhsddmm(rpd, cid, T(grad), T(feat)))[edges]
        digests[f"mhtranspose/{tag}"] = refgold.digest(host(mht.mhtranspose(T(perm), T(e))), np.float32)

    rp, ci, n_cols, X = refgold.scatter_max_inputs()
    out, arg = oracle.ref_module("scatter_max", "cuda").scatter_max_fp(T(rp), T(ci), T(X))
    has = np.diff(rp) > 0
    digests["scatter_max/out"] = refgold.digest(host(out)[has], np.float32)
    digests["scatter_max/arg"] = refgold.digest(host(arg)[has], np.int64)
    return digests, samples


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("part", choices=["cpu", "cuda"])
    ap.add_argument("--out", default=HERE)
    a = ap.parse_args()
    digests, samples = cpu_part() if a.part == "cpu" else cuda_part()
    digests = refgold.merged_digests(digests)
    samples = refgold.merged_samples(samples) if samples else {}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, refgold.DIGESTS), "w") as f:
        json.dump(digests, f, indent=1)
        f.write("\n")
    if samples:
        np.savez_compressed(os.path.join(a.out, refgold.SAMPLES), **samples)
    print(f"{len(digests)} digests, {len(samples)} sampled outputs written to {a.out}")


if __name__ == "__main__":
    main()
