#!/usr/bin/env python
"""bench.py -- SpMM aggregated-edges/s and HBM GB/s (hidden=128) on synthetic power-law CSR graphs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-extras]
                  [--beta B] [--scaling weak|strong] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one synthetic graph:
  N = 1 : BASELINE.json configs[1] -- weighted CSR SpMM, hidden=128, on the ogbn-arxiv-shaped
          graph (169 343 nodes, 1 166 243 edges + self loops, sym-normalised weights, seed 0):
          the aggregation step of GCN layer 1 (`spmm(graph, x)`).
  N > 1 : BASELINE.json configs[4] shape -- every rank owns a contiguous node range of a
          papers100M-shaped graph with locality-controlled columns (--beta, default 0.05); remote
          feature rows are gathered over NVLink INSIDE the SpMM kernel (cogdl_b200.dist).
          --scaling weak (default): 1/8 of papers100M per GPU whatever N (13.9 M rows, 202 M edges);
          --scaling strong: the whole papers100M-shaped graph split N ways.
          value = edges of all ranks / max-over-ranks time.

Timing: CUDA events on the launching (torch current) stream around each step, after W >= 3 warm-up
steps; an L2 flush (512 MiB write) runs between timed steps and is excluded from the intervals;
multi-GPU intervals are max-reduced over ranks.  `value` has the inputs resident in HBM; `e2e` is
the same step through the public API with pinned HOST feature buffers: every step copies X from
pinned host memory to the device, runs `cogdl_b200.spmm(graph, x)` and copies Y back to pinned host
memory; the device->host copy of step k runs on a second stream and overlaps the host->device copy
of step k+1 (PCIe is full duplex), K steps are timed as one interval on the device.  The CSR
structure stays resident as it does across CogDL's training steps (cogdl/trainer/trainer.py:32-45).

Parity inside the run (outside every timed region): N = 1 compares the whole output with the CPU
oracle; N > 1 compares >= 4096 sampled output rows per rank (hub rows and rows with remote columns
included) -- rows not split by the hub plan bit-exactly against oracle.spmm_csr on the gathered
inputs, split (hub) rows against an fp64 sum within 1e-5 of the row scale.  A mismatch fails the run.

The `--impl reference` arm times the reference's own CPU SpMM (cogdl/operators/spmm/spmm_cpu.cpp
compiled unmodified into oracle/_ref/, -O3 build) on the same workload: at N = 1 the whole arxiv
graph, at N > 1 a >= 10 M-edge leading row slice of rank 0's shard (edges/s is size-independent).
It never imports cogdl_b200 (synth.py is loaded by file path), so the only native libraries that arm
loads are under oracle/.  Only that arm, the `cpu_baseline` leg and the parity checks touch oracle/.
"""
import argparse
import importlib.util
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_HIDDEN = 128
FLUSH_BYTES = 512 << 20
METRIC = "spmm_aggregated_edges_per_sec"
CPU_SLICE_EDGES = 12_000_000      # reference arm at N > 1: leading row slice of rank 0's shard
PARITY_ROWS = 4096
DUMP_ROWS = 1 << 16               # --dump-outputs: at most 32 MiB of sampled output rows (hidden=128, fp32)


def load_synth():
    """cogdl_b200/synth.py WITHOUT importing the package (whose __init__ dlopens libcogdl_b200.so)."""
    spec = importlib.util.spec_from_file_location("_cogdl_b200_synth", os.path.join(ROOT, "cogdl_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def profiled_traffic(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the N = 1 SpMM kernel, from the newest
    committed `ncu --set full` summary (profiles/*_spmm_traffic.json, written by tools/ncu_traffic.py from
    the .ncu-rep).  Only used when the profiled kernel is the instantiation that actually ran."""
    pdir = os.path.join(ROOT, "profiles")
    best = None
    for fn in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if fn.endswith("_spmm_traffic.json"):
            best = os.path.join(pdir, fn)
    if best is None:
        return None, "no committed ncu traffic summary (profiles/*_spmm_traffic.json)"
    with open(best) as f:
        d = json.load(f)
    # the instantiation is everything up to the closing '>'; a launch-shape suffix (" block=64": same SASS, other
    # threads per block) moves no DRAM bytes and is not part of the match
    inst = kernel_name[: kernel_name.rfind(">") + 1] if ">" in kernel_name else kernel_name
    want = re.sub(r"\s+", "", d.get("launched_as", ""))
    if want and want != re.sub(r"\s+", "", inst):
        return None, f"{os.path.basename(best)} profiles {d.get('launched_as')}, but this run launched {kernel_name}"
    return int(d["dram_bytes_read"] + d["dram_bytes_write"]), os.path.relpath(best, ROOT)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def spmm_bytes(n, nnz, F, weighted=True):
    """Algorithmic bytes of one SpMM launch (SURVEY 8d): gather one F-float row + colind (+ val) per
    edge, write one row + read one rowptr per node; and the compulsory-traffic bound."""
    per_edge_idx = 8 if weighted else 4
    algo = nnz * (4 * F + per_edge_idx) + n * (4 * F + 4)
    minimum = 4 * (n + 1) + per_edge_idx * nnz + 8 * n * F
    return algo, minimum


def shard_sizes_scaled(synth, world, scaling):
    """Per-GPU (rows, edges); COGDL_B200_BENCH_SHARD_DIV (tests only, printed in the workload string
    through the sizes themselves) shrinks the shard so the plumbing can be exercised on small boxes."""
    rows, edges = synth.shard_sizes(world, scaling)
    div = int(os.environ.get("COGDL_B200_BENCH_SHARD_DIV", "1"))
    return max(rows // div, 1000), max(edges // div, 10000)


def arxiv_workload(synth):
    import torch

    n, e = synth.SHAPES["arxiv"]
    rp, col = synth.powerlaw_csr(n, e, seed=0, self_loops=True)
    w = synth.sym_norm_weights(rp, col)
    x = torch.randn(n, F_HIDDEN, generator=torch.Generator().manual_seed(0))
    return rp, col, w, x


# --------------------------------------------------------------------------------------------- CPU legs
def cpu_thread_sweep(call, set_threads, host_threads, reps=5):
    """Median-of-`reps` time per candidate OpenMP thread count (one untimed warm-up each).  The
    reference loop's `schedule(dynamic)` stops scaling well before all cores on a 128-core host, so
    "all the host threads it can use" = the fastest count, stated in `cores`."""
    cands = sorted({t for t in (host_threads, host_threads // 2, host_threads // 4, 32, 16, 8) if 1 <= t <= host_threads},
                   reverse=True)
    res = {}
    for t in cands:
        set_threads(t)
        call()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        res[t] = statistics.median(ts)
    best = min(res, key=res.get)
    set_threads(best)
    return best, res


def reference_cpu_spmm(rp32, col32, w, x, variant="o3"):
    """(callable, kind): the reference's spmm_cpu.cpp compiled unmodified (oracle/_ref) or the C port."""
    import oracle

    if oracle.ref_available("spmm_cpu", variant):
        fn = oracle.ref_module("spmm_cpu", variant).csr_spmm_cpu
        if w is None:
            import torch
            w = torch.ones(col32.numel(), dtype=torch.float32)     # the reference CPU op always takes values
        return (lambda: fn(rp32, col32, w, x)), "reference"
    a = (rp32.numpy(), col32.numpy(), None if w is None else w.numpy(), x.numpy())
    return (lambda: oracle.spmm_csr(*a)), "port"


def shard_slice_cpu(synth, world, beta, scaling, seed=0):
    """Rank 0's shard, leading rows holding >= CPU_SLICE_EDGES edges, as a CPU problem: local columns
    keep their ids, remote columns are renumbered into a halo block appended to X."""
    import torch

    rows, edges = shard_sizes_scaled(synth, world, scaling)
    rp, col = synth.shard_csr(0, world, rows, edges, beta, seed=seed, device="cpu", max_slice_edges=CPU_SLICE_EDGES)
    remote = col >= rows                      # rank 0 owns [0, rows)
    halo = torch.unique(col[remote])
    col = col.clone()
    col[remote] = rows + torch.searchsorted(halo, col[remote])
    x = torch.empty(rows + int(halo.numel()), F_HIDDEN)
    g = torch.Generator().manual_seed(seed)
    step = 1 << 20
    for s in range(0, x.shape[0], step):      # chunked: keeps the temporary small
        x[s:s + step].normal_(generator=g)
    return rp, col, x, rows, edges


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    import torch
    import oracle

    synth = load_synth()
    host = os.cpu_count() or 1
    torch.set_num_threads(host)
    if world <= 1 and args.gpus <= 1:
        rp, col, w, x = arxiv_workload(synth)
        workload = synth.arxiv_description(int((rp[1:] - rp[:-1]).max()))
        sample = "the full workload, every step (one SpMM over the whole graph)"
        weighted = True
    else:
        n_gpus = max(world, args.gpus)
        rp, col, x, rows, edges = shard_slice_cpu(synth, n_gpus, args.beta, args.scaling)
        w = None
        workload = synth.shard_description(rows, edges, n_gpus, args.beta, 0, F_HIDDEN, args.scaling)
        sample = (f"leading {rp.numel() - 1} rows / {int(rp[-1])} edges of rank 0's shard (same generator and parameters; "
                  f"remote columns read from an appended halo block), every step; edges/s is reported as measured on the slice")
        weighted = False
    rp32, col32 = rp.int(), col.int()
    nnz, n = int(col.numel()), int(rp.numel() - 1)
    call, kind = reference_cpu_spmm(rp32, col32, w, x)
    best_t, sweep = cpu_thread_sweep(call, oracle.set_num_threads, host)
    for _ in range(max(args.warmup, 1)):
        call()
    ts = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        call()
        ts.append(time.perf_counter() - t0)
    t = sum(ts) / len(ts)
    val = nnz / t
    algo, _ = spmm_bytes(n, nnz, F_HIDDEN, weighted)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "edges/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "hidden": F_HIDDEN,
                   "kernel": "reference cogdl/operators/spmm/spmm_cpu.cpp (unmodified, -O3 -fopenmp) via oracle/_ref"
                             if kind == "reference" else "oracle port (oracle/oracle.c)"},
        "algorithmic_GBps": algo / t / 1e9,
        "cpu_baseline": {"value": val, "unit": "edges/s", "cores": best_t, "host_cores": host, "kind": kind,
                         "sample": sample, "threads_sweep_edges_per_s": {str(k): nnz / v for k, v in sweep.items()},
                         "thread_choice": "fastest median of 5 per OpenMP thread count"},
        "e2e": {"value": val, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def cpu_baseline_leg(rp, col, w, x, nnz):
    """Reference CPU SpMM on this box's host cores (rank 0, N = 1 only): same sweep as the reference arm."""
    import oracle

    host = os.cpu_count() or 1
    rp32, col32 = rp.int(), col.int()
    out = {"unit": "edges/s", "host_cores": host}
    call, kind = reference_cpu_spmm(rp32, col32, w, x, "o3")
    best_t, sweep = cpu_thread_sweep(call, oracle.set_num_threads, host)
    out.update({"value": nnz / sweep[best_t], "cores": best_t, "kind": kind,
                "value_all_cores": nnz / sweep[max(sweep)],
                "threads_sweep": {str(t): nnz / v for t, v in sweep.items()},
                "sample": f"full workload (one SpMM over the whole graph) per run, median of 5 runs at the best OpenMP thread "
                          f"count ({best_t} of {host} host cores); reference spmm_cpu.cpp built -O3"
                          if kind == "reference" else "full workload, median of 5, oracle.c"})
    if oracle.ref_available("spmm_cpu", "asis"):
        call2, _ = reference_cpu_spmm(rp32, col32, w, x, "asis")
        oracle.set_num_threads(best_t)
        call2()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            call2()
            ts.append(time.perf_counter() - t0)
        out["as_shipped_value"] = nnz / statistics.median(ts)
    oracle.set_num_threads(host)
    return out


# --------------------------------------------------------------------------------------------- our arm
def time_steps(fn, steps, warmup, flush, torch, dist_on, keep_last=False):
    """Per-step CUDA-event intervals (ms), L2 flushed between steps; max over ranks per step.
    keep_last: also return what the last timed step computed, as (ms, output)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist_on:
        import torch.distributed as dist
        dist.barrier()
    evs = []
    last = None
    for i in range(steps):
        if flush is not None:
            flush.zero_()       # evicts X / Y from the 126 MB L2; outside the timed interval
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        if keep_last and i == steps - 1:
            last = fn()
        else:
            fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    if dist_on:
        import torch.distributed as dist
        dist.barrier()
    ms = torch.tensor([a.elapsed_time(b) for a, b in evs], dtype=torch.float64, device="cuda")
    if dist_on:
        import torch.distributed as dist
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return (ms.cpu().tolist(), last) if keep_last else ms.cpu().tolist()


def time_e2e(torch, dev, x_pin, x_in, run, n_rows, steps, warmup, dist_on, before_h2d=None):
    """End to end through the public API: every step = H2D of X from pinned host memory, run(x_in) ->
    Y, D2H of Y into pinned host memory (double-buffered, on a second stream so that it overlaps the
    next step's H2D).  K steps are one CUDA-event interval on the compute stream, closed only after
    the last D2H has finished; returns (mean ms per step, max over ranks)."""
    s_out = torch.cuda.Stream(dev)
    y_pins = [torch.empty((n_rows, F_HIDDEN), dtype=torch.float32, pin_memory=True) for _ in range(2)]

    def step(i):
        cur = torch.cuda.current_stream(dev)
        if before_h2d is not None:
            before_h2d()                      # N > 1: peers are done reading the shard we overwrite
        x_in.copy_(x_pin, non_blocking=True)
        y = run(x_in)
        ev = torch.cuda.Event()
        ev.record(cur)
        s_out.wait_event(ev)
        with torch.cuda.stream(s_out):
            y_pins[i & 1].copy_(y, non_blocking=True)
        y.record_stream(s_out)

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    if dist_on:
        import torch.distributed as dist
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        step(i)
    done = torch.cuda.Event()
    done.record(s_out)
    torch.cuda.current_stream(dev).wait_event(done)
    b.record()
    torch.cuda.synchronize()
    if dist_on:
        import torch.distributed as dist
        dist.barrier()
    ms = torch.tensor([a.elapsed_time(b) / steps], dtype=torch.float64, device=dev)
    if dist_on:
        import torch.distributed as dist
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms)


def bind_to_gpu_numa(torch, local):
    """Pin this rank's host threads (and so the first-touch placement of its pinned buffers) to the NUMA
    node its GPU hangs off: 8 ranks x 14 GB of pinned traffic per step otherwise cross the socket link."""
    try:
        p = torch.cuda.get_device_properties(local)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA affinity reported for " + bdf}
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus), "pci": bdf}
    except Exception as ex:  # noqa: BLE001
        return {"numa_node": None, "note": f"{type(ex).__name__}: {ex}"}


def dump_output(out_dir, name, y, max_rows):
    """--dump-outputs: `y` (rows x F) as out_dir/<name>.npy in float32.  Above `max_rows` rows, a fixed seeded
    sample of rows in ascending order, with their indices as out_dir/<name>_rows.npy (float64)."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    if y.shape[0] > max_rows:
        rows = torch.randperm(y.shape[0], generator=torch.Generator().manual_seed(0))[:max_rows].sort().values
        np.save(os.path.join(out_dir, name + "_rows.npy"), rows.double().numpy())
        y = y[rows.to(y.device)]
    np.save(os.path.join(out_dir, name + ".npy"), y.float().cpu().numpy())


def elementwise_err(got, ref):
    """max over elements of |a-b| / max(|b|, row scale), row scale = max |b| of the row (numpy)."""
    import numpy as np

    scale = np.maximum(np.abs(ref), np.abs(ref).max(axis=1, keepdims=True))
    scale = np.maximum(scale, 1e-30)
    return float((np.abs(got.astype(np.float64) - ref.astype(np.float64)) / scale).max()) if ref.size else 0.0


def parity_single(torch, rp, col, w, x_host, y_dev, chunk_edges):
    import numpy as np
    import oracle

    ref = oracle.spmm_csr(rp.numpy(), col.numpy(), w.numpy(), x_host.numpy())
    got = y_dev.cpu().numpy()
    deg = np.diff(rp.numpy())
    unsplit = deg <= chunk_edges
    exact = bool(np.array_equal(got[unsplit], ref[unsplit]))
    err = elementwise_err(got, ref)
    return {"rows": int(ref.shape[0]), "rows_unsplit": int(unsplit.sum()), "rows_split": int((~unsplit).sum()),
            "max_rel": err, "bit_exact_unsplit": exact, "tol": 1e-5, "ok": bool(exact and err <= 1e-5),
            "against": "oracle.spmm_csr (pinned bit-exact to the reference spmm_cpu.cpp) on the whole output"}


def parity_dist(torch, part, y, dev):
    """>= PARITY_ROWS sampled output rows of this rank against the oracle on the GATHERED inputs."""
    import numpy as np
    import torch.distributed as dist
    import oracle

    st = part.st
    n_local, F = part.n_local, y.shape[1]
    rp, colind = st.rowptr, st.colind
    deg = rp[1:] - rp[:-1]
    g = torch.Generator(device=dev).manual_seed(1234 + part.part.rank)
    plan = st.plan
    picks = [torch.randint(0, n_local, (PARITY_ROWS,), generator=g, device=dev)]
    if plan.n_hub_rows > 0:       # hub list is sorted by descending degree: the 2 heaviest + a spread of 30
        hubs = plan.hub_rows[: plan.n_hub_rows].long()
        idx = torch.unique(torch.cat([torch.arange(min(2, hubs.numel()), device=dev),
                                      torch.linspace(0, hubs.numel() - 1, 30, device=dev).long()]))
        picks.append(hubs[idx])
    pos = torch.randint(0, st.nnz, (1 << 20,), generator=g, device=dev)          # rows that own remote columns
    pos = pos[colind[pos] >= n_local][:1024]
    if pos.numel() and plan.edge_row is not None:
        picks.append(plan.edge_row[pos].long())
    rows = torch.unique(torch.cat(picks))
    lens = deg[rows].long()
    sub_rp = torch.zeros(rows.numel() + 1, dtype=torch.int64, device=dev)
    torch.cumsum(lens, 0, out=sub_rp[1:])
    total = int(sub_rp[-1])
    epos = torch.repeat_interleave(rp[rows].long() - sub_rp[:-1], lens) + torch.arange(total, device=dev)
    c = colind[epos].long()
    # decode to (owner, row inside the owner's shard)
    rank = part.part.rank
    if part.mode == "p2p":
        shift = part.part.peer_shift
        r = c - n_local
        owner = torch.where(c < n_local, torch.full_like(c, rank), r >> shift)
        orow = torch.where(c < n_local, c, r & ((1 << shift) - 1))
    else:
        bt = torch.tensor(part.part.bounds, device=dev, dtype=torch.int64)
        gid = torch.where(c < n_local, c + part.part.lo, part.part.halo.to(dev)[(c - n_local).clamp_(min=0)])
        owner = torch.searchsorted(bt, gid, right=True) - 1
        orow = gid - bt[owner]
    key = owner * (1 << 40) + orow
    ukey, inv = torch.unique(key, return_inverse=True)
    uowner, urow = ukey >> 40, ukey & ((1 << 40) - 1)
    xs = torch.empty((ukey.numel(), F), dtype=torch.float32, device=dev)
    remote_rows = int((uowner != rank).sum())
    if part.mode == "p2p":
        buf, hdl, _ = part._symm
        hdl.barrier(channel=2)
        for o in range(part.world):
            m = (uowner == o).nonzero().view(-1)
            if m.numel():
                peer = buf if o == rank else hdl.get_buffer(o, tuple(buf.shape), torch.float32)
                xs[m] = peer[urow[m]]
        torch.cuda.synchronize()
        hdl.barrier(channel=2)
    else:   # halo form: the halo rows come from the product's own exchange -- local rows are checked fully
        halo = part.exchange_rows(part.pack(part.x_local), F)
        loc = uowner == rank
        xs[loc] = part.x_local[urow[loc]]
        gid = urow + torch.tensor(part.part.bounds, device=dev)[uowner]
        xs[~loc] = halo[torch.searchsorted(part.part.halo.to(dev), gid[~loc])]
    got = y[rows].cpu().numpy()
    unsplit = (lens <= st.chunk_edges).cpu().numpy()
    ref32 = oracle.spmm_csr(sub_rp.to(torch.int32).cpu().numpy(), inv.to(torch.int32).cpu().numpy(), None, xs.cpu().numpy())
    exact = bool(np.array_equal(got[unsplit], ref32[unsplit]))
    # split (hub) rows: a 1.5 M-edge fp32 sequential sum is itself ~1e-5 off, so the yardstick is an fp64 sum
    err = elementwise_err(got[unsplit], ref32[unsplit]) if unsplit.any() else 0.0
    n_split = int((~unsplit).sum())
    if n_split:
        srows = (~torch.from_numpy(unsplit)).nonzero().view(-1).to(dev)
        ref64 = torch.zeros((n_split, F), dtype=torch.float64, device=dev)
        for k, j in enumerate(srows.tolist()):
            a, b = int(sub_rp[j]), int(sub_rp[j + 1])
            for s in range(a, b, 1 << 20):
                ref64[k] += xs[inv[s:min(b, s + (1 << 20))]].double().sum(0)
        err = max(err, elementwise_err(got[~unsplit], ref64.cpu().numpy()))
    ok = exact and err <= 1e-5
    stats = torch.tensor([rows.numel(), int(unsplit.sum()), n_split, remote_rows, total], dtype=torch.float64, device=dev)
    flags = torch.tensor([float(ok), float(exact), -err], dtype=torch.float64, device=dev)
    dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    return {"rows": int(stats[0]), "rows_unsplit": int(stats[1]), "rows_split": int(stats[2]),
            "distinct_remote_feature_rows_read": int(stats[3]), "edges_checked": int(stats[4]),
            "max_rel": float(-flags[2]), "bit_exact_unsplit": bool(flags[1] > 0.5), "tol": 1e-5, "ok": bool(flags[0] > 0.5),
            "against": "oracle.spmm_csr on the gathered inputs (unsplit rows, bit-exact) / fp64 sum (hub rows, 1e-5 of row scale); "
                       "all ranks, sums / worst over ranks"}


def backward_and_piece_extras(torch, flush, bench, res, g, st, n, nnz, dev):
    """The backward kernels and GAT pieces that had no number in round 1 (arxiv shape)."""
    from cogdl_b200.operators._raw import (edge_softmax_fwd_raw, edge_softmax_bwd_raw, mhspmm_raw, mhsddmm_raw,
                                           spmm_raw, gather_rows_raw, scatter_max_fwd_raw, scatter_max_bwd_raw)

    H, F = 8, 128
    logits = (torch.randn(nnz, H, device=dev) * 3).clamp_(-10, 10)
    att = edge_softmax_fwd_raw(st, logits)
    gatt = torch.randn(nnz, H, device=dev)
    bench("C3_edge_softmax_bwd_H8", lambda: edge_softmax_bwd_raw(st, att, gatt), 3 * 4 * nnz * H + 4 * (n + 1), nnz)
    h = torch.randn(n, H, F, device=dev)
    gout = torch.randn(n, H, F, device=dev)
    bench("C3_mhsddmm_H8_F128", lambda: mhsddmm_raw(st, gout, h), nnz * (4 * H * F + 4 + 4 * H) + n * (4 * H * F + 4), nnz)
    st_t, perm = st.csc()
    st_t.plan
    mh_bytes = nnz * (4 * H * F + 4 + 4 * H + 4) + n * (4 * H * F + 4)
    bench("C3_mhspmm_csc_perm_H8_F128", lambda: mhspmm_raw(st_t, att, gout, perm=perm), mh_bytes, nnz)
    del h, gout, att, gatt, logits
    w = g.raw_edge_weight
    x128 = torch.randn(n, 128, device=dev)
    w_t = gather_rows_raw(perm, w)
    bench("C2_spmm_transpose_F128", lambda: spmm_raw(st_t, w_t, x128), nnz * (4 * 128 + 8) + n * (4 * 128 + 4), nnz)
    xs = torch.rand(n, 128, device=dev) + 0.01
    _, arg = scatter_max_fwd_raw(st, xs)
    gs = torch.randn(n, 128, device=dev)
    bench("C4op_scatter_max_bwd_F128_arxiv", lambda: scatter_max_bwd_raw(gs, arg, n), n * 128 * (4 + 4 + 4 + 4), nnz)


def extras(torch, flush, synth, steps=10):
    """Informational numbers for the other configs (not the headline): C2 layer-2 width, C3 GAT
    pieces on the arxiv shape (H=8, F=128), C4 scatter_max on a products-shaped graph, the backward
    kernels, and the 1-GPU anchor of the multi-GPU weak-scaling shard."""
    import cogdl_b200
    from cogdl_b200.operators._raw import (edge_softmax_fwd_raw, mhspmm_raw, scatter_max_fwd_raw, spmm_raw,
                                           gat_fwd_raw, sddmm_raw)

    peak, _ = measured_peaks()
    dev = torch.device("cuda")
    res = {}
    t_start = time.perf_counter()

    def bench(name, fn, algo_bytes, units):
        try:
            ms = time_steps(fn, steps, 3, flush, torch, False)
            t = statistics.median(ms) / 1e3
            res[name] = {"ms": t * 1e3, "edges_per_s": units / t, "algorithmic_GBps": algo_bytes / t / 1e9,
                         "frac_of_hbm_peak": algo_bytes / t / 1e9 / peak}
        except Exception as ex:  # noqa: BLE001  (secondary numbers must not take the headline down)
            res[name] = {"error": f"{type(ex).__name__}: {ex}"}

    n, e = synth.SHAPES["arxiv"]
    rp, col = synth.powerlaw_csr(n, e, seed=0)
    g = cogdl_b200.Graph(row_ptr=rp, col=col, edge_weight=synth.sym_norm_weights(rp, col), num_nodes=n).to(dev)
    st = g.structure()
    nnz = st.nnz
    w = g.raw_edge_weight
    x40 = torch.randn(n, 40, device=dev)
    bench("C2_spmm_F40", lambda: spmm_raw(st, w, x40), nnz * (4 * 40 + 8) + n * (4 * 40 + 4), nnz)
    x128 = torch.randn(n, 128, device=dev)
    bench("C2_sddmm_F128", lambda: sddmm_raw(st, x128, x128), nnz * (2 * 4 * 128 + 8) + 4 * (n + 1), nnz)
    H, F = 8, 128
    logits = (torch.randn(nnz, H, device=dev) * 3).clamp_(-10, 10)
    bench("C3_edge_softmax_H8", lambda: edge_softmax_fwd_raw(st, logits), 2 * 4 * nnz * H + 4 * (n + 1), nnz)
    att = edge_softmax_fwd_raw(st, logits)
    h = torch.randn(n, H, F, device=dev)
    mh_bytes = nnz * (4 * H * F + 4 + 4 * H) + n * (4 * H * F + 4)
    bench("C3_mhspmm_H8_F128", lambda: mhspmm_raw(st, att, h), mh_bytes, nnz)
    hl, hr = torch.randn(n, H, device=dev), torch.randn(n, H, device=dev)
    bench("C3_fused_gat_H8_F128", lambda: gat_fwd_raw(st, hl, hr, h, 0.2, False), mh_bytes, nnz)
    del h, att, logits, hl, hr
    try:
        backward_and_piece_extras(torch, flush, bench, res, g, st, n, nnz, dev)
    except Exception as ex:  # noqa: BLE001
        res["backward_extras_error"] = f"{type(ex).__name__}: {ex}"
    try:   # fused (A.X).W^T + (A.1) b^T + ReLU with tcgen05 vs SpMM + cuBLAS (SURVEY 8f-3), one 128 -> 128 GCN layer
        from cogdl_b200.operators.fused_gcn import fused_gcn_raw

        lin = torch.nn.Linear(128, 128).to(dev)
        W, b = lin.weight.detach().contiguous(), lin.bias.detach().contiguous()
        layer_bytes = nnz * (4 * 128 + 8) + n * (4 * 128 + 4)
        tf32_was = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False      # the 1e-5 bar rules TF32 out for the unfused comparison
        bench("C2_gcn_layer_fused_tcgen05", lambda: fused_gcn_raw(st, w, x128, W, b, True), layer_bytes, nnz)
        bench("C2_gcn_layer_unfused_fp32_reference_order", lambda: torch.relu_(spmm_raw(st, w, torch.addmm(b, x128, W.t()))),
              layer_bytes, nnz)
        bench("C2_gcn_layer_unfused_fp32_spmm_then_gemm", lambda: torch.relu_(spmm_raw(st, w, x128) @ W.t()), layer_bytes, nnz)
        torch.backends.cuda.matmul.allow_tf32 = True
        bench("C2_gcn_layer_unfused_tf32_reference_order", lambda: torch.relu_(spmm_raw(st, w, torch.addmm(b, x128, W.t()))),
              layer_bytes, nnz)
        torch.backends.cuda.matmul.allow_tf32 = tf32_was
        a = fused_gcn_raw(st, w, x128, W, b, True).double()
        r = torch.relu(torch.sparse_csr_tensor(st.rowptr.long(), st.colind.long(), w.double(), size=(st.n_rows, st.n_cols))
                       @ (x128.double() @ W.double().t() + b.double()))
        scale = torch.maximum(r.abs(), r.abs().amax(dim=1, keepdim=True)).clamp_min(1e-30)
        res["C2_gcn_layer_fused_tcgen05"]["max_rel_err_vs_fp64_reference_order"] = float(((a - r).abs() / scale).max())
        res["C2_gcn_layer_fused_tcgen05"]["kernel"] = cogdl_b200._cabi.last_kernel()
        del a, r, scale, lin
    except Exception as ex:  # noqa: BLE001
        res["fused_gcn_error"] = f"{type(ex).__name__}: {ex}"
    try:   # device neighbour sampler vs the reference's host loop (sample.cpp compiled unmodified), SURVEY 8f-4
        import oracle
        from cogdl_b200 import sampling

        rp64, col64 = g.row_indptr.contiguous(), g.col_indices.contiguous()
        batch = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:4096].to(dev)
        for size, tag in ((10, "k10"), (-1, "full")):
            fn = lambda: sampling.sample_adj(rp64, col64, batch, size, False, seed=1)
            ms = time_steps(fn, steps, 3, None, torch, False)
            t = statistics.median(ms) / 1e3
            out = fn()
            ent = {"ms": t * 1e3, "sampled_edges": int(out[3].numel()), "sampled_edges_per_s": int(out[3].numel()) / t,
                   "what": f"sample_adj: 4096 seed nodes, {'all' if size < 0 else size} neighbours, arxiv shape"}
            if oracle.ref_available("sampler", "o3"):
                smp = oracle.ref_module("sampler", "o3")
                a3 = (rp64.cpu(), col64.cpu(), batch.cpu())
                smp.sample_adj(*a3, size, False)
                ts = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    smp.sample_adj(*a3, size, False)
                    ts.append(time.perf_counter() - t0)
                ent["reference_cpu_ms"] = statistics.median(ts) * 1e3
                ent["speedup_vs_reference_cpu"] = ent["reference_cpu_ms"] / ent["ms"]
            res["C4op_sample_adj_" + tag] = ent
    except Exception as ex:  # noqa: BLE001
        res["sampler_error"] = f"{type(ex).__name__}: {ex}"

    # ---- secondary: whole training steps of the three config models on the arxiv shape (cuBLAS GEMMs +
    # our sparse kernels + autograd: forward, backward, SGD), informational
    def train_step_ms(model, graph, out_dim, reps=5):
        import torch.nn.functional as Fn

        opt = torch.optim.SGD(model.parameters(), lr=0.01)
        y = torch.randint(0, out_dim, (n,), device=dev)
        ts = []
        for i in range(reps + 2):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            opt.zero_grad(set_to_none=True)
            loss = Fn.cross_entropy(model(graph), y)
            loss.backward()
            opt.step()
            b.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(a.elapsed_time(b))
        return statistics.median(ts)

    try:
        from cogdl_b200.layers import GCN, GAT, SAGE

        g.x = torch.randn(n, 128, device=dev)
        res["C2_gcn2_train_step"] = {"ms": train_step_ms(GCN(128, 128, 40, dropout=0.0).to(dev), g, 40),
                                     "what": "2-layer GCN hidden=128, fwd+bwd+SGD, arxiv shape"}
        g2 = cogdl_b200.Graph(x=g.x, row_ptr=rp, col=col, num_nodes=n).to(dev)
        res["C3_gat2_train_step"] = {"ms": train_step_ms(GAT(128, 16, 40, nhead=8, last_nhead=1).to(dev), g2, 40),
                                     "what": "2-layer GAT 8 heads x 16, fwd+bwd+SGD, arxiv shape"}
        res["C4_sage_max2_train_step"] = {"ms": train_step_ms(SAGE(128, 128, 40, aggr="max").to(dev), g2, 40),
                                          "what": "2-layer GraphSAGE aggr=max hidden=128, fwd+bwd+SGD, arxiv shape"}
        del g2
    except Exception as ex:  # noqa: BLE001
        res["train_steps_error"] = f"{type(ex).__name__}: {ex}"
    del x128, x40, g, st
    torch.cuda.empty_cache()
    try:
        n, e = synth.SHAPES["products"]
        rp, col = synth.powerlaw_csr(n, e, seed=0, device=dev, self_loops=False)
        st = cogdl_b200.CSRStructure.from_int64(rp, col, n_cols=n)
        del rp, col
        x = torch.rand(n, 256, device=dev) + 0.01
        bench("C4_scatter_max_F256", lambda: scatter_max_fwd_raw(st, x), e * (4 * 256 + 4) + n * (8 * 256 + 4), e)
        x = x[:, :128].contiguous()
        bench("C4shape_spmm_F128_unweighted", lambda: spmm_raw(st, None, x), e * (4 * 128 + 4) + n * (4 * 128 + 4), e)
        del st, x
        torch.cuda.empty_cache()
    except Exception as ex:  # noqa: BLE001
        res["products_error"] = f"{type(ex).__name__}: {ex}"
    try:    # the 1-GPU anchor of the weak-scaling curve: the same per-GPU shard, every column local (beta = 0)
        rows, edges = synth.shard_sizes(8, "weak")
        rp, col = synth.shard_csr(0, 1, rows, edges, 0.0, seed=0, device=dev)
        st = cogdl_b200.CSRStructure.from_int64(rp, col, n_cols=rows)
        del rp, col
        st.plan
        x = torch.randn(rows, F_HIDDEN, device=dev)
        algo, _ = spmm_bytes(rows, edges, F_HIDDEN, weighted=False)
        bench("C5_shard_1gpu", lambda: spmm_raw(st, None, x), algo, edges)
        res["C5_shard_1gpu"]["what"] = ("one GPU, the multi-GPU weak-scaling shard (13.9 M rows, 202 M edges, hidden=128, "
                                        "unweighted) with every column local (beta = 0): like-for-like anchor for N >= 2")
        del st, x
    except Exception as ex:  # noqa: BLE001
        res["C5_shard_1gpu_error"] = f"{type(ex).__name__}: {ex}"
    res["extras_seconds"] = time.perf_counter() - t_start
    return res


def run_ours(args):
    import torch

    t_begin = time.perf_counter()
    phases = {}
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist_on = world > 1
    numa = bind_to_gpu_numa(torch, local) if dist_on else None
    if dist_on:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"     # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=dev)
    import cogdl_b200
    from cogdl_b200 import _cabi, synth

    _cabi.check(_cabi.load().cogdl_b200_check_device())
    peak, peak_src = measured_peaks()
    flush = torch.empty(FLUSH_BYTES, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(local)
    extra_keys = {}

    if not dist_on:
        rp, col, w, x_host = arxiv_workload(synth)
        n, nnz = int(rp.numel() - 1), int(col.numel())
        g = cogdl_b200.Graph(row_ptr=rp, col=col, edge_weight=w, num_nodes=n).to(dev)
        st = g.structure()
        st.plan  # build once (cached on the graph), outside the timed region
        x_dev = x_host.to(dev)
        workload = synth.arxiv_description(int((rp[1:] - rp[:-1]).max()))
        step = lambda: cogdl_b200.spmm(g, x_dev)
        phases["setup_s"] = time.perf_counter() - t_begin
        # ---- device-resident
        l0 = _cabi.launch_count()
        sampler.start()
        ms, y_last = time_steps(step, args.steps, args.warmup, flush, torch, False, keep_last=True)
        launches_dev = _cabi.launch_count() - l0
        kernel_name = _cabi.last_kernel()
        if args.dump_outputs:
            dump_output(args.dump_outputs, "spmm_out", y_last, DUMP_ROWS)
        del y_last
        # ---- parity of what was just timed, against the oracle (outside the timed regions)
        parity = parity_single(torch, rp, col, w, x_host, step(), st.chunk_edges)
        # ---- end to end: pinned host X -> device, spmm through the public API, Y -> pinned host
        x_pin = x_host.pin_memory()
        x_in = torch.empty_like(x_dev)
        l1 = _cabi.launch_count()
        e2e_steps = args.steps
        ms_e2e = time_e2e(torch, dev, x_pin, x_in, lambda xi: cogdl_b200.spmm(g, xi), n, e2e_steps, args.warmup, False)
        clocks = sampler.stop()      # sampled across both timed regions
        launches = launches_dev + (_cabi.launch_count() - l1)
        total_units = nnz
        algo, bmin = spmm_bytes(n, nnz, F_HIDDEN)
        parallelism = "single GPU"
        h2d = d2h = n * F_HIDDEN * 4
        e2e_l2 = "X is rewritten from pinned host memory by the H2D DMA every step (no L2 flush inside the e2e interval)"
    else:
        from cogdl_b200 import dist as cdist

        rows, edges = shard_sizes_scaled(synth, world, args.scaling)
        part = cdist.synthetic_partition(rank, world, dev, seed=0, rows=rows, edges=edges,
                                         mode=os.environ.get("COGDL_B200_DIST_MODE"), beta=args.beta, scaling=args.scaling)
        workload = part.describe()
        x_dev = part.x_local                       # p2p mode: already inside the symmetric shard
        step = lambda: part.spmm(x_dev)
        phases["setup_s"] = time.perf_counter() - t_begin
        l0 = _cabi.launch_count()
        sampler.start()
        ms, y_last = time_steps(step, args.steps, args.warmup, flush, torch, True, keep_last=True)
        clocks = sampler.stop()
        launches_dev = _cabi.launch_count() - l0
        kernel_name = _cabi.last_kernel()
        if args.dump_outputs:     # this rank's rows of the output
            dump_output(args.dump_outputs, f"spmm_out_rank{rank}", y_last, DUMP_ROWS // world)
        del y_last
        t0 = time.perf_counter()
        parity = parity_dist(torch, part, step(), dev)
        phases["parity_s"] = time.perf_counter() - t0
        # ---- like-for-like 1-GPU anchor measured in the same job: this rank's shard with every column local
        t0 = time.perf_counter()
        try:
            from cogdl_b200.operators._raw import spmm_raw

            rp_a, col_a = synth.shard_csr(rank, world, rows, edges, 0.0, seed=0, device=dev)
            st_a = cogdl_b200.CSRStructure.from_int64(rp_a, col_a - rank * rows, n_cols=rows)
            del rp_a, col_a
            st_a.plan
            xa = part.x_local
            ms_a = time_steps(lambda: spmm_raw(st_a, None, xa), max(3, args.steps // 2), 3, flush, torch, True)
            ta = sum(ms_a) / len(ms_a) / 1e3
            extra_keys["anchor_local_only"] = {
                "what": "same shard shape with every column local (beta = 0), no peer traffic, no barrier: the "
                        "single-GPU anchor of this curve, all ranks at once (max over ranks)",
                "ms_per_step": ta * 1e3, "edges_per_s_all_ranks": part.global_nnz / ta,
                "efficiency_vs_anchor": (sum(ms_a) / len(ms_a)) / (sum(ms) / len(ms))}
            del st_a
            torch.cuda.empty_cache()
        except Exception as ex:  # noqa: BLE001
            extra_keys["anchor_local_only"] = {"error": f"{type(ex).__name__}: {ex}"}
        phases["anchor_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        x_pin = torch.empty(tuple(x_dev.shape), dtype=torch.float32, pin_memory=True)
        x_pin.copy_(x_dev)
        x_in = x_dev if part.mode == "p2p" else torch.empty_like(x_dev)   # H2D lands in the shard itself
        l1 = _cabi.launch_count()
        e2e_steps = max(3, args.steps // 4)
        ms_e2e = time_e2e(torch, dev, x_pin, x_in, lambda xi: part.spmm(xi), part.n_local, e2e_steps, 2, True,
                          before_h2d=part.release if part.mode == "p2p" else None)
        phases["e2e_s"] = time.perf_counter() - t0
        launches = launches_dev + (_cabi.launch_count() - l1)
        total_units = part.global_nnz
        n, nnz = part.n_local, part.nnz_local
        algo, bmin = spmm_bytes(n, nnz, F_HIDDEN, weighted=False)  # per rank, per launch
        parallelism = f"node-range partition x{world}; {part.exchange}; no reduce on the data path"
        h2d = d2h = part.n_local * F_HIDDEN * 4
        e2e_l2 = "X (7.1 GB per rank at weak scaling) is rewritten from pinned host memory every step and exceeds the L2"
        extra_keys["numa"] = numa
        extra_keys["remote_fraction"] = {"beta": args.beta, "expected_remote_edge_fraction": args.beta * (world - 1) / world}

    t = sum(ms) / len(ms) / 1e3
    t_e2e = ms_e2e / 1e3
    value = total_units / t
    kernel_t = t if not dist_on else part.last_kernel_seconds(step, torch)
    achieved = algo / kernel_t / 1e9
    traffic, traffic_src = (None, "not captured at N > 1 (ncu is single-process)") if dist_on else profiled_traffic(kernel_name)
    line = {
        "metric": METRIC, "value": value, "unit": "edges/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "ms_per_step_min": min(ms),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "hidden": F_HIDDEN, "parallelism": parallelism,
                   "l2": "flushed between timed steps (512 MiB write, excluded from the event intervals)",
                   "hub_chunk_edges": cogdl_b200.structure.DEFAULT_CHUNK_EDGES},
        "algorithmic_GBps": achieved,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src, "kernel": kernel_name,
                     "algorithmic_bytes_per_launch": algo, "compulsory_bytes_per_launch": bmin,
                     "frac_compulsory": bmin / kernel_t / 1e9 / peak,
                     "frac_at_profiled_traffic": (traffic / kernel_t / 1e9 / peak) if traffic else None,
                     "l2_resident": (not dist_on),
                     "note": "X (87 MB) fits the 126 MB L2, so algorithmic bytes/time may exceed the HBM peak; "
                             "frac_compulsory / frac_at_profiled_traffic are the DRAM-side fractions" if not dist_on else
                             "per-rank SpMM kernel (max over ranks), X shard >> L2; in p2p mode the same kernel "
                             "also performs the remote-row gather over NVLink"},
        "parity": parity,
        "e2e": {"value": total_units / t_e2e, "unit": "edges/s", "ms_per_step": t_e2e * 1e3, "steps": e2e_steps,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "pcie_GBps_per_rank_each_way": h2d / t_e2e / 1e9,
                "what": "pinned host X -> device, cogdl_b200.spmm(graph, x) (N > 1: PartitionedSpMM.spmm), Y -> pinned host on a "
                        "second stream (overlaps the next step's H2D); CSR resident; K steps timed as one device interval",
                "l2": e2e_l2},
        "gpu_launches": launches, "clocks": clocks,
    }
    line.update(extra_keys)
    if not dist_on:
        t0 = time.perf_counter()
        line["cpu_baseline"] = cpu_baseline_leg(rp, col, w, x_host, nnz)
        phases["cpu_baseline_s"] = time.perf_counter() - t0
        if not args.no_extras:
            del g, st, x_dev, x_in
            torch.cuda.empty_cache()
            line["others"] = extras(torch, flush, synth, args.steps)
    phases["total_s"] = time.perf_counter() - t_begin
    line["phases"] = phases
    if rank == 0:
        print(json.dumps(line))
    if dist_on:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if not parity["ok"]:
        sys.stderr.write(f"bench.py: PARITY FAILED: {json.dumps(parity)}\n")
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--beta", type=float, default=float(os.environ.get("COGDL_B200_DIST_BETA", "0.05")),
                    help="N > 1: probability that a column is drawn over the whole graph instead of the own node range")
    ap.add_argument("--scaling", default=os.environ.get("COGDL_B200_DIST_SCALING", "weak"), choices=["weak", "strong"],
                    help="N > 1: weak = 1/8 of papers100M per GPU; strong = papers100M split N ways")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output of the last one to DIR/*.npy (a fixed seeded row "
                         "sample when larger than %d rows) so that two builds can be compared" % DUMP_ROWS)
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
