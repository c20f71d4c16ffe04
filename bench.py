#!/usr/bin/env python
"""bench.py - graph-steps/sec of the batched ChebConv forward (BASELINE.json metric).

Workload (BASELINE.json configs[1]): one ChebConv layer, K=5, 32 -> 32 features, bias +
leaky_relu, over a batch of 1024 Barabasi-Albert (m=2) graphs of 20..110 nodes.  A "step" is
one pass of the hot path over one such batch.  Weak scaling: every rank gets its own 1024 graphs.

    python bench.py --gpus 1 --steps 200 --warmup 20           # this repo's CUDA path
    python bench.py --impl reference --steps 3 --warmup 1      # the CPU restatement of the reference path
    python bench.py --steps 20 --dump-outputs DIR              # also write the last timed step's output as DIR/*.npy
    torchrun --nproc-per-node N bench.py --gpus N ...          # one rank per GPU

Timing: the K steps (one mho_cheb_forward launch each, round-robin on --streams CUDA streams) are captured ONCE in a
CUDA graph; a timed region is one replay = exactly K steps, bracketed by CUDA events on the launching stream with a
barrier + synchronize on both sides.  --replays of them are timed; `value` comes from the MEDIAN replay (min / max are
reported next to it), max over ranks.  The host launch path (Python -> ctypes -> cudaLaunchKernelEx) is therefore not
inside the timed region; `eager_ms_per_step` gives the old back-to-back eager loop for comparison.  L2 hygiene: step i
uses input/output set i % R with R * bytes > 2 * 126 MB, so no step finds its inputs in L2.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "graph-steps/sec (ChebConv K=5 fwd, BA 20-110 nodes)"
UNIT = "graph-steps/s"
L2_BYTES = 126 * 1024 * 1024
SIZES = np.arange(20, 111, 10)


# --------------------------------------------------------------------------------------------
# workload (pure numpy/networkx; shared by both arms)
# --------------------------------------------------------------------------------------------
def ba_csr(n, seed):
    """CSR of networkx.barabasi_albert_graph(n, 2, seed) (generator of src/offloading_v3.py:40)."""
    import networkx as nx
    g = nx.barabasi_albert_graph(int(n), 2, seed=int(seed))
    indptr = np.zeros(n + 1, dtype=np.int64)
    cols = []
    for i in range(n):
        nb = sorted(g.adj[i])
        cols.append(np.asarray(nb, dtype=np.int64))
        indptr[i + 1] = indptr[i] + len(nb)
    return indptr, (np.concatenate(cols) if cols else np.zeros(0, dtype=np.int64))


def bind_to_gpu_numa_node(torch, local):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off (sysfs), so that cudaHostAlloc'd staging buffers
    are local to the GPU's PCIe root (one rank per GPU: 8 ranks otherwise crowd the first socket).  Best effort."""
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


_BA_CACHE = {}


def make_workload(n_graphs, rank=0, fixed_n=None, K=5, F=32, pack=True, unique=0):
    """unique > 0 (sweep points): only `unique` distinct graphs are generated, the batch cycles through them (every
    instance still has its own feature rows) - networkx needs seconds per thousand 512-node graphs."""
    rng = np.random.default_rng(0 + 7919 * rank)
    sizes = np.full(n_graphs, fixed_n) if fixed_n else rng.choice(SIZES, size=n_graphs)
    if pack and not fixed_n:
        # same multiset of graphs, laid out in tile-packing order (first-fit decreasing): the order of independent
        # graph instances in a batch is the batch builder's choice
        from multihop_offload_b200.batch import pack_order
        perm = pack_order(sizes, 128)
        seeds = (1000 + np.arange(n_graphs) + 100003 * rank)[perm]
        sizes = sizes[perm]
    else:
        seeds = 1000 + np.arange(n_graphs) + 100003 * rank
    goff = np.zeros(n_graphs + 1, dtype=np.int64)
    rps, cis = [np.zeros(1, dtype=np.int64)], []
    noff = zoff = 0
    for i, n in enumerate(sizes):
        if unique:
            key = (int(n), int(seeds[i % unique]))
            if key not in _BA_CACHE:
                _BA_CACHE[key] = ba_csr(*key)
            ip, ci = _BA_CACHE[key]
        else:
            ip, ci = ba_csr(int(n), int(seeds[i]))
        rps.append(ip[1:] + zoff)
        cis.append(ci + noff)
        noff += int(n); zoff += ci.size
        goff[i + 1] = noff
    rowptr = np.concatenate(rps).astype(np.int32)
    colidx = np.concatenate(cis).astype(np.int32)
    X = np.random.default_rng(1 + rank).normal(size=(noff, F)).astype(np.float32)
    lim = np.sqrt(6.0 / (K * F + K * F))
    W = np.random.default_rng(2).uniform(-lim, lim, size=(K, F, F))
    b = np.zeros(F)
    return dict(sizes=sizes, graph_off=goff.astype(np.int32), rowptr=rowptr, colidx=colidx, X=X, W=W, b=b, K=K, F=F)


def algorithmic_bytes(w):
    """SURVEY 8(d): 4 n F_in + 4 n F_out + 4 (n+1) + 8 nnz per graph (fp32 values, int32 ids;
    binary operator => the 4 B/nnz value stream is not read: 4 nnz; T_k stay on chip)."""
    n = int(w["graph_off"][-1]); nnz = int(w["rowptr"][-1]); B = len(w["sizes"]); F = w["F"]
    return 4 * n * F + 4 * n * F + 4 * (n + B) + 4 * nnz


def algorithmic_flops(w):
    n = int(w["graph_off"][-1]); nnz = int(w["rowptr"][-1]); F = w["F"]; K = w["K"]
    return 2 * nnz * F * (K - 1) + 2 * n * K * F * F


# --------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's per-graph fp64 path
# --------------------------------------------------------------------------------------------
def cpu_reference_rate(w, seconds=10.0, threads=0, max_passes=1000):
    """graph-steps/s of the reference's CPU path restated in C (fp64, one graph at a time as the
    reference's eager call does, graphs spread over `threads` OpenMP threads; 0 = all)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    ws = [(w["W"], w["b"])]
    X64 = w["X"].astype(np.float64)
    c_oracle.stack_forward(w["graph_off"], w["rowptr"], w["colidx"], None, ws, [2], 0.2, X64, threads)  # warm
    t0 = time.perf_counter(); passes = 0
    while True:
        c_oracle.stack_forward(w["graph_off"], w["rowptr"], w["colidx"], None, ws, [2], 0.2, X64, threads)
        passes += 1
        dt = time.perf_counter() - t0
        if dt >= seconds or passes >= max_passes:
            break
    cores = threads if threads > 0 else c_oracle.max_threads()
    return len(w["sizes"]) * passes / dt, cores, passes, dt


def host_threads():
    """Threads this process may use: the scheduler affinity mask (cgroup-aware), NOT omp_get_max_threads() - launchers such
    as torch.distributed.run export OMP_NUM_THREADS=1, which would silently turn the CPU arm into a 1-thread run."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    w = make_workload(args.graphs, 0, args.fixed_n, K=args.K, pack=not args.no_pack)
    os.environ.pop("OMP_NUM_THREADS", None)               # the thread count is set explicitly per pass (omp_set_num_threads)
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")   # idle OpenMP threads sleep instead of spinning (CPU quotas)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    ws = [(w["W"], w["b"])]
    X64 = w["X"].astype(np.float64)
    # all the host threads it can USE: more OpenMP threads than the container's CPU quota / the memory system can feed
    # make the pass slower, so the thread count is tuned first (one pass each, halving from the maximum)
    def one_pass(nt):
        t_ = time.perf_counter()
        c_oracle.stack_forward(w["graph_off"], w["rowptr"], w["colidx"], None, ws, [2], 0.2, X64, nt)
        return time.perf_counter() - t_
    avail = host_threads()
    cand, nt = [], avail
    while nt >= 1:
        cand.append(nt)
        nt //= 2
    one_pass(cand[0])
    timing = {nt: min(one_pass(nt), one_pass(nt)) for nt in cand}
    cores = min(timing, key=timing.get)
    if avail > 1 and cores == 1:
        sys.stderr.write("bench.py --impl reference: the best thread count is 1 of %d available - check the CPU quota\n" % avail)
    for _ in range(max(args.warmup, 1)):
        one_pass(cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_pass(cores)
    dt = time.perf_counter() - t0
    val = args.graphs * args.steps / dt
    if args.dump_outputs:
        Y = c_oracle.stack_forward(w["graph_off"], w["rowptr"], w["colidx"], None, ws, [2], 0.2, X64, cores)
        dump_outputs(args.dump_outputs, {"Y": Y})
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, w),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "threads_available": avail, "kind": "port",
                         "threads_tried": {str(k): round(v * 1e3, 2) for k, v in timing.items()},
                         "sample": "%d full passes over the %d-graph batch (oracle/cheb_oracle.c, fp64, one graph at a "
                                   "time, OpenMP over graphs)" % (args.steps, args.graphs)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference hot path is TensorFlow+Spektral (not installable offline): timed arm is the oracle port; the "
                "thread count comes from the affinity mask, never from OMP_NUM_THREADS",
    }
    print(json.dumps(out))
    return 0


def workload_config(args, w):
    """Describes the WORKLOAD only (identical for both arms); how each arm measures is in the line's `method` key."""
    return {"workload": "configs[1]: ChebConv K=%d forward, %d->%d, bias+leaky_relu, batch %d BA(m=2) graphs, n in %s, "
                        "raw-adjacency operator" % (w["K"], w["F"], w["F"], args.graphs,
                                                    "{%d}" % args.fixed_n if args.fixed_n else "{20..110 step 10}"),
            "graphs_per_gpu": args.graphs, "nodes_per_gpu": int(w["graph_off"][-1]), "nnz_per_gpu": int(w["rowptr"][-1]),
            "parallelism": "graph-instance sharding, no data-path collective",
            "l2": "rotating over distinct input/output sets > 2x L2",
            "batch_order": "graphs laid out in tile-packing order (first-fit decreasing, multihop_offload_b200.pack_order)"}


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
class GraphTimer:
    """`steps` forward launches captured in one CUDA graph (round-robin over `n_str` side streams), replayed `replays`
    times; every replay is timed with CUDA events on the launching stream between barrier + synchronize pairs."""

    def __init__(self, torch, dev, launch, steps, n_str, barrier):
        self.torch, self.steps, self.barrier = torch, steps, barrier
        self.g = torch.cuda.CUDAGraph()
        self.s = torch.cuda.Stream(device=dev)
        side = [torch.cuda.Stream(device=dev) for _ in range(n_str)] if n_str > 1 else []
        self.s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self.s):
            with torch.cuda.graph(self.g, stream=self.s):
                if not side:
                    for i in range(steps):
                        launch(i)
                else:
                    for ss in side:
                        ss.wait_stream(self.s)
                    for i in range(steps):
                        with torch.cuda.stream(side[i % n_str]):
                            launch(i)
                    for ss in side:
                        self.s.wait_stream(ss)
        torch.cuda.synchronize()

    def run(self, replays, warm=2):
        torch = self.torch
        for _ in range(warm):
            self.g.replay()
        ms = []
        for _ in range(replays):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.barrier()
            e0.record()
            self.g.replay()
            e1.record()
            self.barrier()
            ms.append(e0.elapsed_time(e1))
        return np.asarray(ms)


def bytes_of(w, survey=False):
    n = int(w["graph_off"][-1]); nnz = int(w["rowptr"][-1]); B = len(w["sizes"]); F = w["F"]
    return 4 * n * F + 4 * n * F + 4 * (n + B) + (8 if survey else 4) * nnz


DUMP_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, arrays, rank=0, world=1):
    """Writes each array as out_dir/<name>.npy (<name>_rank<r>.npy under several ranks), so that two builds can be
    compared output for output on the same seeded inputs.  Device tensors are written as float32, numpy arrays keep
    float64.  All of them together stay within DUMP_BYTES: a larger array is cut to a fixed, seeded sample of its rows."""
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // max(len(arrays), 1) - 4096   # (room for the .npy header)
    for name, a in arrays.items():
        a = np.asarray(a.detach().float().cpu().numpy() if hasattr(a, "detach") else a)
        if a.nbytes > budget:
            row_bytes = a.nbytes // a.shape[0]
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], size=budget // row_bytes, replace=False))]
        np.save(os.path.join(out_dir, name + ("_rank%d" % rank if world > 1 else "") + ".npy"), a)


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    from multihop_offload_b200 import ChebNet, GraphBatch, LayerSpec

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback "
                         "(use --impl reference for the CPU restatement)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.manual_seed(3 + rank)   # the rotating input sets: the same inputs on every run with the same arguments
    numa_node = bind_to_gpu_numa_node(torch, local)   # page-locked staging buffers land next to this rank's GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor(v, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.cpu().numpy()

    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, copy burst)"
    except Exception:
        pass
    n_str = max(1, int(args.streams))
    replays = max(3, int(args.replays))

    def time_layer(w, steps, use_bits=True, reps=replays, warm_steps=3):
        """graph-timed forward of one 32->32 layer over workload w: (median ms per replay, all replay ms, launches, net, sets)"""
        net_ = ChebNet([LayerSpec(w["K"], w["F"], w["F"], 2, 0.2)], device=dev)
        net_.set_weights([(w["W"], w["b"])])
        ab = bytes_of(w)
        R = max(2, min(int(np.ceil(2.2 * L2_BYTES / ab)), 24))
        n_nodes = int(w["graph_off"][-1])
        bt = [GraphBatch(w["graph_off"], w["rowptr"], w["colidx"], None, tile_rows=args.tile_rows, device=dev) for _ in range(R)]
        if not use_bits:
            for b_ in bt:
                b_.dev.pop("adj_bits", None); b_._struct_cache = {}
        X0 = torch.from_numpy(w["X"]).to(dev)
        Xs = [X0] + [torch.randn_like(X0) for _ in range(R - 1)]
        Ys = [torch.empty((n_nodes, w["F"]), dtype=torch.float32, device=dev) for _ in range(R)]

        def launch(i):
            net_.forward(bt[i % R], Xs[i % R], out=Ys[i % R])
        for i in range(max(warm_steps, 3)):
            launch(i)
        barrier()
        l0 = net_.ctx.launch_count()
        gt = GraphTimer(torch, dev, launch, steps, n_str, barrier)
        per_graph = net_.ctx.launch_count() - l0          # launches captured = launches per replay
        ms = gt.run(reps)
        return float(np.median(ms)), ms, per_graph, net_, (bt, Xs, Ys, launch, R)

    # ---------------- headline: configs[1]
    w = make_workload(args.graphs, rank, args.fixed_n, K=args.K, pack=not args.no_pack)
    n_nodes = int(w["graph_off"][-1])
    alg_bytes = bytes_of(w)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    med_ms, all_ms, launches, net, (batches, Xs, Ys, launch, R) = time_layer(w, args.steps, True, replays, max(args.warmup, 3))
    # the eager loop (host launch path inside the timed window), for comparison
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        launch(i)
    ev1.record()
    barrier()
    eager_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    # the graph's launches computed what a lone launch computes (same buffers, same tiles)
    chk = [(args.steps - 1 - d) % R for d in range(min(n_str + 1, args.steps))]
    kept = [Ys[j].clone() for j in chk]
    for j, y in zip(chk, kept):
        net.forward(batches[j], Xs[j], out=Ys[j])
        torch.cuda.synchronize()
        assert torch.equal(Ys[j], y), "overlapped step differs from a single launch"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"Y": Ys[(args.steps - 1) % R]}, rank, world)

    # ---------------- e2e: host buffers in, host buffers out, through the C-ABI host call
    from multihop_offload_b200._lib import PinnedArray, pinned_like
    goff_h, rp_h, ci_h = (pinned_like(np.ascontiguousarray(w[k], dtype=np.int32)) for k in ("graph_off", "rowptr", "colidx"))
    # two calls in flight, each with its own page-locked X / Y: the upload of step i+1 overlaps the download of step i
    Xh = [pinned_like(np.ascontiguousarray(w["X"], dtype=np.float32)) for _ in range(2)]
    Yh = [PinnedArray((n_nodes, w["F"]), np.float32) for _ in range(2)]
    e2e_steps = max(4, min(args.steps, 50))

    def e2e_run(n):
        tickets = [None, None]
        for i in range(n):
            b = i & 1
            if tickets[b] is not None:
                net.host_wait(tickets[b])          # step i-2's result is on the host: its buffers may be reused
            tickets[b] = net.forward_host_async(goff_h.array, rp_h.array, ci_h.array, None, Xh[b].array, Yh[b].array)
        for t_ in tickets:
            if t_ is not None:
                net.host_wait(t_)

    e2e_run(4)
    barrier()
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    h2d = int(Xh[0].array.nbytes + rp_h.array.nbytes + ci_h.array.nbytes)  # graph_off stays on the host (tile planning)
    d2h = int(Yh[0].array.nbytes)

    series = {}
    if not args.no_series:
        # ---- the same layer fed the raw CSR (the kernel derives the adjacency bit rows itself)
        m_csr, _, _, _, _ = time_layer(w, args.steps, use_bits=False, reps=max(3, replays // 2))
        t_csr = float(max_over_ranks([m_csr])[0])
        series["csr_input_K%d" % w["K"]] = {
            "value": world * args.graphs * args.steps / (t_csr * 1e-3), "unit": UNIT, "ms_per_step": t_csr / args.steps,
            "note": "same workload without mho_batch_t.adj_bits: the CSR slice is staged and turned into bit rows in-kernel",
            "frac_of_hbm_roofline": alg_bytes * args.steps / (t_csr * 1e-3) / 1e9 / peak}
        # ---- the north_star's target configuration: all graphs n = 100 (one graph per 128-row tile)
        if not args.fixed_n:
            w100 = make_workload(args.graphs, rank, 100, K=args.K, unique=256)
            m100, _, _, _, _ = time_layer(w100, args.steps, True, max(3, replays // 2))
            t100 = float(max_over_ranks([m100])[0])
            ab100 = bytes_of(w100)
            series["fixed_n100_K%d" % w100["K"]] = {
                "value": world * args.graphs * args.steps / (t100 * 1e-3), "unit": UNIT, "ms_per_step": t100 / args.steps,
                "algorithmic_bytes_per_launch": ab100, "algorithmic_bytes_survey_formula": bytes_of(w100, True),
                "frac_of_hbm_roofline": ab100 * args.steps / (t100 * 1e-3) / 1e9 / peak,
                "frac_survey_formula": bytes_of(w100, True) * args.steps / (t100 * 1e-3) / 1e9 / peak,
                "roofline_graph_steps_per_s_per_gpu_survey": peak * 1e9 / (bytes_of(w100, True) / args.graphs),
                "note": "%d BA(m=2) graphs of exactly 100 nodes per GPU (256 distinct graphs cycled), K=%d, 32->32" % (args.graphs, w100["K"])}
        # ---- the reference's shipped 5-layer stack 4-32-32-32-32-1, K=1, on the same graphs (one fused launch per step)
        from multihop_offload_b200 import reference_stack
        rs = np.random.default_rng(5)
        specs5 = reference_stack(K=1)
        net5 = ChebNet(specs5, device=dev)
        net5.set_weights([((rs.standard_normal((sp_.K, sp_.f_in, sp_.f_out)) * 0.2).astype(np.float32),
                           np.zeros(sp_.f_out, np.float32)) for sp_ in specs5])
        X5 = torch.randn((n_nodes, 4), device=dev)
        Y5 = torch.empty((n_nodes, 1), dtype=torch.float32, device=dev)
        for _ in range(5):
            net5.forward(batches[0], X5, out=Y5)
        barrier()
        X5s = [X5] + [torch.randn_like(X5) for _ in range(min(R, 8) - 1)]
        Y5s = [torch.empty_like(Y5) for _ in range(len(X5s))]
        g5 = GraphTimer(torch, dev, lambda i: net5.forward(batches[i % R], X5s[i % len(X5s)], out=Y5s[i % len(X5s)]), args.steps, n_str, barrier)
        stack5_ms = float(np.median(g5.run(max(3, replays // 2)))) / args.steps
        stack5_ms = float(max_over_ranks([stack5_ms])[0])
        series["reference_stack_4_32_32_32_32_1_K1"] = {
            "value": world * args.graphs / (stack5_ms * 1e-3), "unit": "graph forwards/s (the shipped 5-layer K=1 model, one fused launch per step)",
            "ms_per_step": stack5_ms, "streams": n_str, "kernel": "cheb_mlp_f16_kernel"}
        del g5
        # ---- forward (activations kept) + VJP to one flat gradient per graph + deterministic sum (SURVEY 8a6): graph-timed like
        # the headline; every stream has its own mho context (reduction scratch) and rotates over the same distinct batches
        n_tr = n_str
        nets_t = [ChebNet([LayerSpec(w["K"], w["F"], w["F"], 2, 0.2)], device=dev, private_context=True) for _ in range(n_tr)]
        for nt_ in nets_t:
            nt_.set_weights([(w["W"], w["b"])])
        dYs = [torch.randn((n_nodes, w["F"]), device=dev) for _ in range(min(R, 4))]
        keep_t = {}

        def train_step(i):
            nt_ = nets_t[i % n_tr]
            Yt, saved = nt_.forward(batches[i % R], Xs[i % R], save=True)
            keep_t[i % (2 * n_tr)] = nt_.backward(batches[i % R], Xs[i % R], Yt, saved, dYs[i % len(dYs)])
        for i in range(max(R, 2 * n_tr) + 2):   # (every batch builds its per-graph bit rows on first use)
            train_step(i)
        barrier()
        nt = max(6, min(args.steps, 30))
        l0 = sum(n_.ctx.launch_count() for n_ in nets_t)
        gtt = GraphTimer(torch, dev, train_step, nt, n_tr, barrier)
        train_launches = sum(n_.ctx.launch_count() for n_ in nets_t) - l0
        train_ms = float(np.median(gtt.run(max(3, replays // 2)))) / nt
        train_ms = float(max_over_ranks([train_ms])[0])
        # one stream alone, for the device time of a single step
        gt1 = GraphTimer(torch, dev, train_step, nt, 1, barrier)
        train1_ms = float(np.median(gt1.run(3))) / nt
        series["forward_backward_K%d_32_32" % w["K"]] = {
            "value": world * args.graphs / (train_ms * 1e-3), "unit": "graph forward+VJP steps/s (per-graph gradients + their deterministic sum)",
            "ms_per_step": train_ms, "ms_per_step_one_stream": train1_ms, "streams": n_tr, "launches_per_step": train_launches / nt,
            "kernels": "cheb_f16ws_kernel (forward), cheb_backward_f16_kernel (tensor-core VJP), grads_sum_fused"}
        del gtt, gt1
        # ---- the same for the model the reference ships and trains (AdHoc_train: 4-32-32-32-32-1, K=1): fused forward with kept
        # activations (cheb_mlp_f16_kernel) + VJP of the stack (cheb_mlp_backward_f16_kernel) + gradient sum
        nets5_t = [ChebNet(specs5, device=dev, private_context=True) for _ in range(n_tr)]
        for n5_ in nets5_t:
            n5_.set_flat(net5.get_flat())
        dY5 = torch.randn((n_nodes, 1), device=dev)
        keep5 = {}

        def train_step5(i):
            n5_ = nets5_t[i % n_tr]
            Yt, saved = n5_.forward(batches[i % R], X5s[i % len(X5s)], save=True)
            keep5[i % (2 * n_tr)] = n5_.backward(batches[i % R], X5s[i % len(X5s)], Yt, saved, dY5)
        for i in range(max(R, 2 * n_tr) + 2):
            train_step5(i)
        barrier()
        nt5 = max(4, min(args.steps, 12))
        gt5 = GraphTimer(torch, dev, train_step5, nt5, n_tr, barrier)
        train5_ms = float(np.median(gt5.run(max(3, replays // 2)))) / nt5
        train5_ms = float(max_over_ranks([train5_ms])[0])
        series["reference_stack_forward_backward_K1"] = {
            "value": world * args.graphs / (train5_ms * 1e-3), "unit": "graph forward+VJP steps/s (per-graph gradients + their deterministic sum)",
            "ms_per_step": train5_ms, "streams": n_tr,
            "kernels": "cheb_mlp_f16_kernel (forward), cheb_mlp_backward_f16_kernel (tensor-core VJP of the 5-layer stack), grads_sum_stage1/2"}
        del gt5
        # ---- gradient exchange of AdHoc_train (gnn_offloading_agent.py:156-169 site): NCCL on device tensors
        if world > 1:
            from multihop_offload_b200 import parallel
            series["train_exchange_us"] = parallel.bench_exchange(torch, dist, dev, world, barrier)

    # ---------------- sweep (BASELINE.json configs[4]): n x K x B, one 32->32 layer, per GPU; weak scaling like the headline
    if args.sweep != "off":
        Bs = [256, 4096, 16384] if args.sweep == "full" else [4096]
        pts = []
        for n_ in (20, 100, 200, 512):
            for K_ in (2, 5, 10):
                for B_ in Bs:
                    if n_ * B_ * 32 * 4 * 2 * 2 > 40e9:
                        continue
                    ws_ = make_workload(B_, rank, n_, K=K_, unique=64)
                    st_ = 3 if n_ * B_ >= 2 ** 20 else 6
                    try:
                        m_, _, _, net_s, keep = time_layer(ws_, st_, True, 3, 2)
                    except Exception as e:   # a point that does not fit is reported, not fatal
                        pts.append({"n": n_, "K": K_, "B": B_, "error": str(e)[:120]})
                        continue
                    t_ = float(max_over_ranks([m_])[0])
                    ab_ = bytes_of(ws_)
                    pts.append({"n": n_, "K": K_, "B": B_, "ms_per_step": t_ / st_, "graph_steps_per_s": world * B_ * st_ / (t_ * 1e-3),
                                "frac_of_hbm_roofline": ab_ * st_ / (t_ * 1e-3) / 1e9 / peak,
                                "kernel": ("cheb_f16ws_kernel" if K_ <= 5 else "cheb_f16_kernel") if n_ <= 128 else "cheb_forward_kernel (CSR walk)"})
                    del net_s, keep
                    torch.cuda.empty_cache()
        series["sweep"] = {"unit": UNIT, "points": pts,
                           "note": "cfg-5: BA(m=2) graphs of n nodes (64 distinct graphs cycled, every instance its own features), "
                                   "one ChebConv layer 32->32 of order K, batch B per GPU; graph-timed like the headline (3-6 steps, 3 replays); "
                                   "frac = algorithmic bytes (4 B/nnz variant) / time / measured HBM peak"}

    t = max_over_ranks([med_ms, e2e_s, eager_ms, float(all_ms.min()), float(all_ms.max())])
    med_ms, e2e_s, eager_ms, min_ms, max_ms = (float(x) for x in t)
    value = world * args.graphs * args.steps / (med_ms * 1e-3)
    e2e_val = world * args.graphs * e2e_steps / e2e_s

    if rank == 0:
        per_launch_ms = med_ms / max(launches, 1)
        achieved = alg_bytes / (per_launch_ms * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("dram_bytes_per_launch")
        except Exception:
            pass
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": med_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (fp32 storage and accumulation; both products run on tcgen05 with operands split into two scaled fp16 parts, 22 significand bits)",
            "data": "synthetic",
            "config": workload_config(args, w),
            "method": {"timed_region": "one CUDA-graph replay = exactly %d steps (one mho_cheb_forward launch each), CUDA events on the launching "
                                       "stream, barrier + synchronize on both sides; value from the median of %d replays, max over ranks" % (args.steps, replays),
                       "replay_ms": {"min": min_ms, "median": med_ms, "max": max_ms},
                       "streams": "%d CUDA streams inside the captured graph (independent batches; their head / tail overlap)" % n_str,
                       "eager_ms_per_step": eager_ms / args.steps,
                       "operator_input": "cached per-batch adjacency bit rows (mho_fill_adj_bits, 16 B per node) + tile-packing batch order; "
                                         "series.csr_input_* is the same layer fed the raw CSR",
                       "numa_node": numa_node},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "api": "mho_cheb_forward_host_async + mho_host_wait, two steps in flight (page-locked host buffers from mho_host_alloc; every step uploads X + CSR and downloads Y; chunked upload/kernel/download pipeline)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "cheb_f16ws_kernel<K> (K <= 5; cheb_f16_kernel<K> for K > 5)",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "algorithmic_bytes_survey_formula": bytes_of(w, True),
                         "frac_survey_formula": bytes_of(w, True) / (per_launch_ms * 1e-3) / 1e9 / peak,
                         "tflops_algorithmic": algorithmic_flops(w) / (per_launch_ms * 1e-3) / 1e12},
        }
        if series:
            out["series"] = series
        if world == 1 and not args.no_cpu:
            v, cores, passes, dt = cpu_reference_rate(w, seconds=args.cpu_seconds, threads=1)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                   "sample": "%d passes over the same %d-graph batch in %.1f s (oracle/cheb_oracle.c: fp64, "
                                             "one graph at a time like the reference's eager call, 1 thread)" % (passes, args.graphs, dt)}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--graphs", type=int, default=1024, help="graphs per GPU per step")
    ap.add_argument("--fixed-n", type=int, default=None, help="all graphs of this size (e.g. 100)")
    ap.add_argument("--K", type=int, default=5, help="Chebyshev order of the layer")
    ap.add_argument("--tile-rows", type=int, default=128)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--streams", type=int, default=2, help="independent steps are captured round-robin on this many CUDA streams")
    ap.add_argument("--replays", type=int, default=11, help="timed replays of the K-step graph (median reported)")
    ap.add_argument("--no-pack", action="store_true", help="keep the random graph order instead of tile-packing order")
    ap.add_argument("--no-series", action="store_true", help="headline + e2e only")
    ap.add_argument("--sweep", default="compact", choices=["off", "compact", "full"], help="cfg-5 sweep: n x K (x B with 'full')")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (the layer output Y of the headline batch) as DIR/Y.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
