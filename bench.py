#!/usr/bin/env python
# coding=utf-8
"""bench.py - the headline measurement (BASELINE.json metric):

    edges/sec of GCN + 8-head GAT forward on a synthetic ogbn-products-shaped graph
    (2,449,029 nodes, 123,718,280 directed edges, 100-dim fp32 features), plus the HBM-roofline fraction of the
    dominant kernel and the reference CPU path timed on the same box.

A "step" = one tfg.layers.GCN(128, relu) forward followed by one tfg.layers.GAT(128, num_heads=8, relu) forward over
the whole graph through the public layer API, warm graph.cache (normalised adjacency + destination-sorted CSR built
once, outside the timed region - the regime of the reference's own harness, demo/demo_gcn.py:47,99-105).
edges/sec = (2 * E) / step time: every layer pass streams all E input edges (appended self loops are NOT counted).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config headline|cfg1..cfg5] [--scale S]
                    [--dump-outputs DIR]

--dump-outputs DIR writes the arrays the last timed step returned as DIR/<name>.npy (float32), so that two builds can be
compared output for output on identical seeded inputs; an output above its share of 64 MB is stored as a fixed sample of
its rows (see dump_outputs).  Single-GPU configs of --impl ours only.

--config selects one of BASELINE.json's configs (default: headline = the configuration the metric is quoted on); every
config prints the same JSON contract with its own roofline.  --gpus N > 1 (under torchrun) runs the headline step
destination-partitioned over N GPUs through the same tfg.layers calls; cfg5 (papers100M shape) needs 8 GPUs.

--impl reference times the reference's op sequence on the host CPU cores (oracle/torch_cpu_port.py; TensorFlow and
tf_sparse cannot be installed offline) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PRODUCTS_NODES = 2449029
PRODUCTS_UNDIRECTED = 61859140
FEATURES = 100
UNITS = 128
HEADS = 8
METRIC = "edges/sec GCN+GAT fwd on 2.4M-node/123M-edge synthetic; %HBM roofline"


# BASELINE.json `configs` (SURVEY.md section 8d): sizes, layer(s) per step, and which pass is timed
CONFIGS = {
    "headline": {"nodes": PRODUCTS_NODES, "pairs": PRODUCTS_UNDIRECTED, "features": 100, "kind": "gcn+gat",
                 "what": "GCN(128,relu) fwd + GAT(128, 8 heads, relu) fwd, synthetic ogbn-products shape"},
    "cfg1": {"nodes": 2708, "pairs": 5278, "features": 1433, "kind": "gcn2",
             "what": "demo_gcn.py model (GCN 1433->16 relu -> GCN 16->7) fwd on a Cora-shaped synthetic graph, sparse bag-of-words x"},
    "cfg2": {"nodes": 1000000, "pairs": 10000000, "features": 128, "kind": "gcn",
             "what": "GCN(128,relu) fwd, synthetic 1M nodes / 20M edges / 128 features"},
    "cfg3": {"nodes": 1000000, "pairs": 10000000, "features": 128, "kind": "gat",
             "what": "GAT(128, 8 heads, relu) fwd, synthetic 1M nodes / 20M edges / 128 features"},
    "cfg4": {"nodes": PRODUCTS_NODES, "pairs": PRODUCTS_UNDIRECTED, "features": 100, "kind": "sage_train",
             "what": "MeanGraphSage(256, concat) forward + backward (gradients w.r.t. weights and inputs), ogbn-products shape"},
    "cfg5": {"nodes": 111059956, "edges": 1615685872, "features": 128, "kind": "gcn_partitioned",
             "what": "GCN(128,relu) fwd, synthetic ogbn-papers100M shape, destination-partitioned"},
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS),
                    help="BASELINE.json workload: headline = the metric's own configuration (default); cfg1..cfg5 = configs[0..4]")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (testing only; 1.0 = BASELINE size)")
    ap.add_argument("--cpu-sample-div", type=int, default=0,
                    help="reference arm: graph scaled down by this factor (0 = auto: about two minutes of CPU work in total)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    return ap.parse_args()


# ---- synthetic workload --------------------------------------------------------------------------------------------

def make_graph_device(num_nodes, num_pairs, seed, device):
    """Uniform random undirected pairs u != v, mirrored (SURVEY.md 8d cfg 4 generator), int32 [2, 2*pairs]."""
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    u = torch.randint(0, num_nodes, (num_pairs,), generator=gen, device=device, dtype=torch.int32)
    v = torch.randint(0, num_nodes - 1, (num_pairs,), generator=gen, device=device, dtype=torch.int32)
    v = v + (v >= u).to(torch.int32)                      # v != u, still uniform
    edge_index = torch.empty((2, 2 * num_pairs), dtype=torch.int32, device=device)
    edge_index[0, :num_pairs] = u
    edge_index[0, num_pairs:] = v
    edge_index[1, :num_pairs] = v
    edge_index[1, num_pairs:] = u
    return edge_index


def glorot(shape, seed):
    gen = torch.Generator(device="cpu")
    gen.manual_seed(seed)
    limit = (6.0 / (shape[0] + shape[1])) ** 0.5
    return (torch.rand(shape, generator=gen, dtype=torch.float32) * 2 - 1) * limit


class ClockSampler(object):
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML in a background thread every
    ~2 ms (nvidia-smi -lms cannot resolve a 50 ms region); falls back to one nvidia-smi query if NVML is unavailable."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:
            self.nvml = None

    def _loop(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                try:
                    reasons = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    reasons = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                power = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                self.samples.append((sm, reasons, power))
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        if self.nvml is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        n = self.nvml
        smax = None
        try:
            smax = float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM))
        except Exception:
            pass
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        seen = set()
        for _, r, _ in self.samples:
            for k, bit in names.items():
                if r & bit:
                    seen.add(k)
        sm = [x[0] for x in self.samples]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "power_w_max": max([x[2] for x in self.samples]) if self.samples else None,
                "samples": len(sm), "reasons": sorted(seen)}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# ---- reference arm (CPU) ---------------------------------------------------------------------------------------------

def _cpu_workload(kind, num_nodes, num_pairs, features, seed=0):
    """Builds the reference's op sequence for one step of `kind` on a graph of the given size; returns (step_fn, E,
    edge layer passes per step)."""
    from oracle import torch_cpu_port as port
    from oracle import tfg_oracle as o
    ei = make_graph_device(num_nodes, num_pairs, seed, torch.device("cpu"))
    E = ei.shape[1]
    gen = torch.Generator(device="cpu"); gen.manual_seed(1)
    x = torch.randn((num_nodes, features), generator=gen, dtype=torch.float32)
    # warm cache, like demo_gcn.py:47: normalised adjacency precomputed (numpy oracle), self loops appended for GAT
    normed = o.gcn_norm_adj(o.SparseMatrix(ei.numpy(), None, [num_nodes, num_nodes]))
    n_row = torch.from_numpy(normed.index[0]).long(); n_col = torch.from_numpy(normed.index[1]).long()
    n_val = torch.from_numpy(normed.value)
    b = torch.zeros(UNITS)
    if kind == "gcn+gat":
        wk = glorot((features, UNITS), 2)
        wq_, wk_, wv_ = glorot((features, UNITS), 3), glorot((features, UNITS), 4), glorot((features, UNITS), 5)

        def step():
            port.gcn_forward(x, n_row, n_col, n_val, wk, b)
            port.gat_forward(x, n_row, n_col, wq_, b, wk_, b, wv_, b, HEADS)   # same index: edges + appended self loops
        return step, E, 2
    if kind in ("gcn", "gcn_partitioned"):
        wk = glorot((features, UNITS), 2)
        return (lambda: port.gcn_forward(x, n_row, n_col, n_val, wk, b)), E, 1
    if kind == "gat":
        wq_, wk_, wv_ = glorot((features, UNITS), 3), glorot((features, UNITS), 4), glorot((features, UNITS), 5)
        return (lambda: port.gat_forward(x, n_row, n_col, wq_, b, wk_, b, wv_, b, HEADS)), E, 1
    if kind == "gcn2":
        w1, w2 = glorot((features, 16), 2), glorot((16, 7), 3)
        b1, b2 = torch.zeros(16), torch.zeros(7)

        def step():
            h = port.gcn_forward(x, n_row, n_col, n_val, w1, b1)
            port.gcn_forward(h, n_row, n_col, n_val, w2, b2, relu=False)
        return step, E, 2
    if kind == "sage_train":
        # nn/conv/graph_sage.py:9-60 under autodiff (demo_graph_sage.py:100-106): gather, segment mean, two projections, concat
        row, col = ei[0].long(), ei[1].long()
        ws, wn = glorot((features, UNITS), 2).requires_grad_(True), glorot((features, UNITS), 3).requires_grad_(True)
        bb = torch.zeros(2 * UNITS).requires_grad_(True)
        g = torch.randn((num_nodes, 2 * UNITS), generator=gen)
        cnt = torch.bincount(row, minlength=num_nodes).clamp(min=1).float().unsqueeze(1)
        xg = x.clone().requires_grad_(True)

        def step():
            for t in (ws, wn, bb, xg):
                t.grad = None
            msg = xg.index_select(0, col)
            agg = torch.zeros_like(xg).index_add_(0, row, msg) / cnt
            out = torch.relu(torch.cat([xg @ ws, agg @ wn], dim=1) + bb)
            (out * g).sum().backward()
        return step, E, 1
    raise ValueError(kind)


def cpu_reference(kind, num_nodes, num_pairs, features, steps, warmup, threads=None):
    """The reference's op sequence on the host cores on a bounded graph.  The thread count is swept on a 4x smaller graph
    first (index_add_ / scatter_reduce_ do not scale with threads; 128 threads were 4x slower than 1 in round 1)."""
    ncpu = os.cpu_count() or 1
    sweep = {}
    if threads is None:
        small, _, _ = _cpu_workload(kind, max(num_nodes // 4, 1000), max(num_pairs // 4, 1000), features)
        for t in sorted({1, 4, 8, 16, 32, 64, ncpu}):
            if t > ncpu:
                continue
            torch.set_num_threads(t)
            small()
            t0 = time.perf_counter()
            small()
            sweep[t] = time.perf_counter() - t0
        threads = min(sweep, key=sweep.get)
    torch.set_num_threads(threads)
    step, E, passes = _cpu_workload(kind, num_nodes, num_pairs, features)
    for _ in range(warmup):
        step()
    times = []
    for _ in range(max(steps, 1)):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    dt = float(np.mean(times))
    return {"edges_per_s": passes * E / dt, "ms_per_step": dt * 1e3, "edges": E, "nodes": num_nodes,
            "cores": threads, "host_cores": ncpu, "passes": passes,
            "thread_sweep_s_per_step_quarter_sample": {str(k): v for k, v in sweep.items()},
            "spread": (max(times) - min(times)) / dt if len(times) > 1 else 0.0}


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def config_sizes(args):
    cfg = CONFIGS[args.config]
    n = int(cfg["nodes"] * args.scale)
    pairs = int(cfg.get("pairs", cfg.get("edges", 0) // 2) * args.scale)
    return cfg, n, pairs


def cpu_sample_div(args, passes, budget_s=75.0):
    """Bounded sample for the CPU arm: the op-for-op port does ~1 M edge-layer passes per second on a big host and less on
    a small one, so `passes` executions of the full graph would take hours.  The rate is calibrated on a tiny graph first
    and the sample is sized so that the whole arm (thread sweep + warm-up + timed steps) fits the time budget."""
    if args.cpu_sample_div > 0:
        return args.cpu_sample_div
    cfg, n, pairs = config_sizes(args)
    layers = {"gcn+gat": 2, "gcn2": 2, "sage_train": 3}.get(cfg["kind"], 1)
    tiny_n, tiny_pairs = max(n // 2000, 500), max(pairs // 2000, 2000)
    torch.set_num_threads(min(os.cpu_count() or 1, 16))
    step, tiny_e, _ = _cpu_workload(cfg["kind"], tiny_n, tiny_pairs, cfg["features"])
    step()
    t0 = time.perf_counter()
    step()
    rate = layers * tiny_e / max(time.perf_counter() - t0, 1e-4)          # edge-layer passes per second
    rate *= 0.3                                                           # larger graphs miss cache: be conservative
    per_step_full = 2.0 * pairs * layers
    equivalent_steps = passes + 3.0                                       # + the thread sweep on a quarter-size graph
    return max(1, int(np.ceil(per_step_full * equivalent_steps / (rate * budget_s))))


def run_reference(args, rank, world):
    if rank != 0:
        return
    cfg, n, pairs = config_sizes(args)
    args.cpu_sample_div = cpu_sample_div(args, args.steps + args.warmup)
    ns = max(n // args.cpu_sample_div, min(n, 1000))
    ps = max(pairs // args.cpu_sample_div, min(pairs, 1000))
    res = cpu_reference(cfg["kind"], ns, ps, cfg["features"], args.steps, args.warmup)
    sample = ("same generator and layer shapes at 1/{} scale: {} nodes, {} directed edges; op-for-op torch-CPU port of "
              "the reference op sequence, {} threads (best of a sweep) on {} host cores, {}").format(
                  args.cpu_sample_div, res["nodes"], res["edges"], res["cores"], res["host_cores"], cpu_model_name())
    config = workload_config(args, 1)
    config["reference_sample"] = {"nodes": res["nodes"], "edges": res["edges"], "scale": "1/{}".format(args.cpu_sample_div),
                                  "note": "the CPU arm times a bounded sample of the workload named above"}
    line = {"metric": config_metric(args), "value": res["edges_per_s"], "unit": "edges/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": config,
            "cpu_baseline": {"value": res["edges_per_s"], "unit": "edges/s", "cores": res["cores"], "kind": "port",
                             "sample": sample, "thread_sweep": res["thread_sweep_s_per_step_quarter_sample"],
                             "step_time_spread": res["spread"]},
            "e2e": {"value": res["edges_per_s"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def config_metric(args):
    return METRIC if args.config == "headline" else "edges/sec " + CONFIGS[args.config]["what"]


def workload_config(args, world):
    cfg, n, pairs = config_sizes(args)
    e = 2 * pairs
    passes = {"gcn+gat": 2, "gcn2": 2}.get(cfg["kind"], 1)
    out = {"workload": "{} ({} nodes, {} directed edges, {} features), uniform random undirected pairs mirrored, "
                       "warm graph.cache".format(cfg["what"], n, e, cfg["features"]),
           "name": args.config, "nodes": n, "edges": e, "features": cfg["features"], "units": UNITS, "heads": HEADS,
           "edges_per_step": passes * e, "parallelism": "single GPU" if world == 1 else "dst-partitioned x{}".format(world),
           "l2_policy": "working set (gathered rows + CSR, GBs) exceeds the 126 MB L2; no explicit flush"}
    if cfg["kind"] == "gcn2":
        out["l2_policy"] = "Cora-sized working set fits in L2: this config is latency/launch bound by construction"
    return out


# ---- our arm -----------------------------------------------------------------------------------------------------------

def run_e2e(args, device, x_host, step_fn, n_out_rows, edges_per_layer, barrier=None, passes=2):
    """Host-to-host throughput of the same step: every step copies its input features from pinned host memory and lands
    every output of the step in pinned host memory.  The three engines are pipelined the way a serving loop would do it:
    H2D of step i+1 and D2H of step i's outputs run on their own streams while step i / i+1 compute; device and host
    buffers are double buffered and every dependency is an event.  All copies are inside the timed region.
    (n_out_rows is kept for the callers' bookkeeping; host output buffers take the shapes the step returns.)"""
    s_in, s_out = torch.cuda.Stream(device), torch.cuda.Stream(device)
    main = torch.cuda.current_stream(device)
    x_dev = [torch.empty(x_host.shape, dtype=torch.float32, device=device) for _ in range(2)]
    probe = step_fn(x_dev[0].copy_(x_host))
    outs = [[torch.empty(tuple(o.shape), dtype=torch.float32).pin_memory() for o in probe] for _ in range(2)]
    d2h = sum(o.numel() * 4 for o in probe)
    del probe
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]       # x_dev[slot] no longer read by compute
    ev_out_done = [torch.cuda.Event() for _ in range(2)]   # host output slot drained (previous use)

    def submit(i):
        slot = i & 1
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_free[slot])
            x_dev[slot].copy_(x_host, non_blocking=True)
            ev_in[slot].record(s_in)
        main.wait_event(ev_in[slot])
        results = step_fn(x_dev[slot])                       # public layer API
        ev_free[slot].record(main)
        ev_done = torch.cuda.Event()
        ev_done.record(main)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_done)
            s_out.wait_event(ev_out_done[slot])
            for host, res in zip(outs[slot], results):
                host.copy_(res, non_blocking=True)
            ev_out_done[slot].record(s_out)
        for res in results:
            res.record_stream(s_out)

    for slot in range(2):
        ev_free[slot].record(main)
        ev_out_done[slot].record(s_out)
    for i in range(2):
        submit(i)
    torch.cuda.synchronize(device)
    if barrier is not None:
        barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(main)
    for i in range(args.steps):
        submit(i)
    main.wait_stream(s_out)                                  # the last outputs have landed on the host
    main.wait_stream(s_in)
    t1.record(main)
    torch.cuda.synchronize(device)
    ms = t0.elapsed_time(t1) / args.steps
    return {"value": passes * edges_per_layer / (ms * 1e-3), "unit": "edges/s", "ms_per_step": ms,
            "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": d2h,
            "pipelining": "H2D / compute / D2H on three streams, double buffered, all inside the timed region"}


TIMED_CALLS = ("tfgk_gat_fused_f32", "tfgk_spmm_f32", "tfgk_gemm_f32", "tfgk_gemm_proj_f32")
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of round 2 (constants, NOT
# live counters): profiles/r2_ncu_full_headline_kernels.json; only valid for the full-size products-shape graph
NCU_TRAFFIC = {"gat": 128185916000, "spmm_d128": 63372534000}


def build_workload(args, tfg, device):
    """Graph, features, layers and the step function of args.config on one GPU.  Returns a dict with: x_host, step,
    outputs (a name for each array the step returns), E, passes, kernels = {family: (abi call, algorithmic bytes per
    step, description)}."""
    cfg, n, pairs = config_sizes(args)
    F = cfg["features"]
    kind = cfg["kind"]
    edge_index = make_graph_device(n, pairs, 0, device)
    E = edge_index.shape[1]
    gen = torch.Generator(device="cpu"); gen.manual_seed(1)
    if kind == "gcn2":       # Cora-like bag of words: ~18 non-zeros per row, row-normalised (datasets/planetoid.py:88-92)
        x_host = (torch.rand((n, F), generator=gen) < 18.0 / F).float()
        x_host = (x_host / x_host.sum(1, keepdim=True).clamp(min=1.0)).pin_memory()
    else:
        x_host = torch.randn((n, F), generator=gen, dtype=torch.float32).pin_memory()
    x = x_host.to(device)
    graph = tfg.Graph(x, edge_index)
    e_loop = E + n
    spmm_bytes = lambda d, e, w: e * (4 * d + 4 + (4 if w else 0)) + n * (4 * d + 8)      # noqa: E731  DESIGN.md K1
    gat_bytes = e_loop * (4 * UNITS + 4 * UNITS + 4) + n * (4 * UNITS + 4 * UNITS + 8)       # DESIGN.md K3
    proj_bytes = lambda cols: n * F * 4 + n * cols * 4                                       # noqa: E731
    kernels = {}
    if kind in ("gcn+gat", "gcn", "gat"):
        layers = []
        if "gcn" in kind:
            gcn = tfg.layers.GCN(UNITS, activation=tfg.nn.relu, seed=2)
            gcn.build_cache_for_graph(graph)                   # normalised adjacency + CSR (one-off, untimed)
            layers.append(lambda xd: gcn([xd, graph.edge_index, graph.edge_weight], cache=graph.cache))
            kernels["gcn_spmm"] = ("tfgk_spmm_f32", spmm_bytes(UNITS, e_loop, True), "spmm_gather4_kernel<0,3> (tfgk_spmm_f32)",
                                   NCU_TRAFFIC["spmm_d128"] if args.config == "headline" and args.scale == 1.0 else None)
            kernels["gcn_projection"] = ("tfgk_gemm_f32", proj_bytes(UNITS), "gemm_proj_ts_kernel<STAGES> reached through tfgk_gemm_f32", None)
        if "gat" in kind:
            gat = tfg.layers.GAT(UNITS, num_heads=HEADS, activation=tfg.nn.relu, seed=3)
            layers.append(lambda xd: gat([xd, graph.edge_index], cache=graph.cache))
            kernels["gat_fused"] = ("tfgk_gat_fused_f32", gat_bytes, "gat_gather4_kernel<2> (tfgk_gat_fused_f32)",
                                    NCU_TRAFFIC["gat"] if args.config == "headline" and args.scale == 1.0 else None)
            kernels["gat_projections"] = ("tfgk_gemm_proj_f32", proj_bytes(3 * UNITS),
                                          "gemm_proj_ts_kernel<STAGES>, Q|K|V in one launch (tfgk_gemm_proj_f32)", None)
        step = lambda xd: tuple(f(xd) for f in layers)     # noqa: E731
        outputs = tuple(k for k in ("gcn", "gat") if k in kind)
        passes = len(layers)
    elif kind == "gcn2":
        # sparse bag-of-words features like demo_gcn.py feeds them (tf.SparseTensor, gcn.py:269-272): the pattern is fixed,
        # the values are the per-step input that travels from the host
        nz = torch.nonzero(x_host, as_tuple=True)
        pattern = tfg.SparseMatrix(torch.stack(nz).to(torch.int32).to(device), x_host[nz].to(device), [n, F])
        pattern.csr                                            # feature-matrix CSR (one-off, like the adjacency cache)
        x_host = x_host[nz].contiguous().pin_memory()
        x = x_host.to(device)
        l1 = tfg.layers.GCN(16, activation=tfg.nn.relu, seed=2)
        l2 = tfg.layers.GCN(7, seed=3)
        l1.build_cache_for_graph(graph)
        step = lambda xd: (l2([l1([pattern.with_value(xd), graph.edge_index, graph.edge_weight], cache=graph.cache),     # noqa: E731
                               graph.edge_index, graph.edge_weight], cache=graph.cache),)
        outputs = ("gcn2",)
        nnz = int(x_host.numel())
        kernels["gcn_spmm"] = ("tfgk_spmm_f32", spmm_bytes(16, e_loop, True) + spmm_bytes(7, e_loop, True)
                               + nnz * (4 * 16 + 8) + n * (4 * 16 + 8),
                               "spmm kernels: sparse x @ W (D=16), norm(A) @ h at D=16 and D=7 (tfgk_spmm_f32)", None)
        passes = 2
    elif kind == "sage_train":
        layer = tfg.layers.MeanGraphSage(2 * UNITS, activation=tfg.nn.relu, concat=True, seed=2, trainable=True)
        g = torch.randn((n, 2 * UNITS), generator=torch.Generator(device="cpu").manual_seed(9)).to(device)

        def step(xd):
            xg = xd.detach().requires_grad_(True)
            layer.zero_grad(set_to_none=True)
            out = layer([xg, graph.edge_index])
            loss = (out * g).sum()
            loss.backward()
            return (loss.detach().reshape(1), xg.grad)
        outputs = ("loss", "x_grad")
        # forward mean aggregation (unweighted) + backward aggregation on the transposed CSR (weights 1/deg)
        kernels["sage_spmm"] = ("tfgk_spmm_f32", spmm_bytes(F, E, False) + spmm_bytes(F, E, True),
                                "spmm kernels at D=100, forward + transposed backward (tfgk_spmm_f32)", None)
        kernels["sage_dense"] = ("tfgk_gemm_f32", 0, "forward projections, dX and split-K dW GEMMs (tfgk_gemm_f32)", None)
        passes = 1
    else:
        raise ValueError(kind)
    return {"x_host": x_host, "x": x, "step": step, "outputs": outputs, "E": E, "n": n, "passes": passes, "kernels": kernels,
            "graph": graph}


DUMP_BYTES = 64 * 1000 * 1000


def dump_outputs(directory, names, outputs):
    """Writes each output of one step as <directory>/<name>.npy in float32.  An output whose data exceeds its equal share
    of DUMP_BYTES (less room for the .npy header) is stored as a fixed sample of its rows: the sorted result of
    np.random.RandomState(0).choice(rows, k, replace=False), the same rows for every build at the same arguments."""
    os.makedirs(directory, exist_ok=True)
    share = DUMP_BYTES // len(outputs) - 4096
    for name, out in zip(names, outputs):
        out = out.detach()
        keep = share // (out[0].numel() * 4)
        if keep < out.shape[0]:
            rows = np.sort(np.random.RandomState(0).choice(out.shape[0], keep, replace=False))
            out = out[torch.from_numpy(rows).to(out.device)]
        np.save(os.path.join(directory, name + ".npy"), out.to(torch.float32).cpu().numpy())


def run_ours(args, rank, world, local_rank):
    import tf_geometric_b200 as tfg
    from tf_geometric_b200 import _ffi

    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    cfg = CONFIGS[args.config]
    if args.dump_outputs and (world > 1 or cfg["kind"] == "gcn_partitioned"):
        raise SystemExit("--dump-outputs is implemented for the single-GPU configs only")
    if world > 1 or cfg["kind"] == "gcn_partitioned":
        os.environ.setdefault("NCCL_DEBUG", "WARN")     # keep NCCL's version banner off stdout: one JSON line only
        import torch.distributed as dist
        if world == 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", device_id=device, rank=rank, world_size=world)
        if cfg["kind"] == "gcn_partitioned":
            from tf_geometric_b200.dist import bench_papers
            return bench_papers(args, rank, world, device, config_metric(args), workload_config(args, world))
        if args.config != "headline":
            raise SystemExit("--config {} is a single-GPU workload (BASELINE.json configs); use --gpus 1".format(args.config))
        from tf_geometric_b200.dist import bench_partitioned
        return bench_partitioned(args, rank, world, device, METRIC, workload_config(args, world))

    torch.cuda.synchronize()
    t_cache = time.perf_counter()
    wl = build_workload(args, tfg, device)
    step, x, E, n = wl["step"], wl["x"], wl["E"], wl["n"]
    step(x)                                                # builds the self-looped CSR + weights
    torch.cuda.synchronize()
    t_cache = time.perf_counter() - t_cache

    # ---- device-resident timing ("value") ----
    for _ in range(max(args.warmup, 3)):
        step(x)
    torch.cuda.synchronize()
    trace = _ffi.CallTrace(timed=TIMED_CALLS)
    _ffi.set_trace(trace)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(args.steps):
        outputs = None            # the previous step's outputs are freed before the next step allocates, as when discarded
        outputs = step(x)
    ev[1].record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    _ffi.set_trace(None)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, wl["outputs"], outputs)
    del outputs
    ms_step = ev[0].elapsed_time(ev[1]) / args.steps
    value = wl["passes"] * E / (ms_step * 1e-3)

    call_ms = {name: float(np.sum(trace.elapsed_ms(name))) / args.steps for name in TIMED_CALLS}
    call_n = {name: trace.counts.get(name, 0) / args.steps for name in TIMED_CALLS}
    # one kernel launch per call on the forward paths (no hub rows in these graphs); the training config's split-K dW and
    # column sums launch more, so this is a lower bound there
    launches = sum(trace.counts.get(k, 0) for k in TIMED_CALLS)
    peak, peak_src = measured_peak_gbs()
    fams = {}
    for fam, (call, nbytes, desc, traffic) in wl["kernels"].items():
        ms = call_ms[call]
        fams[fam] = {"kernel": desc, "ms_per_step": ms, "launches_per_step": call_n[call], "algorithmic_bytes_per_step": nbytes,
                     "achieved": (nbytes / (ms * 1e-3) / 1e9) if ms > 0 and nbytes else None,
                     "frac": (nbytes / (ms * 1e-3) / 1e9 / peak) if ms > 0 and nbytes else None, "traffic": traffic}
    dominant = max((f for f in fams if fams[f]["algorithmic_bytes_per_step"]), key=lambda f: fams[f]["ms_per_step"])
    d = fams[dominant]
    roofline = {"bound": "hbm", "kernel": d["kernel"], "achieved": d["achieved"], "peak": peak, "unit": "GB/s",
                "frac": d["frac"], "traffic": d["traffic"],
                "traffic_source": ("constant copied from the committed ncu --set full capture of round 2 "
                                   "(profiles/r2_ncu_full_headline_kernels.json), not measured in this run") if d["traffic"] else None,
                "peak_source": peak_src, "algorithmic_bytes": d["algorithmic_bytes_per_step"] / max(d["launches_per_step"], 1),
                "kernel_ms": d["ms_per_step"] / max(d["launches_per_step"], 1),
                "launches_per_step": d["launches_per_step"],
                "other_kernels": {f: v for f, v in fams.items() if f != dominant}}

    # ---- end to end: host buffers in, host buffers out, through the same public API ----
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, device, wl["x_host"], step, n, E, passes=wl["passes"])

    cpu_base = None
    if not args.no_cpu_baseline:
        _, _, pairs = config_sizes(args)
        args.cpu_sample_div = cpu_sample_div(args, 2, budget_s=40.0)
        ns = max(n // args.cpu_sample_div, min(n, 1000))
        ps = max(pairs // args.cpu_sample_div, min(pairs, 1000))
        res = cpu_reference(cfg["kind"], ns, ps, cfg["features"], steps=1, warmup=1)
        cpu_base = {"value": res["edges_per_s"], "unit": "edges/s", "cores": res["cores"], "kind": "port",
                    "sample": "same generator and layer shapes at 1/{} scale ({} nodes, {} directed edges), 1 step after "
                              "1 warm-up, op-for-op torch-CPU port of the reference op sequence, {} threads (best of a sweep) "
                              "of {} host cores, {}".format(args.cpu_sample_div, res["nodes"], res["edges"], res["cores"],
                                                            res["host_cores"], cpu_model_name()),
                    "thread_sweep": res["thread_sweep_s_per_step_quarter_sample"]}

    line = {"metric": config_metric(args), "value": value, "unit": "edges/s", "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, 1),
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "launches_per_step": launches / args.steps,
            "roofline": roofline, "cpu_baseline": cpu_base,
            "breakdown_ms": dict({f: v["ms_per_step"] for f, v in fams.items()}, cache_build_s=t_cache)}
    emit(line)


class StdoutToStderr(object):
    """Routes file descriptor 1 to stderr while the benchmark runs (NCCL / library banners must not pollute the ONE JSON
    line the driver parses) and restores it for the final print."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def _result_lines():
    # bench.py runs as __main__ and is also imported as `bench` by tf_geometric_b200.dist: share the list through `sys`
    if not hasattr(sys, "_tfgk_bench_lines"):
        sys._tfgk_bench_lines = []
    return sys._tfgk_bench_lines


def emit(line):
    """Collect the JSON line; main() prints it once stdout is restored."""
    _result_lines().append(json.dumps(line))


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    with StdoutToStderr():
        if args.impl == "reference":
            if args.dump_outputs:
                raise SystemExit("--dump-outputs writes the outputs of --impl ours")
            run_reference(args, rank, world)
        else:
            if not torch.cuda.is_available():
                raise SystemExit("bench.py needs a CUDA device for --impl ours (there is no CPU fallback); "
                                 "use --impl reference for the CPU arm")
            run_ours(args, rank, world, local_rank)
    for line in _result_lines():
        print(line, flush=True)


if __name__ == "__main__":
    main()
