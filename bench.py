#!/usr/bin/env python
"""bench.py - GConv-Adapter forward + backward throughput (edges/s) on B200.

    python bench.py --gpus N --steps K --warmup W [--workload arxiv|products|pubmed|cora|molecules]
    python bench.py --impl reference ...        # the CPU oracle timed on the host cores
    python bench.py ... --dump-outputs DIR      # also write the last timed step's outputs as DIR/<name>.npy

A step = one adapter forward + backward over the workload graph.  Default workload (N = 1) is
BASELINE.json configs[3], the ogbn-arxiv-shaped graph the metric is quoted on (169,343 nodes,
1,166,243 edges, hidden 256, rank 16), synthetic data, random weights.  For N > 1 the node rows are
partitioned over the ranks and the r-wide activations are all-gathered (strong scaling).

Prints ONE JSON line (rank 0) with the keys of the driver contract plus `roofline`, `cpu_baseline`,
`e2e`, `clocks`, `gpu_launches`, `phases` and `step_roofline`.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)

import torch  # noqa: E402

METRIC = "gconv_adapter_fwd_bwd_edges_per_sec"
UNIT = "edges/s"
DUMP_BYTES = 64 << 20               # --dump-outputs: upper bound of all arrays written


# ---------------------------------------------------------------------------------------------
def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, help="arxiv (default) | products | pubmed | cora | molecules")
    ap.add_argument("--power-law", action="store_true", help="hub-heavy degree distribution instead of uniform")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--single-adapter", action="store_true",
                    help="molecules / pubmed: ONE adapter fwd+bwd on the workload's graph instead of the host step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (output, input and parameter gradients; "
                         "a fixed sample of rows when larger than %d MB) as DIR/<name>.npy" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs: single-GPU runs of --impl ours only")
    return args


def sample_rows(t, max_rows):
    """A copy of t[rows] for a fixed, seeded sample of at most max_rows rows, kept in row order (all rows when they fit)."""
    if t.size(0) <= max_rows:
        return t.detach().clone()
    rows = torch.randperm(t.size(0), generator=torch.Generator().manual_seed(0))[:max_rows].sort().values
    return t.detach().index_select(0, rows.to(t.device))


def write_outputs(out_dir, arrays):
    """--dump-outputs: DIR/<name>.npy per array, float32 or float64, at most DUMP_BYTES in all."""
    import numpy as np
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    for k, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"--dump-outputs: {k} is {a.dtype}, not float32 / float64")
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def workload(args):
    from gconv_adapter_b200.graphs.synthetic import SHAPES, make_graph
    name = args.workload or "arxiv"
    ei, n = make_graph(name, seed=0, power_law=args.power_law)
    s = SHAPES[name]
    return name, ei, n, s.hidden, s.rank


def workload_string(name, n, e, d, r, power_law=False):
    """config.workload, byte-identical in both arms (ours / --impl reference) so that the driver sees one configuration."""
    return f"{name}-shaped: N={n} E={e} hidden={d} rank={r}" + (" power-law" if power_law else "")


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(n, e_prime, d, r):
    """Minimal HBM bytes per launch of each kernel and of the whole fwd+bwd (DESIGN.md section 5;
    SURVEY.md section 8d: A_min = 28 N d + 52 N r + 16 E' + 32 N)."""
    nd, nr = 4 * n * d, 4 * n * r
    idx = 4 * e_prime + 4 * n          # colidx + rowptr
    dis = 4 * n
    per = {
        "project_fwd": nd + nr + dis,                 # X -> P'
        "hop_fwd": 2 * nr + idx + dis,                # P' -> Z'
        "hop_expand_fwd": 2 * nr + idx + dis + 2 * nd,  # Z' -> H2 ; X -> Y
        "project_bwd": nd + nr + dis,                 # gY -> gH2'
        "wgrad_up": nd + nr,                          # gY, H2 -> gWu partials
        "bwd_up_fused": nd + 2 * nr + dis,            # gY (once) -> gH2' and gWu partials (project_bwd + wgrad_up)
        "hop_bwd": 3 * nr + idx + dis,                # gH2', Z' -> gH1'
        "hop_expand_bwd": 2 * nr + idx + dis + 2 * nd,  # gH1' -> gP ; gY -> gX
        "wgrad_down": 2 * nd + nr,                    # X, gY(dot), gP -> gWd partials
        "finalize": 0,
        # split K3 (operand >> L2, e.g. products-shaped): plain hop kernel + expand-only kernel
        "hop_plain_fwd": 2 * nr + idx + dis, "hop_plain_bwd": 2 * nr + idx + dis,
        "expand_fwd": nr + 2 * nd, "expand_bwd": nr + 2 * nd,
        "bwd_up": nd + 2 * nr + dis,                  # gY (once) -> gH2' and the gWu / gbu partials
        "expand_wgrad_bwd": 3 * nd + nr,              # gY, X (once each), gP -> gX, gWd partials, <gY, X>
    }
    # small graphs: ONE cooperative kernel per direction (gca_small.cu) = the sum of the phases it replaces
    per["small_fwd"] = per["project_fwd"] + per["hop_fwd"] + per["hop_expand_fwd"]
    per["small_bwd"] = per["bwd_up"] + per["hop_bwd"] + per["hop_plain_bwd"] + per["expand_wgrad_bwd"]
    total = 28 * n * d + 52 * n * r + 16 * e_prime + 32 * n
    return per, total


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region and an identical
    1 s continuation of it run (the timed region alone is a few tens of ms)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_step_seconds(ei, n, d, r, params, x, g_out, steps, warmup, threads=None):
    """CPU baseline: the restated reference module (oracle/pyg_restated.py), fwd + bwd, fp32."""
    from oracle.pyg_restated import GConvAdapterRef
    if threads:
        torch.set_num_threads(threads)
    m = GConvAdapterRef(d, r, learnable_scalar=True)
    sd = m.state_dict()
    with torch.no_grad():
        for k, v in params.items():
            sd[k].copy_(v)
    times = []
    for it in range(warmup + steps):
        for p in m.parameters():
            p.grad = None
        xx = x.clone().requires_grad_(True)
        t0 = time.perf_counter()
        y = m(xx, ei)
        y.backward(g_out)
        t1 = time.perf_counter()
        if it >= warmup:
            times.append(t1 - t0)
    return times


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def products_subrecord(lib, dev, steps=8):
    """BASELINE.json configs[4] (products-shaped, hidden 256, rank 32) on this GPU count, measured in the same run as the
    headline so that the 1/2/4/8 curve of the second partitioned config is driver-observed (the N > 1 legs carry the same key)."""
    from gconv_adapter_b200 import GConvAdapter, GraphCache
    from gconv_adapter_b200.graphs.synthetic import SHAPES, input_rows, make_graph, make_inputs
    ei, n = make_graph("products", seed=0)
    s = SHAPES["products"]
    d, r, e = s.hidden, s.rank, ei.size(1)
    _, _, params = make_inputs(8, d, r, seed=0)
    m = GConvAdapter(d, r, learnable_scalar=True)
    sd = m.state_dict()
    with torch.no_grad():
        for k, v in params.items():
            sd[k].copy_(v)
    m = m.to(dev)
    m.graph_cache = GraphCache()
    eid = ei.to(dev)
    del ei
    xd, gd = input_rows(0, n, d, 1234, dev)
    xd.requires_grad_(True)
    e_prime = m.graph_for(eid, n).nnz

    def step():
        xd.grad = None
        for p in m.parameters():
            p.grad = None
        m(xd, eid).backward(gd)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        step()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / steps
    lib.gca_profile_enable(1)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.gca_profile_report(buf, len(buf))
    lib.gca_profile_enable(0)
    prof = json.loads(buf.value.decode())
    per, a_min = algorithmic_bytes(n, e_prime, d, r)
    a_gather = a_min - 16 * n * r + 16 * r * e_prime
    peak, _ = peaks()
    rec = {"workload": workload_string("products", n, e, d, r), "ms_per_step": ms, "value": e / (ms / 1e3), "unit": UNIT, "n_gpus": 1,
           "step_alg_bytes": a_min, "frac_of_measured_peak": round(a_min / 1e6 / ms / peak, 4),
           "gather_bound_bytes": a_gather, "frac_of_measured_peak_on_gather_bound": round(a_gather / 1e6 / ms / peak, 4),
           "phases_ms": {k: round(v["ms"] / max(v["launches"], 1), 4) for k, v in prof.items()},
           "variants": {k: v["variant"] for k, v in prof.items() if v["variant"]}}
    # dominant kernel of this workload: algorithmic bytes against its measured time, and the DRAM bytes ncu saw for it
    dom = max(prof, key=lambda k: prof[k]["ms"])
    dom_ms = prof[dom]["ms"] / max(prof[dom]["launches"], 1)
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("products", {}).get(dom)
    except Exception:
        traffic = None
    rec["roofline"] = {"bound": "hbm", "kernel": dom, "ms_per_launch": round(dom_ms, 5), "alg_bytes_per_launch": per.get(dom, 0),
                       "achieved": round(per.get(dom, 0) / 1e6 / dom_ms, 1), "peak": peak, "unit": "GB/s",
                       "frac": round(per.get(dom, 0) / 1e6 / dom_ms / peak, 4), "traffic": traffic,
                       "traffic_GBs": round(traffic / 1e6 / dom_ms, 1) if traffic else None,
                       "note": "r-wide gather on a random graph whose operand is 2.5x the L2: DRAM traffic (ncu) is ~10x the "
                               "algorithmic bytes and moves at ~90% of the measured peak"}
    del m, eid, xd, gd
    torch.cuda.empty_cache()
    return rec


# ---------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gconv_adapter_b200.graphs.synthetic import make_inputs
    name, ei, n, d, r = workload(args)
    x, g_out, params = make_inputs(n, d, r, seed=0)
    cores = os.cpu_count() or 1
    times = oracle_step_seconds(ei, n, d, r, params, x, g_out, args.steps, args.warmup, threads=cores)
    e = ei.size(1)
    total = sum(times)
    val = e * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(name, n, e, d, r, args.power_law), "inputs": "host memory (CPU run)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"full {name}-shaped fwd+bwd x {len(times)} steps; restated PyG GCNConv op sequence "
                                   f"(torch-geometric is not installable here), {cpu_model()}"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def run_host_workload(args, lib, dev):
    """BASELINE.json configs[1] / configs[2] as they are stated, through the insertion hooks of the reference's host models
    (tests/hosts.py reproduces the hooks around stand-in backbones; the backbones themselves are out of scope):

      molecules: 5-layer GIN-shaped host (hidden 300), post-insertion GConv-Adapter (rank 16) in every layer, a batch of 32
                 molecules per step and a NEW edge_index every step - the graph structure is rebuilt inside the timed region
                 (one K0 launch per step, shared by the five adapters through the graph cache);
      pubmed:    NodeFormer-shaped transductive host (hidden 64, x as [1, N, H]), sequential pre + post adapters x 2 layers on
                 the static PubMed-shaped graph (19,717 nodes, 88,648 edges + one pre-inserted self loop per node).

    value = adapter edges per second = E x (adapter calls per step) / step time of the WHOLE host step (backbone stand-ins,
    loss and autograd included); `adapter_only` is the same adapters timed alone."""
    import functools
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from hosts import MolecularGraphPredictionHost, TransductiveHost          # noqa: PLC0415
    from gconv_adapter_b200 import GConvAdapter, GLOBAL_GRAPH_CACHE
    from gconv_adapter_b200.graphs.synthetic import make_graph, molecule_batch
    name = args.workload
    torch.manual_seed(0)
    if name == "molecules":
        d, r, layers, calls = 300, 16, 5, 5
        host = MolecularGraphPredictionHost(layers, d, 1)
        host.add_adapter(functools.partial(GConvAdapter, bottleneck_size=r, learnable_scalar=True), ["post"], "sequential")
        for a in host.modules():
            if isinstance(a, GConvAdapter):
                a.validate_edge_index = "lazy"      # a new graph every step: no stream synchronisation per build
        pool = []
        for i in range(16):                       # 16 distinct batches > graph-cache capacity (8): every step is a cache miss
            ei, batch, n = molecule_batch(batch_size=32, seed=100 + i)
            g = torch.Generator().manual_seed(i)
            x = torch.stack([torch.randint(0, 120, (n,), generator=g), torch.randint(0, 3, (n,), generator=g)], 1)
            ea = torch.stack([torch.randint(0, 4, (ei.size(1),), generator=g), torch.randint(0, 3, (ei.size(1),), generator=g)], 1)
            pool.append((x, ei, ea, batch))
        e_step = sum(b[1].size(1) for b in pool) / len(pool)
        n_step = sum(b[0].size(0) for b in pool) / len(pool)
        dev_pool = [tuple(t.to(dev) for t in b) for b in pool]
        host_pool = [tuple(t.pin_memory() for t in b) for b in pool]
        graph_note = "new edge_index every step: structure rebuilt in the timed region (16 batches cycle through a cache of 8), node ids validated lazily (no sync)"

        def run(batch):
            x, ei, ea, bt = batch
            return host(x, ei, ea, bt)
    else:
        d, r, layers, calls = 64, 16, 2, 4
        ei, n = make_graph("pubmed", seed=0)
        host = TransductiveHost("nodeformer", 500, d, 3, num_layers=layers)
        host.add_adapter(functools.partial(GConvAdapter, bottleneck_size=r, learnable_scalar=True), ["pre", "post"], "sequential")
        feats = torch.randn(n, 500)
        dev_pool = [(feats.to(dev), ei.to(dev))]
        host_pool = [(feats.pin_memory(), ei.pin_memory())]
        e_step, n_step = ei.size(1), n
        graph_note = "static graph, structure cached across layers, positions and steps"

        def run(batch):
            x, eidx = batch
            return host(x, [eidx])
    host = host.to(dev).train()
    params = [p for p in host.parameters() if p.requires_grad]

    def step(batch):
        for p in params:
            p.grad = None
        out = run(batch)
        loss = out.square().sum()
        loss.backward()
        return loss

    for i in range(max(args.warmup, 3) + len(dev_pool)):
        step(dev_pool[i % len(dev_pool)])
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = lib.gca_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0 = time.perf_counter()
    t0.record()
    for i in range(args.steps):
        loss = step(dev_pool[i % len(dev_pool)])
    t1.record()
    torch.cuda.synchronize()
    ms_step = max(t0.elapsed_time(t1), 1e3 * (time.perf_counter() - c0)) / args.steps
    launches = lib.gca_launch_count() - l0
    dumped = None
    if args.dump_outputs:
        dumped = {"loss": loss.detach().clone()}
        dumped.update({"grad_" + k: p.grad.clone() for k, p in host.named_parameters() if p.grad is not None})
    t_end = time.perf_counter() + 1.0
    i = 0
    while time.perf_counter() < t_end:
        step(dev_pool[i % len(dev_pool)])
        i += 1
    torch.cuda.synchronize()
    clocks = sampler.stop()

    # e2e: every step's inputs come from pinned host memory, the loss goes back
    c0 = time.perf_counter()
    for i in range(args.steps):
        batch = tuple(t.to(dev, non_blocking=True) for t in host_pool[i % len(host_pool)])
        step(batch).item()
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - c0) / args.steps
    h2d = sum(t.numel() * t.element_size() for t in host_pool[0])

    # the adapters alone (same shapes, same number of calls, structure rebuilt per step for molecules)
    adapters = [m for m in host.modules() if isinstance(m, GConvAdapter)]
    if name == "molecules":
        xs = [torch.randn(b[0].size(0), d, device=dev, requires_grad=True) for b in dev_pool]
    else:
        xs = [torch.randn(1, n, d, device=dev, requires_grad=True)]

    def adapter_step(i):
        b = dev_pool[i % len(dev_pool)]
        x = xs[i % len(xs)]
        eidx = b[1]
        h = x
        for a in adapters:
            h = a(h, eidx)
        h.sum().backward()

    for i in range(len(dev_pool) + 3):
        adapter_step(i)
    torch.cuda.synchronize()
    c0 = time.perf_counter()
    t0.record()
    for i in range(args.steps):
        adapter_step(i)
    t1.record()
    torch.cuda.synchronize()
    ad_ms = max(t0.elapsed_time(t1), 1e3 * (time.perf_counter() - c0)) / args.steps

    graphed_ms = None
    if name != "molecules":
        # static graph: forward and backward of every adapter as one CUDA graph each (gconv_adapter_b200.graphed_adapter)
        from gconv_adapter_b200 import graphed_adapter
        fs = [graphed_adapter(a, xs[0], dev_pool[0][1]) for a in adapters]

        def graphed_step():
            h = xs[0]
            for f in fs:
                h = f(h)
            h.sum().backward()

        for _ in range(5):
            graphed_step()
        torch.cuda.synchronize()
        c0 = time.perf_counter()
        t0.record()
        for _ in range(args.steps):
            graphed_step()
        t1.record()
        torch.cuda.synchronize()
        graphed_ms = max(t0.elapsed_time(t1), 1e3 * (time.perf_counter() - c0)) / args.steps

    line = {
        "metric": METRIC, "value": e_step * calls / (ms_step / 1e3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{name}: host step with {calls} adapter calls, N~{int(n_step)} E~{int(e_step)} hidden={d} rank={r}",
                   "host": "tests/hosts.py (reference insertion hooks around stand-in backbones)", "graph": graph_note,
                   "l2": "working set fits L2; no flush (latency-bound config: host issue time is what is measured)",
                   "parallelism": "1 GPU"},
        "adapter_only": {"ms_per_step": ad_ms, "adapter_calls_per_step": calls, "ms_per_adapter_fwd_bwd": ad_ms / calls,
                         "value": e_step * calls / (ad_ms / 1e3), "unit": UNIT,
                         "cuda_graph_ms_per_adapter_fwd_bwd": (graphed_ms / calls) if graphed_ms else None},
        "e2e": {"value": e_step * calls / (e2e_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches), "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": None, "peak": peaks()[0], "unit": "GB/s", "frac": None, "traffic": None,
                     "note": "launch / host-issue bound: a few MB per step; see ms_per_adapter_fwd_bwd"},
        "cpu_baseline": None,
    }
    GLOBAL_GRAPH_CACHE.clear()
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    print(json.dumps(line))


def run_ours(args):
    if args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1:
        from gconv_adapter_b200.partition_bench import run_partitioned   # multi-GPU leg
        return run_partitioned(args, METRIC, UNIT)
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU oracle)")
    from gconv_adapter_b200 import GConvAdapter, GraphCache, _cabi
    from gconv_adapter_b200.graphs.synthetic import make_inputs
    lib = _cabi.load()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    if args.workload in ("molecules", "pubmed") and not args.single_adapter:
        return run_host_workload(args, lib, dev)
    name, ei, n, d, r = workload(args)
    e = ei.size(1)
    x, g_out, params = make_inputs(n, d, r, seed=0)
    m = GConvAdapter(d, r, learnable_scalar=True)
    sd = m.state_dict()
    with torch.no_grad():
        for k, v in params.items():
            sd[k].copy_(v)
    m = m.to(dev)
    m.graph_cache = GraphCache()
    eid = ei.to(dev)
    xd = x.to(dev).requires_grad_(True)
    gd = g_out.to(dev)
    graph = m.graph_for(eid, n)                 # built once; the timed steps reuse it (static graph)
    e_prime = graph.nnz
    holder = {}

    def step():
        xd.grad = None
        for p in m.parameters():
            p.grad = None
        y = m(xd, eid)
        y.backward(gd)
        holder["y"] = y.detach()                # what a caller receives, kept for --dump-outputs (warm-up included)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = lib.gca_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(args.steps):
        step()
    t1.record()
    torch.cuda.synchronize()
    ms_step = t0.elapsed_time(t1) / args.steps
    launches = lib.gca_launch_count() - l0
    dumped = None
    if args.dump_outputs:
        rows = (DUMP_BYTES // 2) // (2 * 4 * d)     # Y and gX share half the budget; the parameter gradients are small
        dumped = {"y": sample_rows(holder["y"], rows), "grad_x": sample_rows(xd.grad, rows)}
        dumped.update({"grad_" + k: p.grad.clone() for k, p in m.named_parameters()})
    # keep the GPU under the same load for ~1 s so nvidia-smi (100 ms period) sees the clocks of this kernel mix
    t_end = time.perf_counter() + 1.0
    while time.perf_counter() < t_end:
        for _ in range(10):
            step()
        torch.cuda.synchronize()
    clocks = sampler.stop()

    # ---- small graphs are host-bound in eager mode: the same step (forward + backward on static tensors) captured in ONE
    # CUDA graph and replayed shows what the kernels cost (reported next to, never instead of, the eager number) ----
    graph_ms = None
    if n <= 65536 and os.environ.get("GCA_BENCH_NO_GRAPH", "0") != "1":
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            cg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(cg):
                step()
            for _ in range(5):
                cg.replay()
            torch.cuda.synchronize()
            t0.record()
            for _ in range(args.steps):
                cg.replay()
            t1.record()
            torch.cuda.synchronize()
            graph_ms = t0.elapsed_time(t1) / args.steps
            del cg
        except Exception as ex:      # noqa: BLE001 - a failed capture only drops the extra number
            print(f"CUDA-graph capture of the step failed ({type(ex).__name__}: {ex})", file=sys.stderr)
            torch.cuda.synchronize()
        for p in m.parameters():     # back to eager-owned gradients
            p.grad = None
        xd.grad = None

    # ---- per-kernel device times (CUDA events on the launching stream, inside libgca) ----
    lib.gca_profile_enable(1)
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.gca_profile_report(buf, len(buf))
    lib.gca_profile_enable(0)
    prof = json.loads(buf.value.decode())
    per_bytes, a_min = algorithmic_bytes(n, e_prime, d, r)
    peak, peak_src = peaks()
    phases = {}
    for k, v in prof.items():
        avg_ms = v["ms"] / max(v["launches"], 1)
        b = per_bytes.get(k, 0)
        phases[k] = {"ms": round(avg_ms, 5), "launches_per_step": v["launches"] / args.steps,
                     "alg_MB": round(b / 1e6, 2), "GBs": round(b / 1e6 / avg_ms, 1) if avg_ms > 0 else None}
    dom = max(prof, key=lambda k: prof[k]["ms"])
    dom_ms = prof[dom]["ms"] / prof[dom]["launches"]
    achieved = per_bytes.get(dom, 0) / 1e6 / dom_ms
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")     # per-launch dram bytes from the ncu --set full capture
    if os.path.isfile(tpath):
        try:
            traffic = json.load(open(tpath)).get(name, {}).get(dom)
        except Exception:
            traffic = None
    kernel_ms = sum(v["ms"] for v in prof.values()) / args.steps
    roofline = {"bound": "hbm", "kernel": dom, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": peak_src,
                "alg_bytes_per_launch": per_bytes.get(dom, 0), "ms_per_launch": round(dom_ms, 5),
                "share_of_step": round(prof[dom]["ms"] / args.steps / kernel_ms, 3)}
    step_gbs = a_min / 1e6 / ms_step
    # A_gather: every neighbour row fetched once per edge (no cache reuse) - the realistic bound when the r-wide
    # operand (4 N r bytes) exceeds L2, e.g. products-shaped (SURVEY.md section 8d)
    a_gather = a_min - 16 * n * r + 16 * r * e_prime
    step_roofline = {"alg_bytes_per_step": a_min, "achieved": round(step_gbs, 1), "unit": "GB/s",
                     "gather_bound_bytes_per_step": a_gather, "achieved_vs_gather_bound": round(a_gather / 1e6 / ms_step, 1),
                     "frac_of_measured_peak": round(step_gbs / peak, 4), "frac_of_8TBs_nominal": round(step_gbs / 8000.0, 4),
                     "sum_of_kernel_ms": round(kernel_ms, 5)}

    # ---- e2e: host inputs, H2D + fwd + bwd + D2H of the loss, through the nn.Module ----
    e2e = None
    if not args.no_e2e:
        # Every step copies its own X from pinned host memory (a fresh 4 N d bytes over PCIe) and reads its loss back.
        # Like a training loop's input prefetch, the copy of step k+1 runs on a copy stream into the second of two device
        # buffers while step k computes; the compute stream waits for the event of the buffer it is about to read.
        x_host = x.pin_memory()
        y_host = torch.empty_like(x_host).pin_memory()           # the step's result travels back too (4 N d bytes)
        x_bufs = [torch.empty_like(xd), torch.empty_like(xd)]
        copy_stream, d2h_stream = torch.cuda.Stream(), torch.cuda.Stream()
        copy_done = [torch.cuda.Event(), torch.cuda.Event()]
        buf_free = [torch.cuda.Event(), torch.cuda.Event()]
        y_ready, y_copied = torch.cuda.Event(), torch.cuda.Event()
        main_stream = torch.cuda.current_stream()

        def issue_copy(i):
            b = i & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(buf_free[b])             # the step that last read this buffer has finished
                x_bufs[b].copy_(x_host, non_blocking=True)
                copy_done[b].record(copy_stream)

        def e2e_step(i):
            for p in m.parameters():
                p.grad = None
            issue_copy(i + 1)
            b = i & 1
            main_stream.wait_event(copy_done[b])
            xin = x_bufs[b].detach().requires_grad_(True)
            y = m(xin, eid)
            y_ready.record(main_stream)
            with torch.cuda.stream(d2h_stream):                  # Y -> pinned host memory under the backward of the same step
                d2h_stream.wait_event(y_ready)
                y_host.copy_(y.detach(), non_blocking=True)
                y.record_stream(d2h_stream)
                y_copied.record(d2h_stream)
            loss = (y * gd).sum()
            loss.backward()
            buf_free[b].record(main_stream)
            val = loss.item()
            y_copied.synchronize()                               # the step is over when its result is on the host
            return val

        for b in range(2):
            buf_free[b].record(main_stream)
        issue_copy(0)
        for i in range(3):
            e2e_step(i)
        torch.cuda.synchronize()
        k2 = max(5, args.steps // 3)
        c0 = time.perf_counter()
        t0.record()
        for i in range(3, 3 + k2):
            e2e_step(i)
        t1.record()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - c0) / k2
        dev_s = t0.elapsed_time(t1) / 1e3 / k2
        e2e = {"value": e / max(wall, dev_s), "unit": UNIT, "h2d_bytes_per_step": x_host.numel() * 4,
               "d2h_bytes_per_step": y_host.numel() * 4 + 4, "ms_per_step": round(1e3 * max(wall, dev_s), 4), "steps": k2,
               "h2d": "one X per step from pinned memory, double-buffered: the copy of step k+1 overlaps step k",
               "d2h": "Y (4 N d bytes, pinned) on its own stream under the backward of the same step + the scalar loss"}

    # ---- CPU baseline (bounded: the oracle at full size takes seconds per step) ----
    cpu = None
    if not args.no_cpu_baseline:
        ksteps = 3 if n > 50_000 else 10
        times = oracle_step_seconds(ei, n, d, r, params, x, g_out, ksteps, 1)
        cpu = {"value": e * len(times) / sum(times), "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"full {name}-shaped fwd+bwd, {len(times)} steps after 1 warm-up, {cpu_model()}",
               "ms_per_step": round(1e3 * sum(times) / len(times), 2)}

    line = {
        "metric": METRIC, "value": e / (ms_step / 1e3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(name, n, e, d, r, args.power_law),
                   "edges_with_self_loops": e_prime,
                   "adapter": "relu, skip, learnable scalar, normalize=True", "graph": "static, structure cached",
                   "l2": "inputs larger than L2 (X, gY, Y, gX are %d MB each)" % (4 * n * d // 1_000_000)
                         if 4 * n * d > 126e6 else "working set fits L2; no flush (latency-bound config)",
                   "parallelism": "1 GPU"},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "roofline": roofline, "step_roofline": step_roofline, "phases": phases, "cpu_baseline": cpu,
    }
    if graph_ms is not None:
        line["cuda_graph_replay"] = {"ms_per_step": round(graph_ms, 5), "value": e / (graph_ms / 1e3), "unit": UNIT,
                                     "note": "the same fwd+bwd step captured in one CUDA graph (static tensors); eager "
                                             "ms_per_step above is bound by Python / autograd dispatch at this size"}
    if args.workload is None and os.environ.get("GCA_BENCH_NO_PRODUCTS", "0") != "1":
        del xd, gd, eid
        holder.clear()
        torch.cuda.empty_cache()
        line["products"] = products_subrecord(lib, dev)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
