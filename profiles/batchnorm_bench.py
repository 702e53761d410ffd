"""normalization='batch_norm': the fused BatchNorm1d + scalar tail (gca_batchnorm.cu) against the stock torch ops
(nn.BatchNorm1d + mul, GConvAdapter.fuse_batch_norm = False) after the same adapter kernels.
    python profiles/batchnorm_bench.py [--reps 7] [--iters 20] > profiles/batchnorm_bench.jsonl

Prints JSON lines:
  * the card (name, power limit, max SM clock), read in this run;
  * per shape (arxiv: 169,343 x 256, r 16; cora: 2,708 x 64, r 8; relu, learnable scalar, skip, train mode): eager
    forward + backward time per step (CUDA events over `iters` steps), fused and stock alternated rep by rep in one
    process; the median and the spread of the reps;
  * the per-kernel times of the fused tail from gca_profile_report (a run of its own: the event brackets cost host time),
    with the bytes each tail kernel must move and the rate that makes at the measured time.
The arxiv tensors (173 MB per [N, d] operand) exceed the 126 MB L2; the cora ones fit in it."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from gconv_adapter_b200 import GConvAdapter, _cabi  # noqa: E402
from gconv_adapter_b200.graphs.synthetic import SHAPES, make_graph, make_inputs  # noqa: E402

TAIL = ("batchnorm_stats", "batchnorm_fwd", "batchnorm_bwd", "batchnorm_bwd_finalize", "batchnorm_bwd_dx")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"card": q[0] if q else torch.cuda.get_device_name(0)}


def module(name, params, fuse):
    s = SHAPES[name]
    m = GConvAdapter(s.hidden, s.rank, normalization="batch_norm", learnable_scalar=True)
    sd = m.state_dict()
    with torch.no_grad():
        for k, v in params.items():
            sd[k].copy_(v)
    m = m.cuda().train()
    m.fuse_batch_norm = fuse
    return m


def shape(name, reps, iters):
    ei, n = make_graph(name, seed=0)
    s = SHAPES[name]
    x, g_out, params = make_inputs(n, s.hidden, s.rank, seed=0)
    eid, xd, gd = ei.cuda(), x.cuda().requires_grad_(True), g_out.cuda()
    mods = {True: module(name, params, True), False: module(name, params, False)}

    def step(m):
        xd.grad = None
        for p in m.parameters():
            p.grad = None
        m(xd, eid).backward(gd)

    for m in mods.values():
        for _ in range(5):
            step(m)
    torch.cuda.synchronize()
    times = {True: [], False: []}
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for fuse, m in mods.items():
            t0.record()
            for _ in range(iters):
                step(m)
            t1.record()
            torch.cuda.synchronize()
            times[fuse].append(t0.elapsed_time(t1) / iters)
    for fuse in (True, False):
        t = times[fuse]
        print(json.dumps({"workload": name, "n": n, "d": s.hidden, "r": s.rank,
                          "tail": "fused BatchNorm1d + scalar" if fuse else "torch BatchNorm1d + mul",
                          "ms_per_fwd_bwd": round(statistics.median(t), 4), "min": round(min(t), 4), "max": round(max(t), 4),
                          "reps": reps, "iters": iters}), flush=True)

    lib = _cabi.load()
    lib.gca_profile_enable(1)
    for _ in range(iters):
        step(mods[True])
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.gca_profile_report(buf, len(buf))
    lib.gca_profile_enable(0)
    prof = json.loads(buf.value.decode())
    nd = 4 * n * s.hidden
    moved = {"batchnorm_stats": nd, "batchnorm_fwd": 2 * nd, "batchnorm_bwd": 2 * nd, "batchnorm_bwd_dx": 3 * nd}
    kernels = {}
    for k in TAIL:
        v = prof.get(k)
        if v is None:
            continue
        us = 1e3 * v["ms"] / iters
        row = {"us_per_step": round(us, 2), "launches_per_step": v["launches"] / iters}
        if k in moved:
            row["gb_moved"] = round(moved[k] / 1e9, 4)
            row["tb_per_s"] = round(moved[k] / (us * 1e-6) / 1e12, 2)
        kernels[k] = row
    others = sum(v["ms"] for k, v in prof.items() if k not in TAIL)
    print(json.dumps({"workload": name, "fused_tail_kernels": kernels,
                      "adapter_kernels_us_per_step": round(1e3 * others / iters, 2)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--shapes", default="arxiv,cora")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batchnorm_bench.py measures on the GPU; no CUDA device found")
    print(json.dumps(card()), flush=True)
    for name in args.shapes.split(","):
        shape(name, args.reps, args.iters)


if __name__ == "__main__":
    main()
