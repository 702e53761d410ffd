"""Parallel insertion fused into the last forward kernel: ``adapter(x, ei, add_to=h)`` against the separate
``h + adapter(x, ei)``.   python profiles/parallel_add_bench.py [--reps 7] [--iters 50]

Prints JSON lines: the card (name, power limit), then
  * arxiv shape (169,343 x 256, r 16, relu, learnable scalar; x and h are 173 MB each, more than the 126 MB L2): device
    time per forward (CUDA events, no autograd graph), the two versions alternated rep by rep;
  * the hop_expand_fwd kernel time with and without the addend (gca_profile_report, a run of its own);
  * cora shape (2,708 x 64, r 8): eager forward + backward wall time per step, ending in a device synchronise;
  * for every timed configuration, whether the fused output has the bits of the separate add."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from gconv_adapter_b200 import GConvAdapter, _cabi  # noqa: E402
from gconv_adapter_b200.graphs.synthetic import make_graph, make_inputs, symmetric_random_graph  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"card": q[0] if q else torch.cuda.get_device_name(0)}


def module(n, d, r, seed):
    _, _, params = make_inputs(n, d, r, seed=seed)
    m = GConvAdapter(d, r, learnable_scalar=True)
    sd = m.state_dict()
    with torch.no_grad():
        for k, v in params.items():
            sd[k].copy_(v)
    return m.cuda()


def arxiv(reps, iters):
    ei, n = make_graph("arxiv", seed=0)
    d, r = 256, 16
    m = module(n, d, r, 0)
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(n, d, device="cuda", generator=gen)
    h = torch.randn(n, d, device="cuda", generator=gen)
    ei = ei.cuda()
    versions = {"separate": lambda: h + m(x, ei), "fused": lambda: m(x, ei, add_to=h)}
    with torch.no_grad():
        same = torch.equal(versions["fused"]().view(torch.int32), versions["separate"]().view(torch.int32))
        for f in versions.values():                      # warm-up of both shapes / kernels
            for _ in range(5):
                f()
        torch.cuda.synchronize()
        times = {k: [] for k in versions}
        for _ in range(reps):
            for k, f in versions.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(iters):
                    f()
                b.record()
                b.synchronize()
                times[k].append(1e3 * a.elapsed_time(b) / iters)
    out = {"shape": f"arxiv {n}x{d} r{r} relu scalar", "bitwise_equal": same}
    for k, v in times.items():
        out[f"{k}_us_median"] = round(statistics.median(v), 2)
        out[f"{k}_us_all"] = [round(t, 2) for t in v]
    out["saved_us"] = round(out["separate_us_median"] - out["fused_us_median"], 2)
    print(json.dumps(out), flush=True)
    # kernel times from the library's own event brackets (a run of its own: the brackets cost host time)
    lib = _cabi.load()
    with torch.no_grad():
        kern = {}
        for k, f in versions.items():
            lib.gca_profile_enable(1)
            for _ in range(iters):
                f()
            torch.cuda.synchronize()
            buf = ctypes.create_string_buffer(1 << 16)
            _cabi.check(lib.gca_profile_report(buf, len(buf)), "gca_profile_report")
            lib.gca_profile_enable(0)
            rep = json.loads(buf.value.decode())
            kern[k] = {name: {"us_per_call": round(1e3 * v["ms"] / v["launches"], 2), "variant": v["variant"]}
                       for name, v in rep.items()}
    print(json.dumps({"shape": "arxiv", "kernels": kern}), flush=True)


def cora(reps, iters):
    n, d, r = 2708, 64, 8
    ei = symmetric_random_graph(n, 5 * n, seed=2).cuda()
    m = module(n, d, r, 3)
    gen = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn(n, d, device="cuda", generator=gen).requires_grad_(True)
    h = torch.randn(n, d, device="cuda", generator=gen).requires_grad_(True)
    g = torch.randn(n, d, device="cuda", generator=gen)
    versions = {"separate": lambda: h + m(x, ei), "fused": lambda: m(x, ei, add_to=h)}
    same = torch.equal(versions["fused"]().detach().view(torch.int32), versions["separate"]().detach().view(torch.int32))

    def step(f):
        x.grad = h.grad = None
        for p in m.parameters():
            p.grad = None
        f().backward(g)

    times = {k: [] for k in versions}
    for f in versions.values():
        for _ in range(20):
            step(f)
    torch.cuda.synchronize()
    for _ in range(reps):
        for k, f in versions.items():
            t0 = time.perf_counter()
            for _ in range(iters):
                step(f)
            torch.cuda.synchronize()
            times[k].append(1e6 * (time.perf_counter() - t0) / iters)
    out = {"shape": f"cora {n}x{d} r{r} fwd+bwd eager wall", "bitwise_equal": same}
    for k, v in times.items():
        out[f"{k}_us_median"] = round(statistics.median(v), 2)
        out[f"{k}_us_all"] = [round(t, 2) for t in v]
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("parallel_add_bench.py measures on the GPU; no CUDA device is visible")
    print(json.dumps(card()), flush=True)
    arxiv(a.reps, a.iters)
    cora(a.reps, 4 * a.iters)


if __name__ == "__main__":
    main()
