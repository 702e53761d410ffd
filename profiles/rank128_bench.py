"""Adapter width 128 against 64, and against the stock PyTorch op chain.   python profiles/rank128_bench.py [--reps 7] [--iters 20]

Prints JSON lines:
  * the card (name, power limit, max SM clock), read in this run;
  * per shape (arxiv: 169,343 x 256, cora: 2,708 x 64; relu, learnable scalar, skip): eager forward + backward wall time
    per step, ending in a device synchronise, for GConvAdapter at r = 64 and r = 128 alternated rep by rep in one process,
    and for the op chain of oracle/pyg_restated.py (PyG's GCNConv restated in torch ops) on the same CUDA tensors;
  * the FLOP and byte bounds of one step from the shapes: 12 N d r flop of the six d-wide products (FFMA at r = 128:
    no tensor-core kernel takes that rank) and A_min = 28 N d + 52 N r + 16 E' + 32 N bytes (DESIGN.md section 5),
    each as time at the data-sheet FP32 rate (75 TFLOP/s, see FP32_TFLOPS) and at 7.7 TB/s, and which one is larger;
  * per-phase kernel times from gca_profile_report (a run of its own: the event brackets cost host time).
The arxiv tensors (173 MB per [N, d] operand) exceed the 126 MB L2; the cora ones fit in it."""
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
from gconv_adapter_b200.graphs.synthetic import make_graph, make_inputs  # noqa: E402
from oracle.pyg_restated import GConvAdapterRef  # noqa: E402

HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU
FP32_TFLOPS = 75.0      # 148 SMs x 128 FP32 lanes x 2 flop x ~1.98 GHz boost: the FFMA ceiling of the d-wide phases


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"card": q[0] if q else torch.cuda.get_device_name(0)}


def build(cls, n, d, r, seed):
    _, _, params = make_inputs(n, d, r, seed=seed)
    m = cls(d, r, learnable_scalar=True)
    sd = m.state_dict()
    with torch.no_grad():
        for k, v in params.items():
            sd[k].copy_(v)
    return m.cuda()


def bounds(n, d, r, e_loops):
    flop = 12 * n * d * r
    a_min = 28 * n * d + 52 * n * r + 16 * e_loops + 32 * n
    t_f, t_b = flop / (FP32_TFLOPS * 1e12) * 1e6, a_min / (HBM_TBPS * 1e12) * 1e6
    return {"r": r, "gflop": round(flop / 1e9, 2), "a_min_gb": round(a_min / 1e9, 3), "ffma_bound_us": round(t_f, 1),
            "hbm_bound_us": round(t_b, 1), "bound": "ffma" if t_f > t_b else "hbm"}


def shape(name, workload, d, reps, iters):
    ei, n = make_graph(workload, seed=0)
    ei = ei.cuda()
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(n, d, device="cuda", generator=gen).requires_grad_(True)
    g = torch.randn(n, d, device="cuda", generator=gen)
    mods = {"libgca_r64": build(GConvAdapter, n, d, 64, 2), "libgca_r128": build(GConvAdapter, n, d, 128, 3),
            "torch_ops_r128": build(GConvAdapterRef, n, d, 128, 3)}

    def step(m):
        x.grad = None
        for p in m.parameters():
            p.grad = None
        m(x, ei).backward(g)

    with torch.no_grad():                          # the two r = 128 implementations agree on this input
        y_ours, y_ref = mods["libgca_r128"](x, ei), mods["torch_ops_r128"](x, ei)
        rel = ((y_ours - y_ref).abs().max() / y_ref.abs().max()).item()
    for m in mods.values():
        for _ in range(3):
            step(m)
    torch.cuda.synchronize()
    times = {k: [] for k in mods}
    for _ in range(reps):
        for k, m in mods.items():
            t0 = time.perf_counter()
            for _ in range(iters):
                step(m)
            torch.cuda.synchronize()
            times[k].append(1e6 * (time.perf_counter() - t0) / iters)
    out = {"shape": f"{name} {n}x{d} relu scalar skip, eager fwd+bwd wall", "y_rel_err_vs_torch_ops": rel}
    for k, v in times.items():
        out[f"{k}_us_median"] = round(statistics.median(v), 1)
        out[f"{k}_us_all"] = [round(t, 1) for t in v]
    e_loops = int(ei.shape[1]) + n
    out["bounds"] = [bounds(n, d, r, e_loops) for r in (64, 128)]
    for r, b in zip((64, 128), out["bounds"]):
        t = out[f"libgca_r{r}_us_median"]
        b["step_share_of_bound"] = round(max(b["ffma_bound_us"], b["hbm_bound_us"]) / t, 3)
    print(json.dumps(out), flush=True)
    # per-phase kernel times
    lib = _cabi.load()
    kern = {}
    for k in ("libgca_r64", "libgca_r128"):
        lib.gca_profile_enable(1)
        for _ in range(iters):
            step(mods[k])
        torch.cuda.synchronize()
        buf = ctypes.create_string_buffer(1 << 16)
        _cabi.check(lib.gca_profile_report(buf, len(buf)), "gca_profile_report")
        lib.gca_profile_enable(0)
        rep = json.loads(buf.value.decode())
        kern[k] = {ph: {"us_per_call": round(1e3 * v["ms"] / v["launches"], 2), "variant": v["variant"]} for ph, v in rep.items()}
    print(json.dumps({"shape": name, "kernels": kern}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rank128_bench.py measures on the GPU; no CUDA device is visible")
    print(json.dumps(card()), flush=True)
    shape("arxiv", "arxiv", 256, a.reps, a.iters)
    shape("cora", "cora", 64, a.reps, 5 * a.iters)


if __name__ == "__main__":
    main()
