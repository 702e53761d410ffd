"""Bottleneck sizes in (64, 128] on the GPU: r = 128 is a native rank of libgca, sizes 65..127 are zero-padded to it.
Oracle parity of Y and every gradient (the tolerances of test_gpu_adapter.compare) over the constructor switches, the
input forms, small / large / hub-heavy graphs and every hidden size r = 64 runs at; every run-time switch in a child
process with the variant each phase reports; pitched and windowed operands through the C ABI; bitwise run-to-run
determinism; partitioned handles (emulated on one GPU, and multi-process where there are GPUs for it)."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

from gconv_adapter_b200 import GConvAdapter, GraphCache, _cabi
from gconv_adapter_b200.graphs.synthetic import make_graph, make_inputs, symmetric_random_graph
from test_gpu_adapter import _oracle_parity
from test_gpu_partition import _emulate, _nccl_abi_worker, _rank_worker
from test_gpu_strides import LAYOUTS, Buffers, Problem, _check_fp64, _run_fused, _run_phases, _same, _u8, _variants
from util import assert_close, load_module_params

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


# ---- module parity ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("r", [128, 96, 100])
@pytest.mark.parametrize("over", [
    dict(), dict(non_linearity="silu"), dict(non_linearity="none"), dict(skip_connection=False),
    dict(learnable_scalar=False), dict(normalization="layer_norm"), dict(normalize=False, non_linearity="silu", skip_connection=False),
])
def test_constructor_variants(r, over):
    n = 3000
    ei = symmetric_random_graph(n, 18000, seed=51)
    _oracle_parity(ei, n, 64, r, seed=52, tag=f"r={r} {over}", **over)


@pytest.mark.parametrize("d", [8, 32, 64, 128, 256, 300, 512, 736])
def test_hidden_sizes(d):
    """Every d r = 64 runs at, up to 736 (the largest d of r = 64's fused hop + expand)."""
    n = 2100
    ei = symmetric_random_graph(n, 12000, seed=53)
    _oracle_parity(ei, n, d, 128, seed=54, tag=f"d={d} r=128")
    if d in (300, 512):
        _oracle_parity(ei, n, d, 100, seed=55, tag=f"d={d} r=100", non_linearity="silu")


@pytest.mark.parametrize("three_d", [False, True])
def test_arxiv_shaped_eighth_scale(three_d):
    """n >= 2048 (21k rows), d = 256: the phase kernels; [N, d] and [1, N, d] inputs."""
    ei, n = make_graph("arxiv", seed=0, scale=1 / 8)
    _oracle_parity(ei, n, 256, 128, seed=56, tag="arxiv/8", three_d=three_d)


def test_cora_shaped_small_path():
    """2,708 rows, d = 64: r d = 8192 takes the fused small-graph kernels at r = 128."""
    lib = _cabi.load()
    ei, n = make_graph("cora", seed=0)
    lib.gca_profile_enable(1)
    _oracle_parity(ei, n, 64, 128, seed=57, tag="cora r=128")
    variants = _variants(lib)
    lib.gca_profile_enable(0)
    assert variants.get("small_fwd") == "fused" and variants.get("small_bwd") == "fused", variants
    _oracle_parity(ei, n, 64, 100, seed=58, tag="cora r=100", normalization="layer_norm")


def test_hub_rows_take_the_work_item_path():
    """A star (hub degree 6000 > 512) and a directed second hub: k_hub_partials<128> in all four hops, with the rank-128
    hub scratch."""
    n = 6001
    leaves = torch.arange(1, n, dtype=torch.int64)
    hub = torch.zeros(n - 1, dtype=torch.int64)
    rnd = symmetric_random_graph(n, 20000, seed=17)
    into7 = torch.randint(1, n, (1500,), generator=torch.Generator().manual_seed(3))
    ei = torch.cat([torch.stack([hub, leaves]), torch.stack([leaves, hub]), rnd,
                    torch.stack([into7, torch.full_like(into7, 7)])], dim=1)
    lib = _cabi.load()
    lib.gca_profile_enable(1)
    _oracle_parity(ei, n, 64, 128, seed=59, tag="hub star r=128")
    variants = _variants(lib)
    lib.gca_profile_enable(0)
    assert "hub_partials" in variants, variants
    _oracle_parity(ei, n, 256, 100, seed=60, tag="hub star r=100 d=256", non_linearity="silu")
    # unnormalized: the hub's gradient rows are sums of 6000 unscaled terms, as in test_gpu_adapter's r = 32 case at d = 64
    _oracle_parity(ei, n, 64, 128, seed=61, tag="hub star r=128 unnormalized", normalize=False)


def test_hub_scratch_queries():
    from gconv_adapter_b200 import GraphStructure
    lib = _cabi.load()
    n = 3000
    ei = torch.cat([torch.stack([torch.zeros(n - 1, dtype=torch.int64), torch.arange(1, n)]),
                    symmetric_random_graph(n, 6000, seed=1)], dim=1)
    g = GraphStructure(ei.cuda(), n, True)
    old = lib.gca_hub_scratch_bytes(g.handle)
    assert old > 0
    for r in (8, 16, 32, 64):
        assert lib.gca_hub_scratch_bytes_r(g.handle, r) == old
    assert lib.gca_hub_scratch_bytes_r(g.handle, 128) >= 2 * old - 256
    assert lib.gca_hub_scratch_bytes_r(g.handle, 0) == 0 and lib.gca_hub_scratch_bytes_r(g.handle, 129) == 0
    hub128 = lib.gca_hub_scratch_bytes_r(g.handle, 128)
    assert lib.gca_forward_workspace_bytes(g.handle, 64, 128) - lib.gca_forward_workspace_bytes(g.handle, 64, 64) >= hub128 - old
    g2 = GraphStructure(symmetric_random_graph(n, 6000, seed=2).cuda(), n, True)
    assert lib.gca_hub_scratch_bytes(g2.handle) == 0 and lib.gca_hub_scratch_bytes_r(g2.handle, 128) == 0


def _module(d, r, params, **kw):
    m = GConvAdapter(d, r, **kw)
    load_module_params(m, params)
    m = m.cuda()
    m.graph_cache = GraphCache()
    return m


def test_batched_input_matches_per_graph_calls():
    """[B, N, d] input: each slice has the bits of the [N, d] call, and the gradients are the sums over the batch."""
    n, d, r, b = 2500, 64, 128, 3
    ei = symmetric_random_graph(n, 15000, seed=61).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=62)
    m = _module(d, r, params, learnable_scalar=True)
    xb = torch.stack([x.cuda() * (1 + 0.1 * i) for i in range(b)]).requires_grad_(True)
    gb = torch.stack([g_out.cuda() * (1 - 0.1 * i) for i in range(b)])
    yb = m(xb, ei)
    yb.backward(gb)
    grads_b = {k: p.grad.clone() for k, p in m.named_parameters()}
    total = {k: torch.zeros_like(v) for k, v in grads_b.items()}
    for i in range(b):
        m.zero_grad()
        xi = xb[i].detach().clone().requires_grad_(True)
        yi = m(xi, ei)
        yi.backward(gb[i])
        assert torch.equal(yi, yb[i]), f"slice {i}: y"
        assert torch.equal(xi.grad, xb.grad[i]), f"slice {i}: g_x"
        for k, p in m.named_parameters():
            total[k] += p.grad
    for k in grads_b:
        assert_close(grads_b[k], total[k], f"batched grad {k}")


@pytest.mark.parametrize("normalization", ["none", "layer_norm"])
def test_add_to_is_the_separate_sum(normalization):
    """add_to=h at r = 128: the bits of h + adapter(x), and the same gradients."""
    n, d, r = 3000, 256, 128
    ei = symmetric_random_graph(n, 18000, seed=63).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=64)
    m = _module(d, r, params, learnable_scalar=True, normalization=normalization)
    h = torch.randn(n, d, device="cuda")
    outs = []
    for fused in (True, False):
        m.zero_grad()
        xi = x.cuda().requires_grad_(True)
        hi = h.clone().requires_grad_(True)
        y = m(xi, ei, add_to=hi) if fused else hi + m(xi, ei)
        y.backward(g_out.cuda())
        outs.append((y.detach(), xi.grad, hi.grad, {k: p.grad.clone() for k, p in m.named_parameters()}))
    (y1, gx1, gh1, g1), (y2, gx2, gh2, g2) = outs
    assert torch.equal(y1, y2) and torch.equal(gx1, gx2) and torch.equal(gh1, gh2)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k


def test_bitwise_determinism():
    ei, n = make_graph("arxiv", seed=1, scale=1 / 16, power_law=True)
    x, g_out, params = make_inputs(n, 256, 128, seed=65)
    m = _module(256, 128, params, learnable_scalar=True)
    runs = []
    for _ in range(2):
        m.zero_grad()
        xi = x.cuda().requires_grad_(True)
        y = m(xi, ei.cuda())
        y.backward(g_out.cuda())
        runs.append((y.detach().clone(), xi.grad.clone(), {k: p.grad.clone() for k, p in m.named_parameters()}))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for k in runs[0][2]:
        assert torch.equal(runs[0][2][k], runs[1][2][k]), k


# ---- run-time switches (child processes) -----------------------------------------------------------------------------
GCA_VARS = ("GCA_DISABLE_TC", "GCA_DISABLE_STREAM", "GCA_DISABLE_TMA", "GCA_DISABLE_PDL", "GCA_SPLIT_MB", "GCA_DISABLE_BWD_FUSE",
            "GCA_DISABLE_SMALL")
# r = 128 has no tensor-core or streaming kernel: under every switch the phases run the FFMA kernels, the second hop of
# each direction as a plain hop + column-block expansion
PHASES = {"project_fwd": "ffma", "hop_fwd": "", "hop_plain_fwd": "", "expand_fwd": "ffma", "project_bwd": "ffma",
          "wgrad_up": "ffma", "hop_bwd": "", "hop_plain_bwd": "", "expand_bwd": "ffma", "wgrad_down": "ffma"}
SMALL = {"small_fwd": "fused", "small_bwd": "fused"}
SWITCHES = {
    "default": {},
    "no_tc": {"GCA_DISABLE_TC": "1"},
    "no_stream": {"GCA_DISABLE_STREAM": "1"},
    "no_tma": {"GCA_DISABLE_TMA": "1"},
    "no_pdl": {"GCA_DISABLE_PDL": "1"},
    "no_small": {"GCA_DISABLE_SMALL": "1"},
    "no_bwd_fuse": {"GCA_DISABLE_BWD_FUSE": "1"},
    "split_k3": {"GCA_SPLIT_MB": "0"},
}


@pytest.mark.parametrize("setting", list(SWITCHES))
@pytest.mark.parametrize("case", ["arxiv_relu", "arxiv_silu_noskip", "cora_relu"])
def test_switches(setting, case):
    env = {k: v for k, v in os.environ.items() if k not in GCA_VARS}
    env.update(SWITCHES[setting])
    res = subprocess.run([sys.executable, os.path.join(HERE, "rank128_runner.py"), case], env=env, capture_output=True,
                         text=True, timeout=900)
    assert res.returncode == 0, f"{case} under {setting}:\n{res.stdout[-3000:]}\n{res.stderr[-6000:]}"
    out = json.loads(res.stdout.strip().splitlines()[-1])
    assert out["ok"]
    expect = SMALL if case == "cora_relu" and setting != "no_small" else PHASES
    got = {k: v for k, v in out["variants"].items() if k != "finalize"}
    assert got == expect, f"{case} under {setting}: {got}"


def test_small_path_after_another_rank_with_the_same_shared_memory():
    """r = 64 at d = 128 and r = 128 at d = 64 give the fused small-graph kernels the same shared memory but different
    occupancy: the co-resident grid limit must be the r = 128 kernel's own (a fresh process, so the order is fixed)."""
    env = {k: v for k, v in os.environ.items() if k not in GCA_VARS}
    res = subprocess.run([sys.executable, os.path.join(HERE, "rank128_runner.py"), "cora_after_r64"], env=env,
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, f"{res.stdout[-3000:]}\n{res.stderr[-6000:]}"
    out = json.loads(res.stdout.strip().splitlines()[-1])
    assert out["variants"].get("small_fwd") == "fused" and out["variants"].get("small_bwd") == "fused", out


# ---- pitched windows through the C ABI ---------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,fused", [(3000, 256, False), (2100, 300, False), (1500, 64, True)])
def test_pitch_sweep_c_abi(n, d, fused):
    """The layouts of test_gpu_strides (contiguous, pitch, offset, rebased) at r = 128: every output bitwise equal to the
    contiguous run, the contiguous run against fp64, pads untouched, the same variant per phase."""
    lib = _cabi.load()
    r = 128
    P = Problem(n, d, r, seed=n + d)
    run = _run_fused if fused else _run_phases
    buffers = Buffers(("x", "gy", "y", "gx"), n, d)
    for act in (_cabi.ACT["none"], _cabi.ACT["silu"]):
        for with_scalar in (True, False):
            base = None
            for layout, _, _ in LAYOUTS:
                tag = f"n={n} d={d} r={r} act={act} scalar={with_scalar} {layout}"
                X, ldx = buffers.window("x", layout, P.x)
                GY, ldg = buffers.window("gy", layout, P.gy)
                Y, ldy = buffers.window("y", layout)
                GX, ldgx = buffers.window("gx", layout)
                lib.gca_profile_enable(1)
                o = run(lib, P, X, ldx, GY, ldg, Y, ldy, GX, ldgx, act, with_scalar, False)
                variants = _variants(lib)
                o.update(y=Y.clone(), gx=GX.clone())
                for name in ("x", "gy", "y", "gx"):
                    buffers.assert_pads_untouched(name, layout, tag)
                assert _same(X, P.x) and _same(GY, P.gy), f"{tag}: an input window was written"
                if base is None:
                    _check_fp64(P, o, o["y"], o["gx"], act, with_scalar, fused, tag)
                    base = (o, variants)
                    assert set(variants.values()) <= {"ffma", "fused", ""}, variants
                    continue
                assert variants == base[1], f"{tag}: variants {variants} vs contiguous {base[1]}"
                for k, t in base[0].items():
                    if t is not None:
                        assert _same(o[k], t), f"{tag}: {k} differs from the contiguous run"
    lib.gca_profile_enable(0)


# ---- partitioned handles -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 4])
def test_emulated_ranks_bitwise_equal_single_gpu_module(world):
    ei, n = make_graph("arxiv", seed=2, scale=1 / 16)
    d, r = 256, 128
    x, g_out, params = make_inputs(n, d, r, seed=66)
    y, gx, grads, _ = _emulate(world, ei, n, d, r, x, g_out, params)
    m = _module(d, r, params, learnable_scalar=True)
    xi = x.cuda().requires_grad_(True)
    ym = m(xi, ei.cuda())
    ym.backward(g_out.cuda())
    assert torch.equal(y, ym.detach()), "emulated partitioned Y differs from the single-GPU module"
    assert_close(gx, xi.grad, "partitioned g_x")
    for k, p in m.named_parameters():
        assert_close(grads[k], p.grad, f"partitioned grad {k}")


def _port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("comm", ["peer", "collective"])
def test_two_process_run_matches_single_gpu(comm):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    n, d, r, world = 20001, 256, 128, 2
    out = mp.Manager().dict()
    mp.spawn(_rank_worker, args=(world, _port(), n, d, r, comm, out), nprocs=world, join=True)
    ei = symmetric_random_graph(n, 8 * n, seed=31)
    x, g_out, params = make_inputs(n, d, r, seed=32)
    m = _module(d, r, params, learnable_scalar=True)
    xi = x.cuda().requires_grad_(True)
    ym = m(xi, ei.cuda())
    ym.backward(g_out.cuda())
    assert torch.equal(torch.cat([out[k]["y"] for k in range(world)]), ym.detach().cpu())
    assert_close(torch.cat([out[k]["gx"] for k in range(world)]), xi.grad, f"{comm}: g_x")
    for k, p in m.named_parameters():
        assert_close(out[0]["grads"][k], p.grad, f"{comm}: grad {k}")


@pytest.mark.parametrize("act", ["relu", "silu"])
def test_nccl_entry_points(act):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_nccl_abi_worker, args=(2, _port(), 6001, 256, 128, act, out), nprocs=2, join=True)   # asserts in the workers
    assert len(out) == 2
