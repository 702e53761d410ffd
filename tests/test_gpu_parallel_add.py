"""Parallel insertion in one pass: ``Y = ... + A`` inside the last forward kernel (gca_fwd_hop2_up_add, gca_forward_add,
gca_layernorm_scale_add_fwd) and ``GConvAdapter(x, ei, add_to=h)`` / ``PartitionedGConvAdapter(..., add_to=h)``.

Every fused result must have the bits of the separate ``A + Y`` of the existing entries on the same kernel variant (the
add is one round-to-nearest fp32 add after Y is formed), take the same variant, work in place (Y == A) and with a pitched
A window whose NaN pads stay untouched.  The module gives exactly ``h + adapter(x)`` and the same gradients; the hosts run
the reference's parallel mode with the one-line edit shown in INTEGRATION.md."""
import ctypes
import json
import os
import socket
import subprocess
import sys

import pytest
import torch
import torch.nn as nn

from gconv_adapter_b200 import GConvAdapter, GraphCache, GraphStructure, _cabi
from gconv_adapter_b200.graphs.synthetic import make_inputs, symmetric_random_graph
from gconv_adapter_b200.partition import CudaPhases, PartitionedGConvAdapter, row_block, shard_size
from hosts import MolecularGNNHost, TransductiveHost
from util import assert_close, load_module_params

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
FILL = 0x7FC5A5A5
RELU, SILU = _cabi.ACT["relu"], _cabi.ACT["silu"]
# the shapes tests/test_gpu_strides.py uses to reach each family, with the hop + expand variant each must take
CASES = {
    "tc16": ((20011, 256, 16), "tcgen05"),
    "tc32": ((20011, 128, 32), "tcgen05"),
    "mma": ((9001, 320, 16), "mma"),
    "ffma": ((9001, 300, 8), "ffma"),
    "small": ((2708, 64, 8), "fused"),
}


def _same(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _u8(nbytes):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device="cuda")


def _variants(lib):
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    _cabi.check(lib.gca_profile_report(buf, len(buf)), "gca_profile_report")
    lib.gca_profile_enable(0)
    return {k: v["variant"] for k, v in json.loads(buf.value.decode()).items()}


class Problem:
    def __init__(self, n, d, r, seed):
        self.n, self.d, self.r = n, d, r
        self.g = GraphStructure(symmetric_random_graph(n, 6 * n, seed=seed).cuda(), n, True)
        gen = torch.Generator(device="cuda").manual_seed(seed)
        rnd = lambda *s: torch.randn(*s, device="cuda", generator=gen)   # noqa: E731
        self.x, self.a = rnd(n, d), rnd(n, d) * 3
        self.wd, self.bd = rnd(r, d) * 0.1, rnd(r) * 0.1
        self.wu, self.bu = rnd(d, r) * 0.1, rnd(d) * 0.1
        self.s = torch.tensor([1.3], device="cuda")


def _forward(lib, P, act, with_scalar, skip, Y, ldy, A=None, lda=0):
    """gca_forward (A None) or gca_forward_add into Y; returns (Z', H2, variants)."""
    n, d, r, g = P.n, P.d, P.r, P.g.handle
    st = torch.cuda.current_stream().cuda_stream
    zp, h2 = torch.empty(n, r, device="cuda"), torch.empty(n, r, device="cuda")
    h1 = torch.empty(n, r, device="cuda") if act == SILU else None
    wf = _u8(lib.gca_forward_workspace_bytes(g, d, r))
    sp = P.s.data_ptr() if with_scalar else None
    args = (g, P.x.data_ptr(), d, P.wd.data_ptr(), P.bd.data_ptr(), P.wu.data_ptr(), P.bu.data_ptr(), sp, act, skip,
            wf.data_ptr(), zp.data_ptr(), h1.data_ptr() if h1 is not None else None, h2.data_ptr())
    lib.gca_profile_enable(1)
    if A is None:
        _cabi.check(lib.gca_forward(*args, Y.data_ptr(), ldy, d, r, st), "gca_forward")
    else:
        _cabi.check(lib.gca_forward_add(*args, A.data_ptr(), lda, Y.data_ptr(), ldy, d, r, st), "gca_forward_add")
    return zp, h2, _variants(lib)


def _hop2_up(lib, P, zp, with_scalar, skip, Y, ldy, A=None, lda=0):
    n, d, r, g = P.n, P.d, P.r, P.g.handle
    st = torch.cuda.current_stream().cuda_stream
    h2 = torch.empty(n, r, device="cuda")
    nh = lib.gca_hub_scratch_bytes(g)
    hub = _u8(nh) if nh else None
    args = (g, zp.data_ptr(), P.x.data_ptr(), d, P.wu.data_ptr(), P.bu.data_ptr(), P.s.data_ptr() if with_scalar else None, skip,
            h2.data_ptr())
    tail = (hub.data_ptr() if hub is not None else None, d, r, st)
    lib.gca_profile_enable(1)
    if A is None:
        _cabi.check(lib.gca_fwd_hop2_up(*args, Y.data_ptr(), ldy, *tail), "gca_fwd_hop2_up")
    else:
        _cabi.check(lib.gca_fwd_hop2_up_add(*args, A.data_ptr(), lda, Y.data_ptr(), ldy, *tail), "gca_fwd_hop2_up_add")
    return h2, _variants(lib)


def _window(n, d, src):
    """src in columns 4 .. 4 + d of a NaN-filled [n + 1, d + 12] buffer: (flat buffer, window, ld)."""
    ld = d + 12
    flat = torch.empty((n + 1) * ld + 4, device="cuda")
    flat.view(torch.int32).fill_(FILL)
    w = flat.as_strided((n, d), (ld, 1), 4)
    w.copy_(src)
    return flat, w, ld


def _pads_untouched(flat, n, d, ld):
    bits = flat.view(torch.int32).clone()
    bits.as_strided((n, d), (ld, 1), 4).fill_(FILL)
    return bool((bits == FILL).all())


def run_case(case):
    """Every act / skip / scalar combination of one shape through gca_forward_add and (phases) gca_fwd_hop2_up_add."""
    lib = _cabi.load()
    (n, d, r), family = CASES[case]
    P = Problem(n, d, r, seed=n + d + r)
    seen = {}                              # phase -> variant
    for act in (RELU, SILU):
        for skip in (1, 0):
            for with_scalar in (True, False):
                tag = f"{case} act={act} skip={skip} scalar={with_scalar}"
                y = torch.empty(n, d, device="cuda")
                zp, _, v0 = _forward(lib, P, act, with_scalar, skip, y, d)
                ref = P.a + y
                yf = torch.empty(n, d, device="cuda")
                _, _, v1 = _forward(lib, P, act, with_scalar, skip, yf, d, P.a, d)
                assert v1 == v0, f"{tag}: gca_forward_add variants {v1} vs {v0}"
                assert _same(yf, ref), f"{tag}: gca_forward_add != A + gca_forward"
                inplace = P.a.clone()
                _forward(lib, P, act, with_scalar, skip, inplace, d, inplace, d)
                assert _same(inplace, ref), f"{tag}: gca_forward_add in place"
                flat, win, ld = _window(n, d, P.a)
                yw = torch.empty(n, d, device="cuda")
                _forward(lib, P, act, with_scalar, skip, yw, d, win, ld)
                assert _same(yw, ref) and _pads_untouched(flat, n, d, ld), f"{tag}: gca_forward_add, pitched A"
                _forward(lib, P, act, with_scalar, skip, win, ld, win, ld)
                assert _same(win, ref) and _pads_untouched(flat, n, d, ld), f"{tag}: gca_forward_add, pitched, in place"
                seen.update(v0)
                if "small_fwd" in v0:
                    continue
                # the K3 entry on its own, from the same Z'
                y3 = torch.empty(n, d, device="cuda")
                _, w0 = _hop2_up(lib, P, zp, with_scalar, skip, y3, d)
                assert _same(y3, y), f"{tag}: gca_fwd_hop2_up differs from gca_forward"
                y3a = torch.empty(n, d, device="cuda")
                _, w1 = _hop2_up(lib, P, zp, with_scalar, skip, y3a, d, P.a, d)
                assert w1 == w0, f"{tag}: gca_fwd_hop2_up_add variants {w1} vs {w0}"
                assert _same(y3a, ref), f"{tag}: gca_fwd_hop2_up_add != A + gca_fwd_hop2_up"
                flat, win, ld = _window(n, d, P.a)
                _hop2_up(lib, P, zp, with_scalar, skip, win, ld, win, ld)
                assert _same(win, ref) and _pads_untouched(flat, n, d, ld), f"{tag}: gca_fwd_hop2_up_add, pitched, in place"
    return seen


@pytest.mark.parametrize("case", list(CASES))
def test_fused_add_entries_bitwise(case):
    seen = run_case(case)
    assert CASES[case][1] in seen.values(), f"{case}: ran as {seen}, expected {CASES[case][1]}"


@pytest.mark.parametrize("env,case,expect", [({"GCA_SPLIT_MB": "0"}, "tc16", "expand_fwd"),
                                             ({"GCA_DISABLE_SMALL": "1"}, "small", "hop_expand_fwd")])
def test_fused_add_under_switches(env, case, expect):
    """The split K3 (plain hop + expand-only tcgen05 kernel) and the phases at small n; the switches are latched per
    process, so each runs in a child (tests/parallel_add_runner.py)."""
    e = dict(os.environ, **env)
    res = subprocess.run([sys.executable, os.path.join(HERE, "parallel_add_runner.py"), case], env=e, capture_output=True,
                         text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    seen = json.loads(res.stdout.strip().splitlines()[-1])
    assert expect in seen, seen


def test_layernorm_scale_add_bitwise():
    lib = _cabi.load()
    st = torch.cuda.current_stream().cuda_stream
    for n, d in ((5000, 256), (33, 516), (777, 1024)):
        gen = torch.Generator(device="cuda").manual_seed(n + d)
        x = torch.randn(n, d, device="cuda", generator=gen) * 3 + 0.5
        a = torch.randn(n, d, device="cuda", generator=gen)
        w = 1 + 0.3 * torch.randn(d, device="cuda", generator=gen)
        b = 0.2 * torch.randn(d, device="cuda", generator=gen)
        s = torch.tensor([1.3], device="cuda")
        stats = [torch.empty(n, device="cuda") for _ in range(4)]
        y = torch.empty(n, d, device="cuda")
        _cabi.check(lib.gca_layernorm_scale_fwd(x.data_ptr(), d, w.data_ptr(), b.data_ptr(), s.data_ptr(), 1e-5, y.data_ptr(), d,
                                                stats[0].data_ptr(), stats[1].data_ptr(), n, d, st), "ln")
        ref = a + y
        flat, win, ld = _window(n, d, a)
        for tag, (A, lda, Y, ldy) in {"contiguous": (a, d, torch.empty(n, d, device="cuda"), d), "pitched in place": (win, ld, win, ld)}.items():
            _cabi.check(lib.gca_layernorm_scale_add_fwd(x.data_ptr(), d, w.data_ptr(), b.data_ptr(), s.data_ptr(), 1e-5, A.data_ptr(),
                                                        lda, Y.data_ptr(), ldy, stats[2].data_ptr(), stats[3].data_ptr(), n, d, st),
                        "ln add")
            torch.cuda.synchronize()
            assert _same(Y, ref), f"layernorm add n={n} d={d} {tag}"
            assert _same(stats[2], stats[0]) and _same(stats[3], stats[1]), f"layernorm add stats n={n} d={d} {tag}"
        assert _pads_untouched(flat, n, d, ld)


# ----------------------------------------------------------------------------------------------------------------------
# module
# ----------------------------------------------------------------------------------------------------------------------
def _module(d, r, params, **kw):
    m = GConvAdapter(d, r, **kw)
    load_module_params(m, params)
    m = m.cuda()
    m.graph_cache = GraphCache()
    return m


def _fwd_bwd(m, x, h, ei, g, fused):
    m.zero_grad(set_to_none=True)
    xx, hh = x.clone().requires_grad_(True), h.clone().requires_grad_(True)
    y = m(xx, ei, add_to=hh) if fused else hh + m(xx, ei)
    y.backward(g.expand(y.shape).to(y.dtype))
    grads = {"x": xx.grad, "h": hh.grad}
    grads.update({k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None})
    return y.detach(), grads


@pytest.mark.parametrize("normalization", ["none", "layer_norm", "batch_norm"])
@pytest.mark.parametrize("n,d,r", [(2708, 64, 8), (20011, 256, 16), (3000, 30, 8)])
@pytest.mark.parametrize("shape", ["2d", "1nd", "bnd"])
def test_module_add_to_matches_separate_add(normalization, n, d, r, shape):
    ei = symmetric_random_graph(n, 6 * n, seed=11).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=12)
    m = _module(d, r, params, normalization=normalization, learnable_scalar=True, non_linearity="silu")
    gen = torch.Generator(device="cuda").manual_seed(13)
    x, g = x.cuda(), g_out.cuda()
    if shape == "1nd":
        x, g = x.unsqueeze(0), g.unsqueeze(0)
    elif shape == "bnd":
        x = torch.stack([x, x.flip(0)])
        g = torch.stack([g, 0.5 * g])
    h = torch.randn(x.shape, device="cuda", generator=gen)
    if normalization == "batch_norm" and shape != "2d":
        pytest.skip("BatchNorm1d rejects 3-D input in the reference as well")
    assert m.fuses_add(x, h) == (normalization != "batch_norm" and d % 4 == 0)
    tag = f"{normalization} n={n} d={d} {shape}"
    m.train(normalization != "batch_norm")
    fused = _fwd_bwd(m, x, h, ei, g, True)
    sep = _fwd_bwd(m, x, h, ei, g, False)
    assert _same(fused[0], sep[0]), f"{tag}: y"
    for k in sep[1]:
        assert _same(fused[1][k], sep[1][k]), f"{tag}: grad {k}"


@pytest.mark.parametrize("kind", ["broadcast", "fp64", "column_window", "stride0"])
def test_module_add_to_operand_forms(kind):
    n, d, r = 20011, 256, 16
    ei = symmetric_random_graph(n, 6 * n, seed=21).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=22)
    m = _module(d, r, params, learnable_scalar=True)
    x, g = x.cuda(), g_out.cuda()
    gen = torch.Generator(device="cuda").manual_seed(23)
    if kind == "broadcast":
        h = torch.randn(d, device="cuda", generator=gen)
    elif kind == "fp64":
        h = torch.randn(n, d, device="cuda", generator=gen, dtype=torch.float64)
    elif kind == "column_window":
        h = torch.randn(n, d + 12, device="cuda", generator=gen)[:, 4:4 + d]
    else:
        h = torch.randn(1, d, device="cuda", generator=gen).expand(n, d)
    assert m.fuses_add(x, h) == (kind in ("column_window", "stride0"))
    m.zero_grad(set_to_none=True)
    xx, hh = x.clone().requires_grad_(True), h.detach().requires_grad_(True)
    y = m(xx, ei, add_to=hh)
    ref_y = h + m(x, ei)
    assert y.shape == ref_y.shape and y.dtype == ref_y.dtype and _same(y.detach(), ref_y.detach()), kind
    y.backward(torch.ones_like(y))
    assert hh.grad.shape == h.shape and torch.equal(hh.grad, torch.ones_like(y).sum_to_size(h.shape)), kind


# ----------------------------------------------------------------------------------------------------------------------
# hosts in parallel mode
# ----------------------------------------------------------------------------------------------------------------------
class FusedMolecularHost(MolecularGNNHost):
    """MolecularGNNHost's parallel mode with the adds done by the adapters (the host edit of INTEGRATION.md)."""

    def forward(self, x, edge_index, edge_attr):
        assert self.adapter_type == "parallel"
        hidden_states = [x]
        for layer in range(self.num_layers):
            key = str(layer)
            h = self.gnn_layers[layer](hidden_states[layer], edge_index, edge_attr)
            if h.size(0) > 1:
                h = self.batch_norm_layers[layer](h)
            t = self.pre_adapters[key](hidden_states[layer], edge_index, edge_attr, add_to=h)     # == h + pre_out
            h = self.post_adapters[key](h, edge_index, edge_attr, add_to=t)                      # == (h + pre) + post
            h = h if layer == self.num_layers - 1 else torch.relu(h)
            hidden_states.append(h)
        return hidden_states[-1]


class FusedTransductiveHost(TransductiveHost):
    def forward(self, x, adjs):
        assert self.adapter_type == "parallel"
        nodeformer = self.kind == "nodeformer"
        if nodeformer:
            x = x.unsqueeze(0)
        z = torch.relu(self.bns[0](self.fcs[0](x)))
        layer_ = [z]
        x = z
        for i, conv in enumerate(self.convs):
            key = str(i)
            if nodeformer:
                z = conv(layer_[i])
                z += layer_[i]
                z = torch.relu(self.bns[i + 1](z))
            else:
                z = conv(x)
                z = self.alpha * z + (1 - self.alpha) * layer_[i]
                z = self.bns[i + 1](z)
            t = self.pre_adapters[key](layer_[i], adjs[0], add_to=z)
            z = self.post_adapters[key](z, adjs[0], add_to=t)
            layer_.append(z)
            x = z
        out = self.fcs[-1](z)
        return out.squeeze(0) if nodeformer else out


def _attach(host, factory):
    if isinstance(host, MolecularGNNHost):
        for position in ("pre", "post"):
            host.add_adapter(factory, position, "parallel")
    else:
        host.add_adapter(factory, ["pre", "post"], "parallel")


def _host_pair(stock_cls, fused_cls, ctor, factory, seed):
    torch.manual_seed(seed)
    stock, fused = stock_cls(*ctor), fused_cls(*ctor)
    _attach(stock, factory)
    _attach(fused, factory)
    fused.load_state_dict(stock.state_dict())
    for a, b in zip(stock.parameters(), fused.parameters()):
        b.requires_grad_(a.requires_grad)
    return stock.cuda(), fused.cuda()


def _host_check(stock, fused, run, tag):
    outs = []
    for host in (stock, fused):
        host.zero_grad(set_to_none=True)
        y = run(host)
        y.square().sum().backward()
        outs.append((y.detach(), {k: p.grad for k, p in host.named_parameters() if p.grad is not None}))
    assert _same(outs[1][0], outs[0][0]), f"{tag}: output"
    assert outs[0][1].keys() == outs[1][1].keys()
    for k, g in outs[0][1].items():
        err = (outs[1][1][k] - g).abs().max().item()
        assert err <= 1e-6 * max(g.abs().max().item(), 1e-30), f"{tag}: grad {k} {err:.3e}"


@pytest.mark.parametrize("normalization", ["none", "layer_norm"])
def test_molecular_host_parallel_mode(normalization):
    n, d = 900, 300
    ei = symmetric_random_graph(n, 4 * n, seed=31)
    ea = torch.stack([torch.randint(0, 4, (ei.shape[1],)), torch.randint(0, 3, (ei.shape[1],))], 1)
    factory = lambda hidden_size: GConvAdapter(hidden_size, 16, normalization=normalization, learnable_scalar=True)  # noqa: E731
    stock, fused = _host_pair(MolecularGNNHost, FusedMolecularHost, (3, d), factory, 32)
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(33)).cuda()
    # the GIN stand-in aggregates with index_add_, whose CUDA kernel adds with atomics: two runs of the stock host differ
    # in the last bits unless the deterministic (sorted) implementation is selected
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        _host_check(stock, fused, lambda h: h(x, ei.cuda(), ea.cuda()), f"molecular {normalization}")
    finally:
        torch.use_deterministic_algorithms(was)


@pytest.mark.parametrize("kind", ["nodeformer", "difformer"])
def test_transductive_host_parallel_mode(kind):
    n, c, hdim = 2708, 40, 64
    ei = symmetric_random_graph(n, 5 * n, seed=41).cuda()
    factory = lambda hidden_size: GConvAdapter(hidden_size, 8, learnable_scalar=True)   # noqa: E731
    stock, fused = _host_pair(TransductiveHost, FusedTransductiveHost, (kind, c, hdim, 7), factory, 42)
    x = torch.randn(n, c, generator=torch.Generator().manual_seed(43)).cuda()
    _host_check(stock, fused, lambda h: h(x, [ei]), kind)


# ----------------------------------------------------------------------------------------------------------------------
# partitioned
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3])
def test_partitioned_add_emulated_ranks(world):
    """Every rank's gca_fwd_hop2_up_add on a partitioned handle, one after the other on one GPU: the rows equal
    h + the 1-GPU module's output bit for bit."""
    n, d, r = 20011, 256, 16
    ei = symmetric_random_graph(n, 6 * n, seed=51).cuda()
    x, _, params = make_inputs(n, d, r, seed=52)
    m = _module(d, r, params, learnable_scalar=True)
    x = x.cuda()
    h = torch.randn(n, d, device="cuda", generator=torch.Generator(device="cuda").manual_seed(53))
    with torch.no_grad():
        ref = m(x, ei, add_to=h)
    be = CudaPhases()
    s = shard_size(n, world)
    blocks = [row_block(n, world, k) for k in range(world)]
    graphs = [be.build_graph(ei, n, True, lo, hi) for lo, hi in blocks]
    P = {k: v.detach().cuda().contiguous() for k, v in m.state_dict().items()}
    wd, bd, wu, bu, sc = (P["conv_down.lin.weight"], P["conv_down.bias"], P["conv_up.lin.weight"], P["conv_up.bias"], P["scalar"])
    p_full, z_full = torch.zeros(world * s, r, device="cuda"), torch.zeros(world * s, r, device="cuda")
    for k, (lo, hi) in enumerate(blocks):
        be.fwd_project(graphs[k], x[lo:hi], wd, p_full[lo:hi])
    for k, (lo, hi) in enumerate(blocks):
        be.fwd_hop1(graphs[k], p_full, bd, RELU, z_full[lo:hi], None)
    ys = []
    for k, (lo, hi) in enumerate(blocks):
        y, ya = torch.empty(hi - lo, d, device="cuda"), torch.empty(hi - lo, d, device="cuda")
        h2 = torch.empty(hi - lo, r, device="cuda")
        be.fwd_hop2_up(graphs[k], z_full, x[lo:hi], wu, bu, sc, True, h2, y)
        be.fwd_hop2_up_add(graphs[k], z_full, x[lo:hi], wu, bu, sc, True, h2, h[lo:hi], ya)
        assert _same(ya, h[lo:hi] + y), f"rank {k} of {world}"
        ys.append(ya)
    torch.cuda.synchronize()
    assert_close(torch.cat(ys), ref.double(), f"world {world} vs the 1-GPU module")


def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("normalization", ["none", "layer_norm"])
def test_partitioned_add_two_processes(normalization):
    res = subprocess.run([sys.executable, os.path.join(HERE, "parallel_add_runner.py"), "partitioned", normalization,
                          str(_free_port())], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
