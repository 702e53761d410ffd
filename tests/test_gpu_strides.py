"""Row pitch and column windows through every kernel family, straight through the C ABI (ctypes), and through the module.

Every dense operand of the ABI (X, Y, gY, gX) has a row pitch.  The TMA-fed kernels encode it in tensor maps (cached per
thread under a key that includes it), the tcgen05 hop + expand reads X / gY and writes Y / gX through tensor maps, and
the mma.sync / FFMA / fused small-graph / LayerNorm / propagate kernels index ``row * ld`` themselves.  Each case below
runs in four layouts of X, gY, Y and gX:

    contiguous  ld = d                                                (the baseline)
    pitch       [:, 0:d] of an [n + 1, d + 4] buffer
    offset      [:, 4:4 + d] of an [n + 1, d + 12] buffer             (base 16 B but not 128 B aligned)
    rebased     the offset window's base pointer with ld = d + 20,    (a stale tensor map cached for the same base
                in the call right after the offset one                 would show here)

and asserts that each phase takes the same kernel variant as in the contiguous run, that every output is bitwise equal
to the contiguous run (same kernel, grid and reduction order), that the pad columns and the extra row n of every buffer
keep their NaN fill bit for bit (nothing written outside the window, and nothing read from outside it: a NaN read would
poison the outputs), and that the input windows are unchanged.  The contiguous run is anchored against fp64.  The
module-level tests cover the layouts autograd produces on its own: broadcast gradients of a sum readout (stride 0),
gradients of ``torch.cat`` outputs, column windows as input, and a single row whose stride(0) is not d."""
import ctypes
import json

import pytest
import torch
import torch.nn.functional as F

from gconv_adapter_b200 import GConvAdapter, GraphCache, GraphStructure, _cabi
from gconv_adapter_b200.graphs.synthetic import make_inputs, symmetric_random_graph
from test_gpu_adapter import compare, run_oracle
from util import assert_close, load_module_params

pytestmark = pytest.mark.gpu

FILL = 0x7FC5A5A5                      # a quiet NaN with a payload: pads must keep exactly these bits
LAYOUTS = (("contiguous", 0, 0), ("pitch", 4, 0), ("offset", 12, 4), ("rebased", 20, 4))   # (name, ld - d, first column)
SILU = _cabi.ACT["silu"]


class Buffers:
    """One flat buffer per operand and layout group; "offset" and "rebased" share theirs, so the rebased window starts at
    the same address as the offset one."""

    def __init__(self, names, n, d):
        self.n, self.d = n, d
        self.flat = {}
        for name in names:
            self.flat[(name, "contiguous")] = torch.empty((n + 1) * d, device="cuda")
            self.flat[(name, "pitch")] = torch.empty((n + 1) * (d + 4), device="cuda")
            self.flat[(name, "offset")] = self.flat[(name, "rebased")] = torch.empty(4 + (n + 1) * (d + 20), device="cuda")

    def window(self, name, layout, src=None):
        """The NaN-filled buffer of ``name`` with the [n, d] window of ``layout`` (holding ``src`` if given): (view, ld)."""
        _, extra, c0 = next(lay for lay in LAYOUTS if lay[0] == layout)
        flat = self.flat[(name, layout)]
        flat.view(torch.int32).fill_(FILL)
        ld = self.d + extra
        w = flat.as_strided((self.n, self.d), (ld, 1), c0)
        if src is not None:
            w.copy_(src)
        return w, ld

    def assert_pads_untouched(self, name, layout, what):
        _, extra, c0 = next(lay for lay in LAYOUTS if lay[0] == layout)
        bits = self.flat[(name, layout)].view(torch.int32).clone()
        bits.as_strided((self.n, self.d), (self.d + extra, 1), c0).fill_(FILL)
        bad = int((bits != FILL).sum())
        assert bad == 0, f"{what}: {bad} elements outside the [{self.n}, {self.d}] window of {name} ({layout}) were changed"


def _nan(*shape):
    return torch.full(shape, float("nan"), device="cuda")


def _u8(nbytes):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device="cuda")


def _variants(lib):
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    _cabi.check(lib.gca_profile_report(buf, len(buf)), "gca_profile_report")
    lib.gca_profile_enable(0)
    return {k: v["variant"] for k, v in json.loads(buf.value.decode()).items()}


def _same(a, b):
    """Bitwise equality (NaN payloads included)."""
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def _rel(a, ref):
    return ((a.double() - ref).abs().max() / ref.abs().max()).item()


def _act(h, act):
    return h * torch.sigmoid(h) if act == SILU else h


def _act_grad(h, act):
    if act != SILU:
        return torch.ones_like(h)
    s = torch.sigmoid(h)
    return s * (1 + h * (1 - s))


class Adjacency:
    """A' (with the self loops the build added) in fp64: rows = targets, columns = their in-neighbours."""

    def __init__(self, g: GraphStructure):
        arr = g.arrays()
        n = arr["rowptr"].numel() - 1
        self.rows = torch.repeat_interleave(torch.arange(n, device="cuda"), arr["rowptr"].diff().long())
        self.cols = arr["colidx"].long()
        self.dis = arr["dis"].double()
        self.n = n

    def fwd(self, f):          # (A' F)[i] = sum over in-neighbours j of F[j]
        return torch.zeros(self.n, f.shape[1], dtype=torch.float64, device="cuda").index_add_(0, self.rows, f.double()[self.cols])

    def adj(self, f):          # (A'^T F)[j] = sum over out-neighbours i of F[i]
        return torch.zeros(self.n, f.shape[1], dtype=torch.float64, device="cuda").index_add_(0, self.cols, f.double()[self.rows])


# ----------------------------------------------------------------------------------------------------------------------
# phase-level sweep
# ----------------------------------------------------------------------------------------------------------------------
# n = 20011 and 9001 leave a partial last tile for every tile height (16, 32, 64, 128).  Each case names the variant
# gca_profile_report must show for the phases it is there to reach; a shape that lands elsewhere is the wrong shape.
CASES = {
    "small": ((2708, 64, 8), {"small_fwd": "fused", "small_bwd": "fused"}),
    "stream16": ((20011, 256, 16), {"project_fwd": "stream_f16", "hop_expand_fwd": "tcgen05", "bwd_up": "stream_f16",
                                    "hop_plain_bwd": "", "expand_wgrad_bwd": "stream_f16"}),
    "stream32": ((20011, 128, 32), {"project_fwd": "stream_f16", "hop_expand_fwd": "tcgen05", "project_bwd": "stream_f16",
                                    "wgrad_up": "stream_f16", "hop_expand_bwd": "tcgen05", "wgrad_down": "stream_f16"}),
    "mma": ((9001, 320, 16), {"project_fwd": "mma", "hop_expand_fwd": "mma", "project_bwd": "mma", "wgrad_up": "mma",
                              "hop_expand_bwd": "mma", "wgrad_down": "mma"}),
    "tc_project": ((9001, 384, 32), {"project_fwd": "tcgen05", "project_bwd": "tcgen05", "hop_expand_fwd": "mma",
                                     "hop_expand_bwd": "mma", "wgrad_up": "mma", "wgrad_down": "mma"}),
    "ffma": ((9001, 300, 8), {"project_fwd": "ffma", "hop_expand_fwd": "ffma", "project_bwd": "ffma", "wgrad_up": "ffma",
                              "hop_expand_bwd": "ffma", "wgrad_down": "ffma"}),
}
FAMILIES = {"stream_f16", "tcgen05", "mma", "ffma", "fused"}
SEEN: dict = {}        # case -> variants of its contiguous runs


class Problem:
    def __init__(self, n, d, r, seed):
        self.n, self.d, self.r = n, d, r
        self.g = GraphStructure(symmetric_random_graph(n, 6 * n, seed=seed).cuda(), n, True)
        self.adjacency = Adjacency(self.g)
        gen = torch.Generator(device="cuda").manual_seed(seed)
        rnd = lambda *s: torch.randn(*s, device="cuda", generator=gen)   # noqa: E731
        self.x, self.gy = rnd(n, d), rnd(n, d)
        self.wd, self.bd = rnd(r, d) * 0.1, rnd(r) * 0.1
        self.wu, self.bu = rnd(d, r) * 0.1, rnd(d) * 0.1
        self.s = torch.tensor([1.3], device="cuda")
        hub = _cabi.load().gca_hub_scratch_bytes(self.g.handle)
        self.hub = _u8(hub) if hub else None


def _run_phases(lib, P: Problem, X, ldx, GY, ldg, Y, ldy, GX, ldgx, act, with_scalar, split):
    """gca_fwd_project -> gca_fwd_hop1 -> gca_fwd_hop2_up, gca_bwd_up (or its two halves) -> gca_bwd_hop2 ->
    gca_bwd_hop1_down -> gca_bwd_finalize; returns every output except Y / gX (they stay in their windows)."""
    n, d, r, g = P.n, P.d, P.r, P.g.handle
    st = torch.cuda.current_stream().cuda_stream
    sp = P.s.data_ptr() if with_scalar else None
    hp = P.hub.data_ptr() if P.hub is not None else None
    o = {k: _nan(n, r) for k in ("pp", "zp", "h2", "gh2", "gh1")}
    o["h1"] = _nan(n, r) if act == SILU else None
    o["gp"] = _nan(n + (n & 1), r)                 # even row count (include/gca.h, gca_bwd_hop1_down)
    o.update(gwd=_nan(r, d), gbd=_nan(r), gwu=_nan(d, r), gbu=_nan(d), gs=_nan(1) if with_scalar else None)
    scratch = _u8(lib.gca_bwd_scratch_bytes(d, r))
    ptr = lambda k: o[k].data_ptr() if o[k] is not None else None   # noqa: E731
    _cabi.check(lib.gca_fwd_project(g, X.data_ptr(), ldx, P.wd.data_ptr(), ptr("pp"), None, d, r, st), "gca_fwd_project")
    _cabi.check(lib.gca_fwd_hop1(g, ptr("pp"), P.bd.data_ptr(), act, ptr("zp"), ptr("h1"), hp, None, r, st), "gca_fwd_hop1")
    _cabi.check(lib.gca_fwd_hop2_up(g, ptr("zp"), X.data_ptr(), ldx, P.wu.data_ptr(), P.bu.data_ptr(), sp, 1, ptr("h2"),
                                    Y.data_ptr(), ldy, hp, d, r, st), "gca_fwd_hop2_up")
    if split:
        _cabi.check(lib.gca_bwd_up_project(g, GY.data_ptr(), ldg, P.wu.data_ptr(), sp, ptr("gh2"), scratch.data_ptr(), None,
                                           d, r, st), "gca_bwd_up_project")
        _cabi.check(lib.gca_bwd_up_wgrad(g, GY.data_ptr(), ldg, ptr("h2"), scratch.data_ptr(), d, r, st), "gca_bwd_up_wgrad")
    else:
        _cabi.check(lib.gca_bwd_up(g, GY.data_ptr(), ldg, ptr("h2"), P.wu.data_ptr(), sp, ptr("gh2"), scratch.data_ptr(), None,
                                   d, r, st), "gca_bwd_up")
    _cabi.check(lib.gca_bwd_hop2(g, ptr("gh2"), ptr("zp"), ptr("h1"), act, ptr("gh1"), scratch.data_ptr(), hp, None, r, st),
                "gca_bwd_hop2")
    _cabi.check(lib.gca_bwd_hop1_down(g, ptr("gh1"), X.data_ptr(), ldx, GY.data_ptr(), ldg, P.wd.data_ptr(), sp, 1, ptr("gp"),
                                      GX.data_ptr(), ldgx, scratch.data_ptr(), hp, d, r, st), "gca_bwd_hop1_down")
    _cabi.check(lib.gca_bwd_finalize(scratch.data_ptr(), P.wu.data_ptr(), P.bu.data_ptr(), sp, 1, ptr("gwd"), ptr("gbd"),
                                     ptr("gwu"), ptr("gbu"), ptr("gs"), d, r, st), "gca_bwd_finalize")
    return o


def _run_fused(lib, P: Problem, X, ldx, GY, ldg, Y, ldy, GX, ldgx, act, with_scalar, split):
    """gca_forward / gca_backward (the fused small-graph kernels at this size)."""
    assert not split
    n, d, r, g = P.n, P.d, P.r, P.g.handle
    st = torch.cuda.current_stream().cuda_stream
    sp = P.s.data_ptr() if with_scalar else None
    o = {k: _nan(n, r) for k in ("zp", "h2")}
    o["h1"] = _nan(n, r) if act == SILU else None
    o.update(gwd=_nan(r, d), gbd=_nan(r), gwu=_nan(d, r), gbu=_nan(d), gs=_nan(1) if with_scalar else None)
    ptr = lambda k: o[k].data_ptr() if o[k] is not None else None   # noqa: E731
    wf = _u8(lib.gca_forward_workspace_bytes(g, d, r))
    wb = _u8(lib.gca_backward_workspace_bytes(g, d, r))
    _cabi.check(lib.gca_forward(g, X.data_ptr(), ldx, P.wd.data_ptr(), P.bd.data_ptr(), P.wu.data_ptr(), P.bu.data_ptr(), sp, act,
                                1, wf.data_ptr(), ptr("zp"), ptr("h1"), ptr("h2"), Y.data_ptr(), ldy, d, r, st), "gca_forward")
    _cabi.check(lib.gca_backward(g, GY.data_ptr(), ldg, X.data_ptr(), ldx, ptr("zp"), ptr("h1"), ptr("h2"), P.wd.data_ptr(),
                                 P.wu.data_ptr(), P.bu.data_ptr(), sp, act, 1, wb.data_ptr(), GX.data_ptr(), ldgx, ptr("gwd"),
                                 ptr("gbd"), ptr("gwu"), ptr("gbu"), ptr("gs"), d, r, st), "gca_backward")
    return o


def _check_fp64(P: Problem, o, y, gx, act, with_scalar, fused, tag):
    """The contiguous run against fp64.  Each phase output is checked against fp64 applied to the kernels' own inputs to
    that phase (the fused path exposes only Z', H1, H2: its other intermediates come from an fp64 chain)."""
    A, dis, n = P.adjacency, P.adjacency.dis[:, None], P.n
    X, GY, WD, WU, BU, BD = (t.double() for t in (P.x, P.gy, P.wd, P.wu, P.bu, P.bd))
    sv = 1.3 if with_scalar else 1.0
    strict = 1e-5 if fused else None           # fused: every dense check through assert_close / 1e-5 sum bounds
    for k, t in o.items():
        if t is not None:
            assert torch.isfinite(t[:n] if k == "gp" else t).all(), f"{tag}: {k} not finite"
    pp = dis * (X @ WD.t())
    if not fused:
        assert _rel(o["pp"], pp) < 1e-6, f"{tag}: P' {_rel(o['pp'], pp):.3e}"
        pp = o["pp"].double()
    h1 = dis * A.fwd(pp) + BD
    assert_close(o["zp"], dis * _act(h1, act), f"{tag}: Z'")
    if act == SILU:
        assert_close(o["h1"], h1, f"{tag}: H1")
        h1 = o["h1"].double()
    assert_close(o["h2"], dis * A.fwd(o["zp"]), f"{tag}: H2")
    H2 = o["h2"].double()
    assert_close(y, sv * (H2 @ WU.t() + BU + X), f"{tag}: Y")
    # backward
    gh2 = dis * sv * (GY @ WU)
    gwu, gbu = sv * (GY.t() @ H2), sv * GY.sum(0)
    for k, ref in (("gwu", gwu), ("gbu", gbu)) + ((("gh2", gh2),) if not fused else ()):
        if strict:
            assert_close(o[k], ref, f"{tag}: {k}")
        else:
            assert _rel(o[k], ref) < 2e-6, f"{tag}: {k} {_rel(o[k], ref):.3e}"
    if not fused:
        gh2 = o["gh2"].double()
    gb_terms = dis * _act_grad(h1, act) * A.adj(gh2)      # d loss / d (pre-activation), per row
    gh1 = dis * gb_terms
    bound = (strict or 2e-6) * gb_terms.abs().sum(0)
    assert ((o["gbd"].double() - gb_terms.sum(0)).abs() <= bound).all(), f"{tag}: gbd"
    if not fused:
        assert_close(o["gh1"], gh1, f"{tag}: gH1'")
        gh1 = o["gh1"].double()
    gp = dis * A.adj(gh1)
    if not fused:
        assert_close(o["gp"][:n], gp, f"{tag}: gP")
        gp = o["gp"][:n].double()
    assert_close(gx, gp @ WD + sv * GY, f"{tag}: gX")
    if strict:
        assert_close(o["gwd"], gp.t() @ X, f"{tag}: gWd")
    else:
        assert _rel(o["gwd"], gp.t() @ X) < 2e-6, f"{tag}: gWd {_rel(o['gwd'], gp.t() @ X):.3e}"
    if with_scalar:
        gs = (GY * X).sum() + ((GY.t() @ H2) * WU).sum() + (GY.sum(0) * BU).sum()
        err = ((o["gs"].double() - gs).abs() / (GY * X).abs().sum()).item()
        assert err < (strict or 2e-6), f"{tag}: gscalar {err:.3e}"


def _sweep_case(case):
    lib = _cabi.load()
    (n, d, r), expect = CASES[case]
    P = Problem(n, d, r, seed=n + d + r)
    fused = case == "small"
    run = _run_fused if fused else _run_phases
    buffers = Buffers(("x", "gy", "y", "gx"), n, d)
    seen = {}
    for act in (_cabi.ACT["none"], SILU):
        for with_scalar in (True, False):
            for split in ((False, True) if case == "stream32" else (False,)):
                base = None
                for layout, _, _ in LAYOUTS:
                    tag = f"{case} n={n} d={d} r={r} act={act} scalar={with_scalar} split={split} {layout}"
                    X, ldx = buffers.window("x", layout, P.x)
                    GY, ldg = buffers.window("gy", layout, P.gy)
                    Y, ldy = buffers.window("y", layout)
                    GX, ldgx = buffers.window("gx", layout)
                    lib.gca_profile_enable(1)
                    o = run(lib, P, X, ldx, GY, ldg, Y, ldy, GX, ldgx, act, with_scalar, split)
                    variants = _variants(lib)
                    o.update(y=Y.clone(), gx=GX.clone())
                    for name in ("x", "gy", "y", "gx"):
                        buffers.assert_pads_untouched(name, layout, tag)
                    assert _same(X, P.x) and _same(GY, P.gy), f"{tag}: an input window was written"
                    if base is None:
                        _check_fp64(P, o, o["y"], o["gx"], act, with_scalar, fused, tag)
                        base = (o, variants)
                        seen.update(variants)
                        if split:       # the two halves of gca_bwd_up give what gca_bwd_up gives
                            assert variants == ref_variants, f"{tag}: {variants} vs {ref_variants}"
                            for k in ref_out:
                                if ref_out[k] is not None:
                                    assert _same(o[k], ref_out[k]), f"{tag}: {k} differs from gca_bwd_up's"
                        else:
                            ref_out, ref_variants = o, variants
                        continue
                    assert variants == base[1], f"{tag}: variants {variants} vs contiguous {base[1]}"
                    for k, t in base[0].items():
                        if t is not None:
                            assert _same(o[k], t), f"{tag}: {k} differs from the contiguous run"
    for k, v in expect.items():
        assert seen.get(k) == v, f"{case}: {k} ran as {seen.get(k)!r}, expected {v!r} (all: {seen})"
    SEEN[case] = seen
    print(f"{case:10s} n={n:5d} d={d:3d} r={r:2d}: " + ", ".join(f"{k}={v or '-'}" for k, v in seen.items()))


@pytest.mark.parametrize("case", list(CASES))
def test_phase_chain_pitch_sweep(case):
    _sweep_case(case)


def test_pitch_sweep_reached_every_kernel_family():
    for case in CASES:
        if case not in SEEN:
            _sweep_case(case)
    seen = {v for variants in SEEN.values() for v in variants.values()}
    assert FAMILIES <= seen, f"the sweep no longer reaches {sorted(FAMILIES - seen)}"


# ----------------------------------------------------------------------------------------------------------------------
# LayerNorm + scalar, propagate
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d", [(5000, 256), (33, 516), (777, 1024)])
def test_layernorm_scale_pitch_sweep(n, d):
    lib = _cabi.load()
    st = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device="cuda").manual_seed(n + d)
    x = torch.randn(n, d, device="cuda", generator=gen) * 3 + 0.5
    gy = torch.randn(n, d, device="cuda", generator=gen)
    w = 1 + 0.3 * torch.randn(d, device="cuda", generator=gen)
    b = 0.2 * torch.randn(d, device="cuda", generator=gen)
    s = torch.tensor([1.3], device="cuda")
    buffers = Buffers(("x", "gy", "y", "gx"), n, d)
    base = None
    for layout, _, _ in LAYOUTS:
        tag = f"layernorm n={n} d={d} {layout}"
        X, ldx = buffers.window("x", layout, x)
        GY, ldg = buffers.window("gy", layout, gy)
        Y, ldy = buffers.window("y", layout)
        GX, ldgx = buffers.window("gx", layout)
        mean, rstd, gw, gb, gs = _nan(n), _nan(n), _nan(d), _nan(d), _nan(1)
        ws = _u8(lib.gca_layernorm_scratch_bytes(d))
        _cabi.check(lib.gca_layernorm_scale_fwd(X.data_ptr(), ldx, w.data_ptr(), b.data_ptr(), s.data_ptr(), 1e-5, Y.data_ptr(), ldy,
                                                mean.data_ptr(), rstd.data_ptr(), n, d, st), "gca_layernorm_scale_fwd")
        _cabi.check(lib.gca_layernorm_scale_bwd(GY.data_ptr(), ldg, X.data_ptr(), ldx, w.data_ptr(), b.data_ptr(), s.data_ptr(),
                                                mean.data_ptr(), rstd.data_ptr(), GX.data_ptr(), ldgx, gw.data_ptr(), gb.data_ptr(),
                                                gs.data_ptr(), ws.data_ptr(), n, d, st), "gca_layernorm_scale_bwd")
        torch.cuda.synchronize()
        out = dict(y=Y.clone(), mean=mean, rstd=rstd, gx=GX.clone(), gw=gw, gb=gb, gs=gs)
        for name in ("x", "gy", "y", "gx"):
            buffers.assert_pads_untouched(name, layout, tag)
        assert _same(X, x) and _same(GY, gy), f"{tag}: an input window was written"
        if base is None:
            ref = [t.double().clone().requires_grad_(True) for t in (x, w, b, s)]
            yr = F.layer_norm(ref[0], (d,), ref[1], ref[2], 1e-5) * ref[3]
            yr.backward(gy.double())
            for k, r_, tol in (("y", yr.detach(), 2e-6), ("gx", ref[0].grad, 5e-6), ("gw", ref[1].grad, 5e-6),
                               ("gb", ref[2].grad, 5e-6)):
                assert _rel(out[k], r_) <= tol, f"{tag}: {k} {_rel(out[k], r_):.3e}"
            floor = 5e-7 * float((gy.abs().double() * yr.detach().abs()).sum()) / 1.3
            assert abs(float(gs) - float(ref[3].grad)) <= 1e-5 * abs(float(ref[3].grad)) + floor, f"{tag}: gscalar"
            base = out
            continue
        for k, t in base.items():
            assert _same(out[k], t), f"{tag}: {k} differs from the contiguous run"


@pytest.mark.parametrize("transpose", [0, 1])
def test_propagate_pitch_sweep(transpose):
    n, D = 20000, 128
    lib = _cabi.load()
    st = torch.cuda.current_stream().cuda_stream
    g = GraphStructure(symmetric_random_graph(n, 6 * n, seed=5).cuda(), n, True)
    A = Adjacency(g)
    x = torch.randn(n, D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(transpose))
    buffers = Buffers(("x", "out"), n, D)
    base = None
    for layout, _, _ in LAYOUTS:
        tag = f"propagate transpose={transpose} {layout}"
        X, ldx = buffers.window("x", layout, x)
        O, ldo = buffers.window("out", layout)
        _cabi.check(lib.gca_propagate(g.handle, transpose, X.data_ptr(), ldx, O.data_ptr(), ldo, None, None, D, st), "gca_propagate")
        torch.cuda.synchronize()
        out = O.clone()
        for name in ("x", "out"):
            buffers.assert_pads_untouched(name, layout, tag)
        assert _same(X, x), f"{tag}: the input window was written"
        if base is None:
            dis = A.dis[:, None]
            assert_close(out, dis * (A.adj(dis * x.double()) if transpose else A.fwd(dis * x.double())), tag)
            base = out
            continue
        assert _same(out, base), f"{tag}: differs from the contiguous run"


# ----------------------------------------------------------------------------------------------------------------------
# the module: layouts autograd hands the kernels
# ----------------------------------------------------------------------------------------------------------------------
SHAPES = [(2708, 64, 8), (20011, 256, 16)]       # fused small-graph kernels; phase kernels


def _module(n, d, r, params, **kw):
    m = GConvAdapter(d, r, non_linearity="silu", **kw)
    load_module_params(m, params)
    m = m.cuda()
    m.graph_cache = GraphCache()
    return m


def _run(m, x, ei, loss_fn):
    """y and the gradients of every leaf after backward of loss_fn(y)."""
    m.zero_grad(set_to_none=True)
    y = m(x, ei)
    loss_fn(y)
    grads = {"x": x.grad.clone() if x.grad is not None else None}
    grads.update({k: p.grad.clone() for k, p in m.named_parameters()})
    x.grad = None
    return y.detach(), grads


def _assert_same(a, b, tag):
    assert _same(a[0], b[0]), f"{tag}: y"
    for k in b[1]:
        assert (a[1][k] is None and b[1][k] is None) or _same(a[1][k], b[1][k]), f"{tag}: grad {k}"


@pytest.mark.parametrize("n,d,r", SHAPES)
@pytest.mark.parametrize("normalization", ["none", "layer_norm"])
@pytest.mark.parametrize("three_d", [False, True])
def test_sum_readout_broadcast_gradient(n, d, r, normalization, three_d):
    """loss = (adapter(x).sum(0) * w).sum() hands y a gradient with stride(0) = 0."""
    ei = symmetric_random_graph(n, 6 * n, seed=1)
    x, _, params = make_inputs(n, d, r, seed=2)
    w = torch.randn(d, generator=torch.Generator().manual_seed(3))
    # the scalar is fused into the adapter without normalization, into the LayerNorm tail with it; the latter's gradient
    # is a near-cancelling sum under this readout, which no fp32 oracle pins, so it is left out there
    m = _module(n, d, r, params, normalization=normalization, learnable_scalar=normalization == "none")
    eic, wc = ei.cuda(), w.cuda()
    xin = (x.cuda().unsqueeze(0) if three_d else x.cuda()).requires_grad_(True)
    readout = _run(m, xin, eic, lambda y: (y.sum(0) * wc).sum().backward())
    dense = _run(m, xin, eic, lambda y: y.backward(wc.expand(n, d).contiguous().reshape(y.shape)))
    tag = f"sum readout n={n} d={d} {normalization} three_d={three_d}"
    _assert_same(readout, dense, tag)
    g_out = w.expand(n, d).contiguous()
    ref = run_oracle(x, ei, params, g_out, non_linearity="silu", normalization=normalization,
                     learnable_scalar=normalization == "none")
    y, grads = readout
    compare((y.reshape(n, d), dict(grads, x=grads["x"].reshape(n, d)), m), ref, tag, g_out=g_out)


@pytest.mark.parametrize("n,d,r", SHAPES)
def test_concatenated_output_gradient_windows(n, d, r):
    """torch.cat([y, z12], 1) hands y a gradient of pitch d + 12, torch.cat([z4, y], 1) one of pitch d + 4 at a 16 B
    offset: the kernels take both in place, with the same result as the dense gradient."""
    ei = symmetric_random_graph(n, 6 * n, seed=4).cuda()
    x, _, params = make_inputs(n, d, r, seed=5)
    m = _module(n, d, r, params, learnable_scalar=True)
    gen = torch.Generator(device="cuda").manual_seed(6)
    xin = x.cuda().requires_grad_(True)
    for width, col in ((12, 0), (4, 4)):
        z = torch.randn(n, width, device="cuda", generator=gen)
        g = torch.randn(n, d + width, device="cuda", generator=gen)
        cat = (lambda y: torch.cat([y, z], 1)) if col == 0 else (lambda y: torch.cat([z, y], 1))
        windowed = _run(m, xin, ei, lambda y: cat(y).backward(g))
        dense = _run(m, xin, ei, lambda y: y.backward(g[:, col:col + d].contiguous()))
        _assert_same(windowed, dense, f"cat n={n} d={d} pitch {d + width} at column {col}")


def test_windowed_input_with_input_gradient():
    """x = h[:, 4:4 + d]: the streaming projection, the tcgen05 skip read and the one-pass backward tail read a pitched X
    at a 16 B offset; Y and every gradient equal those of the same values in a dense tensor."""
    n, d, r = SHAPES[1]
    lib = _cabi.load()
    ei = symmetric_random_graph(n, 6 * n, seed=7).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=8)
    m = _module(n, d, r, params, learnable_scalar=True)
    h = torch.full((n, d + 12), float("nan"), device="cuda")
    h[:, 4:4 + d] = x.cuda()
    xw = h[:, 4:4 + d].requires_grad_(True)
    go = g_out.cuda()
    lib.gca_profile_enable(1)
    windowed = _run(m, xw, ei, lambda y: y.backward(go))
    variants = _variants(lib)
    for k, v in (("project_fwd", "stream_f16"), ("hop_expand_fwd", "tcgen05"), ("expand_wgrad_bwd", "stream_f16")):
        assert variants.get(k) == v, f"{k} ran as {variants.get(k)!r}: {variants}"
    dense = _run(m, x.cuda().requires_grad_(True), ei, lambda y: y.backward(go))
    _assert_same(windowed, dense, "windowed input")


@pytest.mark.parametrize("normalize", [True, False])
def test_single_row_with_row_stride_one(normalize):
    """x = randn(d, 1).t() has strides (1, 1) and is contiguous to PyTorch; one node, no edges."""
    d, r = 64, 8
    ei = torch.zeros(2, 0, dtype=torch.int64, device="cuda")
    _, _, params = make_inputs(1, d, r, seed=9)
    m = _module(1, d, r, params, learnable_scalar=True, normalize=normalize)
    base = torch.randn(d, 1, device="cuda")
    xt = base.t().requires_grad_(True)
    assert xt.stride() == (1, 1) and xt.is_contiguous()
    xd = base.reshape(-1).clone().view(1, d).requires_grad_(True)
    assert xd.stride() == (d, 1)
    go = torch.randn(1, d, device="cuda")
    _assert_same(_run(m, xt, ei, lambda y: y.backward(go)), _run(m, xd, ei, lambda y: y.backward(go)),
                 f"single row normalize={normalize}")
