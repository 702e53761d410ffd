"""normalization='batch_norm': the fused BatchNorm1d + scalar tail (gca_batchnorm.cu) against torch.nn.BatchNorm1d in fp64
(outputs, gradients, batch and running statistics, train and eval), its conditioning, pitched layouts, determinism and
CUDA-graph capture, and the module with the fused tail against the module with the stock ops."""
import copy
import ctypes
import json
import types

import pytest
import torch
import torch.nn as nn

import gconv_adapter_b200.finetune.gconv_adapter as impl
from gconv_adapter_b200 import GConvAdapter, _cabi
from gconv_adapter_b200.graphs.synthetic import make_inputs, symmetric_random_graph
from util import load_module_params

pytestmark = pytest.mark.gpu


def _close(a, b, tag, tol=2e-6, floor=0.0):
    err = float((a.double() - b.double()).abs().max())
    ref = float(b.double().abs().max())
    assert err <= tol * max(ref, 1e-30) + floor + 1e-30, f"{tag}: max err {err:.3e} vs max|ref| {ref:.3e}"


def _tail(bn, scalar):
    """The module's fused tail on its own: GConvAdapter._batch_norm_scale with just the attributes it reads."""
    holder = types.SimpleNamespace(normalization=bn, scalar=scalar)
    return lambda x: GConvAdapter._batch_norm_scale(holder, x)


def _bn(d, affine, momentum, track, seed):
    bn = nn.BatchNorm1d(d, affine=affine, momentum=momentum, track_running_stats=track).cuda()
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        if affine:
            bn.weight.copy_(1 + 0.3 * torch.randn(d, generator=g))
            bn.bias.copy_(0.2 * torch.randn(d, generator=g))
        if track:
            bn.running_mean.copy_(0.5 * torch.randn(d, generator=g))
            bn.running_var.copy_(1 + torch.rand(d, generator=g))
            bn.num_batches_tracked.fill_(4)
    return bn


SETTINGS = {   # name: (train, affine, with_scalar, momentum, track_running_stats)
    "train": (True, True, True, 0.1, True),
    "train_cma_noscalar": (True, True, False, None, True),
    "train_noaffine_mom0": (True, False, True, 0.0, True),
    "train_untracked": (True, True, True, 0.1, False),
    "eval": (False, True, True, 0.1, True),
    "eval_untracked_plain": (False, False, False, 0.1, False),
}
SHAPES = [(2, 4), (3, 64), (257, 300), (5000, 256), (777, 1028), (4099, 2048)]
BIG = (2_449_029, 256)


def _run_fp64_parity(n, d, setting):
    train, affine, with_scalar, momentum, track = SETTINGS[setting]
    bn = _bn(d, affine, momentum, track, seed=n + d).train(train)
    ref_bn = copy.deepcopy(bn).double()
    g = torch.Generator(device="cuda").manual_seed(n * 31 + d)
    x = torch.randn(n, d, device="cuda", generator=g) * 3 + 0.5
    gy = torch.randn(n, d, device="cuda", generator=g)
    s = nn.Parameter(torch.tensor([1.3], device="cuda")) if with_scalar else None
    xl = x.clone().requires_grad_(True)
    y = _tail(bn, s)(xl)
    stats = y.grad_fn.saved_tensors[1].clone()
    y.backward(gy)
    s64 = nn.Parameter(s.detach().double()) if with_scalar else None
    xr = x.double().requires_grad_(True)
    yr = ref_bn(xr)
    ybn = yr.detach()
    if s64 is not None:
        yr = yr * s64
    yr.backward(gy.double())
    _close(y, yr.detach(), "y")
    # gX is a difference of terms of size |s gamma rstd gY| that cancel almost completely at tiny n (at n = 2, xh = +-1
    # whatever x is): the noise floor is a few fp32 ulps of those terms
    gam = ref_bn.weight.detach() if affine else 1.0
    terms = (gy.double() * gam * (s64.detach() if with_scalar else 1.0)).abs().max(0).values
    rstd_ref = ((xr.detach().var(0, unbiased=False) if (train or not track) else ref_bn.running_var) + bn.eps).rsqrt()
    _close(xl.grad, xr.grad, "g_x", tol=5e-6, floor=5e-6 * float((terms * rstd_ref).max()))
    if affine:
        _close(bn.weight.grad, ref_bn.weight.grad, "g_weight", tol=5e-6)
        _close(bn.bias.grad, ref_bn.bias.grad, "g_bias", tol=5e-6)
    else:
        assert bn.weight is None and bn.bias is None
    if with_scalar:
        floor = 5e-7 * float((gy.abs().double() * ybn.abs()).sum())
        assert abs(float(s.grad) - float(s64.grad)) <= 1e-5 * abs(float(s64.grad)) + floor
    batch_stats = train or not track
    xd = x.double()
    if batch_stats:
        mean_ref, var_ref = xd.mean(0), xd.var(0, unbiased=False)
    else:
        mean_ref, var_ref = ref_bn.running_mean, ref_bn.running_var
    _close(stats[0], mean_ref, "mean")
    _close(stats[1], (var_ref + bn.eps).rsqrt(), "rstd")
    if track:
        _close(bn.running_mean, ref_bn.running_mean, "running_mean")
        _close(bn.running_var, ref_bn.running_var, "running_var")
        assert int(bn.num_batches_tracked) == int(ref_bn.num_batches_tracked)
    else:
        assert bn.running_mean is None and bn.running_var is None
    return bn, y, xl.grad, s


@pytest.mark.parametrize("setting", sorted(SETTINGS))
@pytest.mark.parametrize("n,d", SHAPES)
def test_fused_batchnorm_scale_matches_fp64(n, d, setting):
    _run_fp64_parity(n, d, setting)


@pytest.mark.parametrize("setting", ["train", "eval"])
def test_fused_batchnorm_scale_matches_fp64_2_4m_rows(setting):
    _run_fp64_parity(*BIG, setting)


def test_conditioning_large_mean_and_constant_column():
    """|mean| = 100 std: the shifted sums keep running_var / rstd at fp64 accuracy (fp32 E[x^2] - E[x]^2 misses this by
    ~60x); a constant column has x - mean == 0 exactly, so its output is exactly s * beta."""
    n, d = 200_000, 64
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(n, d, device="cuda", generator=g)
    x[:, 3] = 100.0 + torch.randn(n, device="cuda", generator=g)
    x[:, 7] = -250.0 * (1 + 0.01 * torch.randn(n, device="cuda", generator=g))
    x[:, 9] = 3.7
    bn = _bn(d, True, 1.0, True, seed=1).train()     # momentum 1: running_var is the unbiased batch variance
    s = torch.tensor([1.3], device="cuda")
    y = _tail(bn, s)(x)
    rstd = y.grad_fn.saved_tensors[1][1] if y.grad_fn is not None else None
    xd = x.double()
    var_ref = xd.var(0, unbiased=True)
    rstd_ref = (xd.var(0, unbiased=False) + bn.eps).rsqrt()
    for c in (3, 7):
        assert abs(float(bn.running_var[c]) / float(var_ref[c]) - 1) <= 1e-5, c
        if rstd is not None:
            assert abs(float(rstd[c]) / float(rstd_ref[c]) - 1) <= 1e-5, c
    assert torch.equal(y[:, 9], (s * bn.bias.detach())[9].expand(n))
    assert float(bn.running_var[9]) == 0.0


def test_saved_statistics_with_grad():
    n, d = 200_000, 64
    g = torch.Generator(device="cuda").manual_seed(6)
    x = torch.randn(n, d, device="cuda", generator=g)
    x[:, 3] = 100.0 + torch.randn(n, device="cuda", generator=g)
    bn = _bn(d, True, 0.1, True, seed=2).train()
    y = _tail(bn, None)(x.requires_grad_(True))
    mean, rstd = y.grad_fn.saved_tensors[1]
    xd = x.detach().double()
    assert abs(float(rstd[3]) / float((xd[:, 3].var(unbiased=False) + bn.eps).rsqrt()) - 1) <= 1e-5
    assert abs(float(mean[3]) / float(xd[:, 3].mean()) - 1) <= 2e-7


def _nan_window(n, d, pad, gen=None, src=None):
    """[n, d] window at column 4 of an [n, d + pad] NaN-filled tensor (optionally holding src)."""
    full = torch.full((n, d + pad), float("nan"), device="cuda")
    if src is not None:
        full[:, 4:4 + d] = src
    return full, full[:, 4:4 + d]


@pytest.mark.parametrize("training", [1, 0])
def test_pitched_windows_through_the_c_abi(training):
    lib = _cabi.load()
    n, d, pad = 3001, 132, 12
    g = torch.Generator(device="cuda").manual_seed(8)
    x = torch.randn(n, d, device="cuda", generator=g) + 2
    gy = torch.randn(n, d, device="cuda", generator=g)
    gamma = 1 + 0.1 * torch.randn(d, device="cuda", generator=g)
    beta = 0.1 * torch.randn(d, device="cuda", generator=g)
    s = torch.tensor([0.7], device="cuda")
    ws = torch.empty(lib.gca_batchnorm_scratch_bytes(d), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def run(xv, ldx, yv, ldy, gyv, ldg, gxv, ldgx):
        rm, rv = torch.zeros(d, device="cuda"), torch.ones(d, device="cuda")
        stats = torch.empty(2, d, device="cuda")
        assert lib.gca_batchnorm_scale_fwd(xv.data_ptr(), ldx, gamma.data_ptr(), beta.data_ptr(), s.data_ptr(), 1e-5, training,
                                           0.1, rm.data_ptr(), rv.data_ptr(), yv.data_ptr(), ldy, stats[0].data_ptr(),
                                           stats[1].data_ptr(), ws.data_ptr(), n, d, stream) == 0
        gg, gb, gs = torch.empty(d, device="cuda"), torch.empty(d, device="cuda"), torch.empty(1, device="cuda")
        assert lib.gca_batchnorm_scale_bwd(gyv.data_ptr(), ldg, xv.data_ptr(), ldx, gamma.data_ptr(), beta.data_ptr(),
                                           s.data_ptr(), stats[0].data_ptr(), stats[1].data_ptr(), training, gxv.data_ptr(),
                                           ldgx, gg.data_ptr(), gb.data_ptr(), gs.data_ptr(), ws.data_ptr(), n, d, stream) == 0
        return rm, rv, gg, gb, gs

    y, gx = torch.empty(n, d, device="cuda"), torch.empty(n, d, device="cuda")
    dense = run(x, d, y, d, gy, d, gx, d)
    xf, xw = _nan_window(n, d, pad, src=x)
    gyf, gyw = _nan_window(n, d, pad, src=gy)
    yf, yw = _nan_window(n, d, pad)
    gxf, gxw = _nan_window(n, d, pad)
    win = run(xw, d + pad, yw, d + pad, gyw, d + pad, gxw, d + pad)
    torch.cuda.synchronize()
    assert torch.equal(yw, y) and torch.equal(gxw, gx)
    for a, b in zip(dense, win):
        assert torch.equal(a, b)
    for full in (yf, gxf):
        assert torch.isnan(full[:, :4]).all() and torch.isnan(full[:, 4 + d:]).all()
    assert torch.equal(xf[:, 4:4 + d], x) and torch.equal(gyf[:, 4:4 + d], gy)


def _module(d, r, params, fuse=True, **kw):
    m = GConvAdapter(d, r, normalization="batch_norm", learnable_scalar=True, **kw)
    load_module_params(m, params)
    with torch.no_grad():
        m.normalization.weight.copy_(1 + 0.1 * torch.arange(d) / d)
        m.normalization.bias.copy_(0.05 * torch.ones(d))
        m.scalar.fill_(1.2)
    m = m.cuda()
    m.fuse_batch_norm = fuse
    return m


def _step(m, x, ei, g_out, add_to=None):
    m.zero_grad(set_to_none=True)
    xx = x.clone().requires_grad_(True)
    y = m(xx, ei) if add_to is None else m(xx, ei, add_to=add_to)
    y.backward(g_out)
    grads = {"x": xx.grad}
    grads.update({k: p.grad for k, p in m.named_parameters()})
    return y.detach(), grads


def _compare_modules(a, b, g_out, tag):
    (ya, ga), (yb, gb) = a, b
    _close(ya, yb, f"{tag}: y", tol=5e-6)
    for k in gb:
        floor = 1e-6 * float(g_out.abs().sum(0).max()) if k == "conv_up.bias" else 0.0
        _close(ga[k], gb[k], f"{tag}: grad {k}", tol=2e-5 if k == "scalar" else 5e-6, floor=floor)


def _compare_buffers(ma, mb, tag):
    _close(ma.normalization.running_mean, mb.normalization.running_mean, f"{tag}: running_mean", tol=5e-6)
    _close(ma.normalization.running_var, mb.normalization.running_var, f"{tag}: running_var", tol=5e-6)
    assert int(ma.normalization.num_batches_tracked) == int(mb.normalization.num_batches_tracked)


@pytest.mark.parametrize("n,d,r", [(3000, 64, 16), (20000, 256, 16)])
def test_module_with_fused_tail_equals_stock_ops(n, d, r):
    ei = symmetric_random_graph(n, 6 * n, seed=3).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=4)
    x, g_out = x.cuda(), g_out.cuda()
    fused, stock = _module(d, r, params, True), _module(d, r, params, False)
    for step in range(3):
        _compare_modules(_step(fused, x, ei, g_out), _step(stock, x, ei, g_out), g_out, f"step {step}")
        _compare_buffers(fused, stock, f"step {step}")
    assert int(fused.normalization.num_batches_tracked) == 3
    fused.eval(), stock.eval()
    _compare_modules(_step(fused, x, ei, g_out), _step(stock, x, ei, g_out), g_out, "eval")
    _compare_buffers(fused, stock, "eval")


def test_stride0_gradient_through_the_module():
    n, d, r = 5000, 64, 16
    ei = symmetric_random_graph(n, 6 * n, seed=5).cuda()
    x, _, params = make_inputs(n, d, r, seed=6)
    m = _module(d, r, params)
    xx = x.cuda().requires_grad_(True)
    m(xx, ei).sum(0).sum().backward()                                 # gY = ones expanded: stride 0 rows
    dense = _module(d, r, params)
    xd = x.cuda().requires_grad_(True)
    dense(xd, ei).backward(torch.ones(n, d, device="cuda"))
    assert torch.equal(xx.grad, xd.grad)
    for (k, p), (_, q) in zip(m.named_parameters(), dense.named_parameters()):
        assert torch.equal(p.grad, q.grad), k


def _no_fused_tail(monkeypatch):
    class Refuse:
        @staticmethod
        def apply(*a):
            raise AssertionError("the fused BatchNorm tail ran")
    monkeypatch.setattr(impl, "_BatchNormScaleFunction", Refuse)


class _MyBatchNorm(nn.BatchNorm1d):
    pass


@pytest.mark.parametrize("case", ["env", "d30", "1nd", "n1", "subclass"])
def test_fallbacks_take_the_stock_path(case, monkeypatch):
    n, d, r = {"d30": (3000, 30, 8), "n1": (1, 64, 8)}.get(case, (3000, 64, 16))
    ei = symmetric_random_graph(n, 6 * n, seed=9).cuda() if n > 1 else torch.zeros(2, 0, dtype=torch.int64, device="cuda")
    x, g_out, params = make_inputs(n, d, r, seed=10)
    x, g_out = x.cuda(), g_out.cuda()
    if case == "1nd":
        x, g_out = x.unsqueeze(0), g_out.unsqueeze(0)
    outs = []
    for fuse in (True, False):
        m = _module(d, r, params, fuse)
        if case == "subclass":
            m.normalization = _MyBatchNorm(d).cuda()
        if case == "env":
            monkeypatch.setenv("GCA_DISABLE_BN_FUSE", "1")
        with monkeypatch.context() as mp:
            _no_fused_tail(mp)
            outs.append((_step(m, x, ei, g_out), m.normalization.running_mean.clone(), m.normalization.running_var.clone(),
                         int(m.normalization.num_batches_tracked)))
    (ya, ga), *bufa = outs[0]
    (yb, gb), *bufb = outs[1]
    assert torch.equal(ya, yb)
    for k in gb:
        assert (ga[k] is None and gb[k] is None) or torch.equal(ga[k], gb[k]), k
    assert torch.equal(bufa[0], bufb[0]) and torch.equal(bufa[1], bufb[1]) and bufa[2] == bufb[2]
    if case in ("1nd", "n1"):
        assert bufa[2] == 0 and ga["normalization.weight"] is None   # no BatchNorm at all
        assert torch.equal(bufa[0], torch.zeros(d, device="cuda"))


def test_batched_input_is_fused_per_slice():
    n, d, r = 3000, 64, 16
    ei = symmetric_random_graph(n, 6 * n, seed=11).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=12)
    x = torch.stack([x, x.flip(0) * 0.5]).cuda()
    g_out = torch.stack([g_out, 0.5 * g_out]).cuda()
    fused, stock = _module(d, r, params, True), _module(d, r, params, False)
    _compare_modules(_step(fused, x, ei, g_out), _step(stock, x, ei, g_out), g_out.reshape(-1, d), "[2, N, d]")
    _compare_buffers(fused, stock, "[2, N, d]")
    assert int(fused.normalization.num_batches_tracked) == 2


def test_add_to_sits_on_the_fused_tail():
    n, d, r = 20000, 256, 16
    ei = symmetric_random_graph(n, 6 * n, seed=13).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=14)
    x, g_out = x.cuda(), g_out.cuda()
    h = torch.randn(n, d, device="cuda", generator=torch.Generator(device="cuda").manual_seed(15))
    fused, stock = _module(d, r, params, True), _module(d, r, params, False)
    assert not fused.fuses_add(x, h)
    lib = _cabi.load()
    lib.gca_profile_enable(1)
    a = _step(fused, x, ei, g_out, add_to=h)
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.gca_profile_report(buf, len(buf))
    lib.gca_profile_enable(0)
    ran = json.loads(buf.value.decode())
    for k in ("batchnorm_stats", "batchnorm_fwd", "batchnorm_bwd", "batchnorm_bwd_finalize", "batchnorm_bwd_dx"):
        assert k in ran, k
    _compare_modules(a, _step(stock, x, ei, g_out, add_to=h), g_out, "add_to")
    _compare_buffers(fused, stock, "add_to")


def test_determinism_and_cuda_graph_capture():
    """One fwd + bwd step captured in a CUDA graph (momentum 0.1) and replayed three times gives the bits of three eager
    steps from the same start: outputs, gradients, running buffers."""
    n, d, r = 20000, 64, 16      # n d > 2^19: the phase kernels both eager and captured
    ei = symmetric_random_graph(n, 6 * n, seed=17).cuda()
    x, g_out, params = make_inputs(n, d, r, seed=18)
    m = _module(d, r, params)
    bn = m.normalization
    x = x.cuda().requires_grad_(True)
    g_out = g_out.cuda()
    start = (bn.running_mean.clone(), bn.running_var.clone(), bn.num_batches_tracked.clone())

    def reset():
        bn.running_mean.copy_(start[0]); bn.running_var.copy_(start[1]); bn.num_batches_tracked.copy_(start[2])

    holder = {}

    def step():
        y = m(x, ei)
        y.backward(g_out)
        holder["y"] = y.detach()

    def snapshot():
        return [holder["y"].clone(), x.grad.clone()] + [p.grad.clone() for p in m.parameters()] + \
               [bn.running_mean.clone(), bn.running_var.clone(), bn.num_batches_tracked.clone()]

    def zero():
        x.grad = None
        for p in m.parameters():
            p.grad = None

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            zero()
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    zero()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    torch.cuda.synchronize()
    reset()
    replays = []
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        replays.append(snapshot())
    del graph
    reset()
    eager = []
    for _ in range(3):
        zero()
        step()
        eager.append(snapshot())
    reset()
    again = []
    for _ in range(3):
        zero()
        step()
        again.append(snapshot())
    for i in range(3):
        for a, b, c in zip(replays[i], eager[i], again[i]):
            assert torch.equal(b, c), f"eager step {i} is not reproducible"
            assert torch.equal(a, b), f"replay {i} differs from eager step {i}"
    assert int(bn.num_batches_tracked) == int(start[2]) + 3
