"""Drop-in ``GConvAdapter`` backed by the sm_100a kernels of libgca.

Mirrors /root/reference/src/finetune/gconv_adapter.py:5-108: same constructor arguments and
defaults (:23-26), same ``ValueError`` messages (:37,51,61), same parameter names and
``state_dict`` keys (``scalar``, ``conv_down.bias``, ``conv_down.lin.weight``,
``conv_up.bias``, ``conv_up.lin.weight`` [, ``normalization.*``]), same near-identity init
(:73-78, drawing from the torch RNG in the order PyG's constructors + the reference do), same
call signature ``forward(x, edge_index, edge_attr=None)`` (:80) with ``edge_attr`` ignored, x of
shape ``[N, d]`` or ``[1, N, d]``, and the same op order skip -> normalization -> scalar
(:94-106).  ``forward(..., add_to=h)`` returns ``h + forward(...)`` (the reference's parallel insertion), with the
add done in the store of the last kernel where the operands allow.  The arithmetic runs as hand-written CUDA (include/gca.h); there is NO CPU path:
a CPU tensor, or a missing libgca.so, raises ``RuntimeError``.
"""
from __future__ import annotations

import math
import os
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _cabi
from ..graphs.csr import GLOBAL_GRAPH_CACHE, GraphCache, GraphStructure

_FAST_RANKS = (8, 16, 32, 64, 128)

# Test hook: when True the autograd function keeps references to the tensors it saved for the
# backward (scaled activations Z' and H2) in ``LAST_SAVED`` so parity tests can read the ReLU mask.
DEBUG_KEEP_SAVED = False
LAST_SAVED: dict = {}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _sizes(lib, graph: GraphStructure, d: int, r: int):
    """(forward workspace bytes, backward workspace bytes) of one call on this graph - cached on the graph object
    (they depend on its row count and on whether it has hub rows; the C calls are pure functions)."""
    cache = graph.__dict__.setdefault("_ws_sizes", {})
    hit = cache.get((d, r))
    if hit is None:
        hit = (lib.gca_forward_workspace_bytes(graph.handle, d, r), lib.gca_backward_workspace_bytes(graph.handle, d, r))
        cache[(d, r)] = hit
    return hit


def _raw_stream(dev: torch.device) -> int:
    """Make ``dev`` current (libgca launches on the current device) and return its current stream's handle.  The public
    ``torch.cuda.current_stream().cuda_stream`` costs ~10 us per call in Python bookkeeping - a fifth of a tiny-graph
    step (profiles/r2_host_profile.txt) - so the raw accessors are used when this torch build has them."""
    idx = dev.index
    try:
        if torch._C._cuda_getDevice() != idx:
            torch.cuda.set_device(idx)
        return torch._C._cuda_getCurrentRawStream(idx)
    except AttributeError:
        if torch.cuda.current_device() != idx:
            torch.cuda.set_device(idx)
        return torch.cuda.current_stream().cuda_stream


def _align(nbytes: int) -> int:
    return (nbytes + 255) // 256 * 256


def row_pitch(t: torch.Tensor) -> int:
    """Row pitch (elements) to pass with a ``[n, d]`` operand that ``kernel_operand`` accepted.  A single row has no
    pitch: PyTorch calls a ``[1, d]`` tensor with unit inner stride contiguous whatever its stride(0) (``x.t()`` of a
    ``[d, 1]`` tensor has strides ``(1, 1)``), so ``d`` is passed, which the kernels accept."""
    return t.shape[1] if t.shape[0] <= 1 else t.stride(0)


def kernel_operand(t: torch.Tensor) -> tuple[torch.Tensor, int]:
    """``(t, pitch)`` when the kernels can read or write the ``[n, d]`` fp32 tensor ``t`` in place: unit inner stride,
    row pitch >= d and a multiple of 4 elements, base 16 B aligned (include/gca.h).  Otherwise a dense copy and ``d``.
    Column windows of wider tensors and gradients of ``torch.cat`` outputs pass as they are; broadcast gradients
    (stride 0, e.g. of ``y.sum(0)``), odd pitches and misaligned views are copied."""
    n, d = t.shape
    if t.stride(-1) == 1 and t.data_ptr() % 16 == 0:
        ld = row_pitch(t)
        if ld >= d and ld % 4 == 0:
            return t, ld
    return t.clone(memory_format=torch.contiguous_format), d


class _GConvAdapterFunction(torch.autograd.Function):
    """Y = s * (Ahat act(Ahat X Wd^T + bd) Wu^T + bu [+ X]) and its gradients, one graph handle.

    The host side is kept thin on purpose (the small configs are launch-bound): one device allocation per
    direction, carved into the tensors the kernels need, and one C call."""

    @staticmethod
    def forward(ctx, x, w_down, b_down, w_up, b_up, scalar, graph: GraphStructure, act: int, skip: bool, addend=None):
        """``addend`` (optional, [n, d] fp32): Y += addend inside the last kernel (gca_forward_add); its gradient is gY."""
        lib = _cabi.load()
        x, ldx = kernel_operand(x)
        n, d = x.shape
        r = w_down.shape[0]
        dev = x.device
        stream = _raw_stream(dev)
        if not w_down.is_contiguous():
            w_down = w_down.contiguous()
        if not w_up.is_contiguous():
            w_up = w_up.contiguous()
        b_down, b_up = b_down.contiguous(), b_up.contiguous()
        silu = act == _cabi.ACT["silu"]
        y = torch.empty((n, d), dtype=torch.float32, device=dev)
        # one allocation: [Z' | H2 | (H1) | per-call workspace (projection scratch, hub partial sums)]
        rw = _align(4 * max(n, 1) * r)
        ws_bytes = _sizes(lib, graph, d, r)[0]
        buf = torch.empty((3 if silu else 2) * rw + ws_bytes, dtype=torch.uint8, device=dev)
        base = buf.data_ptr()
        zp_ptr, h2_ptr = base, base + rw
        h1_ptr = base + 2 * rw if silu else None
        ws_ptr = base + (3 if silu else 2) * rw
        if addend is None:
            _cabi.check(lib.gca_forward(graph.handle, x.data_ptr(), ldx, w_down.data_ptr(), b_down.data_ptr(),
                                        w_up.data_ptr(), b_up.data_ptr(), _ptr(scalar), act, int(skip), ws_ptr,
                                        zp_ptr, h1_ptr, h2_ptr, y.data_ptr(), y.stride(0), d, r, stream), "gca_forward")
        else:
            addend, lda = kernel_operand(addend)
            _cabi.check(lib.gca_forward_add(graph.handle, x.data_ptr(), ldx, w_down.data_ptr(), b_down.data_ptr(),
                                            w_up.data_ptr(), b_up.data_ptr(), _ptr(scalar), act, int(skip), ws_ptr,
                                            zp_ptr, h1_ptr, h2_ptr, addend.data_ptr(), lda, y.data_ptr(), y.stride(0), d, r,
                                            stream), "gca_forward_add")
        ctx.has_addend = addend is not None
        ctx.graph, ctx.act, ctx.skip = graph, act, skip
        ctx.has_scalar = scalar is not None
        ctx.silu, ctx.rw = silu, rw
        saved = [x, w_down, w_up, b_up, buf]
        if scalar is not None:
            saved.append(scalar)
        ctx.save_for_backward(*saved)
        if DEBUG_KEEP_SAVED:
            nr = n * r
            f = buf[:(3 if silu else 2) * rw].view(torch.float32)
            LAST_SAVED.update(zp=f[:nr].view(n, r), h2=f[rw // 4:rw // 4 + nr].view(n, r),
                              h1=f[2 * rw // 4:2 * rw // 4 + nr].view(n, r) if silu else None)
        return y

    @staticmethod
    def backward(ctx, g_y):
        lib = _cabi.load()
        saved = ctx.saved_tensors
        x, w_down, w_up, b_up, buf = saved[:5]
        scalar = saved[5] if ctx.has_scalar else None
        n, d = x.shape
        r = w_down.shape[0]
        dev = x.device
        g_y_in = g_y
        g_y, ldg = kernel_operand(g_y)
        stream = _raw_stream(dev)
        rw = ctx.rw
        base = buf.data_ptr()
        zp_ptr, h2_ptr = base, base + rw
        h1_ptr = base + 2 * rw if ctx.silu else None
        need_x = ctx.needs_input_grad[0]
        g_a = g_y_in if ctx.has_addend and ctx.needs_input_grad[9] else None     # d(Y + A) / dA = identity
        g_x = torch.empty((n, d), dtype=torch.float32, device=dev) if need_x else None
        # one fresh (non-view) tensor per parameter gradient, so autograd's AccumulateGrad can take ownership
        # of it instead of cloning
        g_wd = torch.empty((r, d), dtype=torch.float32, device=dev)
        g_wu = torch.empty((d, r), dtype=torch.float32, device=dev)
        g_bu = torch.empty((d,), dtype=torch.float32, device=dev)
        g_bd = torch.empty((r,), dtype=torch.float32, device=dev)
        g_s = torch.empty((1,), dtype=torch.float32, device=dev) if scalar is not None else None
        ws = torch.empty(_sizes(lib, ctx.graph, d, r)[1], dtype=torch.uint8, device=dev)
        _cabi.check(lib.gca_backward(ctx.graph.handle, g_y.data_ptr(), ldg, x.data_ptr(), row_pitch(x),
                                     zp_ptr, h1_ptr, h2_ptr, w_down.data_ptr(), w_up.data_ptr(),
                                     b_up.data_ptr(), _ptr(scalar), ctx.act, int(ctx.skip), ws.data_ptr(),
                                     _ptr(g_x), g_x.stride(0) if need_x else d, g_wd.data_ptr(), g_bd.data_ptr(),
                                     g_wu.data_ptr(), g_bu.data_ptr(), _ptr(g_s), d, r, stream), "gca_backward")
        return g_x, g_wd, g_bd, g_wu, g_bu, g_s, None, None, None, g_a


class _LayerNormScaleFunction(torch.autograd.Function):
    """``LayerNorm(x) * scalar`` (gconv_adapter.py:98-106 with normalization='layer_norm') as one pass forward and one
    pass backward over ``[N, d]`` (gca_layernorm.cu) instead of the stock LayerNorm + mul kernels."""

    @staticmethod
    def forward(ctx, x, weight, bias, scalar, eps: float, addend=None):
        """``addend`` (optional, [n, d] fp32): + addend in the same pass (gca_layernorm_scale_add_fwd); its gradient is gY."""
        lib = _cabi.load()
        x, ldx = kernel_operand(x)
        n, d = x.shape
        dev = x.device
        stream = _raw_stream(dev)
        y = torch.empty((n, d), dtype=torch.float32, device=dev)
        stats = torch.empty((2, max(n, 1)), dtype=torch.float32, device=dev)
        weight = weight.contiguous() if weight is not None else None
        bias = bias.contiguous() if bias is not None else None
        if addend is None:
            _cabi.check(lib.gca_layernorm_scale_fwd(x.data_ptr(), ldx, _ptr(weight), _ptr(bias), _ptr(scalar), float(eps),
                                                    y.data_ptr(), y.stride(0), stats[0].data_ptr(), stats[1].data_ptr(), n, d,
                                                    stream), "gca_layernorm_scale_fwd")
        else:
            addend, lda = kernel_operand(addend)
            _cabi.check(lib.gca_layernorm_scale_add_fwd(x.data_ptr(), ldx, _ptr(weight), _ptr(bias), _ptr(scalar), float(eps),
                                                        addend.data_ptr(), lda, y.data_ptr(), y.stride(0), stats[0].data_ptr(),
                                                        stats[1].data_ptr(), n, d, stream), "gca_layernorm_scale_add_fwd")
        ctx.has_addend = addend is not None
        ctx.has = (weight is not None, bias is not None, scalar is not None)
        ctx.save_for_backward(x, stats, *[t for t in (weight, bias, scalar) if t is not None])
        return y

    @staticmethod
    def backward(ctx, g_y):
        lib = _cabi.load()
        saved = list(ctx.saved_tensors)
        x, stats = saved[0], saved[1]
        rest = saved[2:]
        weight = rest.pop(0) if ctx.has[0] else None
        bias = rest.pop(0) if ctx.has[1] else None
        scalar = rest.pop(0) if ctx.has[2] else None
        n, d = x.shape
        dev = x.device
        g_a = g_y if ctx.has_addend and ctx.needs_input_grad[5] else None       # d(Y + A) / dA = identity
        g_y, ldg = kernel_operand(g_y)
        stream = _raw_stream(dev)
        g_x = torch.empty((n, d), dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        g_w = torch.empty((d,), dtype=torch.float32, device=dev) if weight is not None else None
        g_b = torch.empty((d,), dtype=torch.float32, device=dev) if bias is not None else None
        g_s = torch.empty((1,), dtype=torch.float32, device=dev) if scalar is not None else None
        ws = torch.empty(lib.gca_layernorm_scratch_bytes(d), dtype=torch.uint8, device=dev)
        _cabi.check(lib.gca_layernorm_scale_bwd(g_y.data_ptr(), ldg, x.data_ptr(), row_pitch(x), _ptr(weight),
                                                _ptr(bias), _ptr(scalar), stats[0].data_ptr(), stats[1].data_ptr(), _ptr(g_x),
                                                g_x.stride(0) if g_x is not None else d, _ptr(g_w), _ptr(g_b), _ptr(g_s),
                                                ws.data_ptr(), n, d, stream), "gca_layernorm_scale_bwd")
        return g_x, g_w, g_b, g_s, None, g_a


class _BatchNormScaleFunction(torch.autograd.Function):
    """``BatchNorm1d(x) * scalar`` for a 2-D ``x`` (gconv_adapter.py:98-106 with normalization='batch_norm') as one
    statistics pass and one normalizing pass forward, one reduce pass and one gX pass backward (gca_batchnorm.cu) instead
    of the stock BatchNorm + mul kernels.  ``running_mean`` / ``running_var`` (or None) are updated in place when
    ``training``; without ``training`` they are the statistics used."""

    @staticmethod
    def forward(ctx, x, weight, bias, scalar, running_mean, running_var, training: bool, momentum: float, eps: float):
        lib = _cabi.load()
        x, ldx = kernel_operand(x)
        n, d = x.shape
        dev = x.device
        stream = _raw_stream(dev)
        y = torch.empty((n, d), dtype=torch.float32, device=dev)
        stats = torch.empty((2, d), dtype=torch.float32, device=dev)
        ws = torch.empty(lib.gca_batchnorm_scratch_bytes(d), dtype=torch.uint8, device=dev)
        weight = weight.contiguous() if weight is not None else None
        bias = bias.contiguous() if bias is not None else None
        _cabi.check(lib.gca_batchnorm_scale_fwd(x.data_ptr(), ldx, _ptr(weight), _ptr(bias), _ptr(scalar), float(eps),
                                                int(training), float(momentum), _ptr(running_mean), _ptr(running_var),
                                                y.data_ptr(), y.stride(0), stats[0].data_ptr(), stats[1].data_ptr(),
                                                ws.data_ptr(), n, d, stream), "gca_batchnorm_scale_fwd")
        ctx.training = bool(training)
        ctx.has = (weight is not None, bias is not None, scalar is not None)
        ctx.save_for_backward(x, stats, *[t for t in (weight, bias, scalar) if t is not None])
        return y

    @staticmethod
    def backward(ctx, g_y):
        lib = _cabi.load()
        saved = list(ctx.saved_tensors)
        x, stats = saved[0], saved[1]
        rest = saved[2:]
        weight = rest.pop(0) if ctx.has[0] else None
        bias = rest.pop(0) if ctx.has[1] else None
        scalar = rest.pop(0) if ctx.has[2] else None
        n, d = x.shape
        dev = x.device
        g_y, ldg = kernel_operand(g_y)
        stream = _raw_stream(dev)
        g_x = torch.empty((n, d), dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        g_w = torch.empty((d,), dtype=torch.float32, device=dev) if weight is not None else None
        g_b = torch.empty((d,), dtype=torch.float32, device=dev) if bias is not None else None
        g_s = torch.empty((1,), dtype=torch.float32, device=dev) if scalar is not None else None
        ws = torch.empty(lib.gca_batchnorm_scratch_bytes(d), dtype=torch.uint8, device=dev)
        _cabi.check(lib.gca_batchnorm_scale_bwd(g_y.data_ptr(), ldg, x.data_ptr(), row_pitch(x), _ptr(weight), _ptr(bias),
                                                _ptr(scalar), stats[0].data_ptr(), stats[1].data_ptr(), int(ctx.training),
                                                _ptr(g_x), g_x.stride(0) if g_x is not None else d, _ptr(g_w), _ptr(g_b),
                                                _ptr(g_s), ws.data_ptr(), n, d, stream), "gca_batchnorm_scale_bwd")
        return g_x, g_w, g_b, g_s, None, None, None, None, None


class _Lin(nn.Module):
    """Holds ``lin.weight`` [out, in] exactly where PyG's ``GCNConv.lin`` (bias-free Linear) has it."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))


class _GCNConvParams(nn.Module):
    """Parameter container with the attribute layout of ``torch_geometric.nn.GCNConv`` as the
    reference touches it (``.lin.weight``, ``.bias``: gconv_adapter.py:73-78).  Construction
    consumes the RNG like PyG does (glorot on the weight, zeros on the bias)."""

    def __init__(self, in_channels: int, out_channels: int, normalize: bool = True):
        super().__init__()
        self.in_channels, self.out_channels, self.normalize = in_channels, out_channels, normalize
        self.lin = _Lin(in_channels, out_channels)
        self.bias = nn.Parameter(torch.zeros(out_channels))
        a = math.sqrt(6.0 / (in_channels + out_channels))
        with torch.no_grad():
            self.lin.weight.uniform_(-a, a)

    def extra_repr(self) -> str:
        return f"{self.in_channels}, {self.out_channels}, normalize={self.normalize}"


class GConvAdapter(nn.Module):
    """GConv-Adapter (drop-in for ``src.finetune.gconv_adapter.GConvAdapter``).

    Args:
        hidden_size (int): Size of the hidden layer.
        bottleneck_size (int): Size of the bottleneck layer.
        conv_type (str): Type of graph convolution; only 'gcn' can be constructed ('sage' and
            'gat' are accepted names in the reference but its constructor fails for them).
        non_linearity (str): 'relu', 'silu' or 'none'.
        normalization (str): 'batch_norm', 'layer_norm' or 'none'.
        learnable_scalar (bool): multiply the output by a learnable scalar.
        skip_connection (bool): add the input to the output.
        normalize (bool): add self-loops and use symmetric normalisation coefficients.

    Raises:
        ValueError: If an invalid conv_type, non_linearity, or normalization is provided.
    """

    def __init__(self, hidden_size: int, bottleneck_size: int,
                 conv_type: str = 'gcn', non_linearity: str = 'relu',
                 normalization: str = 'none', learnable_scalar: bool = False,
                 skip_connection: bool = True, normalize: bool = True):
        super().__init__()
        if conv_type == 'gcn':
            pass
        elif conv_type in ('sage', 'gat'):
            # reference: SAGEConv / GATConv have no `.lin.weight`, so its own constructor raises
            # AttributeError at gconv_adapter.py:73 (GATConv already rejects `normalize=` at :40).
            raise AttributeError(f"'{conv_type}' convolutions have no attribute 'lin': the reference "
                                 "GConvAdapter cannot be constructed with this conv_type either")
        else:
            raise ValueError("Invalid conv_type. Supported types: 'gcn', 'sage', 'gat'.")
        self.conv_down = _GCNConvParams(hidden_size, bottleneck_size, normalize=normalize)
        self.conv_up = _GCNConvParams(bottleneck_size, hidden_size, normalize=normalize)

        if non_linearity == 'relu':
            self.act_fn = nn.ReLU()
        elif non_linearity == 'silu':
            self.act_fn = nn.SiLU()
        elif non_linearity == 'none':
            self.act_fn = nn.Identity()
        else:
            raise ValueError("Invalid non_linearity. Supported types: 'relu', 'silu', 'none'.")
        self._act = _cabi.ACT[non_linearity]

        if normalization == 'batch_norm':
            self.normalization = nn.BatchNorm1d(hidden_size)
        elif normalization == 'layer_norm':
            self.normalization = nn.LayerNorm(hidden_size)
        elif normalization == 'none':
            self.normalization = None
        else:
            raise ValueError("Invalid normalization. Supported types: 'batch_norm', 'layer_norm', 'none'.")

        if learnable_scalar:
            self.scalar = nn.Parameter(torch.ones(1))
        else:
            self.scalar = None

        self.skip_connection = skip_connection
        self.normalize = normalize
        self.hidden_size = hidden_size
        self.bottleneck_size = bottleneck_size

        torch.nn.init.normal_(self.conv_down.lin.weight, mean=0.0, std=1e-5)
        torch.nn.init.zeros_(self.conv_down.bias)
        torch.nn.init.normal_(self.conv_up.lin.weight, mean=0.0, std=1e-5)
        torch.nn.init.zeros_(self.conv_up.bias)

        # graph structures are shared across adapters / layers / positions through this cache
        self.graph_cache: GraphCache = GLOBAL_GRAPH_CACHE
        # True: check node ids right after the build (one stream synchronisation per NEW edge_index); "lazy": no
        # synchronisation - the check result is picked up at a later call (use it when the graph changes every step);
        # False: never checked (out-of-range ids are then ignored by the build)
        self.validate_edge_index = True
        self.fuse_layer_norm = True       # normalization='layer_norm': LayerNorm + scalar as one fused pass per direction
        self.fuse_batch_norm = True       # normalization='batch_norm': BatchNorm1d + scalar as the fused kernels

    # ------------------------------------------------------------------------------
    def _padded_params(self, d: int, r: int):
        """Kernels take d % 4 == 0 and r in {8,16,32,64,128}; other sizes are zero-padded (exact:
        padded channels carry 0 through bias 0 and relu/silu/identity, and their gradients are
        dropped by autograd's slice)."""
        dp = (d + 3) // 4 * 4
        rp = next((c for c in _FAST_RANKS if c >= r), None)
        if rp is None:
            raise RuntimeError(f"gconv_adapter_b200: bottleneck_size {r} > {_FAST_RANKS[-1]} is not supported by the CUDA kernels")
        wd, bd, wu, bu = self.conv_down.lin.weight, self.conv_down.bias, self.conv_up.lin.weight, self.conv_up.bias
        if dp != d or rp != r:
            wd = F.pad(wd, (0, dp - d, 0, rp - r))
            bd = F.pad(bd, (0, rp - r))
            wu = F.pad(wu, (0, rp - r, 0, dp - d))
            bu = F.pad(bu, (0, dp - d))
        return dp, wd, bd, wu, bu

    def graph_for(self, edge_index: torch.Tensor, num_nodes: int) -> GraphStructure:
        return self.graph_cache.get(edge_index, num_nodes, self.normalize, validate=self.validate_edge_index)

    def _ln_fused(self, d: int) -> bool:
        """normalization='layer_norm' runs as the fused LayerNorm + scalar kernels (else as stock torch ops)."""
        ln = self.normalization
        return (self.fuse_layer_norm and d % 4 == 0 and d <= 1024 and tuple(ln.normalized_shape) == (d,)
                and os.environ.get("GCA_DISABLE_LN_FUSE", "0") != "1")

    def _bn_fused(self, out: torch.Tensor) -> bool:
        """normalization='batch_norm' on the adapter's output ``out`` runs as the fused BatchNorm1d + scalar kernels: a
        plain ``nn.BatchNorm1d`` (not a subclass, whose forward may differ) over ``d`` features, a 2-D fp32 ``out`` with
        more than one row, d % 4 == 0 and fp32 parameters / buffers.  Otherwise the stock ops run.  ``out`` comes from
        the adapter kernels, so it is on the GPU."""
        bn = self.normalization
        if not (self.fuse_batch_norm and type(bn) is nn.BatchNorm1d and out.dim() == 2 and out.dtype == torch.float32):
            return False
        n, d = out.shape
        if n <= 1 or d % 4 != 0 or bn.num_features != d:
            return False
        if any(t is not None and t.dtype != torch.float32 for t in (bn.weight, bn.bias, bn.running_mean, bn.running_var)):
            return False
        return os.environ.get("GCA_DISABLE_BN_FUSE", "0") != "1"

    def _batch_norm_scale(self, out: torch.Tensor) -> torch.Tensor:
        """``self.normalization(out) * self.scalar`` through _BatchNormScaleFunction, with the bookkeeping of
        ``torch.nn.modules.batchnorm._BatchNorm.forward`` (num_batches_tracked, the averaging factor, which statistics and
        buffers are used); the kernels update the running buffers."""
        bn = self.normalization
        factor = 0.0 if bn.momentum is None else bn.momentum
        if bn.training and bn.track_running_stats:
            if bn.num_batches_tracked is not None:
                bn.num_batches_tracked.add_(1)
                if bn.momentum is None:         # cumulative moving average
                    factor = 1.0 / float(bn.num_batches_tracked)
                else:
                    factor = bn.momentum
        bn_training = True if bn.training else (bn.running_mean is None and bn.running_var is None)
        use_buffers = not bn.training or bn.track_running_stats
        return _BatchNormScaleFunction.apply(out, bn.weight, bn.bias, self.scalar,
                                             bn.running_mean if use_buffers else None,
                                             bn.running_var if use_buffers else None, bn_training, factor, bn.eps)

    def fuses_add(self, x: torch.Tensor, h) -> bool:
        """Whether ``forward(x, ..., add_to=h)`` adds ``h`` in the store of its last kernel: ``h`` is an fp32 tensor on
        x's device with exactly x's (= the output's) shape, the hidden size needs no column padding (d % 4 == 0), and
        the tail after the adapter is nothing or the fused LayerNorm.  Any row pitch is fine (odd pitches and broadcast
        strides are copied, as for x).  Otherwise ``h + out`` runs as a stock op, with the same result."""
        if not isinstance(h, torch.Tensor) or h.dtype != torch.float32 or h.device != x.device or h.shape != x.shape:
            return False
        d = x.shape[-1]
        if d % 4 != 0:
            return False
        if self.normalization is None:
            return True
        return isinstance(self.normalization, nn.LayerNorm) and self._ln_fused(d)

    def forward(self, x: torch.Tensor, edge_index: torch.Tensor, edge_attr: torch.Tensor = None, *,
                add_to: Optional[torch.Tensor] = None) -> torch.Tensor:
        """
        Args:
            x: node features ``[N, hidden_size]`` or ``[1, N, hidden_size]`` (fp32, CUDA).
            edge_index: ``[2, num_edges]`` int64, row 0 = source, row 1 = target.
            edge_attr: accepted and ignored, as in the reference (gconv_adapter.py:80,92).
            add_to: optional ``h``: return ``h + adapter(x)`` (parallel insertion, src/models/inductive/gnn.py:120-124),
                with the same value, shape, dtype and gradients as that expression.  See ``fuses_add`` for when the
                add happens inside the last kernel (bitwise the same result as the separate add).
        Returns:
            A new tensor of the same shape as ``x`` (of ``h + out``'s shape and dtype with ``add_to``).
        """
        if add_to is not None and not self.fuses_add(x, add_to):
            return add_to + self._forward(x, edge_index, edge_attr, None)
        return self._forward(x, edge_index, edge_attr, add_to)

    def _forward(self, x: torch.Tensor, edge_index: torch.Tensor, edge_attr, addend: Optional[torch.Tensor]) -> torch.Tensor:
        """The adapter's output (+ ``addend``, which ``fuses_add`` accepted, when given)."""
        if not x.is_cuda:
            raise RuntimeError("gconv_adapter_b200.GConvAdapter runs on CUDA (sm_100a) only; there is no CPU path")
        if x.dtype != torch.float32:
            raise RuntimeError("gconv_adapter_b200.GConvAdapter computes in fp32 like the reference; got " + str(x.dtype))
        if x.dim() == 3 and x.size(0) != 1:
            # PyG's node_dim = -2: a leading batch dimension shares the graph; the fused normalisation / scalar tail is
            # row-wise (LayerNorm) or per-call (BatchNorm1d rejects 3-D like the reference's does), so slices are independent
            return torch.stack([self._forward(x[b], edge_index, edge_attr, None if addend is None else addend[b])
                                for b in range(x.size(0))], dim=0)
        if x.dim() == 3:
            x2 = x[0]
        elif x.dim() == 2:
            x2 = x
        else:
            raise RuntimeError("x must be [N, hidden] or [1, N, hidden]")
        n, d = x2.shape
        if d != self.hidden_size:
            raise RuntimeError(f"expected hidden size {self.hidden_size}, got {d}")
        dp, wd, bd, wu, bu = self._padded_params(d, self.bottleneck_size)
        if dp != d:
            x2 = F.pad(x2, (0, dp - d))
        graph = self.graph_for(edge_index, n)
        fused_scalar = self.scalar if self.normalization is None else None
        add2 = None if addend is None else (addend[0] if addend.dim() == 3 else addend)
        # the addend goes where the adapter's output is finished: the last kernel, or the fused LayerNorm after it
        out = _GConvAdapterFunction.apply(x2, wd, bd, wu, bu, fused_scalar, graph, self._act, self.skip_connection,
                                          add2 if self.normalization is None else None)
        if dp != d:
            out = out[:, :d]
        if x.dim() == 3:
            out = out.unsqueeze(0)

        # normalisation needs batch / row statistics of the finished sum: the fused tails or stock torch ops,
        # then the scalar (which is fused into the adapter kernel only when no normalisation sits between)
        if isinstance(self.normalization, nn.BatchNorm1d):
            if out.size(0) > 1:
                if self._bn_fused(out):
                    # BatchNorm1d + scalar: statistics + one pass forward, one reduce + one gX pass backward
                    return self._batch_norm_scale(out)
                out = self.normalization(out)
        elif isinstance(self.normalization, nn.LayerNorm):
            ln = self.normalization
            if self._ln_fused(d):
                # LayerNorm + scalar in one pass forward / one pass backward (the scalar is part of the kernel)
                flat = _LayerNormScaleFunction.apply(out.reshape(-1, d), ln.weight, ln.bias, self.scalar, ln.eps,
                                                     None if add2 is None else add2.reshape(-1, d))
                return flat.reshape(out.shape)
            out = ln(out)
        if self.normalization is not None and self.scalar is not None:
            out = out * self.scalar
        return out

    def extra_repr(self) -> str:
        return (f"hidden_size={self.hidden_size}, bottleneck_size={self.bottleneck_size}, "
                f"skip_connection={self.skip_connection}, normalize={self.normalize}")
