"""Row-partitioned GConv-Adapter over several GPUs (one process per GPU, torch.distributed / NCCL).

The reference is single-process (SURVEY.md section 2: no torch.distributed anywhere); this is the
scale-out the north star asks for: node rows are split into contiguous blocks, every rank owns the
rows of X / Y / all gradients and the CSR rows (targets) of its block, and only the r-wide operand of
each sparse hop crosses NVLink:

    forward : P' -> gather -> Z' -> gather -> Y                    (2 gathers of [N, r] fp32)
    backward: gH2' -> gather -> gH1' -> gather -> gX, then one all-reduce of the
              2 d r + d + r + 1 parameter-gradient floats.

Communication therefore scales with the adapter rank r, never with the hidden width d.

Two exchange mechanisms (``comm``):

* ``PeerMemoryComm`` (default on CUDA): the kernel that PRODUCES an r-wide operand stores every finished row straight
  into its peers' gathered buffers over NVLink (``gca_push``, peer memory mapped with CUDA IPC), so the "gather" left
  between two phases is a one-warp barrier kernel, and the gradient all-reduce is one kernel over peer memory with a
  fixed rank order.  No NCCL call inside a step: the whole forward + backward can be captured in a CUDA graph.
* ``CollectiveComm``: ``torch.distributed`` all-gather / all-reduce (NCCL or gloo) - the portable path, used by the CPU
  tests of the orchestration and as a fallback when peer mapping is unavailable (GCA_PARTITION_COMM=nccl).

Shards have equal size S = ceil(N / world) (the last ranks may own fewer or zero real rows), so the
gathered buffer is [world * S, r] and a global node id is directly its row in that buffer.

The dense / sparse phases themselves are the C-ABI calls of include/gca.h (``CudaPhases``); the class
takes the phase backend as an argument only so that the orchestration (bounds, buffers, collectives)
can be exercised on CPU with gloo by the tests, which inject their own checker backend.
"""
from __future__ import annotations

import ctypes as C
import os
import warnings
from typing import Optional

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _cabi
from .finetune.gconv_adapter import GConvAdapter, kernel_operand, row_pitch
from .graphs.csr import GraphStructure


# Test hook: when True, the forward keeps this rank's rows of Z' (the ReLU decisions) in LAST_SAVED["zp"].
DEBUG_KEEP_SAVED = False
LAST_SAVED: dict = {}


def shard_size(num_nodes: int, world: int) -> int:
    return (num_nodes + world - 1) // world


def row_block(num_nodes: int, world: int, rank: int) -> tuple[int, int]:
    """[lo, hi) of the rows owned by ``rank``; empty for trailing ranks when N < world * S."""
    s = shard_size(num_nodes, world)
    lo = min(num_nodes, rank * s)
    return lo, min(num_nodes, lo + s)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class CudaPhases:
    """Phase backend = libgca (the product path)."""

    def __init__(self):
        self.lib = _cabi.load()

    @staticmethod
    def _stream(t: torch.Tensor) -> int:
        return torch.cuda.current_stream(t.device).cuda_stream

    @staticmethod
    def _push(push):
        return C.byref(push) if push is not None else None

    def build_graph(self, edge_index, num_nodes, normalize, lo, hi):
        return GraphStructure(edge_index, num_nodes, normalize, lo, hi)

    def hub_scratch(self, g, device, r):
        """Per-call scratch for the rank-r partial sums of hub rows (None when the graph has no row longer than 512)."""
        nbytes = self.lib.gca_hub_scratch_bytes_r(g.handle, r)
        return torch.empty(nbytes, dtype=torch.uint8, device=device) if nbytes else None

    def fwd_project(self, g, x, wd, out_local, push=None):
        d, r = x.shape[1], wd.shape[0]
        _cabi.check(self.lib.gca_fwd_project(g.handle, x.data_ptr(), row_pitch(x), wd.data_ptr(), out_local.data_ptr(),
                                             self._push(push), d, r, self._stream(x)), "gca_fwd_project")

    def fwd_hop1(self, g, p_full, bd, act, z_local, h1_local, hub=None, push=None):
        _cabi.check(self.lib.gca_fwd_hop1(g.handle, p_full.data_ptr(), bd.data_ptr(), act, z_local.data_ptr(),
                                          _ptr(h1_local), _ptr(hub), self._push(push), bd.shape[0], self._stream(p_full)),
                    "gca_fwd_hop1")

    def fwd_hop2_up(self, g, z_full, x, wu, bu, scalar, skip, h2_local, y, hub=None):
        d, r = wu.shape
        _cabi.check(self.lib.gca_fwd_hop2_up(g.handle, z_full.data_ptr(), x.data_ptr(), row_pitch(x), wu.data_ptr(),
                                             bu.data_ptr(), _ptr(scalar), int(skip), h2_local.data_ptr(), y.data_ptr(),
                                             y.stride(0), _ptr(hub), d, r, self._stream(x)), "gca_fwd_hop2_up")

    def fwd_hop2_up_add(self, g, z_full, x, wu, bu, scalar, skip, h2_local, a, y, hub=None):
        """fwd_hop2_up, then y += a in the same kernel (a: the local rows of the parallel-insertion addend)."""
        d, r = wu.shape
        _cabi.check(self.lib.gca_fwd_hop2_up_add(g.handle, z_full.data_ptr(), x.data_ptr(), row_pitch(x), wu.data_ptr(),
                                                 bu.data_ptr(), _ptr(scalar), int(skip), h2_local.data_ptr(), a.data_ptr(),
                                                 row_pitch(a), y.data_ptr(), y.stride(0), _ptr(hub), d, r, self._stream(x)),
                    "gca_fwd_hop2_up_add")

    def bwd_scratch(self, d, r, device):
        return torch.empty(self.lib.gca_bwd_scratch_bytes(d, r), dtype=torch.uint8, device=device)

    def bwd_up(self, g, gy, h2_local, wu, scalar, gh2_local, scratch, push=None):
        d, r = wu.shape
        _cabi.check(self.lib.gca_bwd_up(g.handle, gy.data_ptr(), row_pitch(gy), h2_local.data_ptr(), wu.data_ptr(),
                                        _ptr(scalar), gh2_local.data_ptr(), scratch.data_ptr(), self._push(push), d, r,
                                        self._stream(gy)), "gca_bwd_up")

    def bwd_hop2(self, g, gh2_full, z_local, h1_local, act, gh1_local, scratch, hub=None, push=None):
        r = gh2_full.shape[1]
        _cabi.check(self.lib.gca_bwd_hop2(g.handle, gh2_full.data_ptr(), z_local.data_ptr(), _ptr(h1_local), act,
                                          gh1_local.data_ptr(), scratch.data_ptr(), _ptr(hub), self._push(push), r,
                                          self._stream(gh2_full)), "gca_bwd_hop2")

    def bwd_hop1_down(self, g, gh1_full, x, gy, wd, scalar, skip, gp_local, gx, scratch, hub=None):
        r, d = wd.shape
        _cabi.check(self.lib.gca_bwd_hop1_down(g.handle, gh1_full.data_ptr(), x.data_ptr(), row_pitch(x), gy.data_ptr(),
                                               row_pitch(gy), wd.data_ptr(), _ptr(scalar), int(skip), gp_local.data_ptr(),
                                               _ptr(gx), gx.stride(0) if gx is not None else d, scratch.data_ptr(),
                                               _ptr(hub), d, r, self._stream(x)), "gca_bwd_hop1_down")

    def bwd_finalize(self, scratch, wu, bu, scalar, skip, g_wd, g_bd, g_wu, g_bu, g_s):
        d, r = wu.shape
        _cabi.check(self.lib.gca_bwd_finalize(scratch.data_ptr(), wu.data_ptr(), bu.data_ptr(), _ptr(scalar), int(skip),
                                              g_wd.data_ptr(), g_bd.data_ptr(), g_wu.data_ptr(), g_bu.data_ptr(),
                                              _ptr(g_s), d, r, self._stream(wu)), "gca_bwd_finalize")


# ---------------------------------------------------------------------------------------------------------------
# exchange mechanisms
# ---------------------------------------------------------------------------------------------------------------
GATHERED = ("p", "z", "gh2", "gh1")      # the four r-wide operands that every rank needs in full


class CollectiveComm:
    """torch.distributed collectives (NCCL / gloo): every gather is an in-place all_gather_into_tensor."""

    fused_push = False

    def __init__(self, group=None):
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)

    def buffers(self, rows: int, r: int, device, which):
        return {k: torch.empty((rows, r), dtype=torch.float32, device=device) for k in which}

    def push(self, name, lo, r):
        return None

    def gather(self, full: torch.Tensor, lo: int, s: int) -> None:
        if self.world > 1:
            dist.all_gather_into_tensor(full, full[lo:lo + s], group=self.group)

    def allreduce_(self, flat: torch.Tensor) -> None:
        if self.world > 1:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)


class PeerMemoryComm:
    """NVLink peer memory: gathered buffers live in a symmetric arena (gconv_adapter_b200/peer.py); producers push
    their rows into the peers' copies while they compute, a gather is only the barrier kernel."""

    fused_push = True

    def __init__(self, num_nodes: int, d: int, r: int, group=None, device=None):
        from .peer import PeerGroup
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.rows = self.world * shard_size(num_nodes, self.world)
        self.r = r
        self.buf_bytes = 4 * self.rows * r
        self.pg = PeerGroup([self.buf_bytes] * len(GATHERED), slot_floats=2 * d * r + d + r + 1, group=group, device=device)
        self._views = {k: self.pg.region(i, self.buf_bytes).view(torch.float32).view(self.rows, r) for i, k in enumerate(GATHERED)}

    def buffers(self, rows: int, r: int, device, which):
        assert rows == self.rows and r == self.r
        return {k: self._views[k] for k in which}

    def push(self, name, lo, r):
        return self.pg.push_to_peers(GATHERED.index(name), 4 * lo * r)

    def gather(self, full: torch.Tensor, lo: int, s: int) -> None:
        self.pg.barrier()

    def allreduce_(self, flat: torch.Tensor) -> None:
        self.pg.allreduce_(flat)

    def close(self) -> None:
        self._views = {}
        self.pg.close()


class _PartitionedFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w_down, b_down, w_up, b_up, scalar, graph, act, skip, num_nodes, comm, backend, addend=None):
        world, rank = comm.world, comm.rank
        s = shard_size(num_nodes, world)
        lo = rank * s
        n, d = x.shape
        r = w_down.shape[0]
        dev = x.device
        w_down, b_down, w_up, b_up = (t.contiguous() for t in (w_down, b_down, w_up, b_up))
        # padded rows (beyond N) of the gathered buffers are never referenced by any neighbour id, so the
        # buffers need no initialisation: every real row is written by its owner's kernel or arrives from a peer
        bufs = comm.buffers(world * s, r, dev, ("p", "z"))
        p_full, z_full = bufs["p"], bufs["z"]
        h2 = torch.empty((max(n, 1), r), dtype=torch.float32, device=dev)
        h1 = torch.empty((max(n, 1), r), dtype=torch.float32, device=dev) if act == _cabi.ACT["silu"] else None
        y = torch.empty((n, d), dtype=torch.float32, device=dev)
        hub = backend.hub_scratch(graph, dev, r) if hasattr(backend, "hub_scratch") else None
        if n > 0:
            backend.fwd_project(graph, x, w_down, p_full[lo:lo + n], push=comm.push("p", lo, r))
        comm.gather(p_full, lo, s)
        if n > 0:
            backend.fwd_hop1(graph, p_full, b_down, act, z_full[lo:lo + n], h1, hub, push=comm.push("z", lo, r))
        comm.gather(z_full, lo, s)
        if n > 0:
            if addend is None:
                backend.fwd_hop2_up(graph, z_full, x, w_up, b_up, scalar, skip, h2, y, hub)
            else:
                backend.fwd_hop2_up_add(graph, z_full, x, w_up, b_up, scalar, skip, h2, kernel_operand(addend)[0], y, hub)
        ctx.has_addend = addend is not None
        ctx.graph, ctx.act, ctx.skip, ctx.comm, ctx.backend = graph, act, skip, comm, backend
        ctx.meta = (world, s, lo, n, d, r)
        ctx.has_scalar, ctx.has_h1 = scalar is not None, h1 is not None
        # only this rank's rows of Z' are needed again (activation mask): with shared gathered buffers (peer arena)
        # they are copied out, so that another forward may run before this backward
        z_local = z_full[lo:lo + n].clone() if comm.fused_push else z_full[lo:lo + n]
        saved = [x, w_down, w_up, b_up, z_local, h2]
        if scalar is not None:
            saved.append(scalar)
        if h1 is not None:
            saved.append(h1)
        ctx.save_for_backward(*saved)
        if DEBUG_KEEP_SAVED:
            LAST_SAVED["zp"] = z_local
        return y

    @staticmethod
    def backward(ctx, g_y):
        saved = list(ctx.saved_tensors)
        x, w_down, w_up, b_up, z_local, h2 = saved[:6]
        rest = saved[6:]
        scalar = rest.pop(0) if ctx.has_scalar else None
        h1 = rest.pop(0) if ctx.has_h1 else None
        world, s, lo, n, d, r = ctx.meta
        backend, graph, comm = ctx.backend, ctx.graph, ctx.comm
        dev = x.device
        g_a = g_y if ctx.has_addend and ctx.needs_input_grad[12] else None      # d(Y + A) / dA = identity
        g_y, _ = kernel_operand(g_y)
        bufs = comm.buffers(world * s, r, dev, ("gh2", "gh1"))
        gh2_full, gh1_full = bufs["gh2"], bufs["gh1"]
        gp = torch.empty((max(n + (n & 1), 2), r), dtype=torch.float32, device=dev)     # even row count (gca_bwd_hop1_down)
        need_x = ctx.needs_input_grad[0]
        g_x = torch.empty((n, d), dtype=torch.float32, device=dev) if need_x else None
        # parameter gradients of this rank's rows, packed for ONE all-reduce
        flat = torch.zeros(2 * d * r + d + r + 1, dtype=torch.float32, device=dev)
        g_wd = flat[0:d * r].view(r, d)
        g_wu = flat[d * r:2 * d * r].view(d, r)
        g_bu = flat[2 * d * r:2 * d * r + d]
        g_bd = flat[2 * d * r + d:2 * d * r + d + r]
        g_s = flat[2 * d * r + d + r:]
        hub = backend.hub_scratch(graph, dev, r) if hasattr(backend, "hub_scratch") else None
        if n > 0:
            scratch = backend.bwd_scratch(d, r, dev)
            # one pass over gY: gH2' (pushed to the peers row by row) together with the gWu / gbu partial sums
            backend.bwd_up(graph, g_y, h2, w_up, scalar, gh2_full[lo:lo + n], scratch, push=comm.push("gh2", lo, r))
        comm.gather(gh2_full, lo, s)
        if n > 0:
            backend.bwd_hop2(graph, gh2_full, z_local, h1, ctx.act, gh1_full[lo:lo + n], scratch, hub, push=comm.push("gh1", lo, r))
        comm.gather(gh1_full, lo, s)
        if n > 0:
            backend.bwd_hop1_down(graph, gh1_full, x, g_y, w_down, scalar, ctx.skip, gp, g_x, scratch, hub)
            backend.bwd_finalize(scratch, w_up, b_up, scalar, ctx.skip, g_wd, g_bd, g_wu, g_bu,
                                 g_s if scalar is not None else None)
        comm.allreduce_(flat)
        return (g_x, g_wd, g_bd, g_wu, g_bu, g_s.clone() if scalar is not None else None,
                None, None, None, None, None, None, g_a)


class _AllReduceGrad(torch.autograd.Function):
    """Identity whose backward sums the gradient over the ranks (for parameters used by row-local
    torch ops after the fused kernel: LayerNorm affine, unfused scalar)."""

    @staticmethod
    def forward(ctx, t, group):
        ctx.group = group
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous().clone()
        if dist.get_world_size(ctx.group) > 1:
            dist.all_reduce(g, op=dist.ReduceOp.SUM, group=ctx.group)
        return g, None


class PartitionedGConvAdapter(GConvAdapter):
    """``GConvAdapter`` whose forward takes this rank's ROW BLOCK of x (``row_block(N, world, rank)``)
    and the FULL ``edge_index``; returns the same rows of the output.  Parameter gradients come back
    already summed over ranks, so every replica applies the same optimizer step.  Only the fused
    configuration (normalization='none') is partitioned; LayerNorm is row-local and works unchanged,
    BatchNorm would need cross-rank statistics and is refused.

    ``comm``: "peer" (NVLink peer memory, default for the CUDA backend), "collective" (torch.distributed
    all-gather / all-reduce), or an object with the comm interface.  Every rank must make the same choice."""

    def __init__(self, *args, process_group=None, phase_backend=None, comm=None, **kwargs):
        super().__init__(*args, **kwargs)
        if isinstance(self.normalization, nn.BatchNorm1d):
            raise ValueError("PartitionedGConvAdapter: batch_norm needs global batch statistics; use 'none' or 'layer_norm'")
        self.process_group = process_group
        self._backend = phase_backend
        self._comm_choice = comm
        self._comm = None
        self._comm_key = None
        self._graphs: dict = {}
        self._captured: list = []

    def _graph(self, edge_index: torch.Tensor, num_nodes: int, lo: int, hi: int):
        key = (edge_index.data_ptr(), edge_index._version, tuple(edge_index.shape), num_nodes, lo, hi, self.normalize)
        hit = self._graphs.get(key)
        if hit is None:
            hit = (self._backend.build_graph(edge_index, num_nodes, self.normalize, lo, hi), edge_index)
            self._graphs.clear()
            self._graphs[key] = hit
        return hit[0]

    def _get_comm(self, num_nodes: int, device):
        choice = self._comm_choice
        if choice is None:
            choice = os.environ.get("GCA_PARTITION_COMM") or ("peer" if isinstance(self._backend, CudaPhases) else "collective")
            if choice == "nccl":
                choice = "collective"
        if not isinstance(choice, str):
            return choice
        key = (choice, num_nodes, self.hidden_size, self.bottleneck_size)
        if self._comm is None or self._comm_key != key:
            self.close()
            if choice == "peer" and dist.get_world_size(self.process_group) > 1:
                # mapping the peers' arenas can fail (no peer access between two GPUs, IPC disabled in a container):
                # the ranks agree, and all of them take the torch.distributed exchange instead
                comm, ok = None, 1
                try:
                    comm = PeerMemoryComm(num_nodes, self.hidden_size, self.bottleneck_size, self.process_group, device)
                except Exception as ex:      # noqa: BLE001 - any set-up problem means "use the collectives", on every rank
                    ok = 0
                    warnings.warn(f"NVLink peer-memory exchange unavailable ({type(ex).__name__}: {ex}); using torch.distributed collectives")
                flag = torch.tensor([ok], device=device)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.process_group)
                if flag.item() == 0:
                    if comm is not None:
                        comm.close()
                    comm = CollectiveComm(self.process_group)
                self._comm = comm
            else:
                self._comm = CollectiveComm(self.process_group)
            self._comm_key = key
        return self._comm

    def capture_step(self, step_fn):
        """Capture ``step_fn`` - one training step on STATIC tensors: zero/None the grads, ``y = self(x, ei, N)``,
        ``y.backward(g)`` - in a CUDA graph and return its ``replay`` callable, or None if any rank could not capture
        (the ranks agree, then all stay eager).  With the peer-memory exchange no library collective sits inside a step
        (pushes ride in the producing kernels, barriers and the all-reduce are libgca kernels), so the whole forward +
        backward of every rank is one graph launch.  Collective: every rank calls it at the same point.  The graph is
        owned by the module and destroyed by ``close()`` before the peer arena is unmapped.  Drop every reference to
        outputs / losses of earlier eager steps first: a live autograd graph keeps AccumulateGrad nodes bound to the
        stream they were created on, which invalidates a capture on another stream."""
        if self._comm is None:
            step_fn()                                   # builds the graph handle, the arena and the comm
        if not getattr(self._comm, "fused_push", False):
            return None                                 # NCCL inside the step: left to eager launches
        group, dev = self.process_group, torch.cuda.current_device()
        ok, graph = 1, None
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):               # warm-up on a non-default stream, as capture will run
                step_fn()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            dist.barrier(group)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step_fn()
            torch.cuda.synchronize()
        except Exception as ex:      # noqa: BLE001 - any capture problem means "run eagerly", on every rank
            ok = 0
            warnings.warn(f"CUDA-graph capture of the partitioned step failed ({type(ex).__name__}: {ex}); eager launches")
        flag = torch.tensor([ok], device=torch.device("cuda", dev))
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if flag.item() == 0:
            return None
        self._captured.append(graph)
        graph.replay()
        torch.cuda.synchronize()
        return graph.replay

    def close(self) -> None:
        """Destroy captured steps and unmap the peer arena (collective: call on every rank, before
        destroy_process_group)."""
        if self._captured:
            torch.cuda.synchronize()
            for g in self._captured:
                g.reset()
            self._captured.clear()
        if self._comm is not None and hasattr(self._comm, "close"):
            self._comm.close()
        self._comm, self._comm_key = None, None

    def _ln_fused_partitioned(self, x_local: torch.Tensor) -> bool:
        d = self.hidden_size
        return x_local.is_cuda and self.fuse_layer_norm and d <= 1024 and tuple(self.normalization.normalized_shape) == (d,)

    def fuses_add(self, x_local: torch.Tensor, h) -> bool:
        """Whether ``forward(x_local, ..., add_to=h)`` adds the local rows ``h`` inside the last kernel
        (gca_fwd_hop2_up_add, or the fused LayerNorm): fp32, x_local's device and shape, and a tail that is nothing or the
        fused LayerNorm.  Otherwise ``h + out`` runs as a stock op."""
        if not isinstance(h, torch.Tensor) or h.dtype != torch.float32 or h.device != x_local.device or h.shape != x_local.shape:
            return False
        if self.normalization is None:
            return self._backend is not None and hasattr(self._backend, "fwd_hop2_up_add")
        return isinstance(self.normalization, nn.LayerNorm) and self._ln_fused_partitioned(x_local)

    def forward(self, x_local: torch.Tensor, edge_index: torch.Tensor, num_nodes: int, edge_attr=None, *,
                add_to: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``add_to``: this rank's rows of ``h``; returns ``h + adapter(x)[rows]`` (parallel insertion), fused where
        ``fuses_add`` allows."""
        if self._backend is None:
            self._backend = CudaPhases()
        group = self.process_group
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        lo, hi = row_block(num_nodes, world, rank)
        if x_local.shape != (hi - lo, self.hidden_size):
            raise RuntimeError(f"rank {rank} owns rows [{lo}, {hi}); expected x_local of shape {(hi - lo, self.hidden_size)}")
        if self.hidden_size % 4 != 0 or self.bottleneck_size not in (8, 16, 32, 64, 128):
            raise RuntimeError("PartitionedGConvAdapter needs hidden % 4 == 0 and bottleneck in {8,16,32,64,128}")
        graph = self._graph(edge_index, num_nodes, lo, hi)
        comm = self._get_comm(num_nodes, x_local.device)
        fuse = add_to is not None and self.fuses_add(x_local, add_to)
        addend = add_to if fuse else None
        x_local, _ = kernel_operand(x_local)
        fused_scalar = self.scalar if self.normalization is None else None
        out = _PartitionedFunction.apply(x_local, self.conv_down.lin.weight, self.conv_down.bias,
                                         self.conv_up.lin.weight, self.conv_up.bias, fused_scalar, graph, self._act,
                                         self.skip_connection, num_nodes, comm, self._backend,
                                         addend if self.normalization is None else None)
        if isinstance(self.normalization, nn.LayerNorm):
            ln = self.normalization
            w, b = _AllReduceGrad.apply(ln.weight, group), _AllReduceGrad.apply(ln.bias, group)
            sc = _AllReduceGrad.apply(self.scalar, group) if self.scalar is not None else None
            d = self.hidden_size
            if out.is_cuda and self.fuse_layer_norm and d <= 1024 and tuple(ln.normalized_shape) == (d,):
                from .finetune.gconv_adapter import _LayerNormScaleFunction      # row-local: the fused tail works per shard
                out = _LayerNormScaleFunction.apply(out, w, b, sc, ln.eps, addend)
            else:
                out = torch.nn.functional.layer_norm(out, ln.normalized_shape, w, b, ln.eps)
                if sc is not None:
                    out = out * sc
        if add_to is not None and not fuse:
            out = add_to + out
        return out
