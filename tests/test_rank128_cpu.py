"""Bottleneck sizes up to 128 without a GPU: zero-padding of (64, 128] to the native rank 128, the refusal above 128,
the C ABI's rank set and hub-scratch queries, and PartitionedGConvAdapter at r = 128 over gloo with the CPU phase
double."""
import pytest
import torch
import torch.multiprocessing as mp

from gconv_adapter_b200 import GConvAdapter, _cabi
from gconv_adapter_b200.graphs.synthetic import make_inputs, symmetric_random_graph
from gconv_adapter_b200.partition import PartitionedGConvAdapter
from oracle.pyg_restated import GConvAdapterRef

from test_partition_cpu import _free_port, _worker
from util import load_module_params


@pytest.mark.parametrize("r", [65, 96, 100, 128])
def test_bottleneck_in_64_128_is_padded_to_128(r):
    d = 30
    m = GConvAdapter(d, r)
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert shapes["conv_down.lin.weight"] == (r, d) and shapes["conv_down.bias"] == (r,)
    assert shapes["conv_up.lin.weight"] == (d, r) and shapes["conv_up.bias"] == (d,)
    dp, wd, bd, wu, bu = m._padded_params(d, r)
    assert dp == 32
    assert wd.shape == (128, 32) and bd.shape == (128,) and wu.shape == (32, 128) and bu.shape == (32,)
    # the padding is zeros and the original entries are kept
    assert torch.equal(wd[:r, :d], m.conv_down.lin.weight) and not wd[r:].any() and not wd[:, d:].any()
    assert torch.equal(wu[:d, :r], m.conv_up.lin.weight) and not wu[:, r:].any() and not bd[r:].any()
    # padding does not touch the module's own parameters
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == shapes


def test_bottleneck_64_is_not_padded_further():
    m = GConvAdapter(64, 64)
    assert m._padded_params(64, 64)[1].shape == (64, 64)


@pytest.mark.parametrize("r", [129, 256])
def test_bottleneck_above_128_raises(r):
    m = GConvAdapter(32, r)
    with pytest.raises(RuntimeError, match=f"bottleneck_size {r} > 128"):
        m._padded_params(32, r)


def test_shape_is_fast_accepts_rank_128():
    lib = _cabi.load()
    for r in (8, 16, 32, 64, 128):
        assert lib.gca_shape_is_fast(256, r) == 1
        assert lib.gca_shape_is_fast(300, r) == 1
    for r in (96, 100, 129, 256):
        assert lib.gca_shape_is_fast(256, r) == 0
    assert lib.gca_shape_is_fast(30, 128) == 0


def test_hub_scratch_query_argument_checks():
    lib = _cabi.load()
    assert lib.gca_hub_scratch_bytes(None) == 0
    for r in (-1, 0, 8, 64, 128, 129):
        assert lib.gca_hub_scratch_bytes_r(None, r) == 0
    # the workspace queries still refuse a null graph at r = 128
    assert lib.gca_forward_workspace_bytes(None, 256, 128) == 0
    assert lib.gca_backward_workspace_bytes(None, 256, 128) == 0
    # r-only and d-dependent scratch grow with r
    assert lib.gca_bwd_scratch_bytes(256, 128) > lib.gca_bwd_scratch_bytes(256, 64) > 0
    assert lib.gca_bwd_scratch_bytes(256, 128) % 256 == 0


def _refusal_worker(rank, world, port, out):
    import os
    import torch.distributed as dist
    from cpu_phases import CpuPhases
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n, d = 40, 32
        ei = symmetric_random_graph(n, 4 * n, seed=3)
        for r in (96, 256):
            m = PartitionedGConvAdapter(d, r, phase_backend=CpuPhases())
            try:
                m(torch.randn(n, d), ei, n)
                out[r] = "ran"
            except RuntimeError as ex:
                out[r] = str(ex)
    finally:
        dist.destroy_process_group()


def test_partitioned_refuses_ranks_outside_the_native_set():
    """PartitionedGConvAdapter takes the native ranks only (no padding): 128 is one of them, 96 and 256 are not."""
    out = mp.Manager().dict()
    mp.spawn(_refusal_worker, args=(1, _free_port(), out), nprocs=1, join=True)
    for r in (96, 256):
        assert "bottleneck in {8,16,32,64,128}" in out[r]


@pytest.mark.parametrize("world,n,kw", [
    (2, 301, dict(learnable_scalar=True)),
    (2, 200, dict(non_linearity="silu", normalization="layer_norm")),
])
def test_partitioned_rank128_matches_full_graph_oracle(world, n, kw):
    d, r = 32, 128
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, n, d, r, kw, out), nprocs=world, join=True)
    ei = symmetric_random_graph(n, 6 * n, seed=21)
    x, g_out, params = make_inputs(n, d, r, seed=22)
    ref = GConvAdapterRef(d, r, **kw)
    load_module_params(ref, params)
    xx = x.clone().requires_grad_(True)
    yr = ref(xx, ei)
    yr.backward(g_out)
    y = torch.cat([out[k]["y"] for k in range(world)])
    gx = torch.cat([out[k]["gx"] for k in range(world)])
    assert torch.allclose(y, yr.detach(), rtol=1e-4, atol=1e-5)
    assert torch.allclose(gx, xx.grad, rtol=1e-4, atol=1e-5)
    for k, p in ref.named_parameters():
        for rank in range(world):
            assert out[rank]["grads"][k].shape == p.grad.shape
            assert torch.allclose(out[rank]["grads"][k], p.grad, rtol=1e-4, atol=1e-5 * max(1.0, p.grad.abs().max().item())), (k, rank)
