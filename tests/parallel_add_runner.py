"""Child process of tests/test_gpu_parallel_add.py.

``parallel_add_runner.py <case>``: runs the fused-add checks of one shape (test_gpu_parallel_add.run_case) under the
GCA_* switches of the environment, which libgca latches at first use, and prints ONE JSON line: phase -> variant.

``parallel_add_runner.py partitioned <normalization> <port>``: two ranks (one process per GPU, NCCL) run
PartitionedGConvAdapter(..., add_to=h) and compare their rows with h + the 1-GPU GConvAdapter."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import torch  # noqa: E402


def _rank(rank, world, normalization, port):
    import torch.distributed as dist

    from gconv_adapter_b200 import GConvAdapter, GraphCache
    from gconv_adapter_b200.graphs.synthetic import make_inputs, symmetric_random_graph
    from gconv_adapter_b200.partition import PartitionedGConvAdapter, row_block
    from util import assert_close, load_module_params

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", world_size=world, rank=rank)
    n, d, r = 20011, 256, 16
    ei = symmetric_random_graph(n, 6 * n, seed=61).cuda()
    x, _, params = make_inputs(n, d, r, seed=62)
    x = x.cuda()
    h = torch.randn(n, d, generator=torch.Generator().manual_seed(63)).cuda()
    kw = dict(normalization=normalization, learnable_scalar=True)
    single = GConvAdapter(d, r, **kw)
    part = PartitionedGConvAdapter(d, r, comm="collective", **kw)
    for m in (single, part):
        load_module_params(m, params)
    single, part = single.cuda(), part.cuda()
    single.graph_cache = GraphCache()
    lo, hi = row_block(n, world, rank)
    assert part.fuses_add(x[lo:hi], h[lo:hi])
    hl = h[lo:hi].clone().requires_grad_(True)
    y = part(x[lo:hi], ei, n, add_to=hl)
    y_sep = h[lo:hi] + part(x[lo:hi], ei, n)
    assert torch.equal(y.detach(), y_sep.detach()), "fused != separate add"
    with torch.no_grad():
        ref = single(x, ei, add_to=h)[lo:hi]
    assert_close(y.detach(), ref.double(), f"rank {rank}: vs the 1-GPU module")
    y.sum().backward()
    assert torch.equal(hl.grad, torch.ones_like(hl)), "gradient of add_to"
    part.close()
    dist.destroy_process_group()


def main():
    if sys.argv[1] == "partitioned":
        import torch.multiprocessing as mp
        mp.spawn(_rank, args=(2, sys.argv[2], int(sys.argv[3])), nprocs=2, join=True)
        print(json.dumps({"ok": True}))
        return
    from test_gpu_parallel_add import run_case
    print(json.dumps(run_case(sys.argv[1])))


if __name__ == "__main__":
    main()
