"""CPU tests: the oracle against the committed golden vectors (made with the reference's own
glue class), against the normalisation formulas that live in the reference repo, and against
hand-computed tiny graphs.  PARITY UNPINNED at the PyG boundary - see oracle/__init__.py."""
import numpy as np
import pytest
import torch

from oracle import csr_ref, pyg_restated
from oracle.pyg_restated import GConvAdapterRef, gcn_norm
from gconv_adapter_b200.graphs.synthetic import make_inputs, symmetric_random_graph

from util import assert_close, ctor_kwargs, golden_names, load_golden, load_module_params


def _run_oracle(g):
    cfg = g["cfg"]
    n, d = g["x"].shape if "x" in g else (int(g["num_nodes"]), g["param.conv_up.bias"].shape[0])
    r = g["param.conv_down.bias"].shape[0]
    m = GConvAdapterRef(d, r, **ctor_kwargs(cfg))
    load_module_params(m, {k[6:]: v for k, v in g.items() if k.startswith("param.")})
    m.train()
    return m


@pytest.mark.parametrize("name", [n for n in golden_names() if n != "cora_shaped"])
def test_oracle_matches_golden(name):
    g = load_golden(name)
    m = _run_oracle(g)
    x = torch.from_numpy(g["x"]).clone().requires_grad_(True)
    ei = torch.from_numpy(g["edge_index"])
    three_d = bool(g["cfg"].get("three_d", False))
    xin = x.unsqueeze(0) if three_d else x
    y = m(xin, ei)
    y.backward(torch.from_numpy(g["g_out"]).reshape(y.shape))
    # same code path on the same machine: bit-exact
    assert torch.equal(y.detach().reshape(g["y"].shape), torch.from_numpy(g["y"]))
    assert torch.equal(x.grad, torch.from_numpy(g["g_x"]))
    for k, p in m.named_parameters():
        assert torch.equal(p.grad, torch.from_numpy(g["grad." + k])), k


def test_oracle_matches_golden_cora_shaped():
    g = load_golden("cora_shaped")
    n, d, r = 2708, 64, 8
    ei = symmetric_random_graph(n, 10556, seed=int(g["graph_seed"]))
    x, g_out, _ = make_inputs(n, d, r, seed=int(g["input_seed"]))
    m = _run_oracle(g)
    x = x.clone().requires_grad_(True)
    y = m(x, ei)
    y.backward(g_out)
    rows = torch.from_numpy(g["rows"])
    assert torch.equal(y.detach()[rows], torch.from_numpy(g["y_rows"]))
    assert torch.equal(x.grad[rows], torch.from_numpy(g["g_x_rows"]))
    assert y.detach().double().sum().item() == pytest.approx(float(g["y_sum64"]), rel=1e-12)


def test_gcn_norm_matches_in_repo_formulas():
    """Known answers from formulas that DO live in the reference:
    MolecularGCNConv.norm (src/layers/inductive/gcn_conv.py:36-56) and
    normalize (src/dataset/transductive/data_utils.py:175-183)."""
    n = 60
    ei = symmetric_random_graph(n, 240, seed=4)
    ei2, w = gcn_norm(ei, n)
    # (1) on a symmetric graph with the loops in place, degree-by-row == degree-by-col
    w_mol = pyg_restated.molecular_gcn_norm(ei2, n)
    assert torch.equal(w, w_mol)
    # (2) dense set_diag normalisation on the coalesced (simple) graph: same coefficients, bit for bit
    a = torch.zeros(n, n)
    a[ei[0], ei[1]] = 1
    ce = a.nonzero().t().contiguous()                  # duplicates removed
    dense = pyg_restated.dense_set_diag_normalize(ce, n)
    ce2, wc = gcn_norm(ce, n)
    ours = torch.zeros(n, n).index_put_((ce2[0], ce2[1]), wc)
    assert torch.equal(ours, dense)


def test_tiny_graph_hand_answers():
    # path 0-1-2-3 with loops: deg = [2,3,3,2]
    ei = torch.tensor([[0, 1, 1, 2, 2, 3], [1, 0, 2, 1, 3, 2]])
    ei2, w = gcn_norm(ei, 4)
    assert ei2.size(1) == 10
    dense = torch.zeros(4, 4, dtype=torch.float64).index_put_((ei2[1], ei2[0]), w.double(), accumulate=True)
    expect = torch.tensor([[1 / 2, 1 / 6 ** 0.5, 0, 0], [1 / 6 ** 0.5, 1 / 3, 1 / 3, 0],
                           [0, 1 / 3, 1 / 3, 1 / 6 ** 0.5], [0, 0, 1 / 6 ** 0.5, 1 / 2]], dtype=torch.float64)
    assert torch.allclose(dense, expect, atol=1e-7)
    # existing self loops are replaced by exactly one; duplicates are counted
    ei = torch.tensor([[0, 0, 1, 1, 1], [1, 1, 0, 1, 1]])
    ei2, w = gcn_norm(ei, 2)
    assert ei2.tolist() == [[0, 0, 1, 0, 1], [1, 1, 0, 0, 1]]
    deg = torch.tensor([2.0, 3.0])            # in-degree incl. loop: node0 <- {1, loop}; node1 <- {0, 0, loop}
    assert torch.allclose(w, torch.tensor([1 / 6 ** 0.5] * 3 + [1 / 2, 1 / 3]), atol=1e-7)
    # isolated node: deg = 1 -> weight-1 loop; directed edge uses in-degree on both ends
    ei = torch.tensor([[0], [1]])
    ei2, w = gcn_norm(ei, 3)
    assert torch.allclose(w, torch.tensor([1 / (1 * 2) ** 0.5, 1.0, 0.5, 1.0]))
    # 3-D [1, N, F] input == 2-D input (node_dim = -2)
    m = GConvAdapterRef(8, 4, learnable_scalar=True)
    load_module_params(m, {"conv_down.lin.weight": torch.randn(4, 8) * 0.1, "conv_up.lin.weight": torch.randn(8, 4) * 0.1})
    x = torch.randn(3, 8)
    assert torch.equal(m(x, ei), m(x.unsqueeze(0), ei)[0])
    assert (deg > 0).all()


def test_csr_ref_is_the_oracle_multiset():
    n = 40
    ei = symmetric_random_graph(n, 150, seed=9)
    ei = torch.cat([ei, torch.tensor([[3, 3, 5], [3, 3, 5]])], 1)       # pre-existing loops
    for normalize in (True, False):
        ref = csr_ref.build(ei.numpy(), n, normalize)
        coo = csr_ref.coo_after_loops(ei.numpy(), n, normalize)
        # expand the CSR back to (target, source) pairs and compare multisets
        tgt = np.repeat(np.arange(n), np.diff(ref["rowptr"]))
        got = sorted(zip(tgt.tolist(), ref["colidx"].tolist()))
        want = sorted(zip(coo[1].tolist(), coo[0].tolist()))
        assert got == want
        src = np.repeat(np.arange(n), np.diff(ref["rowptr_t"]))
        assert sorted(zip(src.tolist(), ref["colidx_t"].tolist())) == sorted(zip(coo[0].tolist(), coo[1].tolist()))
    # dis of the restated gcn_norm == 1/sqrt(deg) in IEEE fp32 (what the CUDA build computes)
    ref = csr_ref.build(ei.numpy(), n, True)
    deg = np.diff(ref["rowptr"]).astype(np.float32)
    assert np.array_equal(ref["dis"], (np.float32(1.0) / np.sqrt(deg)).astype(np.float32))
    # partition: two row blocks concatenate to the full structure
    a, b = csr_ref.build(ei.numpy(), n, True, 0, 17), csr_ref.build(ei.numpy(), n, True, 17, n)
    assert np.array_equal(np.concatenate([a["colidx"], b["colidx"]]), ref["colidx"])
    assert np.array_equal(np.concatenate([a["rowptr"][:-1], b["rowptr"] + a["rowptr"][-1]]), ref["rowptr"])


def test_pow_minus_half_is_ieee_div_sqrt():
    """Pins the rounding the CUDA build must reproduce: torch's deg.pow(-0.5) equals
    1.0f / sqrtf(deg) bit for bit on every integer degree we can meet."""
    deg = torch.arange(1, 1 << 20, dtype=torch.float32)
    a = deg.pow(-0.5).numpy()
    b = (np.float32(1.0) / np.sqrt(deg.numpy())).astype(np.float32)
    assert np.array_equal(a, b)
