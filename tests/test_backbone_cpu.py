"""CPU checks of the backbone-propagation widening (SURVEY section 8f rank 3): the oracle restatement against
the golden vectors produced by the reference's own functions, and the host-side guards of the CUDA mirror."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import backbone_ref

GOLD = sorted(p for p in glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "backbone", "*.npz"))
              if not os.path.basename(p).startswith("mol_"))     # mol_*: the molecular layers (tests/test_*molecular*.py)


def _load(path):
    z = np.load(path)
    return {k: torch.from_numpy(z[k]) if z[k].ndim else z[k].item() for k in z.files}


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-4] for p in GOLD])
def test_oracle_restatement_matches_reference_vectors(path):
    g = _load(path)
    x = g["x"].clone().requires_grad_(True)
    y = backbone_ref.gcn_conv(x, g["edge_index"])
    y.backward(g["g_out"])
    assert torch.equal(y.detach(), g["gcn_y"])                 # same op sequence on the same CPU: bit-exact
    assert torch.equal(x.grad, g["gcn_gx"])
    xb = g["x"].unsqueeze(0).clone().requires_grad_(True)
    b = g["b"].clone().requires_grad_(True)
    yb = backbone_ref.add_conv_relational_bias(xb, g["edge_index"], b)
    yb.backward(g["g_out"].unsqueeze(0))
    assert torch.equal(yb.detach(), g["rel_y"])
    assert torch.equal(xb.grad, g["rel_gx"])
    assert torch.allclose(b.grad, g["rel_gb"], rtol=1e-6, atol=1e-6)


def test_propagation_equals_the_adapter_normalisation_on_self_looped_graphs():
    """The precondition the CUDA path relies on: with one self loop per node the reference's matrix is D^-1/2 A' D^-1/2
    of the adapter (oracle.pyg_restated.gcn_norm), up to the rounding of sqrt(1/d) vs d^-1/2."""
    from oracle import pyg_restated
    g = _load(GOLD[0])
    ei, n = g["edge_index"], int(g["num_nodes"])
    ei2, w = pyg_restated.gcn_norm(ei, n)
    x = g["x"].reshape(n, -1)
    dense = torch.zeros(n, x.shape[1]).index_add_(0, ei2[1], w.unsqueeze(1) * x.index_select(0, ei2[0]))
    ref = g["gcn_y"].reshape(n, -1)
    assert (dense - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()


def test_cuda_mirror_has_no_cpu_path_and_rejects_edge_weights():
    from gconv_adapter_b200.layers import propagate
    x = torch.randn(10, 1, 8)
    ei = torch.arange(10).repeat(2, 1)
    with pytest.raises(RuntimeError, match="CUDA"):
        propagate.gcn_conv(x, ei)
    with pytest.raises(NotImplementedError):
        propagate.gcn_conv(x, ei, torch.ones(10))
    with pytest.raises(NotImplementedError):
        propagate.add_conv_relational_bias(x.unsqueeze(0), ei, torch.zeros(1), trans="tanh")
