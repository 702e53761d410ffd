"""CPU checks of the molecular backbone widening (SURVEY section 8f rank 3, inductive half): the oracle restatement of
MolecularGINConv / MolecularGCNConv against the golden vectors produced by the reference's own classes, and the identity the
CUDA layers rest on (sum of edge embeddings = per-node histograms x embedding tables)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import molecular_ref

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "backbone", "mol_*.npz")))
REFS = {"gin": molecular_ref.MolecularGINConvRef, "gcn": molecular_ref.MolecularGCNConvRef}


def load(path):
    z = np.load(path)
    return {k: torch.from_numpy(z[k]) if z[k].ndim else z[k].item() for k in z.files}


def build(cls, g, tag, emb):
    """The layer with the reference's parameters: stored ones (mol_small) or rebuilt from the constructor seed."""
    torch.manual_seed(int(g[tag + "_ctor_seed"]))
    layer = cls(emb)
    stored = {k[len(tag) + 7:]: v for k, v in g.items() if k.startswith(tag + "_param.")}
    if stored:
        sd = layer.state_dict()
        assert sorted(stored) == sorted(sd)                       # same state_dict keys as the reference class
        for k, v in stored.items():
            assert torch.equal(sd[k], v), k                      # ... and the same constructor RNG stream
    return layer


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-4] for p in GOLD])
@pytest.mark.parametrize("tag", ["gin", "gcn"])
def test_oracle_restatement_matches_reference_vectors(path, tag):
    g = load(path)
    emb = g["x"].shape[1]
    layer = build(REFS[tag], g, tag, emb)
    x = g["x"].clone().requires_grad_(True)
    y = layer(x, g["edge_index"], g["edge_attr"])
    y.backward(g["g_out"])
    assert torch.equal(y.detach(), g[tag + "_y"])                # same op sequence on the same CPU: bit-exact
    assert torch.equal(x.grad, g[tag + "_gx"])
    for k, p in layer.named_parameters():
        if f"{tag}_grad.{k}" in g:
            # (nn.Embedding's backward and an indexing backward add the same numbers in different orders)
            want = g[f"{tag}_grad.{k}"]
            assert torch.allclose(p.grad, want, rtol=1e-5, atol=1e-5 * float(want.abs().max())), k


def test_histogram_identity_behind_the_cuda_layers():
    """sum_e emb(type_e) + emb(dir_e) over the incoming edges of a node == counts[node] @ tables (self loop = type 4, dir 0)."""
    from gconv_adapter_b200.graphs.synthetic import molecule_batch
    ei, _, n = molecule_batch(batch_size=8, seed=4)
    gen = torch.Generator().manual_seed(2)
    ea = torch.stack([torch.randint(0, 4, (ei.size(1),), generator=gen), torch.randint(0, 3, (ei.size(1),), generator=gen)], 1)
    wt, wd = torch.randn(6, 12, generator=gen), torch.randn(3, 12, generator=gen)
    x = torch.randn(n, 12, generator=gen)
    full = molecular_ref.gin_aggregate(x, ei, ea, wt, wd)
    plain = torch.zeros_like(x).index_add_(0, torch.cat([ei[1], torch.arange(n)]), x[torch.cat([ei[0], torch.arange(n)])])
    ct = torch.zeros(n, 6).index_put_((ei[1], ea[:, 0]), torch.ones(ei.size(1)), accumulate=True)
    cd = torch.zeros(n, 3).index_put_((ei[1], ea[:, 1]), torch.ones(ei.size(1)), accumulate=True)
    ct[:, 4] += 1
    cd[:, 0] += 1
    assert torch.allclose(full, plain + ct @ wt + cd @ wd, rtol=1e-5, atol=1e-5)
