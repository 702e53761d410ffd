"""CPU tests of parallel insertion (``add_to=h``): which operands the module adds inside its last kernel and which go to
the stock ``h + out``, and the argument checks of the C entries with an addend (no device needed for either)."""
import pytest
import torch

from gconv_adapter_b200 import GConvAdapter, _cabi
from gconv_adapter_b200.partition import PartitionedGConvAdapter

N, D, R = 50, 64, 8


@pytest.mark.parametrize("normalization,fused", [("none", True), ("layer_norm", True), ("batch_norm", False)])
def test_fused_add_decision_by_normalization(normalization, fused):
    m = GConvAdapter(D, R, normalization=normalization)
    x = torch.randn(N, D)
    assert m.fuses_add(x, torch.randn(N, D)) is fused
    assert m.fuses_add(x.unsqueeze(0), torch.randn(1, N, D)) is fused


def test_fused_add_decision_by_operand():
    m = GConvAdapter(D, R)
    x = torch.randn(N, D)
    assert m.fuses_add(x, torch.randn(N, D + 12)[:, 4:4 + D])          # column window: passed in place
    assert m.fuses_add(x, torch.randn(1, D).expand(N, D))               # stride-0 rows: copied, then fused
    assert m.fuses_add(x, torch.randn(D, N).t())                        # column-major: copied, then fused
    assert not m.fuses_add(x, torch.randn(D))                           # broadcast shape
    assert not m.fuses_add(x, torch.randn(1, D))
    assert not m.fuses_add(x, torch.randn(N, D, dtype=torch.float64))   # other dtypes
    assert not m.fuses_add(x, torch.randn(N, D, dtype=torch.bfloat16))
    assert not m.fuses_add(x, torch.randn(N, D, device="meta"))         # another device
    assert not m.fuses_add(x, 1.5)
    assert not m.fuses_add(x.unsqueeze(0), torch.randn(N, D))           # [1, N, d] wants h of the same shape
    assert m.fuses_add(torch.randn(3, N, D), torch.randn(3, N, D))      # [B, N, d]: sliced with x
    assert not m.fuses_add(torch.randn(3, N, D), torch.randn(N, D))


def test_fused_add_decision_padded_hidden_and_unfused_layer_norm(monkeypatch):
    m = GConvAdapter(30, R)
    assert not m.fuses_add(torch.randn(N, 30), torch.randn(N, 30))      # d % 4 != 0: padded columns
    ln = GConvAdapter(D, R, normalization="layer_norm")
    ln.fuse_layer_norm = False
    assert not ln.fuses_add(torch.randn(N, D), torch.randn(N, D))
    ln.fuse_layer_norm = True
    monkeypatch.setenv("GCA_DISABLE_LN_FUSE", "1")
    assert not ln.fuses_add(torch.randn(N, D), torch.randn(N, D))


def test_partitioned_fused_add_needs_a_backend_with_the_add_phase():
    x = torch.randn(N, D)

    class WithAdd:
        def fwd_hop2_up_add(self, *a):
            raise AssertionError

    assert not PartitionedGConvAdapter(D, R, phase_backend=object()).fuses_add(x, torch.randn(N, D))
    assert PartitionedGConvAdapter(D, R, phase_backend=WithAdd()).fuses_add(x, torch.randn(N, D))
    assert not PartitionedGConvAdapter(D, R, phase_backend=WithAdd()).fuses_add(x, torch.randn(N, D, dtype=torch.float64))


def test_add_entries_reject_a_missing_or_short_addend():
    lib = _cabi.load()
    fake = 1 << 20              # never dereferenced: the checks return first
    assert lib.gca_fwd_hop2_up_add(fake, fake, fake, D, fake, fake, None, 1, fake, None, D, fake, D, None, D, R, None) == -1
    assert lib.gca_fwd_hop2_up_add(fake, fake, fake, D, fake, fake, None, 1, fake, fake, D - 4, fake, D, None, D, R, None) == -1
    assert lib.gca_fwd_hop2_up_add(fake, fake, fake, D, fake, fake, None, 1, fake, fake, D + 2, fake, D, None, D, R, None) == -5
    assert lib.gca_fwd_hop2_up_add(None, fake, fake, D, fake, fake, None, 1, fake, fake, D, fake, D, None, D, R, None) == -1
    assert lib.gca_forward_add(fake, fake, D, fake, fake, fake, fake, None, 1, 1, fake, fake, None, fake, None, D, fake, D, D, R,
                               None) == -1
    assert lib.gca_forward_add(None, fake, D, fake, fake, fake, fake, None, 1, 1, fake, fake, None, fake, fake, D, fake, D, D, R,
                               None) == -1
    assert lib.gca_layernorm_scale_add_fwd(fake, D, None, None, None, 1e-5, None, D, fake, D, fake, fake, N, D, None) == -1
    assert lib.gca_layernorm_scale_add_fwd(fake, D, None, None, None, 1e-5, fake, D - 4, fake, D, fake, fake, N, D, None) == -5
