"""CPU tests of the host-side mirror: constructor surface, state_dict contract, init RNG stream,
reference-checkpoint loading, and that a CPU tensor is refused (there is no CPU compute path)."""
import pytest
import torch

import gconv_adapter_b200 as gca
from gconv_adapter_b200 import GConvAdapter
from oracle.pyg_restated import GConvAdapterRef


def test_state_dict_keys_and_shapes_match_reference_contract():
    m = GConvAdapter(64, 16, learnable_scalar=True, normalization="layer_norm")
    ref = GConvAdapterRef(64, 16, learnable_scalar=True, normalization="layer_norm")
    assert list(m.state_dict().keys()) == list(ref.state_dict().keys()) == [
        "scalar", "conv_down.bias", "conv_down.lin.weight", "conv_up.bias", "conv_up.lin.weight",
        "normalization.weight", "normalization.bias"]
    for k, v in ref.state_dict().items():
        assert m.state_dict()[k].shape == v.shape, k
    m = GConvAdapter(32, 8, normalization="batch_norm")
    assert list(m.state_dict().keys()) == list(GConvAdapterRef(32, 8, normalization="batch_norm").state_dict().keys())
    m = GConvAdapter(32, 8)
    assert m.scalar is None and m.normalization is None and m.skip_connection is True
    assert isinstance(m.act_fn, torch.nn.ReLU)
    # a reference-trained checkpoint loads strictly
    m = GConvAdapter(32, 8, learnable_scalar=True)
    m.load_state_dict(GConvAdapterRef(32, 8, learnable_scalar=True).state_dict(), strict=True)


def test_same_seed_gives_reference_init():
    for kw in (dict(), dict(learnable_scalar=True, normalization="layer_norm"), dict(normalization="batch_norm")):
        torch.manual_seed(7)
        a = GConvAdapter(48, 16, **kw)
        torch.manual_seed(7)
        b = GConvAdapterRef(48, 16, **kw)
        for (ka, va), (kb, vb) in zip(a.state_dict().items(), b.state_dict().items()):
            assert ka == kb and torch.equal(va, vb), ka
        assert a.conv_down.lin.weight.abs().max() < 1e-4      # near-identity init, std 1e-5
        assert torch.count_nonzero(a.conv_up.bias) == 0


def test_constructor_errors_match_reference_messages():
    for bad, ref_bad in ((dict(conv_type="foo"), None), (dict(non_linearity="gelu"), None), (dict(normalization="group"), None)):
        with pytest.raises(ValueError) as e1:
            GConvAdapter(8, 4, **bad)
        with pytest.raises(ValueError) as e2:
            GConvAdapterRef(8, 4, **bad)
        assert str(e1.value) == str(e2.value)
    for conv in ("sage", "gat"):          # selectable in the reference, but its constructor cannot finish
        with pytest.raises(AttributeError):
            GConvAdapter(8, 4, conv_type=conv)


def test_freeze_policy_and_moduledict_registration():
    """Hosts keep adapters in nn.ModuleDict and train a parameter iff its module path contains
    'adapter' (/root/reference/src/models/inductive/gnn.py:59-60,230-233)."""
    host = torch.nn.Module()
    host.post_adapters = torch.nn.ModuleDict({str(i): GConvAdapter(16, 8, learnable_scalar=True) for i in range(2)})
    names = [n for n, _ in host.named_parameters()]
    assert "post_adapters.0.scalar" in names and "post_adapters.1.conv_up.lin.weight" in names
    for name, module in host.named_modules():
        for _, p in module.named_parameters(recurse=False):
            p.requires_grad = "adapter" in name
    assert all(p.requires_grad for p in host.parameters())


def test_cpu_tensor_is_refused():
    m = GConvAdapter(16, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.randn(5, 16), torch.zeros(2, 3, dtype=torch.long))


def test_reference_alias_resolves_target_path():
    import importlib
    gca.install_reference_alias()
    mod = importlib.import_module("src.finetune.gconv_adapter")
    assert mod.GConvAdapter is GConvAdapter
