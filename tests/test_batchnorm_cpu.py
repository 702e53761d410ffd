"""CPU tests of normalization='batch_norm': the argument rules of the fused BatchNorm1d + scalar entries and the module's
choice between the fused tail and the stock ops.  No device is needed, and none is touched: every call here returns from
its argument checks (or is an empty no-op) before any CUDA call, so the fake addresses are never dereferenced."""
import pytest
import torch
import torch.nn as nn

from gconv_adapter_b200 import GConvAdapter, _cabi
from gconv_adapter_b200.partition import PartitionedGConvAdapter

N, D, R = 50, 64, 8
F = 1 << 20             # a 256 B aligned address, never dereferenced
INVALID, WORKSPACE, UNSUPPORTED = -1, -2, -5


def _fwd(X=F, ldx=D, eps=1e-5, training=1, rm=F, rv=F, Y=F, ldy=D, mean=F, rstd=F, scratch=F, n=N, d=D):
    return _cabi.load().gca_batchnorm_scale_fwd(X, ldx, None, None, None, eps, training, 0.1, rm, rv, Y, ldy, mean, rstd,
                                                scratch, n, d, None)


def _bwd(gY=F, ldg=D, X=F, ldx=D, mean=F, rstd=F, training=1, gX=F, ldgx=D, gg=None, gb=None, gs=None, scratch=F, n=N, d=D):
    return _cabi.load().gca_batchnorm_scale_bwd(gY, ldg, X, ldx, None, None, None, mean, rstd, training, gX, ldgx, gg, gb, gs,
                                                scratch, n, d, None)


def test_scratch_query():
    lib = _cabi.load()
    assert lib.gca_batchnorm_scratch_bytes(0) == 0 and lib.gca_batchnorm_scratch_bytes(-4) == 0
    for d in (4, 64, 256, 300, 2048):
        b = lib.gca_batchnorm_scratch_bytes(d)
        assert b % 256 == 0
        assert b >= 8 * 2 * d + 4 * 2 * d          # at least one CTA's fp64 statistics / the gradient sums
    assert lib.gca_batchnorm_scratch_bytes(2048) > lib.gca_batchnorm_scratch_bytes(256)


@pytest.mark.parametrize("kw", [dict(X=None), dict(Y=None), dict(mean=None), dict(rstd=None), dict(scratch=None),
                                dict(n=-1), dict(d=0), dict(d=-4), dict(eps=-1e-5), dict(eps=float("nan")),
                                dict(n=1), dict(n=0),                                   # training needs two rows
                                dict(training=0, rm=None), dict(training=0, rv=None)])  # eval needs the buffers
def test_forward_invalid_arguments(kw):
    assert _fwd(**kw) == INVALID


@pytest.mark.parametrize("kw", [dict(d=30), dict(ldx=D - 4), dict(ldx=D + 2), dict(ldy=D - 4), dict(ldy=D + 2),
                                dict(X=F + 4), dict(Y=F + 8)])
def test_forward_unsupported_layouts(kw):
    assert _fwd(**kw) == UNSUPPORTED


def test_forward_workspace_and_empty_eval():
    assert _fwd(scratch=F + 16) == WORKSPACE
    assert _fwd(training=0, n=0) == 0                    # nothing to do, no CUDA call
    assert _fwd(training=1, rm=None, rv=None, n=0) == INVALID


@pytest.mark.parametrize("kw", [dict(gY=None), dict(X=None), dict(mean=None), dict(rstd=None), dict(scratch=None),
                                dict(n=-1), dict(d=0), dict(n=1)])
def test_backward_invalid_arguments(kw):
    assert _bwd(**kw) == INVALID


@pytest.mark.parametrize("kw", [dict(d=30), dict(ldg=D - 4), dict(ldx=D + 2), dict(ldgx=D - 4), dict(ldgx=D + 2),
                                dict(gY=F + 4), dict(X=F + 4), dict(gX=F + 4)])
def test_backward_unsupported_layouts(kw):
    assert _bwd(**kw) == UNSUPPORTED


def test_backward_workspace_and_empty_input():
    assert _bwd(scratch=F + 16) == WORKSPACE
    assert _bwd(n=0, training=0) == 0 and _bwd(n=0, training=1) == 0      # no gradient asked for: no CUDA call


# ---- the module's choice ----
def _bn(d=D, **kw):
    return GConvAdapter(d, R, normalization="batch_norm", learnable_scalar=True, **kw)


def test_fused_by_default_on_a_plain_batchnorm():
    m = _bn()
    assert m.fuse_batch_norm is True
    assert m._bn_fused(torch.randn(N, D))
    assert m._bn_fused(torch.randn(2, D))
    m.eval()
    assert m._bn_fused(torch.randn(N, D))
    assert _bn(d=2048)._bn_fused(torch.randn(3, 2048))               # no d <= 1024 limit, unlike layer_norm
    t = GConvAdapter(D, R, normalization="batch_norm")
    t.normalization = nn.BatchNorm1d(D, affine=False, track_running_stats=False, momentum=None)
    assert t._bn_fused(torch.randn(N, D))


def test_stock_ops_when_fusion_is_off_or_not_possible(monkeypatch):
    m = _bn()
    assert not m._bn_fused(torch.randn(1, D))                         # one row: no BatchNorm at all
    assert not m._bn_fused(torch.randn(1, N, D))                      # [1, N, d]: the reference's size(0) == 1 rule
    assert not m._bn_fused(torch.randn(N, D, dtype=torch.float64))
    assert not _bn(d=30)._bn_fused(torch.randn(N, 30))                # d % 4 != 0
    m.fuse_batch_norm = False
    assert not m._bn_fused(torch.randn(N, D))
    m.fuse_batch_norm = True
    monkeypatch.setenv("GCA_DISABLE_BN_FUSE", "1")
    assert not m._bn_fused(torch.randn(N, D))
    monkeypatch.delenv("GCA_DISABLE_BN_FUSE")

    class MyBatchNorm(nn.BatchNorm1d):
        pass

    m.normalization = MyBatchNorm(D)                                  # a subclass may compute something else
    assert not m._bn_fused(torch.randn(N, D))
    m.normalization = nn.BatchNorm1d(D + 4)                           # features that do not match
    assert not m._bn_fused(torch.randn(N, D))
    m.normalization = nn.BatchNorm1d(D).double()
    assert not m._bn_fused(torch.randn(N, D))


def test_fusion_leaves_add_partitioning_and_state_as_they_were():
    m = _bn()
    x = torch.randn(N, D)
    assert not m.fuses_add(x, torch.randn(N, D))                      # the add stays the stock h + out
    with pytest.raises(ValueError, match="batch_norm"):
        PartitionedGConvAdapter(16, 8, normalization="batch_norm")
    assert list(m.state_dict()) == list(_bn().state_dict())
    assert "normalization.num_batches_tracked" in m.state_dict()
