"""The operand gate of the module (kernel_operand / row_pitch) on CPU tensors: which layouts reach the kernels as they
are, with which row pitch, and which are copied first.  The kernels take a row pitch ld >= d with ld % 4 == 0 and a
16 B aligned base (include/gca.h); everything else must arrive as a dense copy."""
import torch

from gconv_adapter_b200.finetune.gconv_adapter import kernel_operand, row_pitch

D = 64


def _aligned(n, d, extra=0):
    """An [n, d + extra] tensor whose base is 16 B aligned (CPU allocations are at least 64 B aligned)."""
    t = torch.randn(n, d + extra)
    assert t.data_ptr() % 16 == 0
    return t


def _accepted(t, ld):
    out, pitch = kernel_operand(t)
    assert out is t, "an operand the kernels can read in place must not be copied"
    assert pitch == ld == row_pitch(out)
    return out


def _copied(t):
    out, pitch = kernel_operand(t)
    assert out.data_ptr() != t.data_ptr()
    assert out.stride() == (t.shape[1], 1)
    assert pitch == t.shape[1] and out.data_ptr() % 16 == 0
    assert torch.equal(out, t)
    return out


def test_contiguous_tensor_passes_with_pitch_d():
    _accepted(_aligned(10, D), D)


def _grad_of(fn, y):
    """The gradient autograd hands to y's producer for the loss fn(y)."""
    seen = []
    z = y * 1
    z.register_hook(seen.append)
    fn(z).backward()
    return seen[0]


def test_broadcast_gradients_are_copied():
    # a whole-graph sum readout hands y a gradient with stride(0) = 0; the kernels need ld >= d
    y = torch.randn(10, D, requires_grad=True)
    w = torch.randn(D)
    g = _grad_of(lambda z: (z.sum(0) * w).sum(), y)
    assert g.stride() == (0, 1)
    _copied(g)
    g = _grad_of(lambda z: z.sum(), y)
    assert g.stride() == (0, 0)
    _copied(g)


def test_single_row_passes_with_pitch_d_whatever_its_row_stride():
    x = torch.randn(D, 1).t()
    assert x.stride() == (1, 1) and x.is_contiguous() and x.contiguous() is x
    assert row_pitch(x) == D
    _accepted(x, D)
    # a row of a wider tensor, and an empty operand
    _accepted(_aligned(3, D, 4)[1:2, :D], D)
    _accepted(torch.empty(0, D), D)


def test_single_row_with_a_strided_inner_dimension_is_copied():
    _copied(_aligned(1, 2 * D)[:, ::2])


def test_cat_windows():
    y = torch.randn(10, D, requires_grad=True)
    g = _grad_of(lambda z: (torch.cat([z, torch.ones(10, 12)], 1) ** 2).sum() / 2, y)
    assert g.stride() == (D + 12, 1)
    wide = _aligned(10, D, 12)
    _accepted(wide[:, :D], D + 12)                  # offset 0
    _accepted(wide[:, 4:4 + D], D + 12)             # 16 B offset
    _copied(wide[:, 1:1 + D])                       # 4 B offset: misaligned base


def test_pitch_not_a_multiple_of_four_is_copied():
    wide = _aligned(10, D, 2)                       # pitch d + 2 = 2 mod 4
    assert wide.stride(0) % 4 == 2
    _copied(wide[:, :D])


def test_overlapping_rows_are_copied():
    base = _aligned(1, 10 * D)
    t = base.view(-1).as_strided((10, D), (D // 2, 1))   # stride(0) < d: rows overlap
    _copied(t)


def test_contiguous_but_misaligned_view_is_copied_to_an_aligned_one():
    flat = torch.randn(10 * D + 1)
    t = flat[1:].view(10, D)
    assert t.is_contiguous() and t.data_ptr() % 16 != 0
    _copied(t)


def test_inner_stride_other_than_one_is_copied():
    _copied(_aligned(D, 10).t())
