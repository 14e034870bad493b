"""Link-prediction decode ``ops_decode.edge_dot`` (``csrc/decode.cu``) against fp64 torch.

Forward ``(z[a] * z[b]).sum(-1)`` and its autograd gradient, within rel 1e-5 of the summed |terms| of each output.
Widths reach every dispatch branch: 128-bit lanes with GROUP 2/4/8/16/32 (``feat % 4 == 0`` and ``z`` 16-byte
aligned), scalar lanes with GROUP 4/16/32.  Pairs repeat vertices and include self-pairs ``a == b``, whose gradient
the backward kernel accumulates with vector atomics; pair counts cover an empty list, partial warps of lane groups
and more pairs than one grid-stride pass of the kernel takes.
"""
import numpy as np
import pytest
import torch

from oracle import aggregate as A

pytestmark = pytest.mark.gpu

V4 = [4, 8, 12, 16, 32, 36, 64, 68, 128, 132, 256]     # GROUP 2, 2, 4, 4, 8, 16, 16, 32, 32, 32 (two passes), 32
SCALAR = [1, 3, 5, 17, 33, 101]                         # GROUP 4, 4, 16, 32, 32, 32


def _pairs(n, p, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, n, p)
    b = rng.integers(0, n, p)
    b[::5] = a[::5]                                     # self-pairs; n << p repeats every vertex many times
    return torch.from_numpy(a), torch.from_numpy(b)


def _dense(z):
    leaf = z.clone().requires_grad_(True)
    return leaf, leaf, lambda: leaf.grad


def _offset_by_one_float(z):
    """``z`` one float past an aligned address: the scalar path whatever the width."""
    n, f = z.shape
    leaf = torch.cat([torch.zeros(1, device=z.device), z.reshape(-1)]).requires_grad_(True)
    view = leaf[1:].view(n, f)
    assert view.is_contiguous() and view.data_ptr() % 16 == 4
    return leaf, view, lambda: leaf.grad[1:].view(n, f)


def _column_slice(z):
    """``z`` as the first columns of a wider matrix (not contiguous)."""
    n, f = z.shape
    leaf = torch.cat([z, torch.randn(n, 3, device=z.device)], 1).requires_grad_(True)
    view = leaf[:, :f]
    assert not view.is_contiguous()
    return leaf, view, lambda: leaf.grad[:, :f]


def _check(cuda, n, feat, p, seed, idx_dtype=torch.int64, layout=_dense, sum_loss=False):
    from stgraph_b200 import ops_decode

    tg = torch.Generator().manual_seed(seed)
    z_cpu = torch.randn(n, feat, generator=tg)
    g_cpu = torch.ones(p) if sum_loss else torch.randn(p, generator=tg)
    a, b = _pairs(n, p, seed)
    leaf, z, grad = layout(z_cpu.to(cuda))
    out = ops_decode.edge_dot(z, torch.stack([a, b]).to(device=cuda, dtype=idx_dtype))
    assert out.shape == (p,) and out.dtype == torch.float32
    if sum_loss:
        out.sum().backward()                            # grad_out reaches the kernel as an expanded stride-0 tensor
    else:
        out.backward(g_cpu.to(cuda))

    z64 = z_cpu.double().requires_grad_(True)
    ref = (z64[a] * z64[b]).sum(-1)
    ref.backward(g_cpu.double())
    zabs = z_cpu.double().abs().requires_grad_(True)
    mag = (zabs[a] * zabs[b]).sum(-1)                   # sum |terms| of every dot product ...
    mag.backward(g_cpu.double().abs())                  # ... and of every gradient row
    what = f"edge_dot F={feat} P={p}"
    A.assert_close_rel(out.detach().cpu(), ref.detach(), rel=1e-5, abs_terms=mag.detach(), what=what + " forward")
    A.assert_close_rel(grad().cpu(), z64.grad, rel=1e-5, abs_terms=zabs.grad, what=what + " backward")
    return leaf


@pytest.mark.parametrize("feat", V4 + SCALAR)
def test_widths(cuda, feat):
    _check(cuda, 300, feat, 1001, seed=feat)            # 1001 pairs: the last warp holds a partial set of lane groups


@pytest.mark.parametrize("p", [0, 1, 7])
@pytest.mark.parametrize("feat", [4, 12, 36, 132, 3, 33])
def test_short_pair_lists(cuda, feat, p):
    _check(cuda, 50, feat, p, seed=10 * feat + p)


@pytest.mark.parametrize("feat, p", [(4, 700_000), (256, 20_011), (101, 20_011)])
def test_more_pairs_than_one_grid_pass(cuda, feat, p):
    from stgraph_b200 import kernels

    group = {4: 2, 256: 32, 101: 32}[feat]
    assert p > 8 * kernels.device_info(cuda.index or 0)["sm_count"] * 256 // group
    _check(cuda, 5000, feat, p, seed=feat)


@pytest.mark.parametrize("feat", [4, 7, 64])
def test_int32_index(cuda, feat):
    _check(cuda, 400, feat, 3000, seed=feat + 1, idx_dtype=torch.int32)


@pytest.mark.parametrize("feat", [4, 64, 132, 7])
def test_z_off_a_16_byte_boundary(cuda, feat):
    _check(cuda, 400, feat, 3000, seed=feat + 2, layout=_offset_by_one_float)


@pytest.mark.parametrize("feat", [16, 33])
def test_non_contiguous_z(cuda, feat):
    leaf = _check(cuda, 400, feat, 3000, seed=feat + 3, layout=_column_slice)
    assert torch.count_nonzero(leaf.grad[:, feat:]) == 0


@pytest.mark.parametrize("feat", [32, 5])
def test_sum_loss_gives_stride0_grad(cuda, feat):
    _check(cuda, 400, feat, 3000, seed=feat + 4, sum_loss=True)


def test_out_of_range_index_raises(cuda):
    from stgraph_b200 import ops_decode

    z = torch.randn(10, 8, device=cuda)
    for bad in ([[0, 1], [2, 10]], [[0, -1], [2, 3]]):
        with pytest.raises(IndexError):
            ops_decode.edge_dot(z, torch.tensor(bad, device=cuda))


def test_zero_width_z(cuda):
    """``[N, 0]`` rows: torch gives zero scores and a zero gradient; so does ``edge_dot``."""
    from stgraph_b200 import ops_decode

    z = torch.randn(10, 0, device=cuda, requires_grad=True)
    idx = torch.tensor([[0, 3, 9], [1, 3, 2]], device=cuda)
    out = ops_decode.edge_dot(z, idx)
    assert torch.equal(out, (z[idx[0]] * z[idx[1]]).sum(-1)) and out.shape == (3,)
    out.sum().backward()
    assert z.grad is not None and z.grad.shape == (10, 0)
