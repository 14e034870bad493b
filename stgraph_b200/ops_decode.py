"""Link-prediction decode ``(z[a] * z[b]).sum(-1)`` as one fused kernel each way (``csrc/decode.cu``).

Drop-in for ``STGraphTGCN.decode`` of the reference's dynamic-temporal benchmark
(``benchmarking/dynamic-temporal-tgcn/seastar/model.py:18-21``)."""
from __future__ import annotations

import torch

from . import _lib, kernels


class _EdgeDot(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, a, b):
        z = z.contiguous()
        ctx.save_for_backward(z, a, b)
        if z.shape[1] == 0:             # every dot product is empty: zero scores, zero gradient (as torch computes them)
            return torch.zeros(a.shape[0], dtype=torch.float32, device=z.device)
        out = torch.empty(a.shape[0], dtype=torch.float32, device=z.device)
        _lib.call("stg_edge_dot_f32", z.data_ptr(), z.shape[1], a.data_ptr(), b.data_ptr(), a.shape[0], out.data_ptr(),
                  _lib.current_stream_ptr())
        kernels.launch_count += 1
        return out

    @staticmethod
    def backward(ctx, grad_out):
        z, a, b = ctx.saved_tensors
        d_z = torch.zeros_like(z)
        if z.shape[1] == 0:
            return d_z, None, None
        _lib.call("stg_edge_dot_bwd_f32", z.data_ptr(), z.shape[1], a.data_ptr(), b.data_ptr(), a.shape[0],
                  grad_out.contiguous().data_ptr(), d_z.data_ptr(), _lib.current_stream_ptr())
        kernels.launch_count += 1
        return d_z, None, None


def edge_dot(z: torch.Tensor, edge_label_index: torch.Tensor, check: bool = True) -> torch.Tensor:
    """``(z[idx[0]] * z[idx[1]]).sum(-1)`` for ``idx`` of shape ``[2, P]`` (int64 or int32 vertex ids).
    ``check=False`` skips the id range check (one host read-back; not capturable in a CUDA graph)."""
    if z.dim() != 2 or z.dtype != torch.float32 or not z.is_cuda:
        raise TypeError("z must be a [N, F] float32 CUDA tensor (stgraph_b200 has no CPU path)")
    if edge_label_index.dim() != 2 or edge_label_index.shape[0] != 2:
        raise ValueError("edge_label_index must be [2, P]")
    idx = edge_label_index.to(device=z.device, dtype=torch.int64).contiguous()
    if check and idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= z.shape[0]):
        raise IndexError(f"edge_label_index out of range for {z.shape[0]} vertices")
    return _EdgeDot.apply(z, idx[0], idx[1])
