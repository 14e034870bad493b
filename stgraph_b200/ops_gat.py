"""Fused edge-softmax attention aggregation as a torch autograd op (``csrc/gat.cu``).

``out[v,h,:] = sum_{u in in(v)} softmax_u(leaky_relu(el[u,h] + er[v,h])) * feat[u,h,:]`` -- what
``GATConv`` (``stgraph/nn/pytorch/static/gat_conv.py:48-56``) is meant to compute.  Forward is one
online-softmax pass; backward recomputes alpha (no ``[E,H]`` tensor, no atomics).
"""
from __future__ import annotations

import ctypes

import torch

import os

from . import _lib, kernels

#: rows longer than this go to the block-per-row attention kernels (the plain sum splits at csr.HUB_THRESHOLD = 1024).
#: A warp walks a row in groups of 8 (forward) / 4 (backward) neighbour rows per L2 round trip, so on a power-law graph
#: the longest warp-owned row sets the kernel time: config 3 (arxiv shape), 1024 -> 128 (profiles/r01_results.md).
GAT_HUB_THRESHOLD = int(os.environ.get("STG_GAT_HUB_THRESHOLD", "128"))


def _views(graph):
    """(in-edge view, out-edge view) of ``graph`` with the attention kernels' hub threshold."""
    bwd = graph.bwd_view()            # backward first: a dynamic graph builds both views in one go
    fwd = graph.fwd_view()
    f, b = graph._forward_graph, graph._backward_graph
    if hasattr(f, "view_with_hub_threshold") and hasattr(b, "view_with_hub_threshold"):
        return f.view_with_hub_threshold(GAT_HUB_THRESHOLD), b.view_with_hub_threshold(GAT_HUB_THRESHOLD)
    return fwd, bwd


class _GatEdgeSoftmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, graph, el, er, feat, slope):
        n, h, d = feat.shape
        el2 = el.reshape(n, h).contiguous().float()
        er2 = er.reshape(n, h).contiguous().float()
        dtype = kernels.H16_DTYPES.get(feat.dtype)
        if dtype is None:
            feat = feat.contiguous().float()
        else:
            # bf16 / fp16 rows stay 16-bit (the kernels widen them on load).  An 8-byte aligned start gives them the lanes
            # of the fp32 path's fresh copy, so the results are those of the fp32 kernels on feat.float(), bit for bit.
            feat = feat.contiguous()
            if feat.data_ptr() % 8:
                feat = feat.clone()
        out = torch.empty(n, h, d, device=feat.device, dtype=torch.float32)
        row_max = torch.empty(n, h, device=feat.device, dtype=torch.float32)
        row_sum = torch.empty_like(row_max)
        view = ctypes.byref(_views(graph)[0])
        if dtype is None:
            _lib.call("stg_gat_softmax_fwd_f32", view, el2.data_ptr(), er2.data_ptr(), feat.data_ptr(), h, d, float(slope),
                      out.data_ptr(), row_max.data_ptr(), row_sum.data_ptr(), _lib.current_stream_ptr())
        else:
            _lib.call("stg_gat_softmax_fwd_h16", view, el2.data_ptr(), er2.data_ptr(), feat.data_ptr(), h, d, dtype,
                      float(slope), out.data_ptr(), row_max.data_ptr(), row_sum.data_ptr(), _lib.current_stream_ptr())
        kernels.launch_count += 1
        ctx.graph, ctx.slope, ctx.shapes = graph, float(slope), (el.shape, er.shape)
        ctx.timestamp = getattr(graph, "current_timestamp", None)
        ctx.save_for_backward(el2, er2, feat, out, row_max, row_sum)
        return out

    @staticmethod
    def backward(ctx, gout):
        el2, er2, feat, out, row_max, row_sum = ctx.saved_tensors
        g = ctx.graph
        if ctx.timestamp is not None and hasattr(g, "get_backward_graph"):
            g.get_backward_graph(ctx.timestamp)
        n, h, d = feat.shape
        gout = gout.contiguous().float()
        d_feat = torch.empty_like(feat)          # feat's dtype: the 16-bit kernels round d_feat once, when they store it
        d_el = torch.empty_like(el2)
        d_er = torch.empty_like(er2)
        dot = torch.empty_like(el2)
        vf, vb = _views(g)
        args = (el2.data_ptr(), er2.data_ptr(), feat.data_ptr(), out.data_ptr(), gout.data_ptr(), row_max.data_ptr(),
                row_sum.data_ptr(), h, d)
        tail = (ctx.slope, d_feat.data_ptr(), d_el.data_ptr(), d_er.data_ptr(), dot.data_ptr(), _lib.current_stream_ptr())
        dtype = kernels.H16_DTYPES.get(feat.dtype)
        if dtype is None:
            _lib.call("stg_gat_softmax_bwd_f32", ctypes.byref(vf), ctypes.byref(vb), *args, *tail)
        else:
            _lib.call("stg_gat_softmax_bwd_h16", ctypes.byref(vf), ctypes.byref(vb), *args, dtype, *tail)
        kernels.launch_count += 2
        return None, d_el.reshape(ctx.shapes[0]), d_er.reshape(ctx.shapes[1]), d_feat, None


def gat_edge_softmax_aggregate(graph, el, er, feat, negative_slope=0.2):
    """``el, er``: ``[N,H,1]`` or ``[N,H]``; ``feat``: ``[N,H,D]`` -> ``[N,H,D]`` fp32.

    A bf16 / fp16 ``feat`` (``torch.autocast``) is read as it is, without an fp32 copy, and its gradient has its dtype;
    ``out`` and the softmax stay fp32 (``stg_gat_softmax_fwd_h16`` / ``stg_gat_softmax_bwd_h16``)."""
    for name, t in (("el", el), ("er", er), ("feat", feat)):
        if not t.is_cuda:
            raise RuntimeError(f"{name} must live on a CUDA device (stgraph_b200 has no CPU path)")
    if feat.dim() != 3:
        raise ValueError("feat must be [N, heads, dim]")
    return _GatEdgeSoftmax.apply(graph, el, er, feat, negative_slope)
