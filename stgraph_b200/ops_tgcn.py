"""The whole TGCN (GRU) cell as ONE torch autograd op: hand-written backward, no autograd glue between the pieces.

``stgraph/nn/pytorch/temporal/tgcn.py:16-55`` is three ``GCNConv`` + three ``Linear(2H, H)`` + the GRU arithmetic.  Run
through torch autograd piece by piece, one time step of the cell costs about 14 kernels forward and 60 backward (slice
gradients as zero-fill + copy, one bias reduction and one gradient accumulation per parameter use, transposes), and on a
WikiMaths-sized graph the loop is bound by their launches (``profiles/r02_results.md``, config 2).  Here the parameters
are packed once per BPTT window (:func:`pack_parameters`, differentiable, so the gradients reach the module's own
parameters through ONE concatenation backward per window) and the cell is a single ``autograd.Function``:

forward  (6 GEMMs, 1 aggregation, 3 element-wise passes)::

    h = clamp(agg(X @ [W_z|W_r|W_h]) + [b_z|b_r|b_h], +-1e6)          # [N, 3H], column blocks (z | r | h)
    P[:, z|r] = H @ [Lc_z|Lc_r] + [lb_z|lb_r] + h_z @ La_z | h_r @ La_r  # gate pre-activations, one [N, 3H] matrix
    HR = H * sigmoid(P_r);  P[:, h] = HR @ Lc_h + lb_h + h_h @ La_h
    H' = sigmoid(P_z) * H + (1 - sigmoid(P_z)) * tanh(P_h)

(``La_g`` / ``Lc_g`` are the halves of ``linear_g.weight`` that multiply the convolution output and the hidden state.)
backward (12 GEMMs, 1 aggregation on the out-edge CSR, 3 element-wise passes, 2 column sums): every GEMM reads or writes
a column block of ``P`` / ``dP`` / ``h`` / ``dh`` in place, the two bias gradients are one column sum each, the weight
gradients of the hidden-state halves of the z and r gates one GEMM.  The arithmetic per element is that of the reference
cell; sums run in a different order than in the piecewise autograd graph (fp32 rounding only).
Sync-free and allocation-light, so a whole BPTT window stays capturable in a CUDA graph.  (The three per-gate GEMMs on
column blocks as ONE strided-batched ``bmm`` were measured: 8 launches fewer per step, no faster on the WikiMaths shape
and 2.3x slower per epoch at N = 10^6 -- cuBLAS' strided-batched path with a leading dimension of 3H; not kept.)
"""
from __future__ import annotations

import torch

from . import _lib, kernels

CLAMP = 1e6     # tgcn.py:23,31,39
TALL_ROWS = 32768     # vertices from which the weight gradients go through kernels.gemm_tn instead of cuBLAS


def pack_parameters(conv_z, conv_r, conv_h, linear_z, linear_r, linear_h):
    """``(W3 [in,3H], b3 [3H], La [3,H,H], Lc_zr [H,2H], Lc_h [H,H], lb [3H])`` built from the module's parameters with
    differentiable torch ops (``linear.weight`` is ``[H, 2H]``: columns ``[:H]`` multiply the convolution output,
    ``[H:]`` the hidden state, ``tgcn.py:24-25``)."""
    hid = linear_z.weight.shape[0]
    W3 = torch.cat((conv_z.weight, conv_r.weight, conv_h.weight), dim=1)
    b3 = torch.cat((conv_z.bias, conv_r.bias, conv_h.bias))
    La = torch.stack([lin.weight[:, :hid].t() for lin in (linear_z, linear_r, linear_h)])
    Lc_zr = torch.cat((linear_z.weight[:, hid:].t(), linear_r.weight[:, hid:].t()), dim=1)
    Lc_h = linear_h.weight[:, hid:].t().contiguous()
    lb = torch.cat((linear_z.bias, linear_r.bias, linear_h.bias))
    return W3, b3, La, Lc_zr, Lc_h, lb


def _aggregate(csr, view, x, nflat, wflat):
    if getattr(csr, "pack_enabled", False):      # static graph: packed {col, scale} array, built on first use
        return kernels.agg_scaled_sum_graph(csr, x, nflat, wflat, nflat)
    return kernels.agg_scaled_sum(view, x, nflat, wflat, nflat)


def lowp_parameters(packed, dt):
    """The 16-bit GEMM operands of :func:`pack_parameters`' tuple: ``(W3, La, Lc_zr, Lc_h)`` rounded to ``dt``, detached
    (the cell returns the gradients of the fp32 pack).  Made once per pack, not per step."""
    W3, _, La, Lc_zr, Lc_h, _ = packed
    return tuple(t.detach().to(dt).contiguous() for t in (W3, La, Lc_zr, Lc_h))


class _TgcnCell(torch.autograd.Function):
    """``lowp`` is None (fp32 cell) or ``(dt, W3, La, Lc_zr, Lc_h)`` in ``dt`` = bf16 / fp16 (the cell under autocast)."""

    @staticmethod
    def forward(ctx, fwd_view, bwd_view, keepalive, norm, edge_weight, X, H, W3, b3, La, Lc_zr, Lc_h, lb, lowp):
        ctx.lowp = lowp is not None
        if lowp is not None:
            with torch.autocast("cuda", enabled=False):
                return _TgcnCell._forward16(ctx, fwd_view, bwd_view, keepalive, norm, edge_weight, X, H, b3, lb, lowp)
        X, H = X.contiguous(), H.contiguous()
        n, hid = H.shape
        st = _lib.current_stream_ptr()
        nflat = norm.reshape(-1)
        wflat = edge_weight.reshape(-1) if edge_weight is not None else None
        h = _aggregate(keepalive[0], fwd_view, torch.mm(X, W3), nflat, wflat)          # fresh [N, 3H]
        _lib.call("stg_bias_clamp_f32", h.data_ptr(), b3.contiguous().data_ptr(), n, 3 * hid, -CLAMP, CLAMP, st)
        P = torch.empty(n, 3 * hid, device=H.device, dtype=H.dtype)
        torch.addmm(lb[:2 * hid], H, Lc_zr, out=P[:, :2 * hid])
        P[:, :hid].addmm_(h[:, :hid], La[0])
        P[:, hid:2 * hid].addmm_(h[:, hid:2 * hid], La[1])
        HR = torch.empty_like(H)
        _lib.call("stg_tgcn_reset_fwd_f32", P.data_ptr(), H.data_ptr(), HR.data_ptr(), n, hid, st)
        torch.addmm(lb[2 * hid:], HR, Lc_h, out=P[:, 2 * hid:])
        P[:, 2 * hid:].addmm_(h[:, 2 * hid:], La[2])
        out = torch.empty_like(H)
        _lib.call("stg_tgcn_update_fwd_f32", P.data_ptr(), H.data_ptr(), out.data_ptr(), n, hid, st)
        kernels.launch_count += 3
        ctx.views = (bwd_view, keepalive)
        ctx.weighted = wflat is not None
        ctx.save_for_backward(X, H, h, P, HR, W3, La, Lc_zr, Lc_h, nflat, wflat if wflat is not None else nflat)
        return out

    @staticmethod
    def backward(ctx, d_out):
        if ctx.lowp:
            with torch.autocast("cuda", enabled=False):
                return _TgcnCell._backward16(ctx, d_out)
        X, H, h, P, HR, W3, La, Lc_zr, Lc_h, nflat, wflat = ctx.saved_tensors
        bwd_view, keepalive = ctx.views
        need = ctx.needs_input_grad          # (.., X=5, H=6, W3=7, b3=8, La=9, Lc_zr=10, Lc_h=11, lb=12)
        n, hid = H.shape
        st = _lib.current_stream_ptr()
        d_out = d_out.contiguous()
        dP = torch.empty_like(P)
        dH = torch.empty_like(H)
        _lib.call("stg_tgcn_update_bwd_f32", P.data_ptr(), H.data_ptr(), d_out.data_ptr(), dP.data_ptr(), dH.data_ptr(), n, hid, st)
        dHR = torch.mm(dP[:, 2 * hid:], Lc_h.t())
        _lib.call("stg_tgcn_reset_bwd_f32", P.data_ptr(), H.data_ptr(), dHR.data_ptr(), dP.data_ptr(), dH.data_ptr(), n, hid, st)
        if need[6]:
            dH.addmm_(dP[:, :2 * hid], Lc_zr.t())
        dh = torch.empty_like(h)
        for g in range(3):
            torch.mm(dP[:, g * hid:(g + 1) * hid], La[g].t(), out=dh[:, g * hid:(g + 1) * hid])
        # gradient of clamp(a + b): masked in place (element-wise, the kernel reads d_y[i] before it writes d_a[i])
        _lib.call("stg_clamp_bwd_f32", h.data_ptr(), dh.data_ptr(), dh.data_ptr(), dh.numel(), -CLAMP, CLAMP, st)
        kernels.launch_count += 3
        d_b3 = dh.sum(0) if need[8] else None
        # weight gradients: [K, N] x [N, Nc] with N = number of vertices.  On large graphs our split-M kernel (exact fp32,
        # the bias column sums ride along); below TALL_ROWS the cuBLAS call is one or two tiny launches either way.
        tall = n >= TALL_ROWS
        tn = kernels.gemm_tn if tall else (lambda a, b: torch.mm(a.t(), b))
        d_W3 = d_X = None
        if need[5] or need[7]:
            dXW = _aggregate(keepalive[1], bwd_view, dh, nflat, wflat if ctx.weighted else None)
            if need[7]:
                d_W3 = tn(X, dXW)
            if need[5]:
                d_X = torch.mm(dXW, W3.t())
        d_lb = None
        d_Lc_zr = d_Lc_h = None
        if tall and need[12] and need[10] and need[11]:          # the two GEMMs that read all of dP also sum its columns
            d_Lc_zr, lb_zr = kernels.gemm_tn(H, dP[:, :2 * hid], colsum=True)
            d_Lc_h, lb_h = kernels.gemm_tn(HR, dP[:, 2 * hid:], colsum=True)
            d_lb = torch.cat((lb_zr, lb_h))
        else:
            d_lb = dP.sum(0) if need[12] else None
            d_Lc_zr = tn(H, dP[:, :2 * hid]) if need[10] else None
            d_Lc_h = tn(HR, dP[:, 2 * hid:]) if need[11] else None
        d_La = None
        if need[9]:
            d_La = torch.empty_like(La)
            for g in range(3):
                blk = slice(g * hid, (g + 1) * hid)
                if tall:
                    kernels.gemm_tn(h[:, blk], dP[:, blk], out=d_La[g])
                else:
                    torch.mm(h[:, blk].t(), dP[:, blk], out=d_La[g])
        return (None, None, None, None, None, d_X, dH if need[6] else None, d_W3, d_b3, d_La, d_Lc_zr, d_Lc_h, d_lb, None)

    # ---- the cell under autocast (dt = bf16 / fp16).  Every GEMM takes dt operands and accumulates in fp32.  Stored in
    # dt: X·W3, its aggregation A, h = clamp(A + b3), HR, the dt twin dP16 of dP, dh and dXW -- the tensors that are only
    # GEMM operands -- each written by the kernel or GEMM that produces it.  Stored in fp32: P, out, dP, dH and the
    # parameter gradients.  The gate arithmetic is the fp32 kernels' (csrc/gates.cu).
    @staticmethod
    def _forward16(ctx, fwd_view, bwd_view, keepalive, norm, edge_weight, X, H, b3, lb, lowp):
        dt, W3, La, Lc_zr, Lc_h = lowp
        f32 = torch.float32
        code = kernels.H16_DTYPES[dt]
        X16 = X.to(dt).contiguous()                        # X and H: one cast each (none when they come in dt / fp32)
        H32 = H.to(f32).contiguous()
        H16 = H.to(dt).contiguous()
        n, hid = H.shape
        st = _lib.current_stream_ptr()
        nflat = norm.reshape(-1)
        wflat = edge_weight.reshape(-1) if edge_weight is not None else None
        b3 = b3.contiguous()
        A = _aggregate(keepalive[0], fwd_view, torch.mm(X16, W3), nflat, wflat)        # [N, 3H] dt, kept for the mask
        h = torch.empty_like(A)
        _lib.call("stg_tgcn_bias_clamp_h16", A.data_ptr(), b3.data_ptr(), h.data_ptr(), n, 3 * hid, code, -CLAMP, CLAMP, st)
        P = torch.empty(n, 3 * hid, device=H.device, dtype=f32)
        torch.addmm(lb[:2 * hid], H16, Lc_zr, out_dtype=f32, out=P[:, :2 * hid])
        for g in range(2):
            blk = P[:, g * hid:(g + 1) * hid]
            torch.addmm(blk, h[:, g * hid:(g + 1) * hid], La[g], out_dtype=f32, out=blk)
        HR = torch.empty(n, hid, device=H.device, dtype=dt)
        _lib.call("stg_tgcn_reset_fwd_h16", P.data_ptr(), H32.data_ptr(), HR.data_ptr(), n, hid, code, st)
        Ph = P[:, 2 * hid:]
        torch.addmm(lb[2 * hid:], HR, Lc_h, out_dtype=f32, out=Ph)
        torch.addmm(Ph, h[:, 2 * hid:], La[2], out_dtype=f32, out=Ph)
        out = torch.empty(n, hid, device=H.device, dtype=f32)
        _lib.call("stg_tgcn_update_fwd_f32", P.data_ptr(), H32.data_ptr(), out.data_ptr(), n, hid, st)
        kernels.launch_count += 3
        ctx.views = (bwd_view, keepalive)
        ctx.weighted = wflat is not None
        ctx.dt, ctx.x_dtype = dt, X.dtype
        ctx.save_for_backward(X16, H32, H16, A, h, P, HR, W3, b3, La, Lc_zr, Lc_h, nflat,
                              wflat if wflat is not None else nflat)
        return out

    @staticmethod
    def _backward16(ctx, d_out):
        X16, H32, H16, A, h, P, HR, W3, b3, La, Lc_zr, Lc_h, nflat, wflat = ctx.saved_tensors
        bwd_view, keepalive = ctx.views
        need = ctx.needs_input_grad          # (.., X=5, H=6, W3=7, b3=8, La=9, Lc_zr=10, Lc_h=11, lb=12)
        dt, f32 = ctx.dt, torch.float32
        code = kernels.H16_DTYPES[dt]
        n, hid = H32.shape
        st = _lib.current_stream_ptr()
        d_out = d_out.to(f32).contiguous()
        dP = torch.empty_like(P)
        dP16 = torch.empty(n, 3 * hid, device=P.device, dtype=dt)
        dH = torch.empty_like(H32)
        _lib.call("stg_tgcn_update_bwd_h16", P.data_ptr(), H32.data_ptr(), d_out.data_ptr(), dP.data_ptr(), dP16.data_ptr(),
                  dH.data_ptr(), n, hid, code, st)
        dHR = torch.mm(dP16[:, 2 * hid:], Lc_h.t(), out_dtype=f32)
        _lib.call("stg_tgcn_reset_bwd_h16", P.data_ptr(), H32.data_ptr(), dHR.data_ptr(), dP.data_ptr(), dP16.data_ptr(),
                  dH.data_ptr(), n, hid, code, st)
        if need[6]:
            torch.addmm(dH, dP16[:, :2 * hid], Lc_zr.t(), out_dtype=f32, out=dH)
        dh = torch.empty_like(h)
        for g in range(3):
            torch.mm(dP16[:, g * hid:(g + 1) * hid], La[g].t(), out=dh[:, g * hid:(g + 1) * hid])
        # gradient of clamp(A + b3): masked in place on the fp32 value A + b3, not on the rounded h
        _lib.call("stg_tgcn_clamp_bwd_h16", A.data_ptr(), b3.data_ptr(), dh.data_ptr(), dh.data_ptr(), n, 3 * hid, code,
                  -CLAMP, CLAMP, st)
        kernels.launch_count += 3
        d_b3 = dh.sum(0, dtype=f32) if need[8] else None

        def tn(a, b, out=None):          # weight gradients [K, N] x [N, Nc]: dt operands, fp32 result, at every N
            return torch.mm(a.t(), b, out_dtype=f32) if out is None else torch.mm(a.t(), b, out_dtype=f32, out=out)

        d_W3 = d_X = None
        if need[5] or need[7]:
            dXW = _aggregate(keepalive[1], bwd_view, dh, nflat, wflat if ctx.weighted else None)
            if need[7]:
                d_W3 = tn(X16, dXW)
            if need[5]:
                d_X = torch.mm(dXW, W3.t()) if ctx.x_dtype == dt else torch.mm(dXW, W3.t(), out_dtype=f32)
        d_lb = dP.sum(0) if need[12] else None
        d_Lc_zr = tn(H16, dP16[:, :2 * hid]) if need[10] else None
        d_Lc_h = tn(HR, dP16[:, 2 * hid:]) if need[11] else None
        d_La = None
        if need[9]:
            d_La = torch.empty(La.shape, device=La.device, dtype=f32)
            for g in range(3):
                blk = slice(g * hid, (g + 1) * hid)
                tn(h[:, blk], dP16[:, blk], out=d_La[g])
        return (None, None, None, None, None, d_X, dH if need[6] else None, d_W3, d_b3, d_La, d_Lc_zr, d_Lc_h, d_lb, None)


def tgcn_cell(graph, X, H, norm, edge_weight, packed, lowp=None):
    """One step of the TGCN cell on ``graph`` (static graph or the current snapshot of a dynamic one); ``packed`` is
    :func:`pack_parameters`' tuple.  Differentiable w.r.t. ``X``, ``H`` and the packed parameters.

    Under ``torch.autocast("cuda", dtype=dt)`` with ``dt`` bf16 / fp16 the cell runs its 16-bit form: ``X`` and ``H`` may
    be fp32 or ``dt``, the GEMMs take ``dt`` operands (``lowp``: :func:`lowp_parameters` of ``packed``, made here when
    None) with fp32 accumulation, and the returned hidden state is fp32."""
    if not X.is_cuda:
        raise RuntimeError("X must live on a CUDA device (stgraph_b200 has no CPU path)")
    lp = None
    if torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
        if dt not in kernels.H16_DTYPES:
            raise TypeError(f"the fused TGCN cell runs under autocast with bfloat16 or float16, not {dt}")
        if X.dtype not in (torch.float32, dt) or H.dtype not in (torch.float32, dt):
            raise TypeError(f"under {dt} autocast the fused TGCN cell takes float32 or {dt} X and H, got {X.dtype} and {H.dtype}")
        lp = (dt,) + (tuple(lowp) if lowp is not None else lowp_parameters(packed, dt))
    elif X.dtype != torch.float32 or H.dtype != torch.float32:
        raise TypeError("the fused TGCN cell computes in float32")
    bwd = graph.bwd_view()            # backward first: a dynamic graph builds both views in one go
    fwd = graph.fwd_view()
    keep = (graph._forward_graph, graph._backward_graph)
    return _TgcnCell.apply(fwd, bwd, keep, norm, edge_weight, X, H, *packed, lp)
