"""Thin Python wrappers over the C-ABI kernels (tensor checks + stream plumbing).

Argument validation (dtype, contiguity, device) happens here; the C functions
validate pointers/sizes and return error codes (SURVEY.md section 8(b) "errors").
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib

#: number of kernels launched through this module since import (bench.py reports it)
launch_count = 0


def _check(t: torch.Tensor, name: str, dtype=torch.float32):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (stgraph_b200 has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


#: 16-bit feature types of the aggregation (``StgDtype``): fp32 accumulation, one rounding per output element
H16_DTYPES = {torch.bfloat16: 1, torch.float16: 2}


def _agg_h16(view, meta, x, nbr_scale, edge_scale, row_scale, out, accumulate, stream, out_rows=None):
    """16-bit ``x`` (``stg_agg_scaled_sum_h16`` / ``stg_agg_packed_sum_h16``): contiguous, assign-only, ``out`` of ``x``'s
    dtype; the scales stay fp32.  Everything is checked before the launch."""
    global launch_count
    if accumulate is not False:
        raise ValueError(f"accumulate={accumulate!r} is an fp32-only form of the aggregation; {x.dtype} x is assign-only")
    if out_rows is not None:
        raise ValueError(f"out_rows is an fp32-only form of the aggregation (got {x.dtype} x)")
    for nm, t in (("x", x), ("out", out)):
        if isinstance(t, torch.Tensor) and not t.is_contiguous():
            raise ValueError(f"padded / strided rows are an fp32-only form of the aggregation: {x.dtype} {nm} must be contiguous")
    _check(x, "x", x.dtype)
    if x.dim() < 2:
        raise ValueError("x must be [rows, feat...]")
    n = view.num_nodes
    feat = x.numel() // max(x.shape[0], 1)
    for nm, t in (("nbr_scale", nbr_scale), ("edge_scale", edge_scale), ("row_scale", row_scale)):
        if t is not None:
            _check(t, nm)
    if nbr_scale is not None and nbr_scale.numel() != x.shape[0]:
        raise ValueError(f"nbr_scale must have one entry per row of x ({x.shape[0]}), got {nbr_scale.numel()}")
    if row_scale is not None and row_scale.numel() != n:
        raise ValueError(f"row_scale must have {n} elements, got {row_scale.numel()}")
    if edge_scale is not None and edge_scale.numel() < view.num_edges:
        raise ValueError(f"edge_scale has {edge_scale.numel()} elements for {view.num_edges} edges")
    if meta is not None:
        _check(meta, "meta", torch.int32)
        if meta.numel() < 2 * view.num_edges:
            raise ValueError(f"meta has {meta.numel() // 2} entries for {view.num_edges} edges")
    if out is None:
        if x.shape[0] != n:
            raise ValueError(f"x has {x.shape[0]} rows for a view of {n} rows: pass out= for a row slice")
        out = torch.empty_like(x)
    else:
        _check(out, "out", x.dtype)
        if out.shape[0] != n or out.numel() != n * feat:
            raise ValueError(f"out must be [{n}, {feat}], got {tuple(out.shape)}")
    if n == 0 or feat == 0:
        return out
    st = stream if stream is not None else _lib.current_stream_ptr()
    if meta is None:
        _lib.call("stg_agg_scaled_sum_h16", ctypes.byref(view), x.data_ptr(), feat, H16_DTYPES[x.dtype], _lib.ptr(nbr_scale),
                  _lib.ptr(edge_scale), _lib.ptr(row_scale), out.data_ptr(), st)
    else:
        _lib.call("stg_agg_packed_sum_h16", ctypes.byref(view), meta.data_ptr(), x.data_ptr(), feat, H16_DTYPES[x.dtype],
                  _lib.ptr(row_scale), out.data_ptr(), st)
    launch_count += 1 + (1 if view.hub_threshold > 0 else 0)
    return out


def agg_scaled_sum(view: _lib.StgCsrView, x: torch.Tensor, nbr_scale=None, edge_scale=None, row_scale=None,
                   out: torch.Tensor | None = None, accumulate=False, stream=None, out_rows=None) -> torch.Tensor:
    """``out[r] = row_scale[r] * sum_e nbr_scale[c_e] * edge_scale[eid_e] * x[c_e]`` (see ``stg_agg_scaled_sum_f32``).

    ``accumulate``: False (assign), True (``+=``) or ``"red"`` (``red.global.add``).  ``out_rows`` (int32, strictly
    increasing): the view holds a subset of the output rows, view row ``i`` is ``out[out_rows[i]]``
    (``stg_agg_scaled_sum_rows_f32``); ``out`` is then required.

    A bf16 / fp16 ``x`` is summed in fp32 and ``out`` has ``x``'s dtype (``stg_agg_scaled_sum_h16``); that form is
    contiguous and assign-only, and the scales stay fp32.
    """
    global launch_count
    if isinstance(x, torch.Tensor) and x.dtype in H16_DTYPES:
        return _agg_h16(view, None, x, nbr_scale, edge_scale, row_scale, out, accumulate, stream, out_rows)
    _check(x, "x")
    n = view.num_nodes                      # rows of this view (a row slice of a partitioned graph has fewer rows than x)
    if out_rows is not None:
        _check(out_rows, "out_rows", torch.int32)
        if out is None or out_rows.numel() != n:
            raise ValueError("out_rows needs out= and one entry per view row")
        n = out.shape[0]
    if x.dim() < 2:
        raise ValueError("x must be [rows, feat...]")
    feat = x.numel() // max(x.shape[0], 1)
    for nm, t in (("nbr_scale", nbr_scale), ("edge_scale", edge_scale)):
        if t is not None:
            _check(t, nm)
    if nbr_scale is not None and nbr_scale.numel() != x.shape[0]:
        raise ValueError(f"nbr_scale must have one entry per row of x ({x.shape[0]}), got {nbr_scale.numel()}")
    if row_scale is not None:
        _check(row_scale, "row_scale")
        if row_scale.numel() != n:
            raise ValueError(f"row_scale must have {n} elements, got {row_scale.numel()}")
    if edge_scale is not None and edge_scale.numel() < view.num_edges:
        raise ValueError(f"edge_scale has {edge_scale.numel()} elements for {view.num_edges} edges")
    if out is None:
        if x.shape[0] != n:
            raise ValueError(f"x has {x.shape[0]} rows for a view of {n} rows: pass out= for a row slice")
        out = torch.empty_like(x)
    else:
        _check(out, "out")
        if out.shape[0] != n or out.numel() != n * feat:
            raise ValueError(f"out must be [{n}, {feat}], got {tuple(out.shape)}")
    if n == 0 or feat == 0 or view.num_nodes == 0:
        return out
    if out_rows is not None:
        _lib.call("stg_agg_scaled_sum_rows_f32", ctypes.byref(view), out_rows.data_ptr(), x.data_ptr(), feat,
                  _lib.ptr(nbr_scale), _lib.ptr(edge_scale), _lib.ptr(row_scale), out.data_ptr(),
                  {False: 0, True: 1, "red": 2}[accumulate], stream if stream is not None else _lib.current_stream_ptr())
        launch_count += 1 + (1 if view.hub_threshold > 0 else 0)
        return out
    fn = {False: "stg_agg_scaled_sum_f32", True: "stg_agg_scaled_sum_accum_f32", "red": "stg_agg_scaled_sum_red_f32"}[accumulate]
    _lib.call(fn, ctypes.byref(view), x.data_ptr(), feat, _lib.ptr(nbr_scale), _lib.ptr(edge_scale), _lib.ptr(row_scale),
              out.data_ptr(), stream if stream is not None else _lib.current_stream_ptr())
    launch_count += 1 + (1 if view.hub_threshold > 0 else 0)
    return out


def pack_edge_meta(view: _lib.StgCsrView, nbr_scale=None, edge_scale=None, out: torch.Tensor | None = None,
                   device=None) -> torch.Tensor:
    """``meta[e] = {col[e], nbr_scale[col[e]] * edge_scale[eid(e)]}`` per CSR slot as an int32 ``[E, 2]`` tensor
    (``stg_csr_pack_edge_meta_f32``); feed it to :func:`agg_packed_sum`."""
    global launch_count
    for nm, t in (("nbr_scale", nbr_scale), ("edge_scale", edge_scale)):
        if t is not None:
            _check(t, nm)
    if edge_scale is not None and edge_scale.numel() < view.num_edges:
        raise ValueError(f"edge_scale has {edge_scale.numel()} elements for {view.num_edges} edges")
    if out is None:
        ref = nbr_scale if nbr_scale is not None else edge_scale
        dev = device if device is not None else (ref.device if ref is not None else torch.device("cuda", torch.cuda.current_device()))
        out = torch.empty(view.num_edges, 2, dtype=torch.int32, device=dev)
    else:
        _check(out, "out", torch.int32)
        if out.numel() != 2 * view.num_edges:
            raise ValueError(f"meta must be int32 [{view.num_edges}, 2]")
    if view.num_edges == 0:
        return out
    _lib.call("stg_csr_pack_edge_meta_f32", ctypes.byref(view), _lib.ptr(nbr_scale), _lib.ptr(edge_scale), out.data_ptr(),
              _lib.current_stream_ptr())
    launch_count += 1
    return out


def padded_rows(rows: int, feat: int, device, dtype=torch.float32) -> torch.Tensor:
    """``[rows, feat]`` view whose rows start on 128-byte lines (row stride = feat rounded up to 32 floats).

    :func:`agg_packed_sum` takes such views (and any other 2-D view with dense rows) as ``x`` / ``out``.  Measured on
    config 5 (F=100): no faster than the dense layout -- kept for in-place aggregation of column blocks.
    """
    ld = (feat + 31) // 32 * 32
    return torch.empty(rows, ld, dtype=dtype, device=device)[:, :feat]


def _row_stride(t: torch.Tensor, name: str) -> int:
    """Row stride (floats) of a 2-D fp32 CUDA tensor whose rows are dense (``stride(1) == 1``)."""
    if t.dim() == 2 and not t.is_contiguous():
        if not t.is_cuda:
            raise RuntimeError(f"{name} must live on a CUDA device (stgraph_b200 has no CPU path)")
        if t.dtype != torch.float32:
            raise TypeError(f"{name} must be torch.float32, got {t.dtype}")
        if t.shape[1] > 0 and (t.stride(1) != 1 or t.stride(0) < t.shape[1]):
            raise ValueError(f"{name} must have dense rows (stride(1) == 1, stride(0) >= feat)")
        return int(t.stride(0))
    _check(t, name)
    return t.numel() // max(t.shape[0], 1)


def agg_packed_sum(view: _lib.StgCsrView, meta: torch.Tensor, x: torch.Tensor, row_scale=None,
                   out: torch.Tensor | None = None, accumulate=False, stream=None) -> torch.Tensor:
    """``out[r] = row_scale[r] * sum_e meta[e].scale * x[meta[e].col]`` (``stg_agg_packed_sum_strided_f32``): the sums
    of :func:`agg_scaled_sum`, bit for bit, with one coalesced 8-byte load per edge instead of dependent gathers.
    ``x`` / ``out`` may be row-padded 2-D views (:func:`padded_rows`).  A bf16 / fp16 ``x`` takes the 16-bit form of
    :func:`agg_scaled_sum` (``stg_agg_packed_sum_h16``: contiguous, assign-only) with the same ``meta``."""
    global launch_count
    if isinstance(x, torch.Tensor) and x.dtype in H16_DTYPES:
        return _agg_h16(view, meta, x, None, None, row_scale, out, accumulate, stream)
    x_ld = _row_stride(x, "x")
    _check(meta, "meta", torch.int32)
    n = view.num_nodes
    if meta.numel() < 2 * view.num_edges:
        raise ValueError(f"meta has {meta.numel() // 2} entries for {view.num_edges} edges")
    if x.dim() < 2:
        raise ValueError("x must be [rows, feat...]")
    feat = x.shape[1] if x.dim() == 2 else x.numel() // max(x.shape[0], 1)
    if row_scale is not None:
        _check(row_scale, "row_scale")
        if row_scale.numel() != n:
            raise ValueError(f"row_scale must have {n} elements, got {row_scale.numel()}")
    if out is None:
        if x.shape[0] != n:
            raise ValueError(f"x has {x.shape[0]} rows for a view of {n} rows: pass out= for a row slice")
        out = padded_rows(n, feat, x.device) if x_ld != feat else torch.empty_like(x)
    out_ld = _row_stride(out, "out")
    if out.shape[0] != n or out.numel() != n * feat:
        raise ValueError(f"out must be [{n}, {feat}], got {tuple(out.shape)}")
    if n == 0 or feat == 0:
        return out
    _lib.call("stg_agg_packed_sum_strided_f32", ctypes.byref(view), meta.data_ptr(), x.data_ptr(), feat, x_ld,
              _lib.ptr(row_scale), out.data_ptr(), out_ld, {False: 0, True: 1, "red": 2}[accumulate],
              stream if stream is not None else _lib.current_stream_ptr())
    launch_count += 1 + (1 if view.hub_threshold > 0 else 0)
    return out


def agg_packed_sum_rows(view: _lib.StgCsrView, meta: torch.Tensor, out_rows, x: torch.Tensor, row_scale, out: torch.Tensor,
                        accumulate=False, stream=None) -> torch.Tensor:
    """Row-subset form of :func:`agg_packed_sum` (``stg_agg_packed_sum_rows_f32``): view row ``i`` is ``out[out_rows[i]]``
    (``out_rows`` None: identity); ``x`` is the source matrix the packed columns index (any number of rows)."""
    global launch_count
    _check(x, "x")
    _check(out, "out")
    _check(meta, "meta", torch.int32)
    if meta.numel() < 2 * view.num_edges:
        raise ValueError(f"meta has {meta.numel() // 2} entries for {view.num_edges} edges")
    feat = x.numel() // max(x.shape[0], 1)
    if out.numel() != out.shape[0] * feat:
        raise ValueError(f"out must be [rows, {feat}], got {tuple(out.shape)}")
    if out_rows is not None:
        _check(out_rows, "out_rows", torch.int32)
        if out_rows.numel() != view.num_nodes:
            raise ValueError("out_rows needs one entry per view row")
    elif out.shape[0] != view.num_nodes:
        raise ValueError(f"out has {out.shape[0]} rows for a view of {view.num_nodes} rows")
    if row_scale is not None:
        _check(row_scale, "row_scale")
        if row_scale.numel() != out.shape[0]:
            raise ValueError(f"row_scale must have one entry per row of out ({out.shape[0]}), got {row_scale.numel()}")
    if view.num_nodes == 0 or feat == 0:
        return out
    _lib.call("stg_agg_packed_sum_rows_f32", ctypes.byref(view), meta.data_ptr(), _lib.ptr(out_rows), x.data_ptr(), feat,
              _lib.ptr(row_scale), out.data_ptr(), {False: 0, True: 1, "red": 2}[accumulate],
              stream if stream is not None else _lib.current_stream_ptr())
    launch_count += 1 + (1 if view.hub_threshold > 0 else 0)
    return out


def agg_scaled_sum_graph(csr, x: torch.Tensor, nbr_scale=None, edge_scale=None, row_scale=None,
                         out: torch.Tensor | None = None) -> torch.Tensor:
    """:func:`agg_scaled_sum` over one direction of a graph object (``graph/static/csr.py:CSR``).  A static CSR
    keeps the packed ``{col, scale}`` array of the scales it was last called with (``CSR.packed_meta``), so every
    call after the first runs the packed kernel; dynamic snapshots and unscaled sums take the plain kernel."""
    meta = csr.packed_meta(nbr_scale, edge_scale) if getattr(csr, "pack_enabled", False) else None
    if meta is None:
        return agg_scaled_sum(csr.view(), x, nbr_scale, edge_scale, row_scale, out=out)
    return agg_packed_sum(csr.view(), meta, x, row_scale, out=out)


def gemm_tn(a: torch.Tensor, b: torch.Tensor, colsum: bool = False, out: torch.Tensor | None = None):
    """``a^T @ b`` for ``a [M, K]``, ``b [M, Nc]`` with ``M >> K, Nc`` (``stg_gemm_tn_f32``: the weight-gradient GEMM of the
    TGCN cell, exact fp32, deterministic); with ``colsum`` also the column sums of ``b`` (the bias gradient).  ``a`` and
    ``b`` may be column blocks of wider row-major matrices (unit stride along the row)."""
    global launch_count
    for nm, t in (("a", a), ("b", b)):
        if not t.is_cuda or t.dtype != torch.float32 or t.dim() != 2:
            raise TypeError(f"{nm} must be a 2-D float32 CUDA tensor")
        if t.shape[1] > 1 and t.stride(1) != 1:
            raise ValueError(f"{nm} must have unit stride along its rows (got strides {tuple(t.stride())})")
    if a.shape[0] != b.shape[0]:
        raise ValueError(f"a and b must have the same number of rows ({a.shape[0]} vs {b.shape[0]})")
    m, k, nc = a.shape[0], a.shape[1], b.shape[1]
    lda = a.stride(0) if m > 1 else max(k, 1)
    ldb = b.stride(0) if m > 1 else max(nc, 1)
    if out is not None and (out.shape != (k, nc) or not out.is_contiguous() or out.dtype != torch.float32):
        raise ValueError(f"out must be a contiguous float32 [{k}, {nc}] tensor")
    c = out if out is not None else torch.empty(k, nc, device=a.device, dtype=torch.float32)
    cs = torch.empty(nc, device=a.device, dtype=torch.float32) if colsum else None
    need = _lib.call("stg_gemm_tn_workspace_bytes", m, k, nc)
    ws = torch.empty(need // 4, device=a.device, dtype=torch.float32) if need else None
    _lib.call("stg_gemm_tn_f32", a.data_ptr(), lda, b.data_ptr(), ldb, m, k, nc, c.data_ptr(), _lib.ptr(cs), _lib.ptr(ws), need,
              _lib.current_stream_ptr())
    launch_count += 2 if need else 1
    return (c, cs) if colsum else c


def agg_scaled_sum_host(view: _lib.StgCsrView, x_host: torch.Tensor, out_host: torch.Tensor, scratch: torch.Tensor,
                        nbr_scale_host=None, edge_scale_host=None, row_scale_host=None, stream=None):
    """Host-buffer variant (H2D + kernel + D2H inside one C call); buffers should be pinned.

    ``stream`` (a ``torch.cuda.Stream``): enqueue only (``stg_agg_scaled_sum_f32_host_async``) -- ``out_host`` is valid
    after ``stream.synchronize()``; calls on two streams with two scratch buffers overlap H2D with D2H."""
    global launch_count
    n = view.num_nodes
    feat = x_host.numel() // max(n, 1)
    fn = "stg_agg_scaled_sum_f32_host" if stream is None else "stg_agg_scaled_sum_f32_host_async"
    _lib.call(fn, ctypes.byref(view), x_host.data_ptr(), feat,
              _lib.ptr(nbr_scale_host), _lib.ptr(edge_scale_host), _lib.ptr(row_scale_host),
              out_host.data_ptr(), scratch.data_ptr(), scratch.numel() * scratch.element_size(),
              _lib.current_stream_ptr() if stream is None else stream.cuda_stream)
    launch_count += 1 + (1 if view.hub_threshold > 0 else 0)
    return out_host


def host_scratch_bytes(num_nodes: int, num_edges: int, feat: int) -> int:
    up4 = lambda v: (v + 3) // 4 * 4
    return 4 * (2 * up4(num_nodes * feat) + 2 * up4(num_nodes) + up4(num_edges))


def device_info(device: int = 0):
    sm = ctypes.c_int32()
    l2 = ctypes.c_int64()
    maj = ctypes.c_int32()
    mnr = ctypes.c_int32()
    _lib.call("stg_device_info", device, ctypes.byref(sm), ctypes.byref(l2), ctypes.byref(maj), ctypes.byref(mnr))
    return {"sm_count": sm.value, "l2_bytes": l2.value, "cc": (maj.value, mnr.value)}


def agg_scaled_sum_parts(view: _lib.StgCsrView, part_ptrs, part_bounds, feat: int, nbr_scale=None, edge_scale=None,
                         row_scale=None, out: torch.Tensor | None = None) -> torch.Tensor:
    """Aggregation whose source matrix is row-partitioned over ``len(part_ptrs)`` blocks (possibly peer-GPU memory).

    ``part_ptrs``: raw device addresses of the blocks, ``part_bounds``: ``P+1`` global row boundaries.
    See ``stg_agg_scaled_sum_parts_f32``.
    """
    global launch_count
    p = len(part_ptrs)
    assert len(part_bounds) == p + 1
    _check(out, "out")
    ptrs = (ctypes.c_void_p * p)(*[ctypes.c_void_p(int(a)) for a in part_ptrs])
    bounds = (ctypes.c_int32 * (p + 1))(*[int(b) for b in part_bounds])
    _lib.call("stg_agg_scaled_sum_parts_f32", ctypes.byref(view), ptrs, bounds, p, int(feat), _lib.ptr(nbr_scale),
              _lib.ptr(edge_scale), _lib.ptr(row_scale), out.data_ptr(), _lib.current_stream_ptr())
    launch_count += 1 + (1 if view.hub_threshold > 0 else 0)
    return out
