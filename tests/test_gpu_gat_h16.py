"""The fused edge-softmax kernels on 16-bit feature rows (``csrc/gat.cu`` with ``FT`` = bf16 / fp16) and the GAT layers
that reach them under ``torch.autocast``.

The 16-bit kernels lay lanes out as the fp32 kernels do and widen each element exactly on load, so they compute the
same fp32 operations in the same order as the fp32 kernels on ``feat.float()``: ``out``, ``row_max``, ``row_sum``,
``d_el`` and ``d_er`` must be equal bit for bit, and ``d_feat`` must equal the fp32 ``d_feat`` rounded to the 16-bit type.
Each case also checks the fp64 closed form (``oracle/aggregate.py``) on the widened rows.
"""
from __future__ import annotations

import copy
import ctypes
import dataclasses
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import aggregate as A
from oracle import structure as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "stgraph_b200", "lib", "libstgraph_b200.so")

DTYPES = {"bf16": torch.bfloat16, "f16": torch.float16}
CODE = {torch.bfloat16: 1, torch.float16: 2}
U = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
SLOPE = 0.2

# (GROUP, NACC) that dispatch_gat picks for hd / VEC = 1, 2, 4, ..., 128
_SHAPES = [(1, 1), (2, 1), (4, 1), (8, 1), (16, 1), (32, 1), (32, 2), (32, 4)]


def _gat_kernels():
    names = []
    for t in ("__nv_bfloat16", "__half"):
        for v in (4, 1):
            for g, a in _SHAPES:
                names.append(f"gat_fwd_kernel<{t},{v},{g},{a}>")
                names += [f"gat_bwd_kernel<{t},{v},{g},{a},{b}>" for b in ("false", "true")]
                names += [f"gat_hub_kernel<{t},{v},{g},{a},{k}>" for k in (0, 1, 2)]
                if g == 32:
                    names += [f"gat_rows_pipe_kernel<{t},{v},{a},{k},{q}>" for k in (0, 1, 2) for q in ("false", "true")]
    return sorted(names)


# Every 16-bit instantiation of the four fused GAT kernels.
GAT_H16_KERNELS = _gat_kernels()
_KERNEL_RE = re.compile(r"(gat_(?:fwd|bwd|hub|rows_pipe)_kernel)<((?:__nv_bfloat16|__half)[^<>]*)>")
_MANGLED_RE = re.compile(r"\d+(gat_(?:fwd|bwd|hub|rows_pipe)_kernel)I\d+(__nv_bfloat16|__half)((?:L[ib]\d+E)+)E")


def _demangled(text):
    return {f"{m.group(1)}<{m.group(2).replace(' ', '')}>" for m in _KERNEL_RE.finditer(text)}


def _mangled(text):
    def arg(kind, val):
        return val if kind == "i" else ("true" if val == "1" else "false")

    return {f"{m.group(1)}<{m.group(2)},{','.join(arg(k, v) for k, v in re.findall(r'L([ib])(\d+)E', m.group(3)))}>"
            for m in _MANGLED_RE.finditer(text)}


def test_gat_h16_kernel_list_matches_library():
    """``GAT_H16_KERNELS`` names exactly the 16-bit fused GAT kernels compiled into the library."""
    if not os.path.exists(LIB):
        pytest.skip("libstgraph_b200.so is not built")
    tool = shutil.which("cuobjdump")
    if tool is None and shutil.which("nvcc"):
        cand = os.path.join(os.path.dirname(shutil.which("nvcc")), "cuobjdump")
        tool = cand if os.path.exists(cand) else None
    if tool is None:
        pytest.skip("cuobjdump is not available")
    res = subprocess.run([tool, "-symbols", LIB], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, check=True)
    assert len(GAT_H16_KERNELS) == 264
    assert _mangled(res.stdout) == set(GAT_H16_KERNELS)


def test_gat_h16_entry_points_reject_bad_arguments_without_gpu():
    """NULL views, non-positive heads / dim and unknown dtype codes are rejected before anything touches the device."""
    from stgraph_b200 import _lib

    lib = _lib.load()
    v = _lib.StgCsrView()
    v.num_nodes, v.num_edges, v.row_offset = 4, 0, 1      # never dereferenced

    def fwd(view, heads, dim, dtype):
        return lib.stg_gat_softmax_fwd_h16(view, 1, 1, 1, heads, dim, dtype, SLOPE, 1, 1, 1, None)

    def bwd(view, heads, dim, dtype):
        return lib.stg_gat_softmax_bwd_h16(view, view, 1, 1, 1, 1, 1, 1, 1, heads, dim, dtype, SLOPE, 1, 1, 1, 1, None)

    for fn in (fwd, bwd):
        assert fn(None, 2, 4, 1) == -1 and b"NULL" in lib.stg_last_error()
        for heads, dim in ((0, 4), (-1, 4), (2, 0), (2, -3)):
            assert fn(ctypes.byref(v), heads, dim, 1) == -1 and b"positive" in lib.stg_last_error()
        for code in (0, 3, -1):
            assert fn(ctypes.byref(v), 2, 4, code) == -1 and b"dtype" in lib.stg_last_error()


# ------------------------------------------------------------------------------------------------ graphs and cases
def _graph_edges(n, seed):
    """Random edges plus, in both directions, one row of each hub tier (129..1024 and > 1024 edges) and empty rows."""
    rng = np.random.default_rng(seed)
    src = rng.integers(0, n, 6 * n)
    dst = rng.integers(0, n, 6 * n)
    for v, deg in ((1, 1500), (2, 300), (3, 129)):
        other = rng.choice(np.arange(20, n), deg, replace=False)
        src = np.concatenate([src, other, np.full(deg, v + 3)])     # v: hub destination, v + 3: hub source
        dst = np.concatenate([dst, np.full(deg, v), other])
    keep = ~np.isin(dst, [10, 11]) & ~np.isin(src, [12, 13])       # rows without in-edges / without out-edges
    k = np.unique(src[keep] * n + dst[keep])
    return (k // n).astype(np.int32), (k % n).astype(np.int32)


@dataclasses.dataclass(frozen=True)
class Case:
    graph: str        # small (< 4096 rows: one row per lane group) or large (row kernels of the queue / static form)
    view: str         # queue: the views as the op uses them; static: copies without the row queue
    heads: int
    dim: int
    offset: int       # elements between an 8-byte aligned address and feat / d_feat (1: VEC = 1 whatever dim is)
    dtype: str

    @property
    def id(self):
        return f"{self.graph}-{self.view}-{self.dtype}-H{self.heads}xD{self.dim}" + (f"+{self.offset}" if self.offset else "")


# hd / VEC = 1, 2, ..., 128 with VEC = 4, and with VEC = 1 (dim 1 or 2, or feat misaligned)
VEC4 = [(1, 4), (2, 4), (1, 16), (2, 16), (8, 8), (8, 16), (4, 64), (4, 128)]
VEC1 = [(1, 1), (1, 2), (2, 2), (8, 1), (8, 2), (16, 2), (64, 1), (64, 2)]
MISALIGNED = [(4, 8, 1), (2, 4, 1)]


def _cases():
    shapes = [(h, d, 0) for h, d in VEC4 + VEC1] + MISALIGNED
    out = []
    for dt in DTYPES:
        for h, d, o in shapes:
            out.append(Case("small", "queue", h, d, o, dt))
            if h * d // (4 if d % 4 == 0 and not o else 1) >= 32:      # GROUP = 32: the row kernels of large graphs
                out += [Case("large", "queue", h, d, o, dt), Case("large", "static", h, d, o, dt)]
            else:
                out.append(Case("large", "queue", h, d, o, dt))
    return out


CASES = _cases()


def _copy_view(v, **fields):
    from stgraph_b200 import _lib

    c = _lib.StgCsrView()
    for name, _ in _lib.StgCsrView._fields_:
        setattr(c, name, getattr(v, name))
    for name, val in fields.items():
        setattr(c, name, val)
    return c


@pytest.fixture(scope="module")
def ctx(cuda):
    from stgraph_b200 import ops_gat
    from stgraph_b200.graph import StaticGraph

    torch.cuda.set_device(cuda)
    graphs = {}
    for name, n, seed in (("small", 3000, 1), ("large", 6000, 2)):
        src, dst = _graph_edges(n, seed)
        g = StaticGraph(torch.from_numpy(np.stack([src, dst], 1)), None, n)
        vf, vb = ops_gat._views(g)
        assert vf.hub_threshold == ops_gat.GAT_HUB_THRESHOLD and vb.hub_threshold == ops_gat.GAT_HUB_THRESHOLD
        views = {"queue": (vf, vb), "static": (_copy_view(vf, work_queue=None), _copy_view(vb, work_queue=None))}
        queues = (g._forward_graph._work_queue, g._backward_graph._work_queue)
        graphs[name] = {"g": g, "n": n, "views": views, "queues": queues, "csr": S.forward_csr(src, dst, n)}
    return {"graphs": graphs, "device": cuda}


def _aligned(n, h, d, dtype, offset, device, fill=float("nan")):
    """``[n, h, d]`` rows ``offset`` elements past a 16-byte boundary, NaN around them."""
    buf = torch.full((n * h * d + 16,), fill, dtype=dtype, device=device)
    return buf[offset: offset + n * h * d].view(n, h, d)


def _inputs(ctx, c):
    gr = ctx["graphs"][c.graph]
    n, dev, dt = gr["n"], ctx["device"], DTYPES[c.dtype]
    tg = torch.Generator().manual_seed(c.heads * 1000 + c.dim * 10 + c.offset)
    el = (torch.randn(n, c.heads, generator=tg) * 2).to(dev)
    er = (torch.randn(n, c.heads, generator=tg) * 2).to(dev)
    feat = _aligned(n, c.heads, c.dim, dt, c.offset, dev)
    feat.copy_(torch.randn(n, c.heads, c.dim, generator=tg).to(dt))
    gout = torch.randn(n, c.heads, c.dim, generator=tg).to(dev)
    return el, er, feat, gout


def _call(views, el, er, feat, gout, d_feat=None):
    """The fp32 or the 16-bit entry points (by feat's dtype) on the given views: (out, max, sum, d_feat, d_el, d_er)."""
    from stgraph_b200 import _lib

    n, h, d = feat.shape
    vf, vb = views
    out = torch.empty(n, h, d, device=feat.device)
    rmax, rsum = torch.empty(n, h, device=feat.device), torch.empty(n, h, device=feat.device)
    if d_feat is None:
        d_feat = torch.empty_like(feat)
    d_el, d_er, dot = torch.empty_like(el), torch.empty_like(er), torch.empty_like(el)
    st = _lib.current_stream_ptr()
    if feat.dtype == torch.float32:
        _lib.call("stg_gat_softmax_fwd_f32", ctypes.byref(vf), el.data_ptr(), er.data_ptr(), feat.data_ptr(), h, d, SLOPE,
                  out.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), st)
        _lib.call("stg_gat_softmax_bwd_f32", ctypes.byref(vf), ctypes.byref(vb), el.data_ptr(), er.data_ptr(),
                  feat.data_ptr(), out.data_ptr(), gout.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), h, d, SLOPE,
                  d_feat.data_ptr(), d_el.data_ptr(), d_er.data_ptr(), dot.data_ptr(), st)
    else:
        code = CODE[feat.dtype]
        _lib.call("stg_gat_softmax_fwd_h16", ctypes.byref(vf), el.data_ptr(), er.data_ptr(), feat.data_ptr(), h, d, code,
                  SLOPE, out.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), st)
        _lib.call("stg_gat_softmax_bwd_h16", ctypes.byref(vf), ctypes.byref(vb), el.data_ptr(), er.data_ptr(),
                  feat.data_ptr(), out.data_ptr(), gout.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), h, d, code, SLOPE,
                  d_feat.data_ptr(), d_el.data_ptr(), d_er.data_ptr(), dot.data_ptr(), st)
    return out, rmax, rsum, d_feat, d_el, d_er


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _assert_same(a, b, what):
    names = ("out", "row_max", "row_sum", "d_feat", "d_el", "d_er")
    for x, y, nm in zip(a, b, names):
        assert x.dtype == y.dtype and torch.equal(_bits(x), _bits(y)), f"{what}: {nm} differs"


def _run_case(ctx, c):
    gr = ctx["graphs"][c.graph]
    el, er, feat, gout = _inputs(ctx, c)
    # d_feat at the same misalignment as feat: the 16-bit lanes then match those of the fp32 call on misaligned rows
    d_feat = _aligned(*feat.shape, feat.dtype, c.offset, feat.device)
    got = _call(gr["views"][c.view], el, er, feat, gout, d_feat)
    return gr, el, er, feat, gout, got


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_gat_h16_case(ctx, case):
    gr, el, er, feat, gout, got = _run_case(ctx, case)
    dt = DTYPES[case.dtype]
    n, h, d = feat.shape
    # fp32 entry points on the widened rows, at the same misalignment (4-byte elements: offset 1 keeps VEC = 1)
    f32 = _aligned(n, h, d, torch.float32, case.offset, feat.device)
    f32.copy_(feat.float())
    d32 = _aligned(n, h, d, torch.float32, case.offset, feat.device)
    ref32 = _call(gr["views"][case.view], el, er, f32, gout, d32)
    torch.cuda.synchronize()
    for q in gr["queues"]:
        assert q.tolist() == [0, 0]
    rounded = list(ref32)
    rounded[3] = ref32[3].to(dt)
    _assert_same(got, rounded, case.id)
    assert got[3].dtype == dt and torch.isfinite(got[3]).all() and torch.isfinite(got[0]).all()

    again = _call(gr["views"][case.view], el, er, feat, gout)
    _assert_same(again, got, f"{case.id}: repeated call")

    if case.view == "static":
        return          # bit-identical to the queue form (test_gat_h16_static_equals_queue), checked against fp64 there
    # fp64 closed form on the widened rows, with the bounds of test_gpu_layers.py's fused-op tests (+ u |ref| for d_feat)
    f = gr["csr"]
    fc, elc, erc, gc = feat.float().cpu(), el.cpu(), er.cpu(), gout.cpu()
    ref, _, _ = A.gat_softmax_forward(f, elc, erc, fc)
    d_feat, d_el, d_er = A.gat_softmax_backward(f, elc, erc, fc, gc)
    sc = lambda t: t.abs().mean() * torch.ones_like(t) + 1e-12
    A.assert_close_rel(got[0].cpu(), ref, rel=1e-5, abs_terms=sc(ref), what="out")
    A.assert_close_rel(got[4].cpu(), d_el, rel=1e-4, abs_terms=sc(d_el), what="d_el")
    A.assert_close_rel(got[5].cpu(), d_er, rel=1e-4, abs_terms=sc(d_el), what="d_er")
    ref_d = d_feat.double()
    err = (got[3].cpu().double() - ref_d).abs()
    bound = 2e-5 * torch.maximum(ref_d.abs(), sc(ref_d)) + U[dt] * ref_d.abs()
    assert bool((err <= bound).all()), f"d_feat: {int((err > bound).sum())} elements out of bound"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_gat_h16_static_equals_queue(ctx, dtype):
    for c in CASES:
        if c.view == "static" and c.dtype == dtype:
            a = _run_case(ctx, c)[-1]
            b = _run_case(ctx, dataclasses.replace(c, view="queue"))[-1]
            _assert_same(a, b, c.id)


@pytest.mark.gpu
def test_every_gat_h16_instantiation_is_launched(ctx):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for c in CASES:
            _run_case(ctx, c)
        torch.cuda.synchronize()
    launched = set()
    for evt in prof.events():
        launched |= _demangled(evt.name)
    missing = sorted(set(GAT_H16_KERNELS) - launched)
    print(f"16-bit GAT instantiations: {len(GAT_H16_KERNELS)} compiled, {len(launched & set(GAT_H16_KERNELS))} launched, "
          f"{len(missing)} missing")
    assert not missing, f"{len(missing)} instantiations never launched: {missing}"
    assert launched <= set(GAT_H16_KERNELS)


# ------------------------------------------------------------------------------------------------ the autograd op
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("offset", [0, 1])
def test_gat_op_h16_equals_fp32_op_on_widened_rows(ctx, dtype, offset):
    """The op keeps 16-bit feat and its gradient in their dtype and equals the fp32 op on ``feat.float()``: ``out``,
    ``d_el`` and ``d_er`` bit for bit, ``d_feat`` rounded once.  A misaligned feat is copied first."""
    from stgraph_b200 import kernels
    from stgraph_b200.ops_gat import gat_edge_softmax_aggregate

    dt = DTYPES[dtype]
    gr = ctx["graphs"]["large"]
    el, er, feat, gout = _inputs(ctx, Case("large", "queue", 8, 16, offset, dtype))
    res = []
    for x in (feat, feat.float()):
        a, b, f = el.clone().requires_grad_(True), er.clone().requires_grad_(True), x.detach().requires_grad_(True)
        before = kernels.launch_count
        out = gat_edge_softmax_aggregate(gr["g"], a.unsqueeze(-1), b.unsqueeze(-1), f, SLOPE)
        out.backward(gout)
        assert kernels.launch_count == before + 3
        res.append((out.detach(), f.grad, a.grad, b.grad))
    (o16, g16, a16, b16), (o32, g32, a32, b32) = res
    assert o16.dtype == torch.float32 and g16.dtype == dt
    assert torch.equal(o16, o32) and torch.equal(a16, a32) and torch.equal(b16, b32)
    assert torch.equal(g16.view(torch.int16), g32.to(dt).view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_gat_h16_cuda_graph_replay(ctx, dtype):
    gr = ctx["graphs"]["large"]
    c = Case("large", "queue", 8, 16, 0, dtype)
    el, er, feat, gout = _inputs(ctx, c)
    views = gr["views"]["queue"]
    eager = _call(views, el, er, feat, gout)
    bufs = {}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _call(views, el, er, feat, gout)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        bufs["r"] = _call(views, el, er, feat, gout)
    for _ in range(3):
        for t in bufs["r"]:
            t.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        _assert_same(bufs["r"], eager, "graph replay")
        for q in gr["queues"]:
            assert q.tolist() == [0, 0]


@pytest.mark.gpu
def test_shared_row_queue_fp32_and_h16_gat_and_aggregation(ctx):
    """fp32 / 16-bit aggregation and fp32 / 16-bit GAT launches interleaved on one view: each leaves the row queue at
    [0, 0], and the fp32 results equal those of the same launches run alone."""
    from stgraph_b200 import kernels

    gr = ctx["graphs"]["large"]
    views = gr["views"]["queue"]
    vf = gr["g"].fwd_view()
    dev = ctx["device"]
    x32 = torch.randn(gr["n"], 64, device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    el, er, feat, gout = _inputs(ctx, Case("large", "queue", 8, 16, 0, "bf16"))
    f32 = feat.float().contiguous()
    alone = (kernels.agg_scaled_sum(vf, x32), _call(views, el, er, f32, gout))
    torch.cuda.synchronize()

    def rearmed():
        torch.cuda.synchronize()
        for q in gr["queues"]:
            assert q.tolist() == [0, 0]

    for dt in DTYPES.values():
        h = feat.to(dt)
        a32 = kernels.agg_scaled_sum(vf, x32)
        rearmed()
        kernels.agg_scaled_sum(vf, x32.to(dt))
        rearmed()
        g32 = _call(views, el, er, f32, gout)
        rearmed()
        _call(views, el, er, h, gout)
        rearmed()
        assert torch.equal(a32, alone[0])
        _assert_same(g32, alone[1], "fp32 GAT with 16-bit launches in between")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_gat_h16_unsupported_dim_errors_like_fp32(ctx, dtype):
    from stgraph_b200 import kernels
    from stgraph_b200.ops_gat import gat_edge_softmax_aggregate

    g = ctx["graphs"]["small"]["g"]
    n, dev = ctx["graphs"]["small"]["n"], ctx["device"]
    el = torch.randn(n, 2, 1, device=dev)
    msgs = []
    for feat in (torch.randn(n, 2, 6, device=dev), torch.randn(n, 2, 6, device=dev).to(DTYPES[dtype])):
        before = kernels.launch_count
        with pytest.raises(RuntimeError, match="power of two") as info:
            gat_edge_softmax_aggregate(g, el, el, feat)
        assert kernels.launch_count == before
        msgs.append(str(info.value).replace("_h16", "_f32"))
    assert msgs[0] == msgs[1]


# ------------------------------------------------------------------------------------------------ layers
def _autocast(dt, enabled=True):
    if dt == torch.bfloat16:
        return torch.autocast("cuda", dtype=dt, enabled=enabled)
    return torch.autocast("cuda", enabled=enabled)


def _upcast_forward(layer, graph, x):
    """GATConv.forward with the projection widened before the attention: the layer's path before 16-bit rows."""
    from stgraph_b200.ops_gat import gat_edge_softmax_aggregate

    proj, left, right = layer._scores(x)
    if layer.softmax == "fused":
        return gat_edge_softmax_aggregate(graph, left, right, proj.float(), layer.negative_slope)
    return layer._stock_program()(g=graph, n_feats={"el": left, "er": right, "feat_src": proj.float()})


def _snapshots(n, T, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, n, (6 * n, 2))
    out = []
    for _ in range(T):
        e = np.concatenate([base[rng.random(base.shape[0]) > 0.1], rng.integers(0, n, (n, 2))])
        e = e[e[:, 0] != e[:, 1]]
        out.append(np.unique(e, axis=0).astype(np.int32))
    return out


def _grads(layer, x):
    return [p.grad.clone() for p in layer.parameters()] + [x.grad.clone()]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("softmax", ["fused", "stock"])
def test_gatconv_static_under_autocast(cuda, dtype, softmax):
    from stgraph_b200.graph import StaticGraph
    from stgraph_b200.nn.pytorch import GATConv

    dt = DTYPES[dtype]
    n, fin, H, D = 2000, 24, 4, 16
    rng = np.random.default_rng(6)
    g = StaticGraph(torch.from_numpy(np.unique(rng.integers(0, n, (20000, 2)), axis=0)), None, n)
    torch.manual_seed(0)
    layer = GATConv(fin, D, H, softmax=softmax).to(cuda)
    ref = copy.deepcopy(layer)
    fresh = copy.deepcopy(layer)
    x0 = torch.randn(n, fin, device=cuda)
    gout = torch.randn(n, H, D, device=cuda)
    outs = []
    for model, fwd in ((layer, lambda m, x: m(g, x)), (ref, lambda m, x: _upcast_forward(m, g, x))):
        x = x0.clone().requires_grad_(True)
        with _autocast(dt):
            out = fwd(model, x)
        assert out.dtype == torch.float32
        out.backward(gout)
        outs.append((out.detach(), _grads(model, x)))
    assert torch.equal(outs[0][0], outs[1][0])
    for a, b in zip(outs[0][1], outs[1][1]):
        assert torch.equal(a, b)
    # outside autocast afterwards: bit-identical to a fresh fp32 layer (no cache holds a 16-bit program or tensor)
    assert torch.equal(layer(g, x0), fresh(g, x0))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("softmax", ["fused", "stock"])
def test_gatconv_gpma_bptt_under_autocast(cuda, dtype, softmax):
    """GATConv over several GPMAGraph snapshots, one backward at the end (each step's backward at its timestamp)."""
    from stgraph_b200.graph import GPMAGraph
    from stgraph_b200.nn.pytorch import GATConv

    dt = DTYPES[dtype]
    n, F, H, D, T = 500, 16, 2, 8, 4
    G = GPMAGraph(_snapshots(n, T, 9), n)
    torch.manual_seed(0)
    layer = GATConv(F, D, H, softmax=softmax).to(cuda)
    ref = copy.deepcopy(layer)
    fresh = copy.deepcopy(layer)
    xs = torch.randn(T, n, F, device=cuda)
    gouts = [torch.randn(n, H, D, device=cuda) for _ in range(T)]

    def run(model, fwd, autocast=True):
        G.reset_graph()
        x = xs.clone().requires_grad_(True)
        cost, outs = 0, []
        for t in range(T):
            G.get_graph(t)
            G.bwd_view()
            with _autocast(dt, autocast):
                o = fwd(model, G, x[t])
            assert o.dtype == torch.float32
            outs.append(o.detach())
            cost = cost + (o * gouts[t]).sum()
        cost.backward()
        return outs, _grads(model, x)

    native = run(layer, lambda m, g, x: m(g, x))
    upcast = run(ref, _upcast_forward)
    for a, b in zip(native[0] + native[1], upcast[0] + upcast[1]):
        assert torch.equal(a, b)
    plain = run(layer, lambda m, g, x: m(g, x), autocast=False)
    fresh_run = run(fresh, lambda m, g, x: m(g, x), autocast=False)
    for a, b in zip(plain[0], fresh_run[0]):
        assert torch.equal(a, b)
