"""The 16-bit aggregation (``csrc/agg_h16.cu``: bf16 / fp16 rows, fp32 sums) against the fp64 oracle, and the layers
that reach it under ``torch.autocast``.

Bound of every kernel result: ``|got - ref| <= 1e-5 * sum|terms| + u * |ref| + tiny``, where ``ref`` is the fp64 sum of
the 16-bit inputs (upcast exactly) with the fp32 scales, ``u`` the unit roundoff of the stored type (the single rounding
of the fp32 sum) and ``tiny`` its smallest subnormal (underflow).  Every case also requires, bit for bit: packed ==
plain, queue-less copy of the view == global queue, a repeated call and three CUDA-graph replays == the first call; rows
without edges exactly 0; the NaN row of ``x`` (referenced by no edge) nowhere in ``out``; the row queue rearmed.
"""
from __future__ import annotations

import copy
import dataclasses
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "stgraph_b200", "lib", "libstgraph_b200.so")

DTYPES = {"bf16": torch.bfloat16, "f16": torch.float16}
U = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
TINY = {torch.bfloat16: 2.0 ** -133, torch.float16: 2.0 ** -24}

# Every instantiation <T, VEC, NACC, MODE> of the three kernels (MODE 0 plain, 1 packed).
H16_KERNELS = sorted(f"h16_{k}_kernel<{t},{v},{a},{m}>" for k in ("rows", "queue", "hub")
                     for t in ("__nv_bfloat16", "__half") for v in (1, 2, 4, 8) for a in (1, 2, 4) for m in (0, 1))
_KERNEL_RE = re.compile(r"(h16_(?:rows|queue|hub)_kernel)<([^<>]*)>")
_MANGLED_RE = re.compile(r"\d+(h16_(?:rows|queue|hub)_kernel)I\d+(__nv_bfloat16|__half)((?:Li\d+E)+)E")


def _demangled(text):
    return {f"{m.group(1)}<{m.group(2).replace(' ', '')}>" for m in _KERNEL_RE.finditer(text)}


def _mangled(text):
    return {f"{m.group(1)}<{m.group(2)},{','.join(re.findall(r'Li(\d+)E', m.group(3)))}>" for m in _MANGLED_RE.finditer(text)}


def test_h16_kernel_list_matches_library():
    """``H16_KERNELS`` names exactly the 16-bit aggregation kernels compiled into the library."""
    if not os.path.exists(LIB):
        pytest.skip("libstgraph_b200.so is not built")
    tool = shutil.which("cuobjdump")
    if tool is None and shutil.which("nvcc"):
        cand = os.path.join(os.path.dirname(shutil.which("nvcc")), "cuobjdump")
        tool = cand if os.path.exists(cand) else None
    if tool is None:
        pytest.skip("cuobjdump is not available")
    res = subprocess.run([tool, "-symbols", LIB], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, check=True)
    assert len(H16_KERNELS) == 144
    assert _mangled(res.stdout) == set(H16_KERNELS)


def test_h16_entry_points_reject_bad_arguments_without_gpu():
    """NULL view, negative feat and unknown dtype codes are rejected before anything touches the device."""
    import ctypes

    from stgraph_b200 import _lib

    lib = _lib.load()
    assert lib.stg_agg_scaled_sum_h16(None, None, 4, 1, None, None, None, None, None) == -1
    assert b"NULL" in lib.stg_last_error()
    assert lib.stg_agg_packed_sum_h16(None, None, None, 4, 1, None, None, None) == -1
    v = _lib.StgCsrView()
    v.num_nodes, v.num_edges, v.row_offset = 4, 0, 1     # never dereferenced
    for fn, args in (("stg_agg_scaled_sum_h16", lambda f, d: (ctypes.byref(v), 1, f, d, None, None, None, 2, None)),
                     ("stg_agg_packed_sum_h16", lambda f, d: (ctypes.byref(v), None, 1, f, d, None, 2, None))):
        assert getattr(lib, fn)(*args(-1, 1)) == -1 and b"feat" in lib.stg_last_error()
        for code in (0, 3, -1):
            assert getattr(lib, fn)(*args(4, code)) == -1 and b"dtype" in lib.stg_last_error()


# ------------------------------------------------------------------------------------------------ graphs and cases
def _edges(lengths, seed, iso):
    """(src, dst) with exactly ``lengths[v]`` distinct in-neighbours per row ``v``, none of them ``iso``."""
    rng = np.random.default_rng(seed)
    n = lengths.shape[0]
    pool = np.delete(np.arange(n, dtype=np.int64), iso)
    rows = np.repeat(np.arange(n, dtype=np.int64), 2 * lengths + 8)
    key = np.unique(rows * n + pool[rng.integers(0, n - 1, rows.shape[0])])
    r = key // n
    rank = np.arange(key.shape[0]) - np.searchsorted(r, r)
    key = key[rank < lengths[r]]
    have = np.bincount(key // n, minlength=n)
    for v in np.nonzero(have < lengths)[0]:
        key = np.concatenate([key[key // n != v], v * n + rng.choice(pool, lengths[v], replace=False)])
    src, dst = (key % n).astype(np.int32), (key // n).astype(np.int32)
    assert np.array_equal(np.bincount(dst, minlength=n), lengths)
    return src, dst


def _lengths(n, seed, background, prescribed):
    rng = np.random.default_rng(seed)
    lengths = rng.integers(0, background, n)
    lengths[rng.permutation(np.arange(1, n))[: len(prescribed)]] = prescribed
    lengths[0] = 0                  # row 0: no edges, and no edge reads x[0] (it holds NaN)
    return lengths, 0


def _copy_view(v, **fields):
    from stgraph_b200 import _lib

    c = _lib.StgCsrView()
    for name, _ in _lib.StgCsrView._fields_:
        setattr(c, name, getattr(v, name))
    for name, val in fields.items():
        setattr(c, name, val)
    return c


@dataclasses.dataclass
class _V:
    view: object
    csr: object
    queue: torch.Tensor | None


@dataclasses.dataclass(frozen=True)
class Case:
    graph: str
    view: str
    feat: int
    offset: int       # elements between an aligned address and x
    scales: str
    dtype: str

    @property
    def id(self):
        return f"{self.graph}-{self.view}-{self.dtype}-F{self.feat}" + (f"+{self.offset}" if self.offset else "") + \
            f"-{self.scales}"


SCALES = {"all": (True, True, True), "none": (False, False, False), "ns": (True, False, False),
          "es_rs": (False, True, True)}
# vec 8 / 4 / 2 / 1 x 1 / 2 / 4 accumulators, column chunks (1024 / 512 / 256 / 128 elements) and more than two of them
WIDTHS = [1, 2, 3, 4, 7, 8, 16, 47, 63, 64, 65, 66, 100, 128, 130, 132, 255, 256, 257, 260, 264, 1024, 2056]
QUEUE_WIDTHS = [1, 47, 65, 2, 66, 130, 4, 100, 132, 260, 8, 264, 1024]
MISALIGNED = [(8, 1), (64, 1), (100, 1)]


def _cases():
    table = [("small", "fwd", [(f, 0) for f in WIDTHS] + MISALIGNED),
             ("small", "t64", [(f, 0) for f in WIDTHS] + MISALIGNED),     # hub kernel
             ("small", "bwd", [(7, 0), (100, 0)]),
             ("large", "fwd", [(f, 0) for f in QUEUE_WIDTHS] + [(100, 1)]),   # row queue + hub rows up to 8193 edges
             ("large", "bwd", [(7, 0), (100, 0)]),
             ("pcsr", "fwd", [(63, 0), (100, 0)]),
             ("pcsr", "bwd", [(5, 0), (100, 0)])]
    rot = list(SCALES)
    return [Case(g, v, f, o, rot[i % len(rot)], d) for d in DTYPES for g, v, ws in table for i, (f, o) in enumerate(ws)]


CASES = _cases()
WMAX = max(c.feat + c.offset for c in CASES)


@pytest.fixture(scope="module")
def ctx(cuda):
    from stgraph_b200 import kernels
    from stgraph_b200.graph import PCSRGraph, StaticGraph

    torch.cuda.set_device(cuda)
    sm = kernels.device_info(cuda.index or 0)["sm_count"]
    graphs = {}

    def static(n, lengths, seed):
        src, dst = _edges(lengths, seed, 0)
        g = StaticGraph(torch.from_numpy(np.stack([src, dst], 1)), None, n)
        f, b = g._forward_graph, g._backward_graph
        return g, src, dst, {"fwd": _V(g.fwd_view(), f, f._work_queue), "bwd": _V(g.bwd_view(), b, b._work_queue),
                             "t64": _V(f.view_with_hub_threshold(64), f, f._work_queue)}

    lengths, _ = _lengths(600, 1, 24, [0, 1, 2, 31, 32, 33, 63, 64, 65, 128, 300, 599])
    g, _, _, views = static(600, lengths, 10)
    graphs["small"] = (g, views)
    assert 600 < 2 * sm * 32

    n = 2 * sm * 32 + 37
    lengths, _ = _lengths(n, 2, 64, [0, 1, 2, 31, 32, 33, 1024, 1025, 8192, 8193])
    g, src, dst, views = static(n, lengths, 20)
    assert views["fwd"].view.hub_threshold == 1024 and g._forward_graph.num_edges > 1 << 18
    graphs["large"] = (g, views)

    # a PCSR snapshot of the large graph (eid_base 1, eids not the identity)
    rng = np.random.default_rng(30)
    keep = rng.random(src.shape[0]) > 0.02
    pg = PCSRGraph([np.stack([src, dst], 1), np.stack([src[keep], dst[keep]], 1)], n)
    pg.get_graph(1)
    vb, vf = pg.bwd_view(), pg.fwd_view()
    pf, pb = pg._forward_graph, pg._backward_graph
    assert vf.eid_base == 1 and not pf.eids_identity
    graphs["pcsr"] = (pg, {"fwd": _V(vf, pf, getattr(pf, "_work_queue", None)),
                           "bwd": _V(vb, pb, getattr(pb, "_work_queue", None))})

    data = {}
    for name, (g, views) in graphs.items():
        n = g.get_num_nodes()
        tg = torch.Generator().manual_seed(len(name))
        x = torch.randn(n * WMAX, generator=tg)
        ns = (torch.rand(n, generator=tg) + 0.5).to(cuda)
        rs = (torch.rand(n, generator=tg) + 0.5).to(cuda)
        es = (torch.rand(max(v.csr.num_edges for v in views.values()) + 1, generator=tg) + 0.25).to(cuda)
        data[name] = {"x": {d: x.to(d).to(cuda) for d in DTYPES.values()}, "ns": ns, "rs": rs, "es": es}
    return {"graphs": graphs, "data": data, "device": cuda, "metas": {}}


def _inputs(ctx, c):
    g, views = ctx["graphs"][c.graph]
    d = ctx["data"][c.graph]
    dt = DTYPES[c.dtype]
    v = views[c.view]
    n = g.get_num_nodes()
    # dense [n, feat] rows `offset` elements past a 16-byte boundary; NaN in row 0 (no edge reads it) and around x
    buf = torch.full((n * c.feat + 8,), float("nan"), dtype=dt, device=ctx["device"])
    x = buf[c.offset: c.offset + n * c.feat].view(n, c.feat)
    x.copy_(d["x"][dt][: n * c.feat].view(n, c.feat))
    x[0] = float("nan")
    has_ns, has_es, has_rs = SCALES[c.scales]
    es = d["es"][: v.csr.num_edges] if has_es else None
    return v, x, (d["ns"] if has_ns else None), es, (d["rs"] if has_rs else None)


def _oracle(v, x, ns, es, rs):
    """(fp64 reference, fp64 sum of |terms|) on the device."""
    csr = v.csr
    ro = csr.row_offset.long()
    col = csr.column_indices[: csr.num_edges].long()
    rows = torch.repeat_interleave(torch.arange(csr.num_nodes, device=ro.device), ro[1:] - ro[:-1])
    s = torch.ones(col.shape[0], dtype=torch.float64, device=ro.device)
    if ns is not None:
        s = s * ns.double()[col]
    if es is not None:
        eid = (torch.arange(csr.num_edges, device=ro.device) if csr.eids_identity
               else csr.eids[: csr.num_edges].long() - csr.eid_base)
        s = s * es.double()[eid]
    xd = x.double()
    ref = torch.zeros(csr.num_nodes, x.shape[1], dtype=torch.float64, device=ro.device)
    mag = torch.zeros_like(ref)
    ref.index_add_(0, rows, xd[col] * s[:, None])
    mag.index_add_(0, rows, (xd[col] * s[:, None]).abs())
    if rs is not None:
        ref, mag = ref * rs.double()[:, None], mag * rs.double()[:, None]
    return ref, mag, (ro[1:] - ro[:-1]) == 0


def _check_bound(got, ref, mag, dt, what, extra=0.0):
    err = (got.double() - ref).abs()
    bound = 1e-5 * mag + U[dt] * ref.abs() + TINY[dt] + extra
    bad = ~(err <= bound)
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())} elements out of bound, worst excess "
                                 f"{float((err - bound).max()):.3g}")


def _meta(ctx, c, v, ns, es):
    from stgraph_b200 import kernels

    key = (c.graph, c.view, ns is not None, es is not None)
    if key not in ctx["metas"]:
        ctx["metas"][key] = kernels.pack_edge_meta(v.view, ns, es, device=ctx["device"])
    return ctx["metas"][key]


def _launch(ctx, c):
    from stgraph_b200 import kernels

    v, x, ns, es, rs = _inputs(ctx, c)
    out = kernels.agg_scaled_sum(v.view, x, ns, es, rs)
    packed = kernels.agg_packed_sum(v.view, _meta(ctx, c, v, ns, es), x, rs)
    static = kernels.agg_scaled_sum(_copy_view(v.view, work_queue=None), x, ns, es, rs)
    return v, x, ns, es, rs, out, packed, static


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_h16_case(ctx, case):
    from stgraph_b200 import kernels

    v, x, ns, es, rs, out, packed, static = _launch(ctx, case)
    dt = DTYPES[case.dtype]
    assert out.dtype == dt and packed.dtype == dt and out.shape == x.shape
    ref, mag, empty = _oracle(v, x, ns, es, rs)
    _check_bound(out, ref, mag, dt, case.id)
    assert torch.isfinite(out).all(), "the NaN row of x reached out"
    assert (out[empty] == 0).all() and not torch.signbit(out[empty].float()).any()
    assert torch.equal(packed.view(torch.int16), out.view(torch.int16)), "packed != plain"
    assert torch.equal(static.view(torch.int16), out.view(torch.int16)), "queue-less view != global queue"
    again = kernels.agg_scaled_sum(v.view, x, ns, es, rs)
    assert torch.equal(again.view(torch.int16), out.view(torch.int16)), "a repeated call differs"
    if v.queue is not None:
        assert v.queue.tolist() == [0, 0]

    # three CUDA-graph replays of both entry points
    meta = _meta(ctx, case, v, ns, es)
    o1, o2 = torch.empty_like(out), torch.empty_like(out)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        kernels.agg_scaled_sum(v.view, x, ns, es, rs, out=o1)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        kernels.agg_scaled_sum(v.view, x, ns, es, rs, out=o1)
        kernels.agg_packed_sum(v.view, meta, x, rs, out=o2)
    for _ in range(3):
        o1.fill_(float("nan"))
        o2.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(o1.view(torch.int16), out.view(torch.int16)) and torch.equal(o2.view(torch.int16), out.view(torch.int16))
    if v.queue is not None:
        assert v.queue.tolist() == [0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_h16_empty_shapes(cuda, dtype):
    from stgraph_b200 import kernels
    from stgraph_b200.graph import StaticGraph

    dt = DTYPES[dtype]
    g = StaticGraph(torch.tensor([[0, 1], [1, 2]]), None, 3)
    out = kernels.agg_scaled_sum(g.fwd_view(), torch.empty(3, 0, dtype=dt, device=cuda))
    assert out.shape == (3, 0) and out.dtype == dt
    from stgraph_b200 import _lib

    v = _lib.StgCsrView()
    v.row_offset = torch.zeros(1, dtype=torch.int32, device=cuda).data_ptr()
    out = kernels.agg_scaled_sum(v, torch.empty(0, 5, dtype=dt, device=cuda))
    assert out.shape == (0, 5) and out.dtype == dt


@pytest.mark.gpu
def test_every_h16_instantiation_is_launched(ctx):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for c in CASES:
            _launch(ctx, c)
        torch.cuda.synchronize()
    launched = set()
    for evt in prof.events():
        launched |= _demangled(evt.name)
    missing = sorted(set(H16_KERNELS) - launched)
    print(f"16-bit aggregation instantiations: {len(H16_KERNELS)} compiled, {len(launched & set(H16_KERNELS))} launched")
    assert not missing, f"{len(missing)} instantiations never launched: {missing}"
    assert launched <= set(H16_KERNELS)


@pytest.mark.gpu
def test_shared_row_queue_fp32_h16_and_gat(ctx):
    """fp32, 16-bit and fused-GAT launches interleaved on one view's row queue: each leaves it rearmed, and the fp32
    results equal those of the same fp32 launches run alone."""
    from stgraph_b200 import kernels
    from stgraph_b200.ops_gat import gat_edge_softmax_aggregate

    g, views = ctx["graphs"]["large"]
    v = views["fwd"]
    d = ctx["data"]["large"]
    n = g.get_num_nodes()
    x32 = torch.randn(n, 100, device=ctx["device"], generator=torch.Generator(device=ctx["device"]).manual_seed(3))
    es = d["es"][: v.csr.num_edges]
    meta = kernels.pack_edge_meta(v.view, d["ns"], es, device=ctx["device"])

    def fp32():
        return (kernels.agg_scaled_sum(v.view, x32, d["ns"], es, d["rs"]), kernels.agg_packed_sum(v.view, meta, x32, d["rs"]))

    alone = [fp32(), fp32()]
    torch.cuda.synchronize()
    tg = torch.Generator(device=ctx["device"]).manual_seed(5)
    el = torch.randn(n, 4, 1, device=ctx["device"], generator=tg)
    er = torch.randn(n, 4, 1, device=ctx["device"], generator=tg)
    feat = torch.randn(n, 4, 16, device=ctx["device"], generator=tg)
    mixed = []
    for dt in (torch.bfloat16, torch.float16):
        x16 = x32.to(dt)
        h1 = kernels.agg_scaled_sum(v.view, x16, d["ns"], es, d["rs"])
        torch.cuda.synchronize()
        assert v.queue.tolist() == [0, 0]
        mixed.append(fp32())
        torch.cuda.synchronize()
        assert v.queue.tolist() == [0, 0]
        h2 = kernels.agg_packed_sum(v.view, meta, x16, d["rs"])
        gat_edge_softmax_aggregate(g, el, er, feat, 0.2)
        torch.cuda.synchronize()
        assert v.queue.tolist() == [0, 0]
        assert torch.equal(h1.view(torch.int16), h2.view(torch.int16))
    for a, b in zip(mixed, alone):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), "fp32 results moved with 16-bit launches in between"


@pytest.mark.gpu
def test_h16_argument_errors_before_launch(ctx):
    from stgraph_b200 import kernels

    g, views = ctx["graphs"]["small"]
    v = views["fwd"].view
    n = g.get_num_nodes()
    dev = ctx["device"]
    x = torch.randn(n, 16, device=dev).to(torch.bfloat16)
    meta = kernels.pack_edge_meta(v, None, None, device=dev)
    before = kernels.launch_count
    with pytest.raises(TypeError):
        kernels.agg_scaled_sum(v, x, out=torch.empty(n, 16, device=dev))
    with pytest.raises(TypeError):
        kernels.agg_packed_sum(v, meta, x, out=torch.empty(n, 16, device=dev, dtype=torch.float16))
    for acc in (True, "red"):
        with pytest.raises(ValueError, match="fp32-only"):
            kernels.agg_scaled_sum(v, x, out=torch.empty_like(x), accumulate=acc)
        with pytest.raises(ValueError, match="fp32-only"):
            kernels.agg_packed_sum(v, meta, x, out=torch.empty_like(x), accumulate=acc)
    with pytest.raises(ValueError, match="fp32-only"):
        kernels.agg_scaled_sum(v, x, out=torch.empty_like(x), out_rows=torch.arange(n, dtype=torch.int32, device=dev))
    padded = kernels.padded_rows(n, 16, dev, dtype=torch.bfloat16)[:, :12]
    with pytest.raises(ValueError, match="fp32-only"):
        kernels.agg_packed_sum(v, meta, padded)
    with pytest.raises(ValueError, match="fp32-only"):
        kernels.agg_scaled_sum(v, x[:, :12])
    with pytest.raises(TypeError):
        kernels.agg_scaled_sum(v, x, nbr_scale=torch.ones(n, device=dev, dtype=torch.bfloat16))
    assert kernels.launch_count == before


# ------------------------------------------------------------------------------------------------ layers
def _autocast(dt, enabled=True):
    """bf16 autocast, or the default (fp16) one."""
    if dt == torch.bfloat16:
        return torch.autocast("cuda", dtype=dt, enabled=enabled)
    return torch.autocast("cuda", enabled=enabled)


@pytest.fixture
def exact_reductions():
    """16-bit GEMMs whose split-K partial sums stay fp32, so that the gradient bounds below count every rounding."""
    m = torch.backends.cuda.matmul
    old = (m.allow_bf16_reduced_precision_reduction, m.allow_fp16_reduced_precision_reduction)
    m.allow_bf16_reduced_precision_reduction = m.allow_fp16_reduced_precision_reduction = False
    yield
    m.allow_bf16_reduced_precision_reduction, m.allow_fp16_reduced_precision_reduction = old


def _gcn_ref(csr, h, norm, w=None):
    """fp64 ``norm * sum norm[u] (* w) h[u]`` over ``csr`` and its sum of |terms|."""
    v = _V(None, csr, None)
    nf = norm.reshape(-1)
    return _oracle(v, h, nf, None if w is None else w.reshape(-1), nf)[:2]


def _snapshots(n, T, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, n, (6 * n, 2))
    out = []
    for t in range(T):
        e = np.concatenate([base[rng.random(base.shape[0]) > 0.1], rng.integers(0, n, (n, 2))])
        e = e[e[:, 0] != e[:, 1]]
        out.append(np.unique(e, axis=0).astype(np.int32))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("weighted", [False, True])
def test_gcnconv_static_under_autocast(cuda, exact_reductions, dtype, weighted):
    from stgraph_b200.graph import StaticGraph
    from stgraph_b200.nn.pytorch import GCNConv

    dt = DTYPES[dtype]
    u = U[dt]
    n, fin, fout = 3000, 48, 100
    rng = np.random.default_rng(4)
    e = np.unique(rng.integers(0, n, (40000, 2)), axis=0)
    g = StaticGraph(torch.from_numpy(e), None, n)
    g.set_ndata("norm", g.degree_norm())
    norm = g.get_ndata("norm")
    ew = (torch.rand(g.get_num_edges(), 1, device=cuda) + 0.5) if weighted else None
    torch.manual_seed(0)
    layer = GCNConv(fin, fout).to(cuda)
    layer.bias.data.uniform_(-1, 1)
    nobias = GCNConv(fin, fout, bias=False).to(cuda)
    nobias.weight.data.copy_(layer.weight.data)
    fresh = copy.deepcopy(layer)
    x = torch.randn(n, fin, device=cuda, requires_grad=True)
    gout = torch.randn(n, fout, device=cuda)

    with _autocast(dt):
        agg = nobias(g, x.detach(), edge_weight=ew)
        xw = torch.mm(x.detach(), layer.weight)
        out = layer(g, x, edge_weight=ew)
    assert agg.dtype == dt and xw.dtype == dt and out.dtype == torch.float32
    ref, mag = _gcn_ref(g._forward_graph, xw, norm, ew)
    _check_bound(agg, ref, mag, dt, "aggregation")
    b = layer.bias.detach().double()
    # out = fl32(agg16 + bias): one more fp32 rounding
    _check_bound(out.detach().double() - b, ref, mag, dt, "forward + bias",
                 extra=2.0 ** -24 * (out.detach().double().abs() + b.abs()))
    out.backward(gout)

    ref_layer = copy.deepcopy(fresh)
    x32 = x.detach().clone().requires_grad_(True)
    ref_layer(g, x32, edge_weight=ew).backward(gout)
    # Gradient bound.  The 16-bit backward rounds four times: gout to dt, the aggregated gradient once, inside the 16-bit
    # GEMM the other operand (W or X) to dt, and its product.  The fp32 sums of both paths differ by at most
    # (row length + GEMM depth) * 2^-24 of the summed |terms|.  So |dx16 - dx32| <= ((1 + u)^4 - 1 + (L + K) 2^-24) * M
    # with M the product of the |.| operands, computed here in fp64.
    bwd = g._backward_graph
    L = int((bwd.row_offset[1:] - bwd.row_offset[:-1]).max())
    _, gmag = _gcn_ref(bwd, gout.abs(), norm, ew)
    mx = gmag @ layer.weight.detach().double().abs().t()
    mw = x.detach().double().abs().t() @ gmag
    for got, want, m, k, what in ((x.grad, x32.grad, mx, fout, "x.grad"), (layer.weight.grad, ref_layer.weight.grad, mw, n, "weight.grad")):
        assert torch.isfinite(got).all(), what
        bound = ((1 + u) ** 4 - 1 + (L + k) * 2.0 ** -24) * m + TINY[dt]
        assert bool(((got.double() - want.double()).abs() <= bound).all()), what

    # outside autocast afterwards: bit-identical to a fresh fp32 layer (compile and packed-meta caches unpoisoned)
    again = layer(g, x.detach(), edge_weight=ew)
    assert torch.equal(again, fresh(g, x.detach(), edge_weight=ew))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("weighted", [False, True])
def test_gcnconv_gpma_bptt_under_autocast(cuda, exact_reductions, dtype, weighted):
    """GCNConv over several GPMAGraph snapshots, one backward at the end through the executor's state stack."""
    from stgraph_b200.graph import GPMAGraph
    from stgraph_b200.nn.pytorch import GCNConv

    dt = DTYPES[dtype]
    u = U[dt]
    n, F, T = 500, 32, 4
    G = GPMAGraph(_snapshots(n, T, 7), n)
    torch.manual_seed(0)
    layer = GCNConv(F, F, bias=False).to(cuda)
    ref_layer = copy.deepcopy(layer)
    xs = torch.randn(T, n, F, device=cuda)
    gouts = [torch.randn(n, F, device=cuda) for _ in range(T)]

    def run(model, autocast):
        G.reset_graph()
        x = xs.clone().requires_grad_(True)
        cost, bounds = 0, []
        for t in range(T):
            G.get_graph(t)
            G.set_ndata("norm", G.degree_norm())
            G.bwd_view()                  # builds the snapshot's backward CSR
            norm = G.get_ndata("norm")
            w = (torch.rand(G.get_num_edges(), 1, device=cuda, generator=torch.Generator(device=cuda).manual_seed(t))
                 + 0.5) if weighted else None
            with _autocast(dt, autocast):
                o = model(G, x[t], edge_weight=w)
                xw = torch.mm(xs[t], layer.weight)
            if autocast:
                assert o.dtype == dt
                ref, mag = _gcn_ref(G._forward_graph, xw, norm, w)
                _check_bound(o, ref, mag, dt, f"snapshot {t}")
                bwd = G._backward_graph
                L = int((bwd.row_offset[1:] - bwd.row_offset[:-1]).max())
                _, gmag = _gcn_ref(bwd, gouts[t].abs(), norm, w)
                # as in test_gcnconv_static_under_autocast
                bounds.append(((1 + u) ** 4 - 1 + (L + F) * 2.0 ** -24) * (gmag @ layer.weight.detach().double().abs().t())
                              + TINY[dt])
            cost = cost + (o.float() * gouts[t]).sum()
        cost.backward()
        return x.grad, bounds

    gx16, bounds = run(layer, True)
    gx32, _ = run(ref_layer, False)
    assert torch.isfinite(gx16).all() and torch.isfinite(layer.weight.grad).all()
    for t in range(T):
        assert bool(((gx16[t].double() - gx32[t].double()).abs() <= bounds[t]).all()), f"x.grad at snapshot {t}"


@pytest.mark.gpu
def test_tgcn_bptt_under_bf16_autocast(cuda):
    """TGCN under autocast takes its unfused path (three GCNConv), trains, and stays near the fp32 model."""
    from stgraph_b200.graph import StaticGraph
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN

    n, F, H, T = 800, 8, 16, 4
    rng = np.random.default_rng(8)
    g = StaticGraph(torch.from_numpy(np.unique(rng.integers(0, n, (8000, 2)), axis=0)), None, n)
    g.set_ndata("norm", g.degree_norm())
    torch.manual_seed(0)
    model = TGCN(F, H).to(cuda)
    ref = copy.deepcopy(model)
    xs = torch.randn(T, n, F, device=cuda)
    ys = torch.randn(T, n, H, device=cuda)

    def loss_of(m, autocast):
        h = None
        loss = 0
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            for t in range(T):
                h = m(g, xs[t], H=h)
                loss = loss + ((h.float() - ys[t]) ** 2).mean()
        return loss

    l16 = loss_of(model, True)
    l16.backward()
    l32 = loss_of(ref, False)
    l32.backward()
    u = U[torch.bfloat16]
    # Each step rounds to bf16 about eight times on the way to a gate (GEMM inputs, aggregation, gate GEMM inputs), the
    # gates are 1-Lipschitz (sigmoid / tanh), and the errors of T steps add: 8 * T * u relative to the magnitudes.
    k = 8 * T * u
    assert torch.isfinite(l16) and abs(float(l16.detach()) - float(l32.detach())) <= k * float(l32.detach())
    for (name, p16), p32 in zip(model.named_parameters(), ref.parameters()):
        assert p16.grad is not None and torch.isfinite(p16.grad).all(), name
        scale = p32.grad.abs() + p32.grad.abs().mean()
        assert bool(((p16.grad - p32.grad).abs() <= k * scale).all()), name
    opt = torch.optim.SGD(model.parameters(), lr=0.01)
    opt.step()
    opt.zero_grad()
    l2 = loss_of(model, True)
    assert torch.isfinite(l2) and float(l2) < float(l16)
