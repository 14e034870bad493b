"""The one-op TGCN cell under ``torch.autocast`` (``ops_tgcn._TgcnCell`` 16-bit form, ``csrc/gates.cu`` ``cell_*16_kernel``).

Kernel anchors are bit-exact: on 16-bit inputs every fp32 output of a new kernel equals the fp32 kernel's output on the
widened inputs, and every 16-bit output is the rounding of that fp32 output.  The cell is checked against an fp64
restatement of ``temporal/tgcn.py`` over a BPTT window with bounds counted from the roundings on each path, and against
the reference-structured path that autocast ran before.
"""
from __future__ import annotations

import copy
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
CODE = {torch.bfloat16: 1, torch.float16: 2}
U = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
E32 = 2.0 ** -24
CLAMP = 1e6

KINDS = ("bias_clamp", "clamp_bwd", "reset_fwd", "reset_bwd", "update_bwd")
# Every instantiation <FT, V> of the five 16-bit gate kernels (V = 4: vector lanes, V = 1: scalar).
GATE16_KERNELS = sorted(f"cell_{k}16_kernel<{t},{v}>" for k in KINDS for t in ("__nv_bfloat16", "__half") for v in (1, 4))
_KERNEL_RE = re.compile(r"(cell_(?:bias_clamp|clamp_bwd|reset_fwd|reset_bwd|update_bwd)16_kernel)<([^<>]*)>")
_MANGLED_RE = re.compile(r"\d+(cell_(?:bias_clamp|clamp_bwd|reset_fwd|reset_bwd|update_bwd)16_kernel)I\d+(__nv_bfloat16|__half)Li(\d+)E")


def _demangled(text):
    return {f"{m.group(1)}<{m.group(2).replace(' ', '')}>" for m in _KERNEL_RE.finditer(text)}


# ------------------------------------------------------------------------------------------------ CPU checks
def test_tgcn_h16_kernel_list_matches_library():
    """``GATE16_KERNELS`` names exactly the 16-bit gate kernels compiled into the library."""
    if not os.path.exists(LIB):
        pytest.skip("libstgraph_b200.so is not built")
    tool = shutil.which("cuobjdump")
    if tool is None and shutil.which("nvcc"):
        cand = os.path.join(os.path.dirname(shutil.which("nvcc")), "cuobjdump")
        tool = cand if os.path.exists(cand) else None
    if tool is None:
        pytest.skip("cuobjdump is not available")
    res = subprocess.run([tool, "-symbols", LIB], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, check=True)
    found = {f"{m.group(1)}<{m.group(2)},{m.group(3)}>" for m in _MANGLED_RE.finditer(res.stdout)}
    assert len(GATE16_KERNELS) == 20
    assert found == set(GATE16_KERNELS)


def test_tgcn_h16_entry_points_reject_bad_arguments_without_gpu():
    """Shapes, clamp bounds, dtype codes and NULL tensors are rejected before any launch, with the fp32 twins' messages."""
    from stgraph_b200 import _lib

    lib = _lib.load()

    def err(rc):
        assert rc == -1
        return lib.stg_last_error()

    # bad shape: the same message as the fp32 entry point
    assert err(lib.stg_tgcn_reset_fwd_h16(None, None, None, 4, 0, 1, None)) == err(lib.stg_tgcn_reset_fwd_f32(None, None, None, 4, 0, None))
    assert err(lib.stg_tgcn_reset_bwd_h16(None, None, None, None, None, None, -1, 8, 1, None)) == \
        err(lib.stg_tgcn_reset_bwd_f32(None, None, None, None, None, -1, 8, None))
    assert err(lib.stg_tgcn_update_bwd_h16(None, None, None, None, None, None, 4, -3, 2, None)) == \
        err(lib.stg_tgcn_update_bwd_f32(None, None, None, None, None, 4, -3, None))
    assert err(lib.stg_tgcn_bias_clamp_h16(None, None, None, 4, 0, 1, -1.0, 1.0, None)) == \
        err(lib.stg_bias_clamp_f32(None, None, 4, 0, -1.0, 1.0, None))
    assert b"bad shape" in err(lib.stg_tgcn_clamp_bwd_h16(None, None, None, None, -2, 3, 1, -1.0, 1.0, None))
    # clamp bounds
    assert err(lib.stg_tgcn_bias_clamp_h16(None, None, None, 4, 3, 1, 1.0, -1.0, None)) == \
        err(lib.stg_bias_clamp_f32(None, None, 4, 3, 1.0, -1.0, None))
    assert b"clamp bounds" in err(lib.stg_tgcn_clamp_bwd_h16(None, None, None, None, 4, 3, 2, 1.0, -1.0, None))
    # unknown dtype codes, also for empty tensors
    for code in (0, 3, -1):
        for rows in (0, 4):
            for rc in (lib.stg_tgcn_bias_clamp_h16(1, None, 1, rows, 3, code, -1.0, 1.0, None),
                       lib.stg_tgcn_clamp_bwd_h16(1, None, 1, 1, rows, 3, code, -1.0, 1.0, None),
                       lib.stg_tgcn_reset_fwd_h16(1, 1, 1, rows, 4, code, None),
                       lib.stg_tgcn_reset_bwd_h16(1, 1, 1, 1, 1, 1, rows, 4, code, None),
                       lib.stg_tgcn_update_bwd_h16(1, 1, 1, 1, 1, 1, rows, 4, code, None)):
                assert b"unknown dtype code" in err(rc)
    # NULL tensors
    assert err(lib.stg_tgcn_bias_clamp_h16(None, None, 1, 4, 3, 1, -1.0, 1.0, None)) == \
        err(lib.stg_bias_clamp_f32(None, None, 4, 3, -1.0, 1.0, None))
    assert b"NULL" in err(lib.stg_tgcn_bias_clamp_h16(1, None, None, 4, 3, 1, -1.0, 1.0, None))
    assert err(lib.stg_tgcn_clamp_bwd_h16(1, None, None, 1, 4, 3, 2, -1.0, 1.0, None)) == \
        err(lib.stg_clamp_bwd_f32(1, None, 1, 12, -1.0, 1.0, None))
    assert err(lib.stg_tgcn_reset_fwd_h16(1, None, 1, 4, 4, 2, None)) == err(lib.stg_tgcn_reset_fwd_f32(1, None, 1, 4, 4, None))
    assert err(lib.stg_tgcn_reset_bwd_h16(1, 1, 1, 1, None, 1, 4, 4, 1, None)) == \
        err(lib.stg_tgcn_reset_bwd_f32(1, 1, 1, 1, None, 4, 4, None))
    assert err(lib.stg_tgcn_update_bwd_h16(1, 1, 1, None, 1, 1, 4, 4, 1, None)) == \
        err(lib.stg_tgcn_update_bwd_f32(1, 1, 1, None, 1, 4, 4, None))
    # nothing to do: OK without touching a pointer
    assert lib.stg_tgcn_reset_fwd_h16(None, None, None, 0, 4, 1, None) == 0
    assert lib.stg_tgcn_bias_clamp_h16(None, None, None, 0, 3, 2, -1.0, 1.0, None) == 0


# ------------------------------------------------------------------------------------------------ kernel anchors
def _call(name, *args):
    from stgraph_b200 import _lib

    _lib.call(name, *[a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args], _lib.current_stream_ptr())


def _buf(shape, dtype, dev, offset, fill=None, gen=None, scale=1.0):
    """A tensor of ``shape`` that starts ``offset`` elements into its storage (offset 1: no vector alignment)."""
    n = int(np.prod(shape))
    base = torch.empty(n + offset, device=dev, dtype=torch.float32)
    if fill is None:
        base.normal_(generator=gen).mul_(scale)
    else:
        base.fill_(fill)
    base = base.to(dtype)
    return base[offset:].view(shape)


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _same(a, b):
    return a.dtype == b.dtype and torch.equal(_bits(a.contiguous()), _bits(b.contiguous()))


LAYOUTS = {"vec": (517, 64, 0), "odd_hid": (301, 13, 0), "misaligned": (263, 64, 1)}


def _run_anchor(dt, rows, hid, off, dev, seed):
    """Runs every 16-bit gate entry point once next to its fp32 twin and checks the anchors."""
    g = torch.Generator(device=dev).manual_seed(seed)
    c = CODE[dt]
    f32 = torch.float32
    cols = 3 * hid
    # bias + clamp, and its backward (in place and out of place)
    A = _buf((rows, cols), dt, dev, off, gen=g, scale=3.0)
    b3 = _buf((cols,), f32, dev, off, gen=g)
    h = _buf((rows, cols), dt, dev, off, fill=7.0)
    _call("stg_tgcn_bias_clamp_h16", A, b3, h, rows, cols, c, -CLAMP, CLAMP)
    y32 = A.float().contiguous()
    _call("stg_bias_clamp_f32", y32, b3, rows, cols, -CLAMP, CLAMP)
    assert _same(h, y32.to(dt)), "bias_clamp: not the rounding of the fp32 kernel's output"
    assert _same(h, torch.clamp(A.float() + b3, -CLAMP, CLAMP).to(dt))
    d_y = _buf((rows, cols), dt, dev, off, gen=g)
    d_a = _buf((rows, cols), dt, dev, off, fill=5.0)
    _call("stg_tgcn_clamp_bwd_h16", A, b3, d_y, d_a, rows, cols, c, -CLAMP, CLAMP)
    d32 = torch.empty(rows, cols, device=dev)
    _call("stg_clamp_bwd_f32", y32, d_y.float().contiguous(), d32, rows * cols, -CLAMP, CLAMP)
    assert _same(d_a, d32.to(dt)), "clamp_bwd: not the fp32 kernel's output"
    inplace = d_y.clone()
    _call("stg_tgcn_clamp_bwd_h16", A, b3, inplace, inplace, rows, cols, c, -CLAMP, CLAMP)
    assert _same(inplace, d_a)
    # reset forward
    P = _buf((rows, cols), f32, dev, off, gen=g, scale=2.0)
    H = _buf((rows, hid), f32, dev, off, gen=g)
    HR = _buf((rows, hid), dt, dev, off, fill=3.0)
    HR32 = torch.empty(rows, hid, device=dev)
    _call("stg_tgcn_reset_fwd_h16", P, H, HR, rows, hid, c)
    _call("stg_tgcn_reset_fwd_f32", P, H, HR32, rows, hid)
    assert _same(HR, HR32.to(dt)), "reset_fwd"
    # update backward, then reset backward (fp32 outputs bit-identical, the 16-bit twin is their rounding)
    d_out = _buf((rows, hid), f32, dev, off, gen=g)
    d_hr = _buf((rows, hid), f32, dev, off, gen=g)
    dP = _buf((rows, cols), f32, dev, off, fill=9.0)
    dP16 = _buf((rows, cols), dt, dev, off, fill=9.0)
    dH = _buf((rows, hid), f32, dev, off, fill=9.0)
    dP32, dH32 = torch.full((rows, cols), 9.0, device=dev), torch.empty(rows, hid, device=dev)
    _call("stg_tgcn_update_bwd_h16", P, H, d_out, dP, dP16, dH, rows, hid, c)
    _call("stg_tgcn_update_bwd_f32", P, H, d_out, dP32, dH32, rows, hid)
    assert _same(dP, dP32) and _same(dH, dH32), "update_bwd fp32 outputs"
    zh = torch.cat((torch.arange(hid), torch.arange(2 * hid, 3 * hid))).to(dev)
    assert _same(dP16[:, zh], dP32[:, zh].to(dt)), "update_bwd: d_p16 z / h blocks"
    assert bool((dP16[:, hid:2 * hid].float() == 9.0).all()), "update_bwd wrote the r block"
    _call("stg_tgcn_reset_bwd_h16", P, H, d_hr, dP, dP16, dH, rows, hid, c)
    _call("stg_tgcn_reset_bwd_f32", P, H, d_hr, dP32, dH32, rows, hid)
    assert _same(dP, dP32) and _same(dH, dH32), "reset_bwd fp32 outputs"
    assert _same(dP16, dP32.to(dt)), "reset_bwd: d_p16"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_gate16_kernels_equal_fp32_kernels_bit_for_bit(cuda, dtype, layout):
    rows, hid, off = LAYOUTS[layout]
    _run_anchor(DTYPES[dtype], rows, hid, off, cuda, seed=hash(layout) % 1000)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("hid", [4, 5])
def test_clamp_mask_at_the_bounds_and_fp16_overflow(cuda, dtype, hid):
    """The mask is the fp32 cell's ``lo < A + b3 < hi`` on the unrounded sum; the clamped value rounds to dt (fp16: inf)."""
    dt = DTYPES[dtype]
    c = CODE[dt]
    cols = 3 * hid
    a_vals = torch.tensor([0.5, 1.0, 1.5, -0.5, -1.0, -1.5, 0.0], device=cuda)
    rows = a_vals.numel()
    A = a_vals[:, None].expand(rows, cols).contiguous().to(dt)
    b3 = torch.zeros(cols, device=cuda)
    b3[0], b3[1] = CLAMP - 1, -(CLAMP - 1)         # rows 0-2 of column 0: v = 999999.5 (inside), 1e6 (on the bound),
    #                                                1000000.5 (outside); rows 3-5 of column 1 the same at -1e6
    if dt == torch.bfloat16:
        A[:, 2] = 999424.0                              # round_bf16(1e6) = 999424 < 1e6: the rounded h cannot give the mask
        b3[2] = 575.5                                   # v = 999999.5: inside
        b3[3] = 577.0                                   # v = 1000001 (A = 999424): clamped
        A[:, 3] = 999424.0
    h = torch.empty_like(A)
    _call("stg_tgcn_bias_clamp_h16", A, b3, h, rows, cols, c, -CLAMP, CLAMP)
    v = A.float() + b3
    assert _same(h, torch.clamp(v, -CLAMP, CLAMP).to(dt))
    d_y = torch.randn(rows, cols, device=cuda).to(dt)
    d_a = torch.empty_like(d_y)
    _call("stg_tgcn_clamp_bwd_h16", A, b3, d_y, d_a, rows, cols, c, -CLAMP, CLAMP)
    mask = (v > -CLAMP) & (v < CLAMP)
    assert _same(d_a, torch.where(mask, d_y, torch.zeros_like(d_y)))
    assert mask[0, 0] and not mask[1, 0] and not mask[2, 0]          # just inside, on, just outside +1e6
    assert mask[3, 1] and not mask[4, 1] and not mask[5, 1]
    if dt == torch.bfloat16:
        assert float(h[0, 2]) == 999424.0 and mask[0, 2]
        assert float(h[0, 3]) == 999424.0 and not mask[0, 3]          # same rounded h, different mask
    else:
        assert torch.isposinf(h[:, 0].float()).all() and torch.isneginf(h[:, 1].float()).all()


@pytest.mark.gpu
def test_every_gate16_instantiation_is_launched(cuda):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for dt in DTYPES.values():
            for i, (rows, hid, off) in enumerate(LAYOUTS.values()):
                _run_anchor(dt, rows, hid, off, cuda, seed=i)
        torch.cuda.synchronize()
    launched = set()
    for evt in prof.events():
        launched |= _demangled(evt.name)
    missing = sorted(set(GATE16_KERNELS) - launched)
    assert not missing, f"{len(missing)} instantiations never launched: {missing}"
    assert launched <= set(GATE16_KERNELS)


# ------------------------------------------------------------------------------------------------ the cell
def _autocast(dt, enabled=True):
    return torch.autocast("cuda", dtype=dt, enabled=enabled, cache_enabled=False)


def _gamma(u, k):
    return (1 + u) ** k - 1


def _csr_of(csr):
    """fp64-oracle copy of a forward CSR (rows, columns, edge ids): snapshots of a dynamic graph change in place."""
    n = csr.num_nodes
    ro = csr.row_offset.long()
    col = csr.column_indices[: csr.num_edges].long()
    eid = (torch.arange(csr.num_edges, device=ro.device) if csr.eids_identity
           else csr.eids[: csr.num_edges].long() - csr.eid_base)
    rows = torch.repeat_interleave(torch.arange(n, device=ro.device), ro[1:] - ro[:-1])
    return rows, col, eid, n, int((ro[1:] - ro[:-1]).max()) if n else 0


def _agg64(c, x, norm, w):
    rows, col, eid, n, _ = c
    s = norm[col]
    if w is not None:
        s = s * w.reshape(-1).double()[eid]
    return torch.zeros(n, x.shape[1], dtype=x.dtype, device=x.device).index_add(0, rows, x[col] * s[:, None]) * norm[:, None]


def _ref_window(model, steps, H0, u, hid, fin):
    """fp64 restatement of temporal/tgcn.py over the window with autograd, and a first-order bound of the 16-bit cell's
    forward error: every dt rounding (X, W3, X·W3, A, h, H, the gate weights, HR) and fp32 accumulation over the GEMM
    depth / row length, propagated through the gates (sigmoid' <= 1/4, tanh' <= 1, clamp 1-Lipschitz) and over steps."""
    P = {k: p.detach().double().requires_grad_(True) for k, p in model.named_parameters()}
    H = H0.detach().double().requires_grad_(True)
    xs, outs, errs = [], [], []
    eH = torch.zeros_like(H)
    Hc = H
    ab = lambda t: t.detach().abs()   # noqa: E731
    for c, x, norm, w in steps:
        x = x.detach().double().requires_grad_(True)
        xs.append(x)
        nd = norm.reshape(-1).double()
        L = c[4]
        hs, ehs = [], []
        for g in "zrh":
            W = P[f"conv_{g}.weight"]
            xw = x @ W
            a = _agg64(c, xw, nd, w)
            hs.append(torch.clamp(a + P[f"conv_{g}.bias"], -CLAMP, CLAMP))
            mxw = ab(x) @ ab(W)
            e_xw = (_gamma(u, 3) + fin * E32) * mxw
            ma = _agg64(c, mxw, nd.abs(), None if w is None else w.abs())
            e_a = _agg64(c, e_xw, nd.abs(), None if w is None else w.abs()) + (u + L * E32) * ma * (1 + _gamma(u, 3))
            ehs.append(e_a + (u + E32) * (ab(a) + e_a + ab(P[f"conv_{g}.bias"])))
        Hd = ab(Hc)
        lin = {g: (P[f"linear_{g}.weight"][:, :hid], P[f"linear_{g}.weight"][:, hid:], P[f"linear_{g}.bias"]) for g in "zrh"}

        def e_gate(g, hin, e_in, hh, e_hh):     # error of hh @ La^T + hin @ Lc^T + lb; hin is rounded here, hh already was
            La, Lc, lb = lin[g]
            return ((_gamma(u, 2) + 2 * hid * E32) * (ab(hin) @ ab(Lc).t()) + e_in @ ab(Lc).t() * (1 + u)
                    + (u + 2 * hid * E32) * (ab(hh) @ ab(La).t()) + e_hh @ ab(La).t() * (1 + u) + 2 * E32 * ab(lb))

        pz = hs[0] @ lin["z"][0].t() + Hc @ lin["z"][1].t() + lin["z"][2]
        pr = hs[1] @ lin["r"][0].t() + Hc @ lin["r"][1].t() + lin["r"][2]
        e_pz, e_pr = e_gate("z", Hc, eH, hs[0], ehs[0]), e_gate("r", Hc, eH, hs[1], ehs[1])
        R = torch.sigmoid(pr)
        HR = Hc * R
        e_hr = eH * ab(R) + Hd * e_pr / 4
        e_hr = e_hr + u * (ab(HR) + e_hr)
        ph = hs[2] @ lin["h"][0].t() + HR @ lin["h"][1].t() + lin["h"][2]
        La, Lc, lb = lin["h"]
        e_ph = ((u + hid * E32) * (ab(HR) @ ab(Lc).t()) + e_hr @ ab(Lc).t() * (1 + u)
                + (u + 2 * hid * E32) * (ab(hs[2]) @ ab(La).t()) + ehs[2] @ ab(La).t() * (1 + u) + 2 * E32 * ab(lb))
        Z, T = torch.sigmoid(pz), torch.tanh(ph)
        out = Z * Hc + (1 - Z) * T
        eH = ab(Z) * eH + ab(Hc - T) * e_pz / 4 + ab(1 - Z) * e_ph + 16 * E32 * (Hd + 1)
        outs.append(out)
        errs.append(eH)
        Hc = out
    return P, H, xs, outs, errs


def _snapshots(n, T, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, n, (6 * n, 2))
    out = []
    for _ in range(T):
        e = np.concatenate([base[rng.random(base.shape[0]) > 0.1], rng.integers(0, n, (n, 2))])
        e = e[e[:, 0] != e[:, 1]]
        out.append(np.unique(e, axis=0).astype(np.int32))
    return out


def _window(kind, n, T, cuda):
    """(graph, per-step callback that prepares step t and returns (csr copy, norm, edge weight))."""
    from stgraph_b200.graph import GPMAGraph, StaticGraph

    weighted = kind.endswith("weighted")
    if kind.startswith("static"):
        rng = np.random.default_rng(5)
        g = StaticGraph(torch.from_numpy(np.unique(rng.integers(0, n, (10 * n, 2)), axis=0).astype(np.int32)), None, n)
        g.set_ndata("norm", g.degree_norm())
        w = (torch.rand(g.get_num_edges(), 1, device=cuda, generator=torch.Generator(device=cuda).manual_seed(1)) + 0.5
             if weighted else None)

        def step(t):
            return _csr_of(g._forward_graph), g.get_ndata("norm"), w
        return g, step
    G = GPMAGraph(_snapshots(n, T, 7), n)

    def step(t):
        if t == 0:
            G.reset_graph()
        G.get_graph(t)
        G.set_ndata("norm", G.degree_norm())
        G.bwd_view()
        w = (torch.rand(G.get_num_edges(), 1, device=cuda, generator=torch.Generator(device=cuda).manual_seed(t)) + 0.5
             if weighted else None)
        return _csr_of(G._forward_graph), G.get_ndata("norm"), w
    return G, step


def _run(model, g, step, xs, H0, gouts, dt, autocast=True):
    """One BPTT window: returns (outputs, dX, dH0); the parameter gradients are left in ``model``."""
    x = xs.clone().requires_grad_(True)
    H0 = H0.clone().requires_grad_(True)
    h, outs, cost = H0, [], 0
    steps = []
    for t in range(xs.shape[0]):
        c, norm, w = step(t)
        steps.append((c, xs[t], norm, w))
        with _autocast(dt, autocast):
            h = model(g, x[t], edge_weight=w, H=h)
        outs.append(h)
        cost = cost + (h.float() * gouts[t]).sum()
    cost.backward()
    return [o.detach() for o in outs], x.grad, H0.grad, steps


CELL_CASES = {"static": 16, "static_weighted": 13, "gpma": 16}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("kind", list(CELL_CASES))
def test_cell_against_fp64_bptt_window(cuda, dtype, kind):
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN

    dt, u = DTYPES[dtype], U[DTYPES[dtype]]
    n, fin, hid, T = 700, 12, CELL_CASES[kind], 5
    g, step = _window(kind, n, T, cuda)
    torch.manual_seed(0)
    model = TGCN(fin, hid).to(cuda)
    with torch.no_grad():
        for p in model.parameters():
            p.mul_(2.0)
    xs = torch.randn(T, n, fin, device=cuda)
    H0 = 0.5 * torch.randn(n, hid, device=cuda)
    gouts = torch.randn(T, n, hid, device=cuda)
    outs, dX, dH, steps = _run(model, g, step, xs, H0, gouts, dt)
    assert all(o.dtype == torch.float32 for o in outs) and dX.dtype == torch.float32 and dH.dtype == torch.float32
    P, H64, x64, o64, errs = _ref_window(model, steps, H0, u, hid, fin)
    for t in range(T):
        err = (outs[t].double() - o64[t].detach()).abs()
        bound = 1.25 * errs[t] + 2.0 ** -40        # 1.25: second-order terms of the first-order bound
        assert bool((err <= bound).all()), f"out at step {t}: worst excess {float((err - bound).max())}"
    sum(((o * gd.double()).sum() for o, gd in zip(o64, gouts))).backward()
    # Gradients: every path of the backward rounds at most 6 times per step in the forward (as above) and 5 times in
    # the backward (the dt twin of dP, dh, dXW, the weight operand of the GEMM, dX when X is dt), so over T steps the
    # relative error of each product along a path is below gamma(11 T); the gradient is a sum of such products whose
    # magnitude is measured by |g64| plus its mean (cancellation).
    k = _gamma(u, 11 * T)
    got = {"dX": dX, "dH": dH, **{name: p.grad for name, p in model.named_parameters()}}
    want = {"dX": torch.stack([x.grad for x in x64]), "dH": H64.grad, **{name: P[name].grad for name in P}}
    for name, gv in got.items():
        ref = want[name]
        assert gv.dtype == torch.float32 and torch.isfinite(gv).all(), name
        bound = k * (ref.abs() + ref.abs().mean()) + 1e-30
        assert bool(((gv.double() - ref).abs() <= bound).all()), name


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_default_against_reference_structured_path_under_autocast(cuda, dtype):
    """TGCN() against TGCN(fused=False) (the path autocast took before) with the same state_dict: both within their
    rounding bounds of the fp64 model, so within the sum of the two of each other."""
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN

    dt, u = DTYPES[dtype], U[DTYPES[dtype]]
    n, fin, hid, T = 600, 8, 16, 5
    g, step = _window("static", n, T, cuda)
    torch.manual_seed(1)
    a = TGCN(fin, hid).to(cuda)
    b = TGCN(fin, hid, fused=False).to(cuda)
    b.load_state_dict(a.state_dict())
    xs = torch.randn(T, n, fin, device=cuda)
    H0 = 0.5 * torch.randn(n, hid, device=cuda)
    gouts = torch.randn(T, n, hid, device=cuda)
    oa, xa, ha, _ = _run(a, g, step, xs, H0, gouts, dt)
    ob, xb, hb, _ = _run(b, g, step, xs, H0, gouts, dt)
    assert b.conv_z.stgraph._ctx_map and not a.conv_z.stgraph._ctx_map
    # The reference-structured path rounds more often per step: the gate GEMM outputs and the gate activations are dt,
    # about 4 more roundings forward and backward; its bound is gamma(15 T), the fused cell's gamma(11 T).
    k = _gamma(u, 11 * T) + _gamma(u, 15 * T)
    for t in range(T):
        ref = ob[t].float()
        assert bool(((oa[t] - ref).abs() <= k * (ref.abs() + ref.abs().mean())).all()), f"out at step {t}"
    for name, ga, gb in [("dX", xa, xb), ("dH", ha, hb)] + [(nm, p.grad, q.grad) for (nm, p), q in
                                                            zip(a.named_parameters(), b.parameters())]:
        gb = gb.float()
        assert bool(((ga - gb).abs() <= k * (gb.abs() + gb.abs().mean()) + 1e-30).all()), name


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_routing_launches_and_casts(cuda, dtype, monkeypatch):
    """Under autocast TGCN() runs the 16-bit cell (no executor unit), its new kernels, two casts per step (X, H) and the
    16-bit weight copies once per window."""
    from torch.profiler import ProfilerActivity, profile

    from stgraph_b200 import ops_tgcn
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN

    dt = DTYPES[dtype]
    n, fin, hid, T = 500, 8, 16, 4
    g, step = _window("static", n, T, cuda)
    model = TGCN(fin, hid).to(cuda)
    made = []
    orig = ops_tgcn.lowp_parameters
    monkeypatch.setattr(ops_tgcn, "lowp_parameters", lambda packed, d: made.append(d) or orig(packed, d))
    xs = torch.randn(T, n, fin, device=cuda)
    gouts = torch.randn(T, n, hid, device=cuda)

    def window():
        h, cost = None, 0
        for t in range(T):
            with _autocast(dt):
                h = model(g, xs[t], H=h)
            cost = cost + (h * gouts[t]).sum()
        cost.backward()

    window()
    torch.cuda.synchronize()
    assert made == [dt]
    assert not model.conv_z.stgraph._ctx_map and not model.conv_h.stgraph._ctx_map, "an executor unit ran"
    made.clear()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        window()
        torch.cuda.synchronize()
    assert made == [dt], "the 16-bit weight copies are made once per window"
    names = [e.name for e in prof.events()]
    casts = sum(nm == "aten::_to_copy" for nm in names)
    assert casts == 2 * T + 4, f"{casts} casts for {T} steps: X and H per step and the 4 weight copies expected"
    for k in KINDS:
        cnt = sum(f"cell_{k}16_kernel<" in nm for nm in names)
        assert cnt == T, f"cell_{k}16_kernel launched {cnt} times"
    assert sum("cell_update_fwd_kernel<" in nm for nm in names) == T
    assert not any(re.search(r"\bbias_clamp4?_kernel", nm) for nm in names)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_deterministic_and_cuda_graph_replay(cuda, dtype):
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN

    dt = DTYPES[dtype]
    n, fin, hid, T = 500, 8, 16, 4
    g, step = _window("static_weighted", n, T, cuda)
    torch.manual_seed(3)
    model = TGCN(fin, hid).to(cuda)
    xs = torch.randn(T, n, fin, device=cuda)
    H0 = torch.randn(n, hid, device=cuda)
    gouts = torch.randn(T, n, hid, device=cuda)
    w = step(0)[2]

    def window():
        h, cost = H0, 0
        for t in range(T):
            with _autocast(dt):
                h = model(g, xs[t], edge_weight=w, H=h)
            cost = cost + (h * gouts[t]).sum()
        cost.backward()
        return h

    def grads():
        return [p.grad.clone() for p in model.parameters()]

    runs = []
    for _ in range(2):
        model.zero_grad(set_to_none=True)
        out = window().detach().clone()
        runs.append([out] + grads())
    for a, b in zip(*runs):
        assert _same(a, b), "two runs differ"
    # capture a copy whose autograd nodes are all made on the warm-up stream (the eager runs above made the original's
    # on the default stream, which a capture must not wait on)
    model = copy.deepcopy(model)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            model.zero_grad(set_to_none=True)
            window()
    torch.cuda.current_stream().wait_stream(s)
    model.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = window()
    for p in model.parameters():
        p.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip([out] + [p.grad for p in model.parameters()], runs[0]):
        assert _same(a, b), "CUDA-graph replay differs from eager"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_optimizer_steps_and_fp32_after_autocast(cuda, dtype):
    """The packed parameters (and their 16-bit copies) follow optimizer steps under autocast, and an fp32 call after
    autocast is bit-identical to a fresh fp32 copy of the module."""
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN

    dt = DTYPES[dtype]
    n, fin, hid, T = 400, 8, 16, 3
    g, step = _window("static", n, T, cuda)
    torch.manual_seed(4)
    model = TGCN(fin, hid).to(cuda)
    xs = torch.randn(T, n, fin, device=cuda)
    opt = torch.optim.SGD(model.parameters(), lr=0.1)

    def window(m, autocast):
        h, cost = None, 0
        for t in range(T):
            with _autocast(dt, autocast):
                h = m(g, xs[t], H=h)
            cost = cost + (h ** 2).mean()
        return h, cost

    for _ in range(2):
        opt.zero_grad()
        _, cost = window(model, True)
        cost.backward()
        opt.step()
        fresh = TGCN(fin, hid).to(cuda)
        fresh.load_state_dict(model.state_dict())
        with torch.no_grad():
            assert _same(window(model, True)[0], window(fresh, True)[0]), "the pack did not follow the optimizer step"
    fresh = TGCN(fin, hid).to(cuda)
    fresh.load_state_dict(model.state_dict())
    model.zero_grad(set_to_none=True)
    a, ca = window(model, False)
    b, cb = window(fresh, False)
    assert _same(a, b)
    ca.backward()
    cb.backward()
    for p, q in zip(model.parameters(), fresh.parameters()):
        assert _same(p.grad, q.grad)


@pytest.mark.gpu
def test_autocast_contract_edges(cuda):
    """fused=False stays unfused, fused="pieces" raises TypeError, H=None gives fp32 zeros, 16-bit X is accepted."""
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN

    n, fin, hid = 300, 8, 16
    g, step = _window("static", n, 1, cuda)
    torch.manual_seed(5)
    m = TGCN(fin, hid).to(cuda)
    x = torch.randn(n, fin, device=cuda)
    with _autocast(torch.bfloat16):
        out = m(g, x.to(torch.bfloat16))
        assert out.dtype == torch.float32
        ref = m(g, x.to(torch.bfloat16), H=torch.zeros(n, hid, device=cuda))
        assert _same(out, ref)
    pieces = TGCN(fin, hid, fused="pieces").to(cuda)
    with _autocast(torch.bfloat16), pytest.raises(TypeError):
        pieces(g, x)
    unf = TGCN(fin, hid, fused=False).to(cuda)
    with _autocast(torch.float16):
        unf(g, x)
    assert unf.conv_z.stgraph._ctx_map, "fused=False must run the reference-structured path"
    with pytest.raises(TypeError):                     # outside autocast: fp32 only, as before
        TGCN(fin, hid, fused=True).to(cuda)(g, x.to(torch.bfloat16), H=torch.zeros(n, hid, device=cuda))
