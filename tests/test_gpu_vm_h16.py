"""Vertex programs on bf16 / fp16 tensors: the mixed form of the VM kernel (``csrc/vm.cu`` with ``MIXED = true``,
``stg_vm_run_mixed``) and the layers that reach it under ``torch.autocast``.

A LOAD widens each 16-bit element to fp32 and the lanes are those of the fp32 launch on the widened tensors at the same
element offset, so the outputs of a program must equal those of the same program on ``.float()`` copies bit for bit, and
the gradient of a 16-bit input must equal the fp32 run's gradient rounded to the input's dtype.
"""
from __future__ import annotations

import copy
import ctypes
import dataclasses
import os
import re
import shutil
import subprocess
import zlib

import numpy as np
import pytest
import torch
from torch import nn

from oracle import aggregate as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "stgraph_b200", "lib", "libstgraph_b200.so")

DTYPES = {"bf16": torch.bfloat16, "f16": torch.float16}
GROUPS = (1, 2, 4, 8, 16, 32)


def _vm_mixed_kernels():
    """(GROUP, HUB, VEC, U) of every mixed instantiation: the row kernel with float4 lanes (U = 1) and scalar lanes
    (U = 4), the hub kernel with float4 lanes (U = 4 / 2 / 1 by register-file size) and scalar lanes (U = 1)."""
    shapes = [("false", 4, 1), ("false", 1, 4), ("true", 4, 4), ("true", 4, 2), ("true", 4, 1), ("true", 1, 1)]
    return sorted(f"vm_kernel<{g},{h},{v},{u},true>" for g in GROUPS for h, v, u in shapes)


VM_MIXED_KERNELS = _vm_mixed_kernels()
_KERNEL_RE = re.compile(r"vm_kernel<(\d+), ?(true|false), ?(\d+), ?(\d+), ?true>")
_MANGLED_RE = re.compile(r"vm_kernelILi(\d+)ELb([01])ELi(\d+)ELi(\d+)ELb([01])EE")


def _demangled(text):
    return {f"vm_kernel<{m.group(1)},{m.group(2)},{m.group(3)},{m.group(4)},true>" for m in _KERNEL_RE.finditer(text)}


def _mangled(text, mixed):
    return {f"vm_kernel<{m.group(1)},{'true' if m.group(2) == '1' else 'false'},{m.group(3)},{m.group(4)},"
            f"{'true' if mixed else 'false'}>" for m in _MANGLED_RE.finditer(text) if m.group(5) == ("1" if mixed else "0")}


def test_vm_mixed_kernel_list_matches_library():
    """``VM_MIXED_KERNELS`` names exactly the mixed VM kernels compiled into the library, and each has an fp32 twin."""
    if not os.path.exists(LIB):
        pytest.skip("libstgraph_b200.so is not built")
    tool = shutil.which("cuobjdump")
    if tool is None and shutil.which("nvcc"):
        cand = os.path.join(os.path.dirname(shutil.which("nvcc")), "cuobjdump")
        tool = cand if os.path.exists(cand) else None
    if tool is None:
        pytest.skip("cuobjdump is not available")
    res = subprocess.run([tool, "-symbols", LIB], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, check=True)
    assert len(VM_MIXED_KERNELS) == 36
    assert _mangled(res.stdout, True) == set(VM_MIXED_KERNELS)
    assert _mangled(res.stdout, False) == {k.replace(",true>", ",false>") for k in VM_MIXED_KERNELS}


# ------------------------------------------------------------------------------------------------ C ABI, no GPU
def _tiny_program():
    """LOAD t0 (PRE), STORE t1 (POST) on [1, 4] lanes: enough to pass every check; the tensors are never touched."""
    from stgraph_b200 import _lib

    p = _lib.StgVmProgram()
    p.dim0, p.dim1, p.n_tensors, p.n_instr, p.n_regs, p.n_acc, p.n_pre, p.n_loop = 1, 4, 2, 2, 1, 0, 1, 0
    for i in range(2):
        p.tensors[i].side, p.tensors[i].bc0, p.tensors[i].bc1 = 0, 1, 1
    p.instr[0].op, p.instr[0].phase, p.instr[0].dst, p.instr[0].a = 0, 0, 0, 0          # LOAD r0 <- t0
    p.instr[1].op, p.instr[1].phase, p.instr[1].a, p.instr[1].b = 16, 2, 1, 0           # STORE t1 <- r0
    return p


def test_vm_entry_points_check_dtype_codes_without_gpu():
    """Unknown codes and 16-bit STORE targets are rejected by ``stg_vm_run_mixed``, any 16-bit code by
    ``stg_vm_run_f32``; every other check gives the fp32 entry point's message.  All of it before any launch."""
    from stgraph_b200 import _lib

    lib = _lib.load()
    v = _lib.StgCsrView()
    v.num_nodes, v.num_edges, v.row_offset = 4, 0, 1             # never dereferenced
    ptrs = (ctypes.c_void_p * _lib.VM_MAX_TENSORS)()
    ptrs[0], ptrs[1] = 256, 512

    def run(name, prog, view=v):
        return getattr(lib, name)(ctypes.byref(view), ctypes.byref(prog), ptrs, None), lib.stg_last_error()

    for code in (3, -1, 7):
        p = _tiny_program()
        p.tensors[0].dtype = code
        rc, msg = run("stg_vm_run_mixed", p)
        assert rc == -1 and b"unknown dtype code" in msg
    for code in (1, 2):
        p = _tiny_program()
        p.tensors[0].dtype = p.tensors[1].dtype = code
        rc, msg = run("stg_vm_run_mixed", p)
        assert rc == -1 and b"STORE" in msg and b"fp32" in msg
        p.tensors[1].dtype = 0
        rc, msg = run("stg_vm_run_f32", p)
        assert rc == -1 and b"stg_vm_run_mixed" in msg
    # valid codes pass every check: with no rows nothing is launched
    empty = _lib.StgCsrView()
    empty.num_nodes, empty.row_offset = 0, 1
    for code in (0, 1, 2):
        p = _tiny_program()
        p.tensors[0].dtype = code
        assert run("stg_vm_run_mixed", p, empty)[0] == 0
    assert run("stg_vm_run_f32", _tiny_program(), empty)[0] == 0

    # the fp32 entry point's checks, with the same messages
    def broken():
        for field, val in (("dim0", 0), ("n_tensors", 25), ("n_instr", 97), ("n_regs", 49), ("n_acc", 9), ("n_pre", 3)):
            p = _tiny_program()
            setattr(p, field, val)
            yield p
        p = _tiny_program()
        p.instr[0].op = 99
        yield p
        p = _tiny_program()
        p.instr[1].a = 5
        yield p
        p = _tiny_program()
        p.instr[1].op, p.dim1 = 17, 64                                                  # GSUM over 64 lanes
        yield p
        p = _tiny_program()
        p.tensors[0].side = 2                                                           # an edge tensor without eids
        yield p

    nv = _lib.StgCsrView()
    nv.num_nodes, nv.num_edges, nv.row_offset = 4, 8, 1
    for p in broken():
        a, b = run("stg_vm_run_f32", p, nv), run("stg_vm_run_mixed", p, nv)
        assert a[0] == b[0] == -1 and a[1] == b[1], (a, b)
    p = _tiny_program()
    ptrs[0] = None
    assert run("stg_vm_run_f32", p) == run("stg_vm_run_mixed", p) == (-1, b"tensor 0 is NULL")
    assert lib.stg_vm_run_mixed(None, None, None, None) == -1 and b"NULL" in lib.stg_last_error()


# ------------------------------------------------------------------------------------------------ the programs
class Programs(nn.Module):
    """Vertex programs that the lowering sends to the VM kernel (none has the scaled-sum shape)."""

    def __init__(self, F, k=0, dtype=torch.float32, seed=0):
        super().__init__()
        self.k = k
        self.p = nn.Parameter(torch.randn(F, generator=torch.Generator().manual_seed(seed)).to(dtype))
        from stgraph_b200.compiler import STGraph
        from stgraph_b200.compiler.backend.pytorch.torch_callback import STGraphBackendTorch

        self.stgraph = STGraph(STGraphBackendTorch())

    def program(self, name):
        """The compiled vertex program ``name``; its inputs are ``USES[name]`` (``c`` stands for c0 ... c(k-1))."""
        from stgraph_b200.compiler.op.agg import agg_max, agg_mean, agg_min

        if name == "msg":       # centre, neighbour, edge and parameter LOADs; [N,F] and [N,1] broadcasts; a sum
            @self.stgraph.compile(gnn_module=self)
            def msg(v):
                return sum([(nb.h * e.w + self.p) * v.s for nb, e in zip(v.innbs, v.inedges)])

            return msg
        if name == "max":       # the k centre rows stay live in the edge loop: k sets the size of the register file
            @self.stgraph.compile(gnn_module=self)
            def amax(v):
                vals = []
                for nb in v.innbs:
                    x = nb.h
                    for i in range(self.k):
                        x = x * getattr(v, f"c{i}")
                    vals.append(x)
                return agg_max(vals)

            return amax
        if name == "min":
            @self.stgraph.compile(gnn_module=self)
            def amin(v):
                return agg_min([nb.h - v.s for nb in v.innbs])

            return amin

        @self.stgraph.compile(gnn_module=self)
        def amean(v):
            return agg_mean([nb.h * e.w for nb, e in zip(v.innbs, v.inedges)])

        return amean


USES = {"msg": ("h", "s", "w"), "max": ("h", "c"), "min": ("h", "s"), "mean": ("h", "w"),
        "gat": ("el", "er", "feat_src")}
KS = {"max1": 1, "max12": 12, "max20": 20}       # centre rows of the max programs: hub U = 4, 2, 1 with float4 lanes


def _kind(prog):
    return "max" if prog in KS else prog


def _feats(prog, x):
    """(n_feats, e_feats) of a program from a dict holding at least its inputs."""
    names = [k for k in x if k in USES[_kind(prog)] or (k[0] == "c" and "c" in USES[_kind(prog)])]
    return {k: x[k] for k in names if k != "w"}, {k: x[k] for k in names if k == "w"}


@dataclasses.dataclass(frozen=True)
class Case:
    prog: str         # msg | max1 / max12 / max20 (k centre rows) | min | mean | gat (the stock GAT program)
    shape: tuple      # (F,) or (H, D) for gat
    offset: int       # elements between a 16-byte boundary and h / feat_src (2: VEC = 1 whatever F is)
    dtype: str        # bf16 | f16 | mix (h bf16, s fp16, w and p fp32)

    @property
    def id(self):
        return f"{self.prog}-{self.dtype}-{'x'.join(map(str, self.shape))}" + (f"+{self.offset}" if self.offset else "")


VEC4_F = (4, 8, 16, 32, 64, 128, 256)         # lanes 1, 2, 4, 8, 16, 32, 64 with VEC = 4
VEC1_F = (1, 2, 3, 6, 10, 20, 40)             # F % 4 != 0 (or F < 4): VEC = 1, lanes 1 ... 40


def _cases():
    out = []
    for dt in DTYPES:
        out += [Case("msg", (f,), 0, dt) for f in VEC4_F + VEC1_F] + [Case("msg", (16,), 2, dt)]
        out += [Case(p, (f,), 0, dt) for p in ("max12", "max20") for f in VEC4_F]      # hub U = 2 and U = 1
        out += [Case(p, (f,), 0, dt) for p in ("max1", "min", "mean") for f in (16, 6)]
        out += [Case("gat", (8, 16), 0, dt), Case("gat", (4, 6), 0, dt), Case("gat", (2, 4), 2, dt)]
    out += [Case("msg", (32,), 0, "mix"), Case("msg", (10,), 0, "mix")]
    return out


CASES = _cases()


def _graph_edges(n, seed):
    """Random edges plus hub rows (> 96 edges, both directions) and rows without in- or out-edges."""
    rng = np.random.default_rng(seed)
    src = rng.integers(0, n, 6 * n)
    dst = rng.integers(0, n, 6 * n)
    for v, deg in ((1, 700), (2, 300), (3, 97)):
        other = rng.choice(np.arange(20, n), deg, replace=False)
        src = np.concatenate([src, other, np.full(deg, v + 3)])
        dst = np.concatenate([dst, np.full(deg, v), other])
    keep = ~np.isin(dst, [10, 11]) & ~np.isin(src, [12, 13])
    k = np.unique(src[keep] * n + dst[keep])
    return (k // n).astype(np.int32), (k % n).astype(np.int32)


@pytest.fixture(scope="module")
def graph(cuda):
    from stgraph_b200.graph import StaticGraph

    torch.cuda.set_device(cuda)
    n = 3000
    src, dst = _graph_edges(n, 4)
    return {"g": StaticGraph(torch.from_numpy(np.stack([src, dst], 1)), None, n), "n": n, "src": src, "dst": dst,
            "device": cuda}


def _aligned(shape, dtype, offset, device):
    """A tensor of ``shape`` ``offset`` elements past a 16-byte boundary, NaN around it."""
    numel = int(np.prod(shape))
    buf = torch.full((numel + 16,), float("nan"), dtype=dtype, device=device)
    return buf[offset: offset + numel].view(*shape)


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _same(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _inputs(c, n, e, device):
    """{name: (tensor in the case's dtype, requires grad)} and the parameter dtype."""
    tg = torch.Generator().manual_seed(zlib.crc32(c.id.encode()))
    rand = lambda *s: torch.randn(*s, generator=tg)
    dts = {k: DTYPES.get(c.dtype, torch.bfloat16) for k in ("h", "s", "w", "p", "c", "feat", "el")}
    if c.dtype == "mix":
        dts.update(s=torch.float16, w=torch.float32, p=torch.float32)
    # gradients: AggMin / AggMean have none (as in the reference); max20's backward needs more than 48 registers
    grads = {"msg": ("h", "s"), "max1": ("h",), "max12": ("h",), "gat": ("feat_src", "el", "er")}.get(c.prog, ())
    if c.prog == "gat":
        H, D = c.shape
        x = {"feat_src": rand(n, H, D), "el": rand(n, H, 1), "er": rand(n, H, 1)}
        dt = {"feat_src": dts["feat"], "el": dts["el"], "er": dts["el"]}
        offs = {"feat_src": c.offset}
    else:
        (F,) = c.shape
        x = {"h": rand(n, F), "s": rand(n, 1) * 0.5 + 1, "w": rand(e, 1)}
        dt = {"h": dts["h"], "s": dts["s"], "w": dts["w"]}
        for i in range(KS.get(c.prog, 0)):
            x[f"c{i}"] = rand(n, F) * 0.25 + 1
            dt[f"c{i}"] = dts["c"]
        offs = {"h": c.offset}
    out16, out32 = {}, {}
    for name, t in x.items():
        a = _aligned(t.shape, dt[name], offs.get(name, 0), device)
        a.copy_(t.to(dt[name]))
        b = _aligned(t.shape, torch.float32, offs.get(name, 0), device)
        b.copy_(a.float())
        out16[name], out32[name] = a, b
    for name in grads:
        out16[name].requires_grad_(True)
        out32[name].requires_grad_(True)
    return out16, out32, dts["p"]


def _call(c, gr, x, module):
    if c.prog == "gat":
        return module._stock_program()(g=gr["g"], n_feats={k: x[k] for k in USES["gat"]})
    nf, ef = _feats(c.prog, x)
    return module.program(_kind(c.prog))(g=gr["g"], n_feats=nf, e_feats=ef)


def _module(c, dtype):
    if c.prog == "gat":
        from stgraph_b200.nn.pytorch import GATConv

        H, D = c.shape
        return GATConv(4, D, H).to("cuda")
    return Programs(c.shape[0], KS.get(c.prog, 0), dtype, seed=len(c.id)).to("cuda")


def _run_case(gr, c):
    """Both runs of a case: (output, {input: grad}, parameter grad) for the 16-bit and for the widened inputs."""
    n, e = gr["n"], gr["g"].get_num_edges()
    x16, x32, pdt = _inputs(c, n, e, gr["device"])
    res, mods = [], []
    for x, dt in ((x16, pdt), (x32, torch.float32)):
        m = _module(c, dt)
        if mods and c.prog != "gat":
            with torch.no_grad():
                m.p.copy_(mods[0].p.float())        # the widened parameter
        mods.append(m)
        out = _call(c, gr, x, m)
        grads = {}
        if any(t.requires_grad for t in x.values()):
            gout = torch.randn(out.shape, generator=torch.Generator().manual_seed(7)).to(out.device)
            out.backward(gout)
            grads = {k: t.grad for k, t in x.items() if t.requires_grad}
        pg = getattr(m, "p", None)
        res.append((out.detach(), grads, None if pg is None else pg.grad))
    return x16, res


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_vm_h16_program_equals_widened_run(graph, case):
    from stgraph_b200 import kernels

    before = kernels.launch_count
    x16, ((o16, g16, p16), (o32, g32, p32)) = _run_case(graph, case)
    assert kernels.launch_count > before
    assert o16.dtype == torch.float32 and _same(o16, o32), f"{case.id}: output differs"
    has_in = torch.from_numpy(np.bincount(graph["dst"], minlength=graph["n"]) > 0).to(o16.device)
    assert torch.isfinite(o16[has_in]).all()
    assert set(g16) == set(g32)
    for k in g16:
        dt = x16[k].dtype
        assert g16[k].dtype == dt and _same(g16[k], g32[k].to(dt)), f"{case.id}: gradient of {k} differs"
    if p16 is not None and p32 is not None:
        assert _same(p16, p32.to(p16.dtype)), f"{case.id}: parameter gradient differs"
    elif case.prog == "msg":
        pytest.fail("the parameter received no gradient")


@pytest.mark.gpu
def test_every_vm_mixed_instantiation_is_launched(graph):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for c in CASES:
            _run_case(graph, c)
        torch.cuda.synchronize()
    launched = set()
    for evt in prof.events():
        launched |= _demangled(evt.name)
    missing = sorted(set(VM_MIXED_KERNELS) - launched)
    print(f"mixed VM instantiations: {len(VM_MIXED_KERNELS)} compiled, {len(launched & set(VM_MIXED_KERNELS))} launched")
    assert not missing, f"{len(missing)} instantiations never launched: {missing}"
    assert launched <= set(VM_MIXED_KERNELS)


@pytest.mark.gpu
def test_vm_mixed_program_against_fp64_oracle(graph):
    """The mixed-dtype message program against the fp64 IR interpreter on the widened inputs, within DESIGN §5's fp32
    bound ``|x - ref| <= 1e-5 * max(|ref|, sum |terms|)``."""
    from oracle.ir_interp import Interp

    c = Case("msg", (32,), 0, "mix")
    n = graph["n"]
    x16, _, pdt = _inputs(c, n, graph["g"].get_num_edges(), graph["device"])
    m = _module(c, pdt)
    out = _call(c, graph, x16, m).detach().cpu()
    ctx = m.stgraph._ctx_map[next(iter(m.stgraph._ctx_map))]
    # the CSR's edge ids: forward eid i is the i-th edge in (dst, src) order
    order = np.lexsort((graph["src"], graph["dst"]))
    src, dst = graph["src"][order], graph["dst"][order]

    def oracle(f):
        env = {"Vhinb": f(x16["h"]), "Vscen": f(x16["s"]), "Vw": f(x16["w"]), "Vp": f(m.p)}
        env = Interp(src, dst, n).run_units(ctx.forward_units, env)
        return env[ctx.forward_units[-1].unit_rets()[0].id]

    ref = oracle(lambda t: t.detach().double().cpu())
    terms = oracle(lambda t: t.detach().double().cpu().abs())
    A.assert_close_rel(out, ref, rel=1e-5, abs_terms=terms, what="mixed program vs fp64")


# ------------------------------------------------------------------------------------------------ end to end
def _autocast(dt, enabled=True):
    if dt == torch.bfloat16:
        return torch.autocast("cuda", dtype=dt, enabled=enabled)
    return torch.autocast("cuda", enabled=enabled)


class UserLayer(nn.Module):
    """A user's layer: two projections under autocast feed a vertex program with an fp32 edge weight."""

    def __init__(self, fin, F):
        super().__init__()
        self.fc = nn.Linear(fin, F)
        self.gate = nn.Linear(fin, 1)
        self.p = nn.Parameter(torch.randn(F))
        from stgraph_b200.compiler import STGraph
        from stgraph_b200.compiler.backend.pytorch.torch_callback import STGraphBackendTorch

        self.stgraph = STGraph(STGraphBackendTorch())

    def forward(self, g, x, w, widen=False):
        h, s = self.fc(x), torch.sigmoid(self.gate(x)) + 0.5
        if widen:
            h, s = h.float(), s.float()

        @self.stgraph.compile(gnn_module=self)
        def nb(v):
            return sum([(nb.h * e.w + self.p) * v.s for nb, e in zip(v.innbs, v.inedges)])

        return nb(g=g, n_feats={"h": h, "s": s}, e_feats={"w": w})


def _grads(model, x):
    return [p.grad.clone() for p in model.parameters()] + [x.grad.clone()]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_user_program_static_under_autocast(graph, dtype):
    dt = DTYPES[dtype]
    g, n, dev = graph["g"], graph["n"], graph["device"]
    torch.manual_seed(0)
    layer = UserLayer(12, 24).to(dev)
    ref, fresh = copy.deepcopy(layer), copy.deepcopy(layer)
    x0 = torch.randn(n, 12, device=dev)
    w = torch.rand(g.get_num_edges(), 1, device=dev)
    gout = torch.randn(n, 24, device=dev)
    outs = []
    for model, widen in ((layer, False), (ref, True)):
        x = x0.clone().requires_grad_(True)
        with _autocast(dt):
            out = model(g, x, w, widen)
        assert out.dtype == torch.float32
        out.backward(gout)
        outs.append((out.detach(), _grads(model, x)))
    assert all(p.grad is not None and p.grad.abs().sum() > 0 for p in layer.fc.parameters())
    assert _same(outs[0][0], outs[1][0])
    for a, b in zip(outs[0][1], outs[1][1]):
        assert _same(a, b)
    assert _same(layer(g, x0, w), fresh(g, x0, w))       # outside autocast afterwards: the fp32 program, unchanged


def _snapshots(n, T, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, n, (6 * n, 2))
    out = []
    for _ in range(T):
        e = np.concatenate([base[rng.random(base.shape[0]) > 0.1], rng.integers(0, n, (n, 2))])
        e = e[e[:, 0] != e[:, 1]]
        out.append(np.unique(e, axis=0).astype(np.int32))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_user_program_gpma_bptt_under_autocast(cuda, dtype):
    """The user layer over several GPMAGraph snapshots, one backward at the end (each step's backward at its timestamp)."""
    from stgraph_b200.graph import GPMAGraph

    dt = DTYPES[dtype]
    n, fin, F, T = 500, 12, 16, 4
    G = GPMAGraph(_snapshots(n, T, 9), n)
    torch.manual_seed(0)
    layer = UserLayer(fin, F).to(cuda)
    ref, fresh = copy.deepcopy(layer), copy.deepcopy(layer)
    xs = torch.randn(T, n, fin, device=cuda)
    gouts = [torch.randn(n, F, device=cuda) for _ in range(T)]

    def run(model, widen, autocast=True):
        model.zero_grad(set_to_none=True)
        G.reset_graph()
        x = xs.clone().requires_grad_(True)
        cost, outs = 0, []
        for t in range(T):
            G.get_graph(t)
            w = torch.linspace(0.5, 1.5, G.get_num_edges(), device=cuda).unsqueeze(1)
            with _autocast(dt, autocast):
                o = model(G, x[t], w, widen)
            assert o.dtype == torch.float32
            outs.append(o.detach())
            cost = cost + (o * gouts[t]).sum()
        cost.backward()
        return outs, _grads(model, x)

    native, widened = run(layer, False), run(ref, True)
    for a, b in zip(native[0] + native[1], widened[0] + widened[1]):
        assert _same(a, b)
    plain, fresh_run = run(layer, False, autocast=False), run(fresh, False, autocast=False)
    for a, b in zip(plain[0] + plain[1], fresh_run[0] + fresh_run[1]):
        assert _same(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_vm_mixed_cuda_graph_replay(graph, dtype):
    c = Case("msg", (32,), 0, dtype)
    x16, _, pdt = _inputs(c, graph["n"], graph["g"].get_num_edges(), graph["device"])
    x = {k: t.detach() for k, t in x16.items()}
    m = _module(c, pdt)
    with torch.no_grad():
        eager = _call(c, graph, x, m).clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            _call(c, graph, x, m)
        torch.cuda.current_stream().wait_stream(side)
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            out = _call(c, graph, x, m)
        for _ in range(3):
            out.fill_(float("nan"))
            cg.replay()
            torch.cuda.synchronize()
            assert _same(out, eager)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_stock_gatconv_reads_the_16bit_projection(graph, dtype):
    """Under autocast the stock layer launches no cast of the projection, and the state stack holds the 16-bit
    projection itself for backward: no fp32 ``[N, H, D]`` tensor but the layer's own output."""
    from torch.profiler import ProfilerActivity, profile

    from stgraph_b200.nn.pytorch import GATConv

    dt = DTYPES[dtype]
    g, n, dev = graph["g"], graph["n"], graph["device"]
    H, D = 8, 16
    torch.manual_seed(0)
    layer = GATConv(24, D, H).to(dev)
    x = torch.randn(n, 24, device=dev, requires_grad=True)

    def upcast(m, x):
        proj, left, right = m._scores(x)
        return m._stock_program()(g=g, n_feats={"el": left, "er": right, "feat_src": proj.float()})

    def kernels_of(fwd):
        with _autocast(dt):
            fwd(layer, x)                                     # warm: traced, graph views built
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            with _autocast(dt):
                fwd(layer, x)
            torch.cuda.synchronize()
        return [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]

    native, widened = kernels_of(lambda m, x: m(g, x)), kernels_of(upcast)
    assert len(native) == len(widened) - 1, ([e.name for e in native], [e.name for e in widened])

    fc_out = {}
    hook = layer.fc.register_forward_hook(lambda mod, i, o: fc_out.__setitem__("o", o))
    with _autocast(dt):
        out = layer(g, x)
    hook.remove()
    ex = layer._stock_program()._executor_cache
    saved = ex.ts.tensor_map_stack.top()
    feat = saved["Vfeat_srcinb"]
    assert feat.dtype == dt and feat.data_ptr() == fc_out["o"].data_ptr()
    for t in saved.values():
        if t.dtype == torch.float32 and tuple(t.shape) == (n, H, D):
            assert t.data_ptr() == out.data_ptr(), "an fp32 [N, H, D] tensor besides the output is held for backward"
    out.sum().backward()
    while len(ex.ts.tensor_map_stack):                         # the warm-up forwards above had no backward
        ex.ts.tensor_map_stack.pop()


# ------------------------------------------------------------------------------------------------ lowering, no GPU
class _FakeGraph:
    def __init__(self, n, e):
        self.n, self.e = n, e

    def get_num_nodes(self):
        return self.n

    def get_num_edges(self):
        return self.e


def _lowered(ctx):
    out = []
    for units in (ctx.forward_units, ctx.backward_units):
        for u in units:
            if not u.compiled:
                out.append(("torch", tuple(s.op_name for s in u.program)))
                continue
            for la in u.launches:
                assert la.kind == "vm"
                p = la.program
                out.append((la.center.name, p.dim0, p.dim1, p.n_regs, p.n_acc, p.n_pre, p.n_loop,
                            tuple(p.acc_init[i] for i in range(p.n_acc)), tuple(p.acc_kind[i] for i in range(p.n_acc)),
                            tuple((p.tensors[i].side, p.tensors[i].bc0, p.tensors[i].bc1) for i in range(p.n_tensors)),
                            tuple((ins.op, ins.phase, ins.dst, ins.a, ins.b, ins.imm) for ins in p.instr[:p.n_instr]),
                            tuple(v.id for v in la.tensor_vars)))
    return out


@pytest.mark.parametrize("prog", ["msg", "max12", "max20", "min", "mean", "gat"])
def test_16bit_trace_lowers_to_the_fp32_program(prog):
    """A program traced with bf16 inputs lowers to the VM instructions of its fp32 trace: the premise of the bit-identity
    of the two runs.  Every launch goes to the VM kernel (none has the scaled-sum shape)."""
    from stgraph_b200.nn.pytorch import GATConv

    n, e, F = 10, 30, 8
    got = []
    for dt in (torch.float32, torch.bfloat16):
        grads = {"msg": ("h", "s"), "max12": ("h",), "gat": ("el", "er", "feat_src")}.get(prog, ())
        if prog == "gat":
            x = {"el": torch.randn(n, 8, 1), "er": torch.randn(n, 8, 1), "feat_src": torch.randn(n, 8, 16).to(dt)}
            ctx = GATConv(12, 16, 8)._stock_program()
            nf, ef = x, {}
        else:
            x = {"h": torch.randn(n, F), "s": torch.randn(n, 1), "w": torch.randn(e, 1)}
            x.update({f"c{i}": torch.randn(n, F) for i in range(KS.get(prog, 0))})
            x = {k: t.to(dt) for k, t in x.items()}
            ctx = Programs(F, KS.get(prog, 0), dt).program(_kind(prog))
            nf, ef = _feats(prog, x)
        for k in grads:
            x[k].requires_grad_(True)
        ctx._setup_executor(g=_FakeGraph(n, e), n_feats=nf, e_feats=ef)
        got.append(_lowered(ctx))
    assert got[0] == got[1]
    assert len(got[0]) >= 1
