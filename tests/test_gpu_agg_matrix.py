"""Every aggregation kernel instantiation of ``csrc/agg.cu`` against the fp64 oracle.

One call of ``agg_scaled_sum_device`` chooses among 186 kernel instantiations: the vector width (from ``feat``, the
alignment of ``x`` / ``out`` and their row strides, and the 33..64-float ``vec = 2`` override on large graphs that
carry a row queue), the lane group and accumulator count, feature chunks above ``32 * 4 * vec`` floats, the schedule
(one row per lane group below ``2 * sm_count * 32`` rows; at or above it the software-pipelined row queue, from
static block ranges or from the view's global queue), the edge-record mode (plain, packed, row-partitioned sources),
the write mode, an ``out_rows`` map, and the hub kernel in its one-CTA and whole-cluster tiers, overlapped with the
row kernel by programmatic dependent launch on graphs of at least 2^18 edges.

``CASES`` is a table of (graph, view, width, misalignment of ``x``, scales) that together reach every instantiation
of ``AGG_KERNELS`` that the default configuration can launch; ``test_every_instantiation_is_launched`` proves it
with the profiler and ``test_kernel_list_matches_library`` keeps the list equal to the library's symbols, so a new
template instantiation fails the suite until a case reaches it.

Every case runs every entry point and write mode on the same inputs and checks:

* rel 1e-5 of the summed |terms| of ``oracle/aggregate.scaled_sum`` (fp64; ``eid_base`` passed through);
* packed == plain, padded rows == dense rows, global-queue == static-block schedule: bit for bit;
* ``+=`` and ``red.global.add`` into a random ``init`` == ``init + assign``, and a repeated call: bit for bit;
* rows outside ``out_rows`` and the padding columns of a padded ``out`` keep their sentinels;
* the view's row-queue counters read ``[0, 0]`` afterwards;
* every output is finite, although ``x`` holds NaN in a row no edge references, in the padding columns of padded
  rows and in the floats around a misaligned ``x`` (the NaN isolation of the pair form, for every schedule and width).

Graphs have prescribed in-degrees: row lengths at the edges of an edge batch (31/32/33, 63/64/65), of the hub
thresholds (64/65, 1024/1025) and of the hub tiers (8192/8193), over a random background, with distinct sources per
row so that the CSR keeps every edge.
"""
from __future__ import annotations

import dataclasses
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import aggregate as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "stgraph_b200", "lib", "libstgraph_b200.so")

# Template instantiations <VEC, GROUP, NACC, MODE> / <VEC, GROUP, NACC, MODE, PAIR> /
# <VEC, GROUP, NACC, MINB, UNROLL, MODE, PAIR, GQ>; MODE 0 plain, 1 row-partitioned sources, 2 packed.
AGG_KERNELS = [
    "agg_hub_kernel<1,1,1,0>", "agg_hub_kernel<1,1,1,1>", "agg_hub_kernel<1,1,1,2>", "agg_hub_kernel<1,16,1,0>",
    "agg_hub_kernel<1,16,1,1>", "agg_hub_kernel<1,16,1,2>", "agg_hub_kernel<1,2,1,0>", "agg_hub_kernel<1,2,1,1>",
    "agg_hub_kernel<1,2,1,2>", "agg_hub_kernel<1,32,1,0>", "agg_hub_kernel<1,32,1,1>", "agg_hub_kernel<1,32,1,2>",
    "agg_hub_kernel<1,32,2,0>", "agg_hub_kernel<1,32,2,1>", "agg_hub_kernel<1,32,2,2>", "agg_hub_kernel<1,32,4,0>",
    "agg_hub_kernel<1,32,4,1>", "agg_hub_kernel<1,32,4,2>", "agg_hub_kernel<1,4,1,0>", "agg_hub_kernel<1,4,1,1>",
    "agg_hub_kernel<1,4,1,2>", "agg_hub_kernel<1,8,1,0>", "agg_hub_kernel<1,8,1,1>", "agg_hub_kernel<1,8,1,2>",
    "agg_hub_kernel<2,1,1,0>", "agg_hub_kernel<2,1,1,1>", "agg_hub_kernel<2,1,1,2>", "agg_hub_kernel<2,16,1,0>",
    "agg_hub_kernel<2,16,1,1>", "agg_hub_kernel<2,16,1,2>", "agg_hub_kernel<2,2,1,0>", "agg_hub_kernel<2,2,1,1>",
    "agg_hub_kernel<2,2,1,2>", "agg_hub_kernel<2,32,1,0>", "agg_hub_kernel<2,32,1,1>", "agg_hub_kernel<2,32,1,2>",
    "agg_hub_kernel<2,32,2,0>", "agg_hub_kernel<2,32,2,1>", "agg_hub_kernel<2,32,2,2>", "agg_hub_kernel<2,32,4,0>",
    "agg_hub_kernel<2,32,4,1>", "agg_hub_kernel<2,32,4,2>", "agg_hub_kernel<2,4,1,0>", "agg_hub_kernel<2,4,1,1>",
    "agg_hub_kernel<2,4,1,2>", "agg_hub_kernel<2,8,1,0>", "agg_hub_kernel<2,8,1,1>", "agg_hub_kernel<2,8,1,2>",
    "agg_hub_kernel<4,1,1,0>", "agg_hub_kernel<4,1,1,1>", "agg_hub_kernel<4,1,1,2>", "agg_hub_kernel<4,16,1,0>",
    "agg_hub_kernel<4,16,1,1>", "agg_hub_kernel<4,16,1,2>", "agg_hub_kernel<4,2,1,0>", "agg_hub_kernel<4,2,1,1>",
    "agg_hub_kernel<4,2,1,2>", "agg_hub_kernel<4,32,1,0>", "agg_hub_kernel<4,32,1,1>", "agg_hub_kernel<4,32,1,2>",
    "agg_hub_kernel<4,32,2,0>", "agg_hub_kernel<4,32,2,1>", "agg_hub_kernel<4,32,2,2>", "agg_hub_kernel<4,32,4,0>",
    "agg_hub_kernel<4,32,4,1>", "agg_hub_kernel<4,32,4,2>", "agg_hub_kernel<4,4,1,0>", "agg_hub_kernel<4,4,1,1>",
    "agg_hub_kernel<4,4,1,2>", "agg_hub_kernel<4,8,1,0>", "agg_hub_kernel<4,8,1,1>", "agg_hub_kernel<4,8,1,2>",
    "agg_rows_kernel<1,1,1,0,false>", "agg_rows_kernel<1,1,1,1,false>", "agg_rows_kernel<1,1,1,2,false>",
    "agg_rows_kernel<1,16,1,0,false>", "agg_rows_kernel<1,16,1,1,false>", "agg_rows_kernel<1,16,1,2,false>",
    "agg_rows_kernel<1,2,1,0,false>", "agg_rows_kernel<1,2,1,1,false>", "agg_rows_kernel<1,2,1,2,false>",
    "agg_rows_kernel<1,32,1,0,false>", "agg_rows_kernel<1,32,1,1,false>", "agg_rows_kernel<1,32,1,2,false>",
    "agg_rows_kernel<1,32,2,0,false>", "agg_rows_kernel<1,32,2,1,false>", "agg_rows_kernel<1,32,2,2,false>",
    "agg_rows_kernel<1,32,4,0,false>", "agg_rows_kernel<1,32,4,1,false>", "agg_rows_kernel<1,32,4,2,false>",
    "agg_rows_kernel<1,4,1,0,false>", "agg_rows_kernel<1,4,1,1,false>", "agg_rows_kernel<1,4,1,2,false>",
    "agg_rows_kernel<1,8,1,0,false>", "agg_rows_kernel<1,8,1,1,false>", "agg_rows_kernel<1,8,1,2,false>",
    "agg_rows_kernel<2,1,1,0,false>", "agg_rows_kernel<2,1,1,1,false>", "agg_rows_kernel<2,1,1,2,false>",
    "agg_rows_kernel<2,16,1,0,false>", "agg_rows_kernel<2,16,1,1,false>", "agg_rows_kernel<2,16,1,2,false>",
    "agg_rows_kernel<2,2,1,0,false>", "agg_rows_kernel<2,2,1,1,false>", "agg_rows_kernel<2,2,1,2,false>",
    "agg_rows_kernel<2,32,1,0,false>", "agg_rows_kernel<2,32,1,1,false>", "agg_rows_kernel<2,32,1,2,false>",
    "agg_rows_kernel<2,32,2,0,false>", "agg_rows_kernel<2,32,2,1,false>", "agg_rows_kernel<2,32,2,2,false>",
    "agg_rows_kernel<2,32,4,0,false>", "agg_rows_kernel<2,32,4,1,false>", "agg_rows_kernel<2,32,4,2,false>",
    "agg_rows_kernel<2,4,1,0,false>", "agg_rows_kernel<2,4,1,1,false>", "agg_rows_kernel<2,4,1,2,false>",
    "agg_rows_kernel<2,8,1,0,false>", "agg_rows_kernel<2,8,1,1,false>", "agg_rows_kernel<2,8,1,2,false>",
    "agg_rows_kernel<4,1,1,0,false>", "agg_rows_kernel<4,1,1,1,false>", "agg_rows_kernel<4,1,1,2,false>",
    "agg_rows_kernel<4,16,1,0,false>", "agg_rows_kernel<4,16,1,1,false>", "agg_rows_kernel<4,16,1,2,false>",
    "agg_rows_kernel<4,2,1,0,false>", "agg_rows_kernel<4,2,1,1,false>", "agg_rows_kernel<4,2,1,2,false>",
    "agg_rows_kernel<4,32,1,0,false>", "agg_rows_kernel<4,32,1,0,true>", "agg_rows_kernel<4,32,1,1,false>",
    "agg_rows_kernel<4,32,1,2,false>", "agg_rows_kernel<4,32,1,2,true>", "agg_rows_kernel<4,32,2,0,false>",
    "agg_rows_kernel<4,32,2,1,false>", "agg_rows_kernel<4,32,2,2,false>", "agg_rows_kernel<4,32,4,0,false>",
    "agg_rows_kernel<4,32,4,1,false>", "agg_rows_kernel<4,32,4,2,false>", "agg_rows_kernel<4,4,1,0,false>",
    "agg_rows_kernel<4,4,1,1,false>", "agg_rows_kernel<4,4,1,2,false>", "agg_rows_kernel<4,8,1,0,false>",
    "agg_rows_kernel<4,8,1,1,false>", "agg_rows_kernel<4,8,1,2,false>",
    "agg_rows_pipe_kernel<1,32,1,4,8,0,false,false>", "agg_rows_pipe_kernel<1,32,1,4,8,0,false,true>",
    "agg_rows_pipe_kernel<1,32,1,4,8,2,false,false>", "agg_rows_pipe_kernel<1,32,1,4,8,2,false,true>",
    "agg_rows_pipe_kernel<1,32,2,4,4,0,false,false>", "agg_rows_pipe_kernel<1,32,2,4,4,0,false,true>",
    "agg_rows_pipe_kernel<1,32,2,4,4,2,false,false>", "agg_rows_pipe_kernel<1,32,2,4,4,2,false,true>",
    "agg_rows_pipe_kernel<1,32,4,4,2,0,false,false>", "agg_rows_pipe_kernel<1,32,4,4,2,0,false,true>",
    "agg_rows_pipe_kernel<1,32,4,4,2,2,false,false>", "agg_rows_pipe_kernel<1,32,4,4,2,2,false,true>",
    "agg_rows_pipe_kernel<2,32,1,4,8,0,false,false>", "agg_rows_pipe_kernel<2,32,1,4,8,0,false,true>",
    "agg_rows_pipe_kernel<2,32,1,4,8,2,false,false>", "agg_rows_pipe_kernel<2,32,1,4,8,2,false,true>",
    "agg_rows_pipe_kernel<2,32,2,4,4,0,false,false>", "agg_rows_pipe_kernel<2,32,2,4,4,0,false,true>",
    "agg_rows_pipe_kernel<2,32,2,4,4,2,false,false>", "agg_rows_pipe_kernel<2,32,2,4,4,2,false,true>",
    "agg_rows_pipe_kernel<2,32,4,4,2,0,false,false>", "agg_rows_pipe_kernel<2,32,4,4,2,0,false,true>",
    "agg_rows_pipe_kernel<2,32,4,4,2,2,false,false>", "agg_rows_pipe_kernel<2,32,4,4,2,2,false,true>",
    "agg_rows_pipe_kernel<4,32,1,4,8,0,false,false>", "agg_rows_pipe_kernel<4,32,1,4,8,0,false,true>",
    "agg_rows_pipe_kernel<4,32,1,4,8,0,true,false>", "agg_rows_pipe_kernel<4,32,1,4,8,0,true,true>",
    "agg_rows_pipe_kernel<4,32,1,4,8,2,false,false>", "agg_rows_pipe_kernel<4,32,1,4,8,2,false,true>",
    "agg_rows_pipe_kernel<4,32,1,4,8,2,true,false>", "agg_rows_pipe_kernel<4,32,1,4,8,2,true,true>",
    "agg_rows_pipe_kernel<4,32,2,4,4,0,false,false>", "agg_rows_pipe_kernel<4,32,2,4,4,0,false,true>",
    "agg_rows_pipe_kernel<4,32,2,4,4,2,false,false>", "agg_rows_pipe_kernel<4,32,2,4,4,2,false,true>",
    "agg_rows_pipe_kernel<4,32,4,4,2,0,false,false>", "agg_rows_pipe_kernel<4,32,4,4,2,0,false,true>",
    "agg_rows_pipe_kernel<4,32,4,4,2,2,false,false>", "agg_rows_pipe_kernel<4,32,4,4,2,2,false,true>",
]

# Reached only with STG_AGG_PAIR=0, which is read once per process: with the pair form on, a vec-4 tile of one
# 32-lane group and one accumulator is 68..128 floats wide and always takes the pair form (launch_agg).
UNREACHABLE = {
    "agg_rows_kernel<4,32,1,0,false>": "vec 4, GROUP 32, NACC 1 is wider than 64 floats: always the pair form",
    "agg_rows_kernel<4,32,1,2,false>": "vec 4, GROUP 32, NACC 1 is wider than 64 floats: always the pair form",
    "agg_rows_pipe_kernel<4,32,1,4,8,0,false,false>": "vec 4, GROUP 32, NACC 1 on the row queue: always the pair form",
    "agg_rows_pipe_kernel<4,32,1,4,8,0,false,true>": "vec 4, GROUP 32, NACC 1 on the row queue: always the pair form",
    "agg_rows_pipe_kernel<4,32,1,4,8,2,false,false>": "vec 4, GROUP 32, NACC 1 on the row queue: always the pair form",
    "agg_rows_pipe_kernel<4,32,1,4,8,2,false,true>": "vec 4, GROUP 32, NACC 1 on the row queue: always the pair form",
}

_KERNEL_RE = re.compile(r"(agg_(?:rows_pipe|rows|hub)_kernel)<([^<>]*)>")
_MANGLED_RE = re.compile(r"\d+(agg_(?:rows_pipe|rows|hub)_kernel)I((?:L[ib]\d+E)+)E")


def _demangled_agg_names(text):
    """``agg_*_kernel<args>`` with the spaces removed, from demangled kernel names."""
    return {f"{m.group(1)}<{m.group(2).replace(' ', '')}>" for m in _KERNEL_RE.finditer(text)}


def _mangled_agg_names(text):
    """The same names from Itanium-mangled symbols (template arguments ``Li<int>E`` / ``Lb<0|1>E``)."""
    out = set()
    for m in _MANGLED_RE.finditer(text):
        args = [("true" if v == "1" else "false") if t == "b" else v for t, v in re.findall(r"L([ib])(\d+)E", m.group(2))]
        out.add(f"{m.group(1)}<{','.join(args)}>")
    return out


def test_kernel_list_matches_library():
    """``AGG_KERNELS`` names exactly the aggregation kernels compiled into the library."""
    if not os.path.exists(LIB):
        pytest.skip("libstgraph_b200.so is not built")
    tool = shutil.which("cuobjdump")
    if tool is None and shutil.which("nvcc"):
        cand = os.path.join(os.path.dirname(shutil.which("nvcc")), "cuobjdump")
        tool = cand if os.path.exists(cand) else None
    if tool is None:
        pytest.skip("cuobjdump is not available")
    res = subprocess.run([tool, "-symbols", LIB], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, check=True)
    built = _mangled_agg_names(res.stdout)
    assert len(AGG_KERNELS) == len(set(AGG_KERNELS)) == 186
    assert set(UNREACHABLE) <= set(AGG_KERNELS)
    assert built == set(AGG_KERNELS), (f"in the library, not in AGG_KERNELS: {sorted(built - set(AGG_KERNELS))}; "
                                       f"in AGG_KERNELS, not in the library: {sorted(set(AGG_KERNELS) - built)}")


# ------------------------------------------------------------------------------------------------ case table
W4 = [4, 8, 16, 32, 64, 100, 128, 132, 256, 260, 512, 612, 1028]     # vec 4 (612 = 512 + a pair-form 100)
W2 = [2, 6, 14, 30, 34, 62, 66, 130, 258, 514]                        # vec 2
W1 = [1, 3, 7, 15, 31, 33, 63, 65, 127, 129, 257]                     # vec 1
# (feat, floats by which x is shifted off a 16-byte boundary): the alignment, not the width, selects vec
MISALIGNED = [(2, 1), (4, 1), (4, 2), (8, 2), (64, 2), (132, 1), (260, 2)]
WMAX = 1028

# scale set -> (nbr_scale, edge_scale, row_scale) present
SCALES = {"all": (True, True, True), "none": (False, False, False), "ns": (True, False, False),
          "es_rs": (False, True, True)}


@dataclasses.dataclass(frozen=True)
class Case:
    graph: str       # "small" (per-row kernel), "large" (row queue, >= 2^18 edges), "pcsr" (dynamic snapshot)
    view: str        # key of _Graph.views
    feat: int
    offset: int      # floats between a 16-byte boundary and x
    scales: str

    @property
    def id(self):
        return f"{self.graph}-{self.view}-F{self.feat}" + (f"+{self.offset}" if self.offset else "") + f"-{self.scales}"


def _cases():
    table = [
        ("small", "fwd", [(f, 0) for f in W4 + W2 + W1] + MISALIGNED),     # per-row kernels, every cell, every mode
        ("small", "t64", [(f, 0) for f in W4 + W2 + W1] + MISALIGNED),     # hub kernels (one-CTA tier), every cell
        ("small", "bwd", [(f, 0) for f in (4, 7, 30, 100, 260, 612)]),
        # row queue: global queue and (static copy) block ranges; 48 / 64 take the narrow vec-2 override
        ("large", "fwd", [(f, 0) for f in (1, 2, 4, 6, 31, 33, 34, 48, 62, 64, 65, 66, 100, 127, 128, 130, 132, 256,
                                            258, 260, 512, 612, 1028)] + [(48, 1), (64, 2), (132, 2)]),
        ("large", "nohub", [(f, 0) for f in (4, 64, 100, 612)]),
        ("large", "t64", [(f, 0) for f in (3, 16, 34, 64, 100, 132, 260, 612)] + [(8, 2)]),   # hundreds of hub rows
        ("large", "bwd", [(f, 0) for f in (7, 64, 100, 260)]),
        ("pcsr", "fwd", [(f, 0) for f in (1, 48, 64, 100, 130, 612)]),
        ("pcsr", "bwd", [(f, 0) for f in (5, 100)]),
    ]
    rot = list(SCALES)
    cases = []
    for graph, view, widths in table:
        for i, (f, off) in enumerate(widths):
            # wide oracles are the expensive ones: above 260 floats the large graphs use one scale set
            sc = "all" if graph != "small" and f > 260 else rot[i % len(rot)]
            cases.append(Case(graph, view, f, off, sc))
    return cases


CASES = _cases()


# ------------------------------------------------------------------------------------------------ graphs
def _prescribed_edges(lengths, seed, iso):
    """(src, dst) with exactly ``lengths[v]`` distinct in-neighbours per vertex ``v``, none of them ``iso``."""
    rng = np.random.default_rng(seed)
    n = lengths.shape[0]
    rows = np.repeat(np.arange(n, dtype=np.int64), 2 * lengths + 16)
    src = rng.integers(0, n - 1, rows.shape[0])
    src[src >= iso] += 1
    key = rng.permutation(np.unique(rows * n + src))
    key = key[np.argsort(key // n, kind="stable")]
    r = key // n
    rank = np.arange(key.shape[0]) - np.searchsorted(r, r)
    key = key[rank < lengths[r]]
    short = np.nonzero(np.bincount(key // n, minlength=n) < lengths)[0]
    pool = np.delete(np.arange(n, dtype=np.int64), iso)
    extra = [v * n + rng.choice(pool, lengths[v], replace=False) for v in short]
    key = np.concatenate([key[~np.isin(key // n, short)]] + extra)
    src, dst = (key % n).astype(np.int32), (key // n).astype(np.int32)
    assert np.array_equal(np.bincount(dst, minlength=n), lengths)
    return src, dst


def _lengths(n, seed, background, prescribed, medium):
    """Random background in-degrees, the ``prescribed`` ones spread over the rows, ``medium`` rows of 65..160 edges."""
    rng = np.random.default_rng(seed)
    lengths = rng.integers(0, background, n)
    slots = rng.permutation(np.arange(1, n))
    lengths[slots[: len(prescribed)]] = prescribed
    lengths[slots[len(prescribed): len(prescribed) + medium]] = rng.integers(65, 161, medium)
    iso = 0                                  # no edges at all: x[iso] is never read
    lengths[iso] = 0
    return lengths, iso


@dataclasses.dataclass
class _View:
    view: object
    direction: str          # "fwd" / "bwd": which CSR (and oracle) the view describes
    csr: object
    queue: torch.Tensor | None
    static: object = None   # the same view without its row queue (static block ranges)
    sub: object = None      # sub-CSR of selected rows (see _sub), built on first use


@dataclasses.dataclass
class _Graph:
    n: int
    iso: int
    owner: object
    views: dict
    ns: torch.Tensor
    es: dict               # direction -> edge_scale (indexed by eid - eid_base)
    rs: torch.Tensor
    x: torch.Tensor        # [n, WMAX] fp32 on the device, NaN in row iso
    x_cpu: torch.Tensor


def _copy_view(v, **fields):
    from stgraph_b200 import _lib

    c = _lib.StgCsrView()
    for name, _ in _lib.StgCsrView._fields_:
        setattr(c, name, getattr(v, name))
    for name, val in fields.items():
        setattr(c, name, val)
    return c


def _no_hubs(v):
    return _copy_view(v, hub_rows=None, hub_count=None, hub_threshold=0, hub_capacity=0)


def _queue_of(csr, v):
    q = getattr(csr, "_work_queue", None)
    if v.work_queue is None:
        return None
    assert q is not None and q.data_ptr() == v.work_queue
    return q


def _entry(csr, v, direction):
    q = _queue_of(csr, v)
    return _View(v, direction, csr, q, static=_copy_view(v, work_queue=None) if q is not None else None)


def _scales(n, e_fwd, e_bwd, seed, device):
    tg = torch.Generator().manual_seed(seed)
    ns = torch.rand(n, generator=tg) + 0.5
    rs = torch.rand(n, generator=tg) + 0.5
    es = torch.rand(max(e_fwd, e_bwd), generator=tg) + 0.25
    return ns.to(device), {"fwd": es[:e_fwd].to(device), "bwd": es[:e_bwd].to(device)}, rs.to(device)


def _features(n, iso, seed, device):
    x = torch.randn(n, WMAX, generator=torch.Generator().manual_seed(seed))
    x[iso] = float("nan")
    return x.to(device), x


def _static_graph(n, lengths, iso, seed, device):
    from stgraph_b200.graph import StaticGraph

    src, dst = _prescribed_edges(lengths, seed, iso)
    g = StaticGraph(torch.from_numpy(np.stack([src, dst], 1)), None, n)
    f, b = g._forward_graph, g._backward_graph
    assert np.array_equal(np.diff(f.row_offset.cpu().numpy()), lengths)
    views = {"fwd": _entry(f, g.fwd_view(), "fwd"), "bwd": _entry(b, g.bwd_view(), "bwd"),
             "t64": _entry(f, f.view_with_hub_threshold(64), "fwd")}
    views["nohub"] = _View(_no_hubs(g.fwd_view()), "fwd", f, views["fwd"].queue)
    ns, es, rs = _scales(n, f.num_edges, b.num_edges, seed + 1, device)
    x, x_cpu = _features(n, iso, seed + 2, device)
    return _Graph(n, iso, g, views, ns, es, rs, x, x_cpu), (src, dst)


@pytest.fixture(scope="module")
def ctx(cuda):
    from stgraph_b200 import kernels
    from stgraph_b200.graph import PCSRGraph

    torch.cuda.set_device(cuda)
    sm = kernels.device_info(cuda.index or 0)["sm_count"]
    queue_rows = 2 * sm * 4 * 8                 # launch_agg: the row queue starts at two waves of 4 blocks x 8 warps
    hub_pass = 2 * (sm // 8) * 8                # hub rows one pass of the hub grid takes (2 CTAs per SM below 2^24 edges)
    graphs = {}

    n = 600
    lengths, iso = _lengths(n, 1, 24, [0, 1, 2, 31, 32, 33, 63, 64, 65, 128, 129, 300, 599], 40)
    graphs["small"], _ = _static_graph(n, lengths, iso, 10, cuda)
    assert n < queue_rows

    n = queue_rows + 37                         # the last queue slot and the last block are partial
    lengths, iso = _lengths(n, 2, 40, [0, 1, 2, 31, 32, 33, 63, 64, 65, 1024, 1025, 8192, 8193], 3 * hub_pass)
    large, (src, dst) = _static_graph(n, lengths, iso, 20, cuda)
    graphs["large"] = large
    e = src.shape[0]
    assert e >= 1 << 18                         # the hub kernel overlaps the row kernel (programmatic launch)
    f = large.owner._forward_graph
    assert int(f._alt_views[64][2].item()) > hub_pass      # the threshold-64 view needs more than one pass

    # a dynamic snapshot of the same graph: PCSR rows back to front, eids from 1, unsorted hub list on the stream
    rng = np.random.default_rng(30)
    background = lengths < 64
    drop = (rng.random(e) < 0.02) & background[dst]
    k_old = dst.astype(np.int64) * n + src
    cand = rng.integers(1, n, (2, e // 40))
    cand = cand[:, background[cand[1]] & (cand[0] != cand[1])]
    k_new = np.setdiff1d(cand[1].astype(np.int64) * n + cand[0], k_old)
    k1 = np.concatenate([k_old[~drop], k_new])
    snaps = [np.stack([src, dst], 1), rng.permutation(np.stack([k1 % n, k1 // n], 1).astype(np.int32))]
    pg = PCSRGraph(snaps, n)
    pg.get_graph(1)
    vb = pg.bwd_view()                          # builds both directions
    vf = pg.fwd_view()
    pf, pb = pg._forward_graph, pg._backward_graph
    assert pf.eid_base == 1 and pb.eid_base == 1 and vf.eid_base == 1 and not pf.eids_identity
    assert pf.num_edges >= 1 << 18 and int(pf.row_degrees.max()) == 8193 and vf.hub_threshold > 0
    ns, es, rs = _scales(n, pf.num_edges, pb.num_edges, 31, cuda)
    x, x_cpu = _features(n, iso, 32, cuda)
    graphs["pcsr"] = _Graph(n, iso, pg, {"fwd": _entry(pf, vf, "fwd"), "bwd": _entry(pb, vb, "bwd")},
                            ns, es, rs, x, x_cpu)

    widths = {}                                 # oracle key -> widest case that needs it
    for c in CASES:
        k = _oracle_key(graphs[c.graph], c)
        widths[k] = max(widths.get(k, 0), c.feat)
    return {"graphs": graphs, "widths": widths, "oracles": {}, "device": cuda, "sm": sm}


def _oracle_key(g, c):
    has_ns, has_es, _ = SCALES[c.scales]
    return (c.graph, g.views[c.view].direction, has_ns, has_es)


def _oracle(ctx, c):
    """(fp64 reference, fp64 sum of |terms|) on the device, ``[n, feat]``, row scale applied."""
    g = ctx["graphs"][c.graph]
    entry = g.views[c.view]
    key = _oracle_key(g, c)
    if key not in ctx["oracles"]:
        csr = entry.csr
        ro = csr.row_offset.cpu()
        col = csr.column_indices.cpu()
        eids = (torch.arange(csr.num_edges, dtype=torch.int64) + csr.eid_base) if csr.eids_identity else csr.eids.cpu()
        ns = g.ns.cpu() if key[2] else None
        es = g.es[key[1]].cpu() if key[3] else None
        refs, mags = [], []
        for c0 in range(0, ctx["widths"][key], 64):     # the oracle is exact per column: bound its [E, F] messages
            xs = g.x_cpu[:, c0:min(ctx["widths"][key], c0 + 64)].double()
            refs.append(A.scaled_sum(ro, col, eids, xs, ns, es, None, eid_base=csr.eid_base))
            mags.append(A.scaled_sum(ro, col, eids, xs.abs(), ns, es, None, eid_base=csr.eid_base))
        ctx["oracles"][key] = (torch.cat(refs, 1).to(ctx["device"]), torch.cat(mags, 1).to(ctx["device"]))
    ref, mag = ctx["oracles"][key]
    ref, mag = ref[:, : c.feat], mag[:, : c.feat]
    if SCALES[c.scales][2]:
        rs = g.rs.double().reshape(-1, 1)
        ref, mag = ref * rs, mag * rs
    return ref, mag


def _sub(ctx, g, entry):
    """A CSR of all rows but every (n // 20)-th (as a row-partitioned pass builds it), with the view's hub threshold
    and its own row queue when the view has one; view row i is output row ``out_rows[i]``."""
    from stgraph_b200 import _lib

    if entry.sub is not None:
        return entry.sub
    dev = ctx["device"]
    csr, v, n = entry.csr, entry.view, g.n
    keep = torch.ones(n, dtype=torch.bool, device=dev)
    keep[3:: max(n // 20, 2)] = False
    sel = torch.nonzero(keep).reshape(-1)
    ro = csr.row_offset.long()
    beg, deg = ro[sel], ro[sel + 1] - ro[sel]
    sro = torch.zeros(sel.numel() + 1, dtype=torch.int64, device=dev)
    sro[1:] = torch.cumsum(deg, 0)
    idx = torch.repeat_interleave(beg - sro[:-1], deg) + torch.arange(int(sro[-1]), device=dev)
    cols = csr.column_indices[idx].contiguous()
    eids = ((idx + csr.eid_base) if csr.eids_identity else csr.eids[idx].long()).int().contiguous()
    sro = sro.int().contiguous()
    s = _lib.StgCsrView()
    s.row_offset, s.column_indices, s.eids, s.node_ids = sro.data_ptr(), cols.data_ptr(), eids.data_ptr(), None
    s.num_nodes, s.num_edges, s.eid_base, s.eids_identity = int(sel.numel()), int(cols.shape[0]), csr.eid_base, 0
    keep_alive = [sro, cols, eids]
    s.hub_rows = s.hub_count = None
    s.hub_threshold = s.hub_capacity = 0
    if v.hub_threshold > 0:
        cap = int(cols.shape[0]) // v.hub_threshold + 1
        hr = torch.empty(cap, dtype=torch.int32, device=dev)
        hc = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.call("stg_csr_hub_rows", sro.data_ptr(), s.num_nodes, v.hub_threshold, hr.data_ptr(), cap, hc.data_ptr(),
                  _lib.current_stream_ptr())
        s.hub_rows, s.hub_count, s.hub_threshold, s.hub_capacity = hr.data_ptr(), hc.data_ptr(), v.hub_threshold, cap
        keep_alive += [hr, hc]
    q = None
    if v.work_queue is not None:
        q = torch.zeros(2, dtype=torch.int32, device=dev)
        s.work_queue = q.data_ptr()
    else:
        s.work_queue = None
    entry.sub = (s, sel.int().contiguous(), q, keep, keep_alive)
    return entry.sub


# ------------------------------------------------------------------------------------------------ running a case
SENTINEL = -7.0


def _x_at(g, feat, offset):
    """``x[:, :feat]`` as a contiguous [n, feat] tensor ``offset`` floats past an aligned address, NaN around it."""
    buf = torch.full((offset + g.n * feat + 4,), float("nan"), device=g.x.device)
    x = buf[offset: offset + g.n * feat].view(g.n, feat)
    x.copy_(g.x[:, :feat])
    return x


def _padded(kernels, n, feat, fill, device):
    t = kernels.padded_rows(n, feat, device)
    torch.as_strided(t, (n, t.stride(0)), (t.stride(0), 1)).fill_(fill)
    return t


def _launch(ctx, c):
    """Run one case through every entry point and write mode; returns the outputs (checked by ``_check``)."""
    from stgraph_b200 import kernels

    dev = ctx["device"]
    g = ctx["graphs"][c.graph]
    entry = g.views[c.view]
    v, n, feat = entry.view, g.n, c.feat
    has_ns, has_es, has_rs = SCALES[c.scales]
    ns = g.ns if has_ns else None
    es = g.es[entry.direction] if has_es else None
    rs = g.rs if has_rs else None
    x = _x_at(g, feat, c.offset)
    gen = torch.Generator(device=dev).manual_seed(feat * 7 + c.offset)
    init = torch.randn(n, feat, device=dev, generator=gen)
    r = {"init": init}
    r["assign"] = kernels.agg_scaled_sum(v, x, ns, es, rs)
    r["queue_first"] = entry.queue.clone() if entry.queue is not None else None
    r["again"] = kernels.agg_scaled_sum(v, x, ns, es, rs)
    r["accum"] = kernels.agg_scaled_sum(v, x, ns, es, rs, out=init.clone(), accumulate=True)
    r["red"] = kernels.agg_scaled_sum(v, x, ns, es, rs, out=init.clone(), accumulate="red")
    meta = kernels.pack_edge_meta(v, ns, es, device=dev)
    r["packed"] = kernels.agg_packed_sum(v, meta, x, rs)
    r["packed_accum"] = kernels.agg_packed_sum(v, meta, x, rs, out=init.clone(), accumulate=True)
    r["packed_red"] = kernels.agg_packed_sum(v, meta, x, rs, out=init.clone(), accumulate="red")
    if c.offset == 0:
        xp = _padded(kernels, n, feat, float("nan"), dev)
        xp.copy_(x)
        op = _padded(kernels, n, feat, SENTINEL, dev)
        kernels.agg_packed_sum(v, meta, xp, rs, out=op)
        r["padded"] = op
    if entry.static is not None:
        r["static"] = kernels.agg_scaled_sum(entry.static, x, ns, es, rs)
        r["static_packed"] = kernels.agg_packed_sum(entry.static, meta, x, rs)
    s, out_rows, sq, keep, _ = _sub(ctx, g, entry)
    r["rows"] = kernels.agg_scaled_sum(s, x, ns, es, rs, out=torch.full((n, feat), SENTINEL, device=dev), out_rows=out_rows)
    r["rows_accum"] = kernels.agg_scaled_sum(s, x, ns, es, rs, out=init.clone(), accumulate=True, out_rows=out_rows)
    smeta = kernels.pack_edge_meta(s, ns, es, device=dev)
    r["rows_packed"] = kernels.agg_packed_sum_rows(s, smeta, out_rows, x, rs, torch.full((n, feat), SENTINEL, device=dev))
    r["rows_keep"], r["rows_queue"] = keep, sq
    bounds = [0, n // 3, 2 * n // 3, n]
    r["parts"] = kernels.agg_scaled_sum_parts(v, [x[b].data_ptr() for b in bounds[:3]], bounds, feat, ns, es, rs,
                                              out=torch.full((n, feat), SENTINEL, device=dev))
    r["queue_last"] = entry.queue
    return r


def _narrow_override(c):
    """33..64 floats, feat % 4 == 0, 16-byte aligned: vec 2 on the global queue, vec 4 without a queue."""
    return c.offset == 0 and c.feat % 4 == 0 and 32 < c.feat <= 64


def _check(ctx, c, r):
    ref, mag = _oracle(ctx, c)
    what = c.id
    a = r["assign"]
    assert bool(torch.isfinite(a).all()), f"{what}: non-finite output (NaN from a row no edge references?)"
    A.assert_close_rel(a, ref, rel=1e-5, abs_terms=mag, what=what)
    init = r["init"]

    def same(key, exp):
        assert torch.equal(r[key], exp), f"{what}: {key} differs from its expected bits ({int((r[key] != exp).sum())} elements)"

    same("again", a)
    same("accum", init + a)
    same("red", init + a)
    same("packed", a)
    same("packed_accum", init + a)
    same("packed_red", init + a)
    if "padded" in r:
        op = r["padded"]
        assert torch.equal(op, a), f"{what}: padded rows differ from dense rows"
        full = torch.as_strided(op, (op.shape[0], op.stride(0)), (op.stride(0), 1))
        assert bool((full[:, c.feat:] == SENTINEL).all()), f"{what}: padding columns of out were written"
    if "static" in r:
        if _narrow_override(c):
            A.assert_close_rel(r["static"], ref, rel=1e-5, abs_terms=mag, what=what + " static schedule")
        else:
            same("static", a)
        same("static_packed", r["static"])
    keep = r["rows_keep"]
    rows = r["rows"]
    A.assert_close_rel(rows[keep], ref[keep], rel=1e-5, abs_terms=mag[keep], what=what + " out_rows")
    assert bool((rows[~keep] == SENTINEL).all()), f"{what}: out_rows wrote rows outside the map"
    same("rows_packed", rows)
    acc = r["rows_accum"]
    assert torch.equal(acc[keep], init[keep] + rows[keep]) and torch.equal(acc[~keep], init[~keep]), \
        f"{what}: out_rows += is not init + assign"
    A.assert_close_rel(r["parts"], ref, rel=1e-5, abs_terms=mag, what=what + " row-partitioned sources")
    for key in ("queue_first", "queue_last", "rows_queue"):
        if r[key] is not None:
            assert r[key].tolist() == [0, 0], f"{what}: {key} counters not re-armed: {r[key].tolist()}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_case_matches_oracle(ctx, case):
    _check(ctx, case, _launch(ctx, case))


@pytest.mark.gpu
def test_every_instantiation_is_launched(ctx):
    """The case table launches every reachable instantiation (and none of the unreachable ones)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for c in CASES:
            _launch(ctx, c)
        torch.cuda.synchronize()
    launched = set()
    for evt in prof.events():
        launched |= _demangled_agg_names(evt.name)
    expected = set(AGG_KERNELS) - set(UNREACHABLE)
    missing = sorted(expected - launched)
    print(f"aggregation instantiations: {len(AGG_KERNELS)} compiled, {len(expected & launched)} launched, "
          f"{len(UNREACHABLE)} unreachable by design, {len(missing)} missing")
    assert not missing, f"{len(missing)} instantiations never launched: {missing}"
    assert not (launched & set(UNREACHABLE)), f"launched although listed unreachable: {sorted(launched & set(UNREACHABLE))}"
    assert launched <= set(AGG_KERNELS), f"launched but not in AGG_KERNELS: {sorted(launched - set(AGG_KERNELS))}"


@pytest.mark.gpu
def test_row_queue_protocol_across_kernels_and_graph_capture(ctx):
    """The global row queue is shared by the aggregation and the GAT kernels of one view; every launch must leave
    its two counters re-armed, or the next launch on the view silently skips rows."""
    from stgraph_b200 import kernels
    from stgraph_b200.ops_gat import gat_edge_softmax_aggregate

    dev = ctx["device"]
    g = ctx["graphs"]["large"]
    entry = g.views["fwd"]
    v, q = entry.view, entry.queue
    assert q is not None
    widths = (34, 64, 100, 132, 260, 612)
    xs = {f: _x_at(g, f, 0) for f in widths}
    meta = kernels.pack_edge_meta(v, g.ns, g.es["fwd"], device=dev)
    outs = {("plain", f): torch.empty(g.n, f, device=dev) for f in widths}
    outs.update({("packed", f): torch.empty(g.n, f, device=dev) for f in widths})

    def run():
        for f in widths:
            kernels.agg_scaled_sum(v, xs[f], g.ns, g.es["fwd"], g.rs, out=outs[("plain", f)])
        for f in widths:
            kernels.agg_packed_sum(v, meta, xs[f], g.rs, out=outs[("packed", f)])

    run()
    torch.cuda.synchronize()
    first = {k: t.clone() for k, t in outs.items()}
    assert q.tolist() == [0, 0]
    for f in widths:
        assert torch.equal(first[("plain", f)], first[("packed", f)]), f
        c = Case("large", "fwd", f, 0, "all")
        ref, mag = _oracle(ctx, c)
        A.assert_close_rel(first[("plain", f)], ref, rel=1e-5, abs_terms=mag, what=f"queue sequence F={f}")

    tg = torch.Generator(device=dev).manual_seed(5)
    heads, dim = 4, 16
    el = torch.randn(g.n, heads, 1, device=dev, generator=tg)
    er = torch.randn(g.n, heads, 1, device=dev, generator=tg)
    feat = torch.randn(g.n, heads, dim, device=dev, generator=tg).requires_grad_(True)
    att = gat_edge_softmax_aggregate(g.owner, el, er, feat, 0.2)
    att.backward(torch.randn_like(att))
    torch.cuda.synchronize()
    assert q.tolist() == [0, 0], "the GAT kernels left the shared row queue armed"
    att2 = gat_edge_softmax_aggregate(g.owner, el, er, feat.detach(), 0.2)
    assert torch.equal(att.detach(), att2)

    run()
    torch.cuda.synchronize()
    for k, t in outs.items():
        assert torch.equal(t, first[k]), f"{k} changed after the GAT kernels ran on the same queue"

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run()
    for k in outs:
        outs[k].fill_(SENTINEL)
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        for k, t in outs.items():
            assert torch.equal(t, first[k]), f"{k}: a CUDA-graph replay differs from the eager result"
            t.fill_(SENTINEL)
    assert q.tolist() == [0, 0]
