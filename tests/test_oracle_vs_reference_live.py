"""Pinning of the oracle against the reference's OWN code, on random inputs.

Aggregation and GAT: the outputs of the CUDA kernels the reference's code generator emits, run on these tests' seeded
inputs, are stored in ``tests/golden/ref_kernels_live.npz`` (``oracle/make_golden.py``); the tests rebuild the inputs
from their seeds and compare the oracle with the stored rows.

Structure: ``oracle/build_ref.py`` compiles the reference's ``csr.cu`` and ``pcsr.cu`` from its sources into
``oracle/_ref/*.so`` (host code; no GPU needed to run it).  Where those libraries are built, these tests drive them on
seeded random graphs / streams and demand bit-identical arrays from ``oracle/structure.py``; elsewhere they skip, and
the committed fixtures ``tests/golden/ref_structure.npz`` / ``ref_pcsr.npz`` (tests/test_golden_oracle.py) are such runs.
"""
import os

import numpy as np
import pytest
import torch

from oracle import aggregate as A
from oracle import make_golden as MG
from oracle import ref_emulate as RE
from oracle import structure as S

GOLD = os.path.join(os.path.dirname(__file__), "golden")
HAVE_CSR = os.path.exists(os.path.join(RE.REF_DIR, "ref_csr.so"))
HAVE_PCSR = os.path.exists(os.path.join(RE.REF_DIR, "ref_pcsr.so"))


@pytest.mark.skipif(not HAVE_CSR, reason="oracle/_ref/ref_csr.so not built (oracle/build_ref.py needs the reference's sources)")
@pytest.mark.parametrize("n,e,seed", [(1, 0, 0), (2, 1, 1), (7, 20, 2), (50, 400, 3), (300, 5000, 4), (1000, 3000, 5)])
def test_static_structure_oracle_equals_reference_csr_builder(n, e, seed):
    src, dst = MG.live_graph(n, e, seed)
    if e == 0:
        src, dst = np.zeros(0, np.int32), np.zeros(0, np.int32)
    w = np.random.default_rng(seed + 100).uniform(0.1, 1.0, size=src.shape[0]).astype(np.float32)
    fwd, bwd = RE.reference_static_graph(src, dst, w, n)
    f, b = S.forward_csr(src, dst, n), S.backward_csr(src, dst, n)
    for name in ("row_offset", "column_indices", "eids"):
        np.testing.assert_array_equal(getattr(f, name), getattr(fwd, name), err_msg=f"fwd {name}")
        np.testing.assert_array_equal(getattr(b, name), getattr(bwd, name), err_msg=f"bwd {name}")
    np.testing.assert_array_equal(f.row_degrees, fwd.out_degrees)         # CSR::out_degrees = row lengths
    np.testing.assert_array_equal(f.col_degrees, fwd.in_degrees)
    np.testing.assert_array_equal(b.row_degrees, bwd.out_degrees)
    for ids, deg in ((fwd.node_ids, f.row_degrees), (bwd.node_ids, b.row_degrees)):
        assert sorted(ids.tolist()) == list(range(n)) and np.all(np.diff(deg[ids]) <= 0)
    np.testing.assert_array_equal(S.weighted_in_degrees(src, dst, w, n), fwd.weighted_out_degrees.astype(np.int32))


def _stream(n, t_count, base, churn, seed):
    rng = np.random.default_rng(seed)
    cur = set()
    while len(cur) < base:
        a, b = rng.integers(0, n, 2)
        if a != b:
            cur.add((int(a), int(b)))
    snaps = []
    for _ in range(t_count):
        snaps.append(sorted(cur))
        curl = sorted(cur)
        for i in rng.choice(len(curl), size=min(churn, len(curl)), replace=False):
            cur.discard(curl[i])
        while len(cur) < base:
            a, b = rng.integers(0, n, 2)
            if a != b:
                cur.add((int(a), int(b)))
    return snaps


@pytest.mark.skipif(not HAVE_PCSR, reason="oracle/_ref/ref_pcsr.so not built (oracle/build_ref.py needs the reference's sources)")
@pytest.mark.parametrize("n,T,base,churn,seed", [(5, 4, 6, 3, 0), (16, 6, 60, 30, 1), (40, 5, 200, 200, 2), (120, 8, 900, 150, 3)])
def test_pcsr_oracle_equals_reference_pcsr_on_random_streams(n, T, base, churn, seed):
    """Forward roll, then backward roll, like PCSRGraph (pcsr_graph.py:45-166); `churn == base` replaces every edge."""
    snaps = _stream(n, T, base, churn, seed)
    keys = S.snapshot_edge_sets(snaps)
    ups = S.snapshot_updates(snaps)
    ref = RE.RefPcsr(n, len({e for s in snaps for e in s}))
    try:
        def same(t, reverse):
            exp = (S.labelled_backward_view if reverse else S.labelled_forward_view)(keys[t], n, descending_rows=True)
            ro, col, eid, nid, ind, outd = ref.build(reverse)
            np.testing.assert_array_equal(ro.astype(np.int32), exp.row_offset, err_msg=f"t={t} rev={reverse} row_offset")
            np.testing.assert_array_equal(col.astype(np.int32), exp.column_indices, err_msg=f"t={t} rev={reverse} cols")
            np.testing.assert_array_equal(eid.astype(np.int32), exp.eids, err_msg=f"t={t} rev={reverse} labels")
            if not reverse:
                np.testing.assert_array_equal(outd.astype(np.int32), exp.row_degrees)
                np.testing.assert_array_equal(ind.astype(np.int32), exp.col_degrees)

        for t in range(T):
            ref.step(ups[t]["add"], ups[t]["delete"])
            same(t, False)
            same(t, True)
        for t in range(T - 1, 0, -1):
            ref.step(ups[t]["delete"], ups[t]["add"])
            same(t - 1, True)
            same(t - 1, False)
    finally:
        ref.close()


@pytest.fixture(scope="module")
def gl():
    return np.load(os.path.join(GOLD, "ref_kernels_live.npz"))


def _stored(gl, key):
    """(row ids, rows) of one reference output kept in the fixture."""
    return torch.from_numpy(gl[f"{key}/rows"]).long(), torch.from_numpy(gl[key])


@pytest.mark.parametrize("case,feat,weighted", [("gcn_f16", 16, False), ("gcn_f100", 100, False), ("gcn_f128", 128, False),
                                                ("gcnw_f7", 7, True)])
@pytest.mark.parametrize("n,e,seed", [(12, 30, 0), (100, 1500, 1), (400, 6000, 2)])
def test_aggregation_oracle_equals_reference_kernels_live(gl, case, feat, weighted, n, e, seed):
    """The CUDA kernels the reference's code generator emits for GCNConv (forward K0 on the in-edge CSR, backward K1 on
    the out-edge CSR), executed on the CPU by the SIMT shim with the reference's own launch geometry, against
    oracle/aggregate.py on random graphs (a star around vertex 0 makes one long row and many short ones).  The kernels'
    outputs on these seeded inputs are stored in tests/golden/ref_kernels_live.npz (a seeded sample of rows)."""
    src, dst, w, norm, h, gin = MG.live_gcn_inputs(feat, n, e, seed)
    f, b = S.forward_csr(src, dst, n), S.backward_csr(src, dst, n)
    ht, gt, nt = torch.from_numpy(h), torch.from_numpy(gin), torch.from_numpy(norm).reshape(-1)
    wt = torch.from_numpy(w) if weighted else None
    cols = 4 if feat == 7 else feat          # trap T1: for F=7 the reference launches 4 lanes per node
    key = f"gcn/{case}/{n}_{e}_{seed}"
    for direction, run in (("forward", A.gcn_forward), ("backward", A.gcn_backward)):
        rows, ref = _stored(gl, f"{key}/{direction}")
        csr, x = (f, ht) if direction == "forward" else (b, gt)
        mine, mag = run(csr, x, nt, wt)[rows], run(csr, x.abs(), nt, wt)[rows]
        A.assert_close_rel(mine[:, :cols], ref[:, :cols], rel=3e-6, abs_terms=mag[:, :cols], what=f"{case} {direction}")
        if feat == 7 and direction == "forward":
            assert torch.count_nonzero(ref[:, 4:]) == 0      # the columns the reference never writes


@pytest.mark.parametrize("case,heads,dim", [("gat_h2d4", 2, 4), ("gat_h8d16", 8, 16)])
@pytest.mark.parametrize("n,e,seed", [(30, 150, 0), (200, 2500, 1)])
def test_stock_gat_oracle_equals_reference_kernels_live(gl, case, heads, dim, n, e, seed):
    """The three kernels the reference emits for GATConv as shipped (trap T2: a mean), forward and backward; their
    outputs on these seeded inputs are stored in tests/golden/ref_kernels_live.npz (a seeded sample of rows)."""
    src, dst, el, er, feat, gout = MG.live_gat_inputs(heads, dim, n, e, seed)
    t = torch.from_numpy
    f = S.forward_csr(src, dst, n)
    key = f"gat/{case}/{n}_{e}_{seed}"
    scale = lambda x: x.abs().mean() * torch.ones_like(x) + 1e-12

    def check(role, mine, rel, abs_terms, what=""):
        rows, ref = _stored(gl, f"{key}/{role}")
        A.assert_close_rel(mine[rows], ref.reshape((-1,) + tuple(mine.shape[1:])), rel=rel, abs_terms=abs_terms[rows], what=what)

    out, o3, o4 = A.gat_stock_forward(f, t(el), t(er), t(feat))
    check("v3", o3, 1e-6, scale(o3))
    check("v4", o4, 1e-6, scale(o4))
    check("out", out, 3e-6, scale(out))
    d_feat, d_el, d_er, m_feat, m_el, m_er = A.gat_stock_backward(f, t(el), t(er), t(feat), t(gout), return_mag=True)
    ref_dfeat_scale = float(gl[f"{key}/d_feat_abs_mean"]) * torch.ones_like(d_feat) + 1e-12
    check("d_feat", d_feat, 5e-6, ref_dfeat_scale, what="d_feat")
    check("d_el", d_el, 2e-5, m_el, what="d_el")
    check("d_er", d_er, 2e-5, m_er, what="d_er")
