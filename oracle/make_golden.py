"""Generate ``tests/golden/*.npz`` from the reference itself (run in the build container).

TEST INFRASTRUCTURE ONLY.  Requires ``oracle/_ref`` (``python oracle/build_ref.py``).  Every array
written here was computed by reference code: the CSR arrays by ``CSR::CSR`` from
``/root/reference/stgraph/graph/static/csr.cu``, the feature/gradient tensors by the CUDA kernels the
reference's code generator emits for ``GCNConv`` / ``GATConv`` (executed on the CPU through
``oracle/simt_shim.h``).  Inputs are seeded; the fixtures are small (N=40, E=200).
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_emulate as RE  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def make_graph(n=40, e=200, seed=0):
    rng = np.random.default_rng(seed)
    key = rng.choice(n * n, size=e, replace=False)
    return (key // n).astype(np.int32), (key % n).astype(np.int32)


def dynamic_stream(n, t_count, base, churn, seed):
    """Snapshot edge lists with churn, duplicates, one edge that is deleted and later re-added, and a near-empty step."""
    rng = np.random.default_rng(seed)
    cur = set()
    while len(cur) < base:
        a, b = rng.integers(0, n, 2)
        if a != b:
            cur.add((int(a), int(b)))
    pinned = sorted(cur)[0]                       # deleted at t=1, re-added at t=3
    snaps = []
    for t in range(t_count):
        now = set(cur)
        if t in (1, 2):
            now.discard(pinned)
        else:
            now.add(pinned)
        if t == t_count - 2:
            now = set(sorted(now)[:3])            # almost everything deleted at once, then re-inserted
        lst = sorted(now)
        rng.shuffle(lst)
        snaps.append(lst + lst[: max(1, len(lst) // 10)])          # duplicates collapse (dynamic_graph.py:58-63)
        curl = sorted(cur)
        for i in rng.choice(len(curl), size=min(churn, len(curl)), replace=False):
            cur.discard(curl[i])
        while len(cur) < base:
            a, b = rng.integers(0, n, 2)
            if a != b:
                cur.add((int(a), int(b)))
    return snaps


def make_pcsr_golden():
    """Drive the reference's PCSR exactly like ``PCSRGraph`` does (forward roll over all timestamps, then the
    backward roll ``_update_graph_backward`` T-1 -> 0) and record the CSR it builds at every stop."""
    from oracle import structure as S

    out = {}
    for tag, (n, T, base, churn, seed) in {"a": (60, 7, 300, 40, 3), "b": (24, 6, 70, 25, 11)}.items():
        snaps = dynamic_stream(n, T, base, churn, seed)
        ups = S.snapshot_updates(snaps)
        max_edges = len({e for s in snaps for e in s})
        flat = np.array([e for s in snaps for e in s], dtype=np.int32).reshape(-1, 2)
        out[f"{tag}/num_nodes"] = np.int32(n)
        out[f"{tag}/snap_edges"] = flat
        out[f"{tag}/snap_sizes"] = np.array([len(s) for s in snaps], dtype=np.int32)
        ref = RE.RefPcsr(n, max_edges)
        for t in range(T):
            ref.step(ups[t]["add"], ups[t]["delete"])
            for d, rev in (("fwd", False), ("bwd", True)):
                ro, col, eid, nid, ind, outd = ref.build(rev)
                out[f"{tag}/{d}/{t}/row_offset"], out[f"{tag}/{d}/{t}/column_indices"] = ro, col
                out[f"{tag}/{d}/{t}/eids"], out[f"{tag}/{d}/{t}/node_ids"] = eid, nid
                out[f"{tag}/{d}/{t}/pcsr_in_degrees"], out[f"{tag}/{d}/{t}/pcsr_out_degrees"] = ind, outd
        for t in range(T - 1, 0, -1):             # pcsr_graph.py:146-166: add the deletions, delete the additions of t
            ref.step(ups[t]["delete"], ups[t]["add"])
            ro, col, eid, nid, _, _ = ref.build(True)
            out[f"{tag}/rewind/{t - 1}/row_offset"], out[f"{tag}/rewind/{t - 1}/column_indices"] = ro, col
            out[f"{tag}/rewind/{t - 1}/eids"] = eid
        ref.close()
    np.savez_compressed(os.path.join(GOLD, "ref_pcsr.npz"), **out)
    print("wrote", os.path.join(GOLD, "ref_pcsr.npz"), len(out), "arrays")


def reference_graph_updates(snaps, n):
    """``graph_updates`` exactly as the reference computes them: its own ``DynamicGraph._preprocess_graph_structure``
    (``/root/reference/stgraph/graph/dynamic/dynamic_graph.py:56-79``, pure Python) is loaded from where it lies and run
    on the snapshot lists; only its base-class import is stubbed (the ABC pulls in the CUDA-backed graph modules)."""
    import importlib.util
    import types

    saved = {k: sys.modules.get(k) for k in ("stgraph", "stgraph.graph", "stgraph.graph.stgraph_base")}
    base = types.ModuleType("stgraph.graph.stgraph_base")

    class STGraphBase:              # stand-in for the abstract base (no behaviour on this path)
        def __init__(self):
            pass

    base.STGraphBase = STGraphBase
    sys.modules["stgraph"] = types.ModuleType("stgraph")
    sys.modules["stgraph.graph"] = types.ModuleType("stgraph.graph")
    sys.modules["stgraph.graph.stgraph_base"] = base
    try:
        spec = importlib.util.spec_from_file_location(
            "_ref_dynamic_graph", "/root/reference/stgraph/graph/dynamic/dynamic_graph.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)

        class Concrete(mod.DynamicGraph):
            def _get_cached_graph(self, timestamp):
                return False

            def __getattr__(self, name):        # the remaining abstract hooks are never reached here
                raise AttributeError(name)

        Concrete.__abstractmethods__ = frozenset()
        g = Concrete([[tuple(map(int, e)) for e in s] for s in snaps], n)
        return g.graph_updates
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def make_updates_golden():
    """a9: per-timestamp add / delete lists of three update streams, computed by the reference's own preprocessing."""
    out = {}
    for tag, (n, T, base, churn, seed) in {"a": (60, 7, 300, 40, 3), "b": (24, 6, 70, 25, 11), "c": (500, 8, 4000, 700, 29)}.items():
        snaps = dynamic_stream(n, T, base, churn, seed)
        ups = reference_graph_updates(snaps, n)
        out[f"{tag}/num_nodes"] = np.int32(n)
        out[f"{tag}/snap_edges"] = np.array([e for s in snaps for e in s], dtype=np.int32).reshape(-1, 2)
        out[f"{tag}/snap_sizes"] = np.array([len(s) for s in snaps], dtype=np.int32)
        for t in range(T):
            for kind in ("add", "delete"):
                out[f"{tag}/{t}/{kind}"] = np.array(ups[str(t)][kind], dtype=np.int32).reshape(-1, 2)
    np.savez_compressed(os.path.join(GOLD, "ref_updates.npz"), **out)
    print("wrote", os.path.join(GOLD, "ref_updates.npz"), len(out), "arrays")


def live_graph(n, e, seed):
    """Random directed graph of ``min(e, n*n)`` distinct edges (self loops allowed) for the randomized oracle tests."""
    rng = np.random.default_rng(seed)
    key = rng.choice(n * n, size=min(e, n * n), replace=False)
    return (key // n).astype(np.int32), (key % n).astype(np.int32)


def live_gcn_inputs(feat, n, e, seed):
    """Inputs of ``test_aggregation_oracle_equals_reference_kernels_live``: a random graph plus a star around vertex 0
    (one long row and many short ones), no self loops; ``(src, dst, edge_weight_by_eid, norm [N,1], h, grad_in)``."""
    src, dst = live_graph(n, e, seed)
    star = np.arange(1, n, dtype=np.int32)
    k = np.unique(np.concatenate([src.astype(np.int64) * n + dst, star.astype(np.int64) * n, star.astype(np.int64)]))
    src, dst = (k // n).astype(np.int32), (k % n).astype(np.int32)
    keep = src != dst
    src, dst = src[keep], dst[keep]
    rng = np.random.default_rng(seed + 7)
    w = rng.uniform(0.1, 1.0, size=src.shape[0]).astype(np.float32)
    norm = rng.uniform(0.2, 1.0, size=(n, 1)).astype(np.float32)
    h = rng.standard_normal((n, feat)).astype(np.float32)
    gin = rng.standard_normal((n, feat)).astype(np.float32)
    return src, dst, w, norm, h, gin


def live_gat_inputs(heads, dim, n, e, seed):
    """Inputs of ``test_stock_gat_oracle_equals_reference_kernels_live``: ``(src, dst, el, er, feat, grad_out)``."""
    src, dst = live_graph(n, e, seed)
    keep = src != dst
    src, dst = src[keep], dst[keep]
    rng = np.random.default_rng(seed + 11)
    f32 = lambda *s: rng.standard_normal(s).astype(np.float32)
    return (src, dst) + (f32(n, heads, 1), f32(n, heads, 1), f32(n, heads, dim), f32(n, heads, dim))


LIVE_GCN_CASES = (("gcn_f16", 16, False), ("gcn_f100", 100, False), ("gcn_f128", 128, False), ("gcnw_f7", 7, True))
LIVE_GCN_GRAPHS = ((12, 30, 0), (100, 1500, 1), (400, 6000, 2))
LIVE_GAT_CASES = (("gat_h2d4", 2, 4), ("gat_h8d16", 8, 16))
LIVE_GAT_GRAPHS = ((30, 150, 0), (200, 2500, 1))


def sample_rows(num_rows, row_width, seed, budget=2048):
    """Rows of one output kept in the fixture: the first and the last row plus a seeded sample, ~``budget`` values."""
    k = min(num_rows, max(4, budget // max(row_width, 1)))
    pick = np.random.default_rng(seed).choice(num_rows, size=k, replace=False)
    return np.unique(np.concatenate([[0, num_rows - 1], pick])).astype(np.int32)


def make_live_golden():
    """The reference kernels' outputs on the seeded inputs of the randomized oracle tests (``ref_kernels_live.npz``).

    The emitted kernels read only ``row_offsets``, ``column_indices`` and ``eids`` of a CSR (``node_ids`` is never
    indexed), and ``oracle/structure.py`` reproduces those three arrays of the reference's ``CSR::CSR`` bit for bit
    (``ref_structure.npz``), so the kernels run on the oracle's CSRs here.  Only a seeded sample of rows of every output
    is stored (``<key>/rows`` holds the row ids) to keep the fixture small; the inputs are rebuilt from their seeds."""
    from oracle import structure as S

    out = {}

    def run(case, tensors, grads, src, dst, n):
        kernels, lib = RE.load_case(case)
        ne = src.shape[0]
        fwd, bwd = S.forward_csr(src, dst, n), S.backward_csr(src, dst, n)
        for kern in kernels:
            for name, vt, shp in zip(kern["args"], kern["arg_types"], kern["arg_shapes"]):
                if name not in tensors:
                    lead = ne if vt == "EDGE" else n
                    tensors[name] = np.zeros([lead] + shp, np.float32) if name in kern["rets"] else grads.pop(0)
            RE.run_reference_kernel(lib, kern, tensors, fwd if kern["parallel_mode"] == "DstParallel" else bwd, n)
        return kernels

    def store(key, arr, seed):
        arr = arr.reshape(arr.shape[0], -1)
        rows = sample_rows(arr.shape[0], arr.shape[1], seed)
        out[f"{key}/rows"] = rows
        out[key] = arr[rows]

    for case, feat, weighted in LIVE_GCN_CASES:
        for n, e, seed in LIVE_GCN_GRAPHS:
            src, dst, w, norm, h, gin = live_gcn_inputs(feat, n, e, seed)
            tensors = {"Vhinb": h, "Vnormcen": norm, "Vnorminb": norm}
            if weighted:
                tensors["Vedge_weight"] = w.reshape(-1, 1).copy()
            kernels = run(case, tensors, [gin], src, dst, n)
            for kern in kernels:
                store(f"gcn/{case}/{n}_{e}_{seed}/{kern['direction']}", tensors[kern["rets"][0]], seed)
    for case, heads, dim in LIVE_GAT_CASES:
        for n, e, seed in LIVE_GAT_GRAPHS:
            src, dst, el, er, feat, gout = live_gat_inputs(heads, dim, n, e, seed)
            tensors = {"Velinb": el, "Vercen": er, "Vfeat_srcinb": feat}
            k0, k1, k2 = run(case, tensors, [gout], src, dst, n)
            rets = [tensors[r] for r in k2["rets"]]
            d_feat = [r for r in rets if r.shape[-1] == dim and r.ndim == 3 and r.shape[1] == heads][0]
            small = [r for r in rets if r.shape[-1] == 1]
            key = f"gat/{case}/{n}_{e}_{seed}"
            out[f"{key}/d_feat_abs_mean"] = np.float64(np.abs(d_feat.astype(np.float64)).mean())
            for role, arr in (("v3", tensors[k0["rets"][0]]), ("v4", tensors[k0["rets"][1]]), ("out", tensors[k1["rets"][0]]),
                              ("d_feat", d_feat), ("d_el", max(small, key=lambda x: float(np.abs(x).max()))),
                              ("d_er", min(small, key=lambda x: float(np.abs(x).max())))):
                store(f"{key}/{role}", arr, seed)
    np.savez_compressed(os.path.join(GOLD, "ref_kernels_live.npz"), **out)
    print("wrote", os.path.join(GOLD, "ref_kernels_live.npz"), len(out), "arrays")


def main():
    os.makedirs(GOLD, exist_ok=True)
    make_updates_golden()
    n, e = 40, 200
    src, dst = make_graph(n, e, 0)
    rng = np.random.default_rng(1)
    w = rng.uniform(0.1, 1.0, size=e).astype(np.float32)
    fwd, bwd = RE.reference_static_graph(src, dst, w, n)
    out = {"src": src, "dst": dst, "num_nodes": np.int32(n), "edge_weight_by_eid": w}
    for tag, c in (("fwd", fwd), ("bwd", bwd)):
        for f in ("row_offset", "column_indices", "eids", "node_ids", "in_degrees", "out_degrees", "weighted_out_degrees"):
            out[f"{tag}_{f}"] = getattr(c, f)
    # a graph with isolated vertices / empty rows and a multi-edge, for the row-offset back-fill path
    src2 = np.array([5, 5, 1, 7, 7, 7, 2], dtype=np.int32)
    dst2 = np.array([1, 3, 5, 1, 3, 9, 9], dtype=np.int32)
    f2, b2 = RE.reference_static_graph(src2, dst2, np.ones(7, np.float32), 12)
    out.update({"sparse_src": src2, "sparse_dst": dst2, "sparse_num_nodes": np.int32(12)})
    for tag, c in (("sparse_fwd", f2), ("sparse_bwd", b2)):
        for f in ("row_offset", "column_indices", "eids", "in_degrees", "out_degrees"):
            out[f"{tag}_{f}"] = getattr(c, f)
    np.savez_compressed(os.path.join(GOLD, "ref_structure.npz"), **out)

    kout = {}
    f32 = lambda *s: rng.standard_normal(s).astype(np.float32)
    norm = (rng.uniform(0.2, 1.0, size=(n, 1))).astype(np.float32)

    def run_case(case, inputs, grads):
        kernels, lib = RE.load_case(case)
        tensors = dict(inputs)
        for k in kernels:
            for name, vt, shp in zip(k["args"], k["arg_types"], k["arg_shapes"]):
                if name not in tensors:
                    lead = e if vt == "EDGE" else n
                    if name in k["rets"]:
                        tensors[name] = np.zeros([lead] + shp, np.float32)       # executor.new_zeros
                    else:                                                          # incoming gradient
                        tensors[name] = grads.pop(0)
            csr = fwd if k["parallel_mode"] == "DstParallel" else bwd
            launch = RE.run_reference_kernel(lib, k, tensors, csr, n)
            kout[f"{case}/{k['name']}/launch"] = np.array(launch, np.int32)
            kout[f"{case}/{k['name']}/args"] = np.array(k["args"])
            kout[f"{case}/{k['name']}/rets"] = np.array(k["rets"])
            kout[f"{case}/{k['name']}/mode"] = np.array(k["parallel_mode"])
            kout[f"{case}/{k['name']}/program"] = np.array(k["program"])
        for name, t in tensors.items():
            kout[f"{case}/tensor/{name}"] = t
        kout[f"{case}/kernels"] = np.array([k["name"] for k in kernels])

    h16 = f32(n, 16)
    run_case("gcn_f16", {"Vhinb": h16, "Vnormcen": norm, "Vnorminb": norm}, [f32(n, 16)])
    h7 = f32(n, 7)
    run_case("gcnw_f7", {"Vhinb": h7, "Vnormcen": norm, "Vnorminb": norm, "Vedge_weight": w.reshape(e, 1).copy()},
             [f32(n, 7)])
    for case, (hh, dd) in (("gat_h8d16", (8, 16)), ("gat_h2d4", (2, 4))):
        el, er, feat = f32(n, hh, 1), f32(n, hh, 1), f32(n, hh, dd)
        run_case(case, {"Velinb": el, "Vercen": er, "Vfeat_srcinb": feat}, [f32(n, hh, dd)])
    make_pcsr_golden()
    make_live_golden()
    np.savez_compressed(os.path.join(GOLD, "ref_kernels.npz"), **kout)
    print("wrote", os.path.join(GOLD, "ref_structure.npz"), "and ref_kernels.npz:", len(kout), "arrays")


if __name__ == "__main__":
    main()
