"""Synthetic graphs shaped like the BASELINE.json configs (no network: no real datasets).

Stands in for ``stgraph.dataset`` on the measured path (the loaders there download
JSON; SURVEY.md section 2 #15).  All generators are seeded and run with torch ops,
so they work on CPU (tests, golden fixtures) and on the GPU (full-size bench inputs).

Shapes pinned by the reference's own tests:
Cora 2708 nodes / 10556 edges / 1433 feats / 7 classes
(``tests/dataset/static/test_CoraDataLoader.py:5-12``), WikiMaths 1068 nodes /
27079 edges / 731 timestamps (``tests/dataset/temporal/test_WikiMathDataLoader.py:6-11``).
"""
from __future__ import annotations

import math

import torch


def _gen(seed: int, device) -> torch.Generator:
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    return g


def _unique_pairs(a: torch.Tensor, b: torch.Tensor, directed: bool):
    """Drop self loops and duplicates; keeps first-seen order irrelevant (returns sorted keys order)."""
    keep = a != b
    a, b = a[keep], b[keep]
    if not directed:
        lo, hi = torch.minimum(a, b), torch.maximum(a, b)
        a, b = lo, hi
    key = a.to(torch.int64) * (1 << 32) + b.to(torch.int64)
    key = torch.unique(key)
    return (key >> 32), (key & 0xFFFFFFFF)


def uniform_undirected(num_nodes: int, num_pairs: int, seed: int = 0, device="cpu"):
    """``num_pairs`` distinct undirected pairs, symmetrised -> ``2*num_pairs`` directed edges (config 1, Cora-shaped)."""
    g = _gen(seed, device)
    a = torch.empty(0, dtype=torch.int64, device=device)
    b = a.clone()
    need = num_pairs
    while True:
        k = int(need * 1.3) + 16
        na = torch.randint(0, num_nodes, (k,), generator=g, device=device)
        nb = torch.randint(0, num_nodes, (k,), generator=g, device=device)
        a, b = _unique_pairs(torch.cat([a, na]), torch.cat([b, nb]), directed=False)
        if a.shape[0] >= num_pairs:
            break
        need = num_pairs - a.shape[0]
    perm = torch.randperm(a.shape[0], generator=g, device=device)[:num_pairs]
    a, b = a[perm], b[perm]
    src = torch.cat([a, b]).to(torch.int32)
    dst = torch.cat([b, a]).to(torch.int32)
    return src, dst


def uniform_directed(num_nodes: int, num_edges: int, seed: int = 0, device="cpu"):
    """``num_edges`` distinct directed edges without self loops (config 2, WikiMaths-shaped)."""
    g = _gen(seed, device)
    a = torch.empty(0, dtype=torch.int64, device=device)
    b = a.clone()
    need = num_edges
    while True:
        k = int(need * 1.3) + 16
        na = torch.randint(0, num_nodes, (k,), generator=g, device=device)
        nb = torch.randint(0, num_nodes, (k,), generator=g, device=device)
        a, b = _unique_pairs(torch.cat([a, na]), torch.cat([b, nb]), directed=True)
        if a.shape[0] >= num_edges:
            break
        need = num_edges - a.shape[0]
    perm = torch.randperm(a.shape[0], generator=g, device=device)[:num_edges]
    return a[perm].to(torch.int32), b[perm].to(torch.int32)


def _zipf_weights(num_nodes: int, alpha: float, max_frac: float, g, device, shuffle: bool = True):
    """Per-vertex sampling weights with a power-law tail: degree pdf ~ d^-alpha."""
    rank = torch.arange(1, num_nodes + 1, dtype=torch.float64, device=device)
    w = rank.pow(-1.0 / (alpha - 1.0))
    w = w / w.sum()
    if max_frac is not None:
        for _ in range(8):  # water-filling clip so no vertex exceeds max_frac of the endpoints
            w = torch.clamp(w, max=max_frac)
            w = w / w.sum()
    if shuffle:
        w = w[torch.randperm(num_nodes, generator=g, device=device)]
    return w


def _sample(cdf: torch.Tensor, k: int, g, device):
    u = torch.rand(k, generator=g, device=device, dtype=torch.float64)
    return torch.searchsorted(cdf, u).clamp_(max=cdf.shape[0] - 1)


def power_law_graph(num_nodes: int, num_edges: int, alpha: float = 2.1, symmetric: bool = True,
                    locality: float = 0.0, window: int = 4096, max_degree: int | None = None,
                    seed: int = 0, device="cpu"):
    """Power-law graph with optional community structure.

    ``locality`` = probability that an edge's second endpoint is drawn from a
    Laplace-distributed id offset of scale ``window`` around the first (vertex ids
    are ordered by community, as in a co-purchase graph stored in crawl order);
    the rest are drawn from the global power-law weights.  ``locality=0`` gives a
    locality-free graph.  ``symmetric=True`` emits both directions of every pair
    (ogbn-products-shaped, config 5); ``symmetric=False`` draws power-law *sources
    and destinations* (config 3: in-degree Zipf, clipped by ``max_degree``).
    Returns int32 ``(src, dst)`` with exactly ``num_edges`` distinct directed edges.
    """
    g = _gen(seed, device)
    pairs = num_edges // 2 if symmetric else num_edges
    max_frac = None
    if max_degree is not None:
        max_frac = max_degree / float(pairs * (2 if symmetric else 1))
    w = _zipf_weights(num_nodes, alpha, max_frac, g, device)
    cdf = torch.cumsum(w, 0)
    cdf = cdf / cdf[-1]
    a = torch.empty(0, dtype=torch.int64, device=device)
    b = a.clone()
    need = pairs
    while True:
        k = int(need * 1.15) + 1024
        u = _sample(cdf, k, g, device)
        v = _sample(cdf, k, g, device)
        if locality > 0:
            local = torch.rand(k, generator=g, device=device) < locality
            mag = -torch.log1p(-torch.rand(k, generator=g, device=device, dtype=torch.float64)) * window
            sign = torch.randint(0, 2, (k,), generator=g, device=device) * 2 - 1
            off = (mag.to(torch.int64) + 1) * sign
            vl = u + off
            # reflect at the borders
            vl = torch.where(vl < 0, -vl, vl)
            vl = torch.where(vl >= num_nodes, 2 * (num_nodes - 1) - vl, vl).clamp_(0, num_nodes - 1)
            v = torch.where(local, vl, v)
        a, b = _unique_pairs(torch.cat([a, u]), torch.cat([b, v]), directed=not symmetric)
        if a.shape[0] >= pairs:
            break
        need = pairs - a.shape[0]
    perm = torch.randperm(a.shape[0], generator=g, device=device)[:pairs]
    a, b = a[perm], b[perm]
    if symmetric:
        src = torch.cat([a, b])
        dst = torch.cat([b, a])
    else:
        src, dst = a, b   # b (destination) carries the clipped power-law in-degree
    return src.to(torch.int32), dst.to(torch.int32)


def cora_shaped(seed: int = 0, device="cpu"):
    """Config 1: N=2708, 5278 undirected pairs -> E=10556; X [N,1433] Bernoulli(18/1433) row-normalised; 7 classes."""
    n = 2708
    src, dst = uniform_undirected(n, 5278, seed=seed, device=device)
    g = _gen(seed + 1, device)
    x = (torch.rand(n, 1433, generator=g, device=device) < (18.0 / 1433.0)).float()
    x = x / x.sum(dim=1, keepdim=True).clamp_(min=1.0)
    labels = torch.randint(0, 7, (n,), generator=g, device=device)
    return {"num_nodes": n, "src": src, "dst": dst, "features": x, "labels": labels, "num_classes": 7}


def wikimaths_shaped(seed: int = 0, device="cpu", num_timestamps: int = 731, lags: int = 8):
    """Config 2: N=1068, E=27079 directed, weights U(0.1,1) in (dst,src) order, 731 snapshots, 8 lags."""
    n, e = 1068, 27079
    src, dst = uniform_directed(n, e, seed=seed, device=device)
    g = _gen(seed + 1, device)
    w = torch.rand(e, generator=g, device=device) * 0.9 + 0.1
    targets = torch.randn(num_timestamps, n, generator=g, device=device)
    return {"num_nodes": n, "src": src, "dst": dst, "edge_weight": w, "targets": targets,
            "num_timestamps": num_timestamps, "lags": lags}


def arxiv_shaped(seed: int = 0, device="cpu", scale: float = 1.0):
    """Config 3: N=169,343, E=1,166,243 directed, in-degree Zipf(2.1) clipped to 13k, 128 feats."""
    n = max(64, int(169343 * scale))
    e = max(256, int(1166243 * scale))
    src, dst = power_law_graph(n, e, alpha=2.1, symmetric=False, max_degree=max(16, int(13000 * scale)),
                               seed=seed, device=device)
    return {"num_nodes": n, "src": src, "dst": dst, "in_feats": 128, "heads": 8, "out_feats": 16}


def products_shaped(seed: int = 0, device="cpu", scale: float = 1.0, locality: float = 0.9, window: int = 8192):
    """Config 5: N=2,449,029, E=61,859,140 symmetric power-law, 100 feats (ogbn-products-shaped)."""
    n = max(64, int(2449029 * scale))
    e = max(256, int(61859140 * scale)) // 2 * 2
    src, dst = power_law_graph(n, e, alpha=2.4, symmetric=True, locality=locality, window=window,
                               max_degree=max(32, int(17500 * scale)), seed=seed, device=device)
    return {"num_nodes": n, "src": src, "dst": dst, "feats": 100, "num_classes": 47,
            "locality": locality, "window": window}


def temporal_stream(num_nodes: int, num_events: int, alpha: float = 1.8, seed: int = 0, device="cpu",
                    distinct: bool = False, max_frac: float | None = None):
    """Config 4 input: exactly ``num_events`` temporal edges with Zipf endpoints, no self loops
    (sx-mathoverflow / wiki-talk shaped; repeated interactions are frequent, snapshots de-duplicate them).

    ``distinct=True``: every (src, dst) pair occurs once in the stream, in random order, so that a sliding window of
    ``base`` events holds exactly ``base`` live edges and every slide adds and deletes exactly ``slide`` of them
    (SURVEY.md section 8(d) C4: ~10^7 live edges, +-10^5 per step); ``max_frac`` caps the share of the endpoints one
    vertex may take (a Zipf(1.8) head vertex would otherwise need more distinct partners than there are vertices)."""
    g = _gen(seed, device)
    w = _zipf_weights(num_nodes, alpha, max_frac, g, device)
    cdf = torch.cumsum(w, 0)
    cdf = cdf / cdf[-1]
    if distinct:
        keys = torch.empty(0, dtype=torch.int64, device=device)
        while keys.shape[0] < num_events:
            k = int((num_events - keys.shape[0]) * 1.3) + 4096
            u = _sample(cdf, k, g, device)
            v = _sample(cdf, k, g, device)
            keep = u != v
            keys = torch.unique(torch.cat([keys, u[keep] * num_nodes + v[keep]]))
        keys = keys[torch.randperm(keys.shape[0], generator=g, device=device)[:num_events]]
        return (keys // num_nodes).to(torch.int32), (keys % num_nodes).to(torch.int32)
    us, vs, have = [], [], 0
    while have < num_events:
        k = int((num_events - have) * 1.05) + 1024
        u = _sample(cdf, k, g, device)
        v = _sample(cdf, k, g, device)
        keep = u != v
        us.append(u[keep])
        vs.append(v[keep])
        have += int(keep.sum())
    u, v = torch.cat(us)[:num_events], torch.cat(vs)[:num_events]
    return u.to(torch.int32), v.to(torch.int32)


def sliding_window_snapshots(src, dst, base: int, slide: int, num_snapshots: int | None = None):
    """Snapshot t = events [t*slide, base + t*slide) (``benchmarking/dataset/preprocessing/preprocess_temporal_data.py:46-131``)."""
    total = int(src.shape[0])
    snaps = []
    t = 0
    while base + t * slide <= total and (num_snapshots is None or t < num_snapshots):
        lo, hi = t * slide, base + t * slide
        snaps.append((src[lo:hi], dst[lo:hi]))
        t += 1
    return snaps


def gcn_algorithmic_bytes(num_nodes: int, num_edges: int, feat: int, weighted: bool = False, elem_bytes: int = 4) -> int:
    """Compulsory traffic of one fused aggregation launch (SURVEY.md section 8(d)); ``elem_bytes`` is the size of one
    element of the feature rows read and written (2 for bf16 / fp16 rows; indices and scales stay 4 bytes)."""
    b = elem_bytes * 2 * num_nodes * feat + 4 * (num_edges + (num_nodes + 1) + 2 * num_nodes)
    if weighted:
        b += 4 * num_edges
    return b
