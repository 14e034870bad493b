"""Experiment: how does the aggregation time respond to neighbour locality (Laplace window)?"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200 import kernels
from stgraph_b200.graph import StaticGraph
from stgraph_b200.utils import synthetic
dev = torch.device('cuda')
for loc, win in ((1.0, 16), (1.0, 64), (0.95, 64), (0.9, 256), (0.9, 1024), (0.9, 8192), (0.9, 65536), (0.5, 8192)):
    d = synthetic.products_shaped(seed=0, device=dev, locality=loc, window=win)
    n = d['num_nodes']; e = d['src'].shape[0]
    g = StaticGraph(torch.stack([d['src'], d['dst']], 1), None, n)
    norm = g.degree_norm().reshape(-1)
    F = 100
    x = torch.randn(n, F, device=dev); out = torch.empty_like(x)
    view = g.fwd_view()
    for _ in range(3): kernels.agg_scaled_sum(view, x, norm, None, norm, out=out)
    s = torch.cuda.Event(enable_timing=True); t = torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(10): kernels.agg_scaled_sum(view, x, norm, None, norm, out=out)
    t.record(); torch.cuda.synchronize()
    ms = s.elapsed_time(t) / 10
    b = synthetic.gcn_algorithmic_bytes(n, e, F)
    print(f'loc={loc} win={win}: {ms:.3f} ms alg {b/ms/1e6:.0f} GB/s ({b/ms/1e6/6549.4*100:.1f}%) gather {4*(e*F+n*F+e)/ms/1e6:.0f} GB/s maxdeg {int(g.in_degrees_tensor().max())}', flush=True)
    del g, x, out, d
