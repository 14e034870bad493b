"""Profiling driver: a few launches of the F=100 forward aggregation on the config-5 graph."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200 import kernels
from stgraph_b200.graph import StaticGraph
from stgraph_b200.utils import synthetic
dev = torch.device('cuda')
loc = float(sys.argv[1]) if len(sys.argv) > 1 else 0.9
F = int(sys.argv[2]) if len(sys.argv) > 2 else 100
d = synthetic.products_shaped(seed=0, device=dev, locality=loc)
n = d['num_nodes']
g = StaticGraph(torch.stack([d['src'], d['dst']], 1), None, n)
norm = g.degree_norm().reshape(-1)
x = torch.randn(n, F, device=dev); out = torch.empty_like(x)
plain = len(sys.argv) > 3 and sys.argv[3] == 'plain'
for _ in range(4):
    if plain:
        kernels.agg_scaled_sum(g.fwd_view(), x, norm, None, norm, out=out)
    else:   # packed {col, scale} metadata (what a static graph runs; the pack kernel is launch 0)
        kernels.agg_scaled_sum_graph(g._forward_graph, x, norm, None, norm, out=out)
torch.cuda.synchronize()
