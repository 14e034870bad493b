"""A/B timing of the aggregation kernel variants on the config-5 graph (F=100 and F=128)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200 import kernels
from stgraph_b200.graph import StaticGraph
from stgraph_b200.utils import synthetic
dev = torch.device('cuda')
loc = float(os.environ.get('LOC', '0.9'))
d = synthetic.products_shaped(seed=0, device=dev, locality=loc)
n = d['num_nodes']; e = d['src'].shape[0]
g = StaticGraph(torch.stack([d['src'], d['dst']], 1), None, n)
norm = g.degree_norm().reshape(-1)
tag = ' '.join(f'{k}={v}' for k, v in os.environ.items() if k.startswith('STG_'))
for F in (100, 128, 64):
    x = torch.randn(n, F, device=dev); out = torch.empty_like(x)
    view = g.fwd_view()
    for _ in range(3): kernels.agg_scaled_sum(view, x, norm, None, norm, out=out)
    s = torch.cuda.Event(enable_timing=True); t = torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(10): kernels.agg_scaled_sum(view, x, norm, None, norm, out=out)
    t.record(); torch.cuda.synchronize()
    ms = s.elapsed_time(t) / 10
    b = synthetic.gcn_algorithmic_bytes(n, e, F)
    print(f'[{tag}] loc={loc} F={F}: {ms:.3f} ms alg {b/ms/1e6:.0f} GB/s ({b/ms/1e6/6549.4*100:.1f}%) gather {4*(e*F+n*F+e)/ms/1e6:.0f} GB/s', flush=True)
