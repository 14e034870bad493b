import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200 import kernels
from stgraph_b200.graph import StaticGraph
from stgraph_b200.utils import synthetic
dev = torch.device('cuda')
for loc in (0.9, 0.0):
    t0 = time.time()
    d = synthetic.products_shaped(seed=0, device=dev, locality=loc)
    torch.cuda.synchronize(); t1 = time.time()
    n = d['num_nodes']; e = d['src'].shape[0]
    g = StaticGraph(torch.stack([d['src'], d['dst']], 1), None, n)
    torch.cuda.synchronize(); t2 = time.time()
    print(f'locality={loc} N={n} E={e} gen {t1-t0:.2f}s build {t2-t1:.2f}s maxdeg {int(g.in_degrees_tensor().max())} hubs {int(g._forward_graph._hub_count.item())}')
    norm = g.degree_norm().reshape(-1)
    for F in (100, 16, 128, 48):
        x = torch.randn(n, F, device=dev); out = torch.empty_like(x)
        for view, nm in ((g.fwd_view(), 'fwd'), (g.bwd_view(), 'bwd')):
            for _ in range(3): kernels.agg_scaled_sum(view, x, norm, None, norm, out=out)
            s = torch.cuda.Event(enable_timing=True); t = torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(10): kernels.agg_scaled_sum(view, x, norm, None, norm, out=out)
            t.record(); torch.cuda.synchronize()
            ms = s.elapsed_time(t) / 10
            b = synthetic.gcn_algorithmic_bytes(n, e, F)
            print(f'  F={F} {nm}: {ms:.3f} ms  alg {b/ms/1e6:.0f} GB/s ({b/ms/1e6/6549.4*100:.1f}%)  gather-model {4*(e*F+n*F+e)/ms/1e6:.0f} GB/s')
