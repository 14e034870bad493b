"""A/B on the config-5 graph: plain kernel, plain kernel without the neighbour-scale gather, packed {col, scale} kernel."""
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
w = torch.rand(e, device=dev) + 0.5


def timed(fn, reps=10):
    for _ in range(3): fn()
    s = torch.cuda.Event(enable_timing=True); t = torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps): fn()
    t.record(); torch.cuda.synchronize()
    return s.elapsed_time(t) / reps


for F in [int(f) for f in os.environ.get('FEATS', '100,128,64,16,47').split(',')]:
    x = torch.randn(n, F, device=dev); out = torch.empty_like(x)
    b = synthetic.gcn_algorithmic_bytes(n, e, F)
    for dname, csr in (('fwd', g._forward_graph), ('bwd', g._backward_graph)):
        view = csr.view()
        meta = kernels.pack_edge_meta(view, norm, None)
        meta_w = kernels.pack_edge_meta(view, norm, w)
        res = {
            'plain': timed(lambda: kernels.agg_scaled_sum(view, x, norm, None, norm, out=out)),
            'plain_no_ns': timed(lambda: kernels.agg_scaled_sum(view, x, None, None, norm, out=out)),
            'packed': timed(lambda: kernels.agg_packed_sum(view, meta, x, norm, out=out)),
            'plain_w': timed(lambda: kernels.agg_scaled_sum(view, x, norm, w, norm, out=out)),
            'packed_w': timed(lambda: kernels.agg_packed_sum(view, meta_w, x, norm, out=out)),
            'pack': timed(lambda: kernels.pack_edge_meta(view, norm, None, out=meta)),
        }
        xp = kernels.padded_rows(n, F, dev); xp.copy_(x)
        op = kernels.padded_rows(n, F, dev)
        res['packed_padded'] = timed(lambda: kernels.agg_packed_sum(view, meta, xp, norm, out=op))
        res['packed_padded_in'] = timed(lambda: kernels.agg_packed_sum(view, meta, xp, norm, out=out))
        assert torch.equal(op, kernels.agg_packed_sum(view, meta, x, norm)), 'padded layout changed the result'
        del xp, op
        same = torch.equal(kernels.agg_scaled_sum(view, x, norm, None, norm), kernels.agg_packed_sum(view, meta, x, norm))
        print(f'pair={os.environ.get("STG_AGG_PAIR", "1")} loc={loc} F={F} {dname}: ' + ' '.join(f'{k}={v:.3f}ms' for k, v in res.items())
              + f' | packed: alg {b/res["packed"]/1e6:.0f} GB/s ({b/res["packed"]/1e6/6549.4*100:.1f}%)'
              + f' gather {4*(e*F+n*F+2*e)/res["packed"]/1e6:.0f} GB/s bit-identical={same}', flush=True)
        del meta, meta_w
