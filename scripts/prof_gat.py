"""Profiling driver: fused edge-softmax GAT forward + backward on the arxiv-shaped graph (config 3)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200.graph import StaticGraph
from stgraph_b200.ops_gat import gat_edge_softmax_aggregate
from stgraph_b200.utils import synthetic
dev = torch.device('cuda')
d = synthetic.arxiv_shaped(seed=0, device=dev)
n = d['num_nodes']
g = StaticGraph(torch.stack([d['src'], d['dst']], 1), None, n)
feat = torch.randn(n, 8, 16, device=dev, requires_grad=True)
el = torch.randn(n, 8, 1, device=dev, requires_grad=True)
er = torch.randn(n, 8, 1, device=dev, requires_grad=True)
gout = torch.randn(n, 8, 16, device=dev)
for _ in range(int(sys.argv[1]) if len(sys.argv) > 1 else 3):
    y = gat_edge_softmax_aggregate(g, el, er, feat)
    y.backward(gout)
torch.cuda.synchronize()
print('hub rows fwd/bwd:', int(g._forward_graph._hub_count.item()), int(g._backward_graph._hub_count.item()),
      'max in/out degree', int(g.in_degrees_tensor().max()), int(g.out_degrees_tensor().max()))
