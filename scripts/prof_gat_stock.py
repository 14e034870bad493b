import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200.graph import StaticGraph
from stgraph_b200.nn.pytorch import GATConv
from stgraph_b200.utils import synthetic
dev = torch.device('cuda')
d = synthetic.arxiv_shaped(seed=0, device=dev)
n = d['num_nodes']
g = StaticGraph(torch.stack([d['src'], d['dst']], 1), None, n)
x = torch.randn(n, 128, device=dev); gout = torch.randn(n, 8, 16, device=dev)
layer = GATConv(128, 16, 8).to(dev)
for _ in range(3):
    layer.zero_grad(); y = layer(g, x); y.backward(gout)
torch.cuda.synchronize()
