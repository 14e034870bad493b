import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200.graph import GPMAGraph
from stgraph_b200.nn.pytorch import TGCN
from stgraph_b200.utils import synthetic
dev = torch.device('cuda'); n = 1_000_000; base, slide, T = 10_000_000, 100_000, 24
src, dst = synthetic.temporal_stream(n, base + slide * (T - 1), alpha=1.8, seed=0, device=dev)
snaps = [torch.stack([s, d], 1) for s, d in synthetic.sliding_window_snapshots(src, dst, base, slide, T)]
G = GPMAGraph(snaps, n)
model = TGCN(32, 64, fused=True).to(dev); opt = torch.optim.Adam(model.parameters(), lr=1e-2)
x = torch.randn(n, 32, device=dev)
def epoch():
    G.reset_graph(); h = None; cost = 0
    for t in range(len(snaps)):
        G.get_graph(t); G.set_ndata("norm", G.degree_norm())
        h = model(G, x, None, h); cost = cost + (h ** 2).mean()
        if (t + 1) % 12 == 0:
            opt.zero_grad(); cost.backward(); opt.step(); h, cost = h.detach(), 0
epoch(); torch.cuda.synchronize()
t0 = time.perf_counter(); epoch(); torch.cuda.synchronize(); print('epoch ms', (time.perf_counter() - t0) * 1e3, 'per step', (time.perf_counter() - t0) * 1e3 / T)
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    epoch(); torch.cuda.synchronize()
print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=22, max_name_column_width=60))
