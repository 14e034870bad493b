"""Device time of the fused edge-softmax kernels on the arxiv-shaped graph (config 3): raw C-ABI calls on
preallocated buffers, 20 back-to-back iterations between two CUDA events (no per-call Python allocation)."""
import ctypes, json, os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200 import _lib, ops_gat
from stgraph_b200.graph import StaticGraph
from stgraph_b200.utils import synthetic
dev = torch.device('cuda')
d = synthetic.arxiv_shaped(seed=0, device=dev)
n, e = d['num_nodes'], int(d['src'].shape[0])
g = StaticGraph(torch.stack([d['src'], d['dst']], 1), None, n)
H, D = 8, 16
feat = torch.randn(n, H, D, device=dev); el = torch.randn(n, H, device=dev); er = torch.randn(n, H, device=dev)
gout = torch.randn(n, H, D, device=dev)
out = torch.empty_like(feat); rmax = torch.empty(n, H, device=dev); rsum = torch.empty_like(rmax)
dfeat = torch.empty_like(feat); d_el = torch.empty_like(el); d_er = torch.empty_like(er); dot = torch.empty_like(el)
vf, vb = ops_gat._views(g)
st = _lib.current_stream_ptr()
fwd = lambda: _lib.call("stg_gat_softmax_fwd_f32", ctypes.byref(vf), el.data_ptr(), er.data_ptr(), feat.data_ptr(), H, D, 0.2,
                        out.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), st)
bwd = lambda: _lib.call("stg_gat_softmax_bwd_f32", ctypes.byref(vf), ctypes.byref(vb), el.data_ptr(), er.data_ptr(), feat.data_ptr(),
                        out.data_ptr(), gout.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), H, D, 0.2, dfeat.data_ptr(),
                        d_el.data_ptr(), d_er.data_ptr(), dot.data_ptr(), st)


def timed(fn, reps=20):
    for _ in range(3): fn()
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


hd = H * D
b_fwd = 4 * (2 * n * hd + 4 * n * H + e + n + 1)
b_bwd = 4 * (4 * n * hd + 6 * n * H + 2 * (e + n + 1))
tf, tb = timed(fwd), timed(bwd)
print(json.dumps({"gat_hub_threshold": ops_gat.GAT_HUB_THRESHOLD, "fwd_ms": tf, "bwd_ms": tb, "fwd_alg_gbs": b_fwd / tf / 1e6,
                  "bwd_alg_gbs": b_bwd / tb / 1e6, "fwd_frac_hbm": b_fwd / tf / 1e6 / 6549.4, "bwd_frac_hbm": b_bwd / tb / 1e6 / 6549.4,
                  "gather_fwd_gbs": 4.0 * e * hd / tf / 1e6}))
