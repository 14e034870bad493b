"""Single-GPU timing of one rank's share of the 8-way partitioned aggregation (no communication):
own-source pass, halo-source pass, alone and concurrently -- isolates kernel efficiency at slice size."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200 import _lib, kernels
from stgraph_b200.dist.partition import edge_balanced_bounds
from stgraph_b200.graph import StaticGraph
from stgraph_b200.graph.static.csr import HUB_THRESHOLD
from stgraph_b200.utils import synthetic

dev = torch.device('cuda'); P = int(sys.argv[1]) if len(sys.argv) > 1 else 8; F = 100
d = synthetic.products_shaped(seed=0, device=dev)
n = d['num_nodes']
g = StaticGraph(torch.stack([d['src'], d['dst']], 1), None, n)
norm = g.degree_norm().reshape(-1).contiguous()
x = torch.randn(n, F, device=dev)
csr = g._forward_graph
bounds = edge_balanced_bounds(csr.row_offset, P)
keep = []
USE_QUEUE = os.environ.get('STG_SLICE_QUEUE', '1') != '0'

def mkview(ro, cols, n_rows):
    cap = int(cols.shape[0]) // HUB_THRESHOLD + 1
    hr = torch.empty(cap, dtype=torch.int32, device=dev); hc = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.call("stg_csr_hub_rows", ro.data_ptr(), n_rows, HUB_THRESHOLD, hr.data_ptr(), cap, hc.data_ptr(), _lib.current_stream_ptr())
    has = int(hc.item()) > 0
    keep.append((hr, hc, ro, cols))
    v = _lib.StgCsrView()
    v.row_offset, v.column_indices, v.eids, v.node_ids = ro.data_ptr(), cols.data_ptr(), None, None
    v.num_nodes, v.num_edges, v.eid_base, v.eids_identity = n_rows, int(cols.shape[0]), 0, 1
    v.hub_rows = hr.data_ptr() if has else None; v.hub_count = hc.data_ptr() if has else None
    v.hub_threshold = HUB_THRESHOLD if has else 0; v.hub_capacity = cap if has else 0
    if USE_QUEUE:
        q = torch.zeros(2, dtype=torch.int32, device=dev); keep.append(q); v.work_queue = q.data_ptr()
    return v

def timeit(fn, reps=20):
    for _ in range(3): fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps

for rank in (0, P // 2):
    lo, hi = bounds[rank], bounds[rank + 1]
    ro = csr.row_offset[lo:hi + 1].long(); e0, e1 = int(ro[0]), int(ro[-1])
    cols = csr.column_indices[e0:e1].long()
    local = (cols >= lo) & (cols < hi)
    halo_ids = torch.unique(cols[~local])
    nr = hi - lo
    rows = torch.repeat_interleave(torch.arange(nr, device=dev), ro[1:] - ro[:-1])
    def sub(m, vals):
        cnt = torch.bincount(rows[m], minlength=nr)
        sro = torch.zeros(nr + 1, dtype=torch.int32, device=dev); sro[1:] = torch.cumsum(cnt, 0).int()
        return sro.contiguous(), vals[m].int().contiguous()
    oro, ocols = sub(local, cols - lo)
    hro, hcols = sub(~local, torch.searchsorted(halo_ids, cols))
    v_own, v_halo = mkview(oro, ocols, nr), mkview(hro, hcols, nr)
    v_all = mkview((ro - e0).int().contiguous(), cols.int().contiguous(), nr)
    x_own = x[lo:hi].contiguous(); halo = x[halo_ids].contiguous()
    ns_own, ns_halo, rs = norm[lo:hi].contiguous(), norm[halo_ids].contiguous(), norm[lo:hi].contiguous()
    out = torch.empty(nr, F, device=dev)
    side = torch.cuda.Stream(priority=-1)
    t_all = timeit(lambda: kernels.agg_scaled_sum(v_all, x, norm, None, rs, out=out))
    t_own = timeit(lambda: kernels.agg_scaled_sum(v_own, x_own, ns_own, None, rs, out=out))
    t_own_red = timeit(lambda: kernels.agg_scaled_sum(v_own, x_own, ns_own, None, rs, out=out, accumulate="red"))
    t_halo_rmw = timeit(lambda: kernels.agg_scaled_sum(v_halo, halo, ns_halo, None, rs, out=out, accumulate=True))
    t_halo_red = timeit(lambda: kernels.agg_scaled_sum(v_halo, halo, ns_halo, None, rs, out=out, accumulate="red"))
    def both():
        cur = torch.cuda.current_stream()
        out.zero_()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            kernels.agg_scaled_sum(v_halo, halo, ns_halo, None, rs, out=out, accumulate="red", stream=side.cuda_stream)
        kernels.agg_scaled_sum(v_own, x_own, ns_own, None, rs, out=out, accumulate="red")
        cur.wait_stream(side)
    t_both = timeit(both)
    t_zero = timeit(lambda: out.zero_())
    print(f"P={P} rank {rank}: rows {nr} own_edges {int(ocols.shape[0])} halo_edges {int(hcols.shape[0])} halo_rows {int(halo_ids.shape[0])} | "
          f"all-edges(global x) {t_all:.3f}  own {t_own:.3f}  own_red {t_own_red:.3f}  halo_rmw {t_halo_rmw:.3f}  halo_red {t_halo_red:.3f}  "
          f"zero+both_concurrent {t_both:.3f}  zero {t_zero:.3f} ms", flush=True)
