#!/usr/bin/env python
"""Benchmark of the hot path: fused GCN neighbour aggregation (forward + backward) on the
ogbn-products-shaped synthetic graph of BASELINE.json (config 5: 2,449,029 V / 61,859,140 E, F=100).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference ...                     # CPU reference (torch index_add), rank 0 only

One step = one forward aggregation over the in-edge CSR + one backward aggregation over the
out-edge CSR (SURVEY.md section 8(d): "primary measurement = the F=100 aggregation fwd+bwd").
``value`` = algorithmic bytes of the whole job / max-over-ranks device time (GB/s); ``e2e`` = the same
with HOST buffers (H2D of the step's inputs and D2H of its results inside the timed region);
``roofline`` = the forward launch against the measured HBM peak (per GPU); ``cpu_baseline`` = the oracle
port on the host cores; ``reference_gpu`` = the reference's own emitted kernels on the same inputs.
At N>1 the vertices are partitioned (cost-balanced, contiguous), every rank aggregates its own rows and the
remote source rows travel as halo over NVLink (``stgraph_b200/dist``): strong scaling, total work fixed.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "gcn_fused_aggregation_fwd_bwd_algorithmic_hbm_gbs"
UNIT = "GB/s"
FEAT = 100
WORKLOAD = "config5: GCN aggregation fwd+bwd, ogbn-products-shaped synthetic graph"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=float(os.environ.get("STG_BENCH_SCALE", "1.0")),
                    help="shrink the graph (debug only; the judged number is scale=1)")
    ap.add_argument("--locality", type=float, default=0.9)
    ap.add_argument("--window", type=int, default=8192)
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / e2e / reference_gpu / other-config legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's forward and backward aggregation as DIR/fwd_aggregate.npy "
                         "and DIR/bwd_aggregate.npy (float32; a fixed seeded sample of rows when the arrays exceed 60 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return args


DUMP_BYTES = 60_000_000     # all arrays --dump-outputs writes, together


def dump_rows(num_rows, row_bytes, n_arrays):
    """Row ids --dump-outputs writes: every row when the arrays fit in DUMP_BYTES, else a fixed seeded sample (sorted),
    the same for every run and build with the same graph size."""
    cap = DUMP_BYTES // (row_bytes * n_arrays)
    if num_rows <= cap:
        return torch.arange(num_rows)
    return torch.randperm(num_rows, generator=torch.Generator().manual_seed(0))[:cap].sort().values


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes per forward launch (row + hub kernel) from this round's ncu capture of the same command
    (profiles/r02_traffic.json; single GPU only -- a rank of a partitioned run walks 1/N of the rows)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get("fwd_launch_dram_bytes")
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(args, dev):
    from stgraph_b200.utils import synthetic

    return synthetic.products_shaped(seed=0, device=dev, scale=args.scale, locality=args.locality, window=args.window)


# ----------------------------------------------------------------------------------------------- CPU reference
class CpuReference:
    """The reference's GPU-only vertex program restated as torch-CPU ``index_add_`` (oracle/aggregate.py, fp32), on
    the WHOLE graph, both directions, all host threads.  The edge list is walked in destination-row blocks of
    ~``block_edges`` edges so that the gathered [edges, F] message tensor stays bounded (the full one is 24.7 GB);
    every edge of the graph is still aggregated every step."""

    def __init__(self, src, dst, n, feat, block_edges=4_000_000, threads=None):
        import numpy as np

        self.threads = threads or os.cpu_count()
        torch.set_num_threads(self.threads)
        self.n, self.feat = n, feat
        dev = src.device                      # torch ops only (sort on the GPU when there is one): no product code
        key_f = dst.to(torch.int64) * n + src.to(torch.int64)
        key_b = src.to(torch.int64) * n + dst.to(torch.int64)
        self.dirs = []
        for key in (key_f, key_b):
            k = torch.sort(key).values
            rows = (k // n)
            cols = (k % n).cpu()
            deg = torch.bincount(rows, minlength=n).cpu()
            ro = torch.zeros(n + 1, dtype=torch.int64)
            ro[1:] = torch.cumsum(deg, 0)
            ro_np = ro.numpy()
            cuts = [0]
            while cuts[-1] < n:
                nxt = int(np.searchsorted(ro_np, ro_np[cuts[-1]] + block_edges, side="left"))
                cuts.append(min(max(nxt, cuts[-1] + 1), n))
            self.dirs.append((ro_np, cols.numpy(), cuts))
            del k, rows
        self.num_edges = int(src.shape[0])
        g = torch.Generator().manual_seed(1)
        self.x = torch.randn(n, feat, generator=g)
        self.gout = torch.randn(n, feat, generator=g)
        indeg = (torch.from_numpy(self.dirs[0][0][1:] - self.dirs[0][0][:-1])).float()
        self.norm = torch.where(indeg > 0, indeg.pow(-0.5), torch.zeros_like(indeg))
        self.out = torch.empty(n, feat)

    def aggregate(self, d, x, max_rows=None):
        from oracle import aggregate as A

        ro, cols, cuts = self.dirs[d]
        edges = 0
        for a, b in zip(cuts[:-1], cuts[1:]):
            if max_rows is not None and a >= max_rows:
                break
            e0, e1 = int(ro[a]), int(ro[b])
            self.out[a:b] = A.scaled_sum(ro[a:b + 1] - e0, cols[e0:e1], None, x, self.norm, None, self.norm[a:b],
                                         dtype=torch.float32)
            edges += e1 - e0
        return edges

    def step(self):
        self.aggregate(0, self.x)
        self.aggregate(1, self.gout)


def run_reference(args):
    """--impl reference: same graph (same generator stream when a GPU is there to run it), same F, forward + backward."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from stgraph_b200.utils import synthetic

    gen_dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    d = synthetic.products_shaped(seed=0, device=gen_dev, scale=args.scale, locality=args.locality, window=args.window)
    n, e = d["num_nodes"], int(d["src"].shape[0])
    ref = CpuReference(d["src"], d["dst"], n, FEAT)
    del d
    if torch.cuda.is_available():
        torch.cuda.empty_cache()
    b_step = 2 * synthetic.gcn_algorithmic_bytes(n, e, FEAT)
    ts = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        ref.step()
        if i >= args.warmup:
            ts.append(time.perf_counter() - t0)
    t_step = sum(ts) / len(ts)
    value = b_step / t_step / 1e9
    sample = (f"the whole workload every step: forward + backward torch-CPU index_add (fp32) over all {e} edges x 2 directions, "
              f"F={FEAT}, in destination-row blocks of ~4M edges (bounded memory), {ref.threads} threads")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "num_nodes": n, "num_edges": e, "feat": FEAT, "locality": args.locality,
                       "window": args.window, "scale": args.scale, "graph_generated_on": str(gen_dev),
                       "same_graph_as_cuda_arm": gen_dev.type == "cuda"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------ the reference's own GPU kernels
def reference_gpu_leg(graph, x, gout, norm, out_f, out_b, feat):
    """The CUDA kernels the reference's code generator emits for GCNConv (K0 forward, K1 backward), built by
    oracle/build_ref.py as generic compute_100 code like its JIT would, launched with the reference's own geometry
    (execution_unit.py:92-106) on the SAME inputs; baseline only, nothing of the product runs through it."""
    import ctypes

    from oracle import ref_emulate as RE

    case = f"gcn_f{feat}"
    so = os.path.join(RE.REF_DIR, case + "_gpu.so")
    if not os.path.exists(so):
        return {"unavailable": f"{os.path.relpath(so, ROOT)} not built (oracle/build_ref.py needs /root/reference)"}
    kernels_meta, _ = RE.load_case(case)
    lib = ctypes.CDLL(so)
    n = graph.get_num_nodes()
    norm2 = norm.reshape(-1, 1).contiguous()
    res = {}
    stream = torch.cuda.current_stream().cuda_stream
    total = 0.0
    for k in kernels_meta:
        fwd = k["parallel_mode"] == "DstParallel"
        csr = graph._forward_graph if fwd else graph._backward_graph
        ours = out_f if fwd else out_b
        src_t = x if fwd else gout
        ref_out = torch.zeros(n, feat, device=x.device)
        tensors = {name: (ref_out if name in k["rets"] else norm2 if "norm" in name else src_t) for name in k["args"]}
        arr = (ctypes.c_void_p * len(k["args"]))(*[ctypes.c_void_p(tensors[a].data_ptr()) for a in k["args"]])
        nblks, nthrs, group, npb = RE.reference_launch_params(feat, n)
        fn = getattr(lib, "launch_" + k["name"])
        fn.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int] * 7 + [ctypes.c_void_p]

        def launch():
            rc = fn(arr, csr.row_offset.data_ptr(), csr.eids.data_ptr(), csr.column_indices.data_ptr(),
                    csr.node_ids.data_ptr(), n, feat, 1, group, npb, nblks, nthrs, stream)
            assert rc == 0, rc

        for _ in range(2):
            launch()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            launch()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 5
        scale = float(ours.abs().max())
        res[k["direction"]] = {"kernel": k["name"], "ms": ms, "launch": [nblks, nthrs, group, npb],
                               "max_abs_diff_vs_ours_over_max": float((ours - ref_out).abs().max()) / max(scale, 1e-30)}
        total += ms
        del ref_out
    res["ms_per_step"] = total
    res["kind"] = "the reference's emitted K0/K1 (tpl_fa_csr_unsorted.jinja) compiled as compute_100 PTX, CUDA events, 5 launches"
    return res


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from stgraph_b200 import kernels
    from stgraph_b200.dist import PartitionedGraph
    from stgraph_b200.graph import StaticGraph
    from stgraph_b200.utils import synthetic

    d = make_workload(args, dev)
    if world > 1:   # every rank must hold the same graph: rank 0's
        dist.broadcast(d["src"], src=0)
        dist.broadcast(d["dst"], src=0)
    n, e = d["num_nodes"], int(d["src"].shape[0])
    graph = StaticGraph(torch.stack([d["src"], d["dst"]], 1), None, n)
    norm = graph.degree_norm().reshape(-1).contiguous()
    gen = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(n, FEAT, device=dev, generator=gen)
    gout = torch.randn(n, FEAT, device=dev, generator=gen)
    b_alg_one = synthetic.gcn_algorithmic_bytes(n, e, FEAT)
    b_alg_step = 2 * b_alg_one

    halo_info = parity = segments = None
    if world > 1:
        pg = PartitionedGraph(graph, rank, world)
        lo, hi = pg.own_lo, pg.own_hi
        # single-GPU result of this rank's rows, to check the partitioned path after the warm-up steps
        ref_rows = kernels.agg_scaled_sum(graph.fwd_view(), x, norm, None, norm)[lo:hi].clone()
        mag_rows = kernels.agg_scaled_sum(graph.fwd_view(), x.abs(), norm, None, norm)[lo:hi].clone()
        x_own, g_own = x[lo:hi].clone(), gout[lo:hi].clone()
        nl = norm[lo:hi].contiguous()
        out_f = torch.empty(pg.n_own, FEAT, device=dev)
        out_b = torch.empty(pg.n_own, FEAT, device=dev)
        ex_f, ex_b = pg.exchange("fwd", FEAT, nl), pg.exchange("bwd", FEAT, nl)
        hf = ex_f.plan
        halo_info = {"mode": {"ce": "halo rows packed by our gather kernel and shipped by the copy engines into the peers' "
                                    "symmetric-memory halo buffers during the own-source pass, arrival flags instead of a "
                                    "barrier, then the halo-source pass; no NCCL on the data path",
                              "sm": "halo rows pushed by our SM kernel (posted NVLink stores) during the own-source pass, "
                                    "arrival flags, then the halo-source pass; no NCCL on the data path"}[ex_f.mode],
                     "halo_rows_fwd": hf.n_halo, "halo_rows_bwd": ex_b.plan.n_halo, "own_rows": pg.n_own,
                     "full_allgather_rows": n - pg.n_own, "halo_edges_fwd": int(hf.halo_cols.shape[0]),
                     "own_edges_fwd": int(hf.own_cols.shape[0]), "bounds": pg.bounds}
        del x, gout

        def step(ev=None):
            if ev:
                ev[0].record()
            pg.aggregate("fwd", x_own, nl, nl, out=out_f)
            if ev:
                ev[1].record()
            pg.aggregate("bwd", g_own, nl, nl, out=out_b)
    else:
        out_f = torch.empty_like(x)
        out_b = torch.empty_like(x)
        vf, vb = graph.fwd_view(), graph.bwd_view()
        # the public path of a static graph (GCNConv -> executor -> kernels.agg_scaled_sum_graph): the {col, scale}
        # array of this norm is packed on the first (warm-up) call and reused, like the CSR arrays themselves
        fcsr, bcsr = graph._forward_graph, graph._backward_graph

        def step(ev=None):
            if ev:
                ev[0].record()
            kernels.agg_scaled_sum_graph(fcsr, x, norm, None, norm, out=out_f)
            if ev:
                ev[1].record()
            kernels.agg_scaled_sum_graph(bcsr, gout, norm, None, norm, out=out_b)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    if world > 1:
        torch.cuda.synchronize()
        ex_f.check()
        ex_b.check()
        ok = bool(((out_f - ref_rows).abs() <= 1e-5 * mag_rows + 1e-30).all())
        t_ok = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        parity = bool(int(t_ok.item()))
        assert parity, "partitioned aggregation disagrees with the single-GPU result"
        del ref_rows, mag_rows
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = kernels.launch_count
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_beg.record()
    for i in range(args.steps):
        step(kev[i])
    t_end.record()
    barrier()
    launches = kernels.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # out_f / out_b still hold the last timed step's results: the legs below reuse these buffers
        import numpy as np

        rows = dump_rows(n, FEAT * out_f.element_size(), 2)
        dumped = {}
        for name, out in (("fwd_aggregate", out_f), ("bwd_aggregate", out_b)):
            if world > 1:   # every rank holds a contiguous, ascending range of rows
                mine = rows[(rows >= lo) & (rows < hi)]
                parts = [None] * world
                dist.all_gather_object(parts, out[(mine - lo).to(dev)].cpu())
                dumped[name] = torch.cat(parts)
            else:
                dumped[name] = out[rows.to(dev)].cpu()
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, t in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), t.numpy())
        del dumped
    ms_total = t_beg.elapsed_time(t_end)
    ms_fwd_kernel = sum(a.elapsed_time(b) for a, b in kev) / args.steps
    ms_fwd_own = ms_fwd_kernel
    if world > 1:
        t = torch.tensor([ms_total, ms_fwd_kernel], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_fwd_kernel = float(t[0]), float(t[1])
        # per-rank device time of every segment of one aggregation (untimed extra iterations)
        ex_f.profile, ex_b.profile = [], []
        for _ in range(6):
            step()
        summ = {"rank": rank, "fwd": ex_f.profile_summary(), "bwd": ex_b.profile_summary(), "rows": pg.n_own,
                "own_edges_fwd": int(hf.own_cols.shape[0]), "halo_edges_fwd": int(hf.halo_cols.shape[0]),
                "halo_rows_in_fwd": hf.n_halo, "rows_sent_fwd": int(hf.send_index.numel()), "fwd_aggregate_ms": ms_fwd_own}
        ex_f.profile = ex_b.profile = None
        allsum = [None] * world
        dist.all_gather_object(allsum, summ)
        segments = [{k: (round(v, 4) if isinstance(v, float) else ({a: round(b, 4) for a, b in v.items()} if isinstance(v, dict) else v))
                     for k, v in s.items()} for s in allsum]
    ms_step = ms_total / args.steps
    value = b_alg_step / (ms_step * 1e-3) / 1e9

    extras = {}
    # ---- end to end with HOST buffers: every step copies its inputs host->device and its results device->host ----
    if not args.no_extras:
        k = max(3, min(args.steps, 8))
        if world == 1:
            xh, gh, nh = x.cpu().pin_memory(), gout.cpu().pin_memory(), norm.cpu().pin_memory()
            oh, oh2 = torch.empty(n, FEAT).pin_memory(), torch.empty(n, FEAT).pin_memory()
            scratch = torch.empty(kernels.host_scratch_bytes(n, e, FEAT), dtype=torch.uint8, device=dev)
            scratch2 = torch.empty_like(scratch)
            for _ in range(2):
                kernels.agg_scaled_sum_host(vf, xh, oh, scratch, nh, None, nh)
            torch.cuda.synchronize()
            # (a) one blocking call after the other: H2D, kernel, D2H strictly in sequence
            t0 = time.perf_counter()
            for _ in range(k):
                kernels.agg_scaled_sum_host(vf, xh, oh, scratch, nh, None, nh)
                kernels.agg_scaled_sum_host(vb, gh, oh2, scratch, nh, None, nh)
            torch.cuda.synchronize()
            e2e_serial_ms = (time.perf_counter() - t0) / k * 1e3
            # (b) the forward and the backward call enqueued on two streams (two scratch buffers): one call's H2D
            # overlaps the other's D2H; every step still copies all of its inputs in and all of its results out
            sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
            for _ in range(2):
                kernels.agg_scaled_sum_host(vf, xh, oh, scratch, nh, None, nh, stream=sa)
                kernels.agg_scaled_sum_host(vb, gh, oh2, scratch2, nh, None, nh, stream=sb)
            torch.cuda.synchronize()
            oh.zero_()
            t0 = time.perf_counter()
            for _ in range(k):
                kernels.agg_scaled_sum_host(vf, xh, oh, scratch, nh, None, nh, stream=sa)
                kernels.agg_scaled_sum_host(vb, gh, oh2, scratch2, nh, None, nh, stream=sb)
            sa.synchronize()
            sb.synchronize()
            e2e_ms = (time.perf_counter() - t0) / k * 1e3
            h2d = 2 * (n * FEAT * 4 + 2 * n * 4)
            d2h = 2 * n * FEAT * 4
            extras["e2e"] = {"value": b_alg_step / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": e2e_ms,
                             "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                             "api": "stg_agg_scaled_sum_f32_host_async: forward and backward calls on two streams (pinned host "
                                    "buffers; H2D + kernels + D2H per call, one call's H2D overlapping the other's D2H)",
                             "blocking_calls_ms_per_step": e2e_serial_ms,
                             "blocking_calls_value": b_alg_step / (e2e_serial_ms * 1e-3) / 1e9}
            assert torch.equal(oh, out_f.cpu()), "host-buffer path and device path disagree"
            del scratch, scratch2
        else:
            # every rank: pinned host rows -> device, PartitionedGraph.aggregate (the public call), results -> pinned host
            xh, gh = x_own.cpu().pin_memory(), g_own.cpu().pin_memory()
            oh, oh2 = torch.empty(pg.n_own, FEAT).pin_memory(), torch.empty(pg.n_own, FEAT).pin_memory()
            xd, gd = torch.empty_like(x_own), torch.empty_like(g_own)

            def e2e_step():
                xd.copy_(xh, non_blocking=True)
                pg.aggregate("fwd", xd, nl, nl, out=out_f)
                oh.copy_(out_f, non_blocking=True)
                gd.copy_(gh, non_blocking=True)
                pg.aggregate("bwd", gd, nl, nl, out=out_b)
                oh2.copy_(out_b, non_blocking=True)

            for _ in range(2):
                e2e_step()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(k):
                e2e_step()
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b) / k, float(2 * pg.n_own * FEAT * 4)], device=dev)
            tmax = t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            e2e_ms = float(tmax[0])
            extras["e2e"] = {"value": b_alg_step / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": e2e_ms,
                             "h2d_bytes_per_step": int(t[1]), "d2h_bytes_per_step": int(t[1]),
                             "api": "per rank: pinned host rows -> device, PartitionedGraph.aggregate fwd + bwd, results -> "
                                    "pinned host; device time, max over ranks; bytes summed over ranks"}

    # ---- 2-layer GCN 100 -> 100 -> 47 training epoch on the same graph through the layer API (GCNConv on a StaticGraph /
    # on a PartitionedGraph; fwd + bwd + gradient all-reduce + Adam), the whole-model figure SURVEY.md section 8(e) asks
    # to report beside the aggregation-only scaling
    if not args.no_extras:
        try:
            from stgraph_b200.dist import all_reduce_gradients
            from stgraph_b200.nn.pytorch import GCNConv

            torch.manual_seed(7)
            l1, l2 = GCNConv(FEAT, 100, activation=torch.relu).to(dev), GCNConv(100, 47).to(dev)
            params = list(l1.parameters()) + list(l2.parameters())
            if world > 1:
                for p_ in params:
                    dist.broadcast(p_.data, 0)
                gg, xin = pg, x_own
                pg.set_ndata("norm", nl.reshape(-1, 1))
            else:
                gg, xin = graph, x
                graph.set_ndata("norm", norm.reshape(-1, 1))
            labels = torch.randint(0, 47, (xin.shape[0],), device=dev)
            opt = torch.optim.Adam(params, lr=1e-2)

            def epoch():
                opt.zero_grad()
                # per-row losses + one parallel sum: torch's reduction="sum" / "mean" kernel is a single-block loop over
                # the rows (2.6 ms forward + 1.4 ms backward on 2.4 M rows, scripts/r3_gcn_epoch_prof.py)
                loss = torch.nn.functional.cross_entropy(l2(gg, l1(gg, xin)), labels, reduction="none").sum() / n
                loss.backward()
                if world > 1:
                    all_reduce_gradients(params)
                opt.step()
                return loss

            for _ in range(2):
                epoch()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                loss = epoch()
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b) / 3, float(loss)], device=dev)
            if world > 1:
                tm = t.clone()
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
                t[0] = tm[0]
            extras["gcn_2layer_epoch"] = {"ms_per_epoch": float(t[0]), "loss": float(t[1]),
                                          "model": "GCNConv(100,100,relu) -> GCNConv(100,47), cross-entropy on random labels, Adam",
                                          "api": "stgraph_b200.nn.pytorch.GCNConv on " + ("PartitionedGraph (local rows; weight "
                                                 "gradients all-reduced)" if world > 1 else "StaticGraph")}
            del l1, l2, opt, params
        except Exception as ex:
            extras["gcn_2layer_epoch"] = {"error": repr(ex)[:300]}

    if rank == 0 and world == 1 and not args.no_extras:
        # ---- the plain kernel (column load + dependent norm gather per edge) on the same inputs, for the record ----
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(2):
            kernels.agg_scaled_sum(vf, x, norm, None, norm, out=out_f)
        a.record()
        for _ in range(5):
            kernels.agg_scaled_sum(vf, x, norm, None, norm, out=out_f)
            kernels.agg_scaled_sum(vb, gout, norm, None, norm, out=out_b)
        b.record()
        torch.cuda.synchronize()
        ms_plain = a.elapsed_time(b) / 5
        extras["plain_kernel"] = {"ms_per_step": ms_plain, "value": b_alg_step / (ms_plain * 1e-3) / 1e9, "unit": UNIT,
                                  "note": "stg_agg_scaled_sum_f32 (no packed edge metadata)"}
        # ---- the reference's own GPU kernels on the same inputs (out_f / out_b hold our results of these inputs) ----
        try:
            extras["reference_gpu"] = reference_gpu_leg(graph, x, gout, norm, out_f, out_b, FEAT)
        except Exception as ex:
            extras["reference_gpu"] = {"error": repr(ex)[:300]}
        # ---- locality-free variant of the same shape (secondary figure, SURVEY.md section 8(e)) ----
        try:
            d0 = synthetic.products_shaped(seed=0, device=dev, scale=args.scale, locality=0.0)
            g0 = StaticGraph(torch.stack([d0["src"], d0["dst"]], 1), None, n)
            nm0 = g0.degree_norm().reshape(-1).contiguous()
            f0, b0 = g0._forward_graph, g0._backward_graph
            for _ in range(3):
                kernels.agg_scaled_sum_graph(f0, x, nm0, None, nm0, out=out_f)
                kernels.agg_scaled_sum_graph(b0, gout, nm0, None, nm0, out=out_b)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(5):
                kernels.agg_scaled_sum_graph(f0, x, nm0, None, nm0, out=out_f)
                kernels.agg_scaled_sum_graph(b0, gout, nm0, None, nm0, out=out_b)
            b.record()
            torch.cuda.synchronize()
            ms0 = a.elapsed_time(b) / 5
            extras["locality_free"] = {"ms_per_step": ms0, "value": b_alg_step / (ms0 * 1e-3) / 1e9, "unit": UNIT}
            del g0, d0
        except Exception as ex:  # secondary figure only
            extras["locality_free"] = {"error": str(ex)[:200]}
        # ---- CPU baseline: the oracle port on the host cores, bounded sample of the same workload ----
        try:
            cpu = CpuReference(d["src"], d["dst"], n, FEAT)
            t0 = time.perf_counter()
            e_s = cpu.aggregate(0, cpu.x) + cpu.aggregate(1, cpu.gout)
            t_cpu = time.perf_counter() - t0
            extras["cpu_baseline"] = {"value": b_alg_step * (e_s / (2.0 * e)) / t_cpu / 1e9, "unit": UNIT, "cores": cpu.threads,
                                      "kind": "port",
                                      "sample": f"ONE full step (no sampling): torch-CPU index_add (fp32), forward + backward over all "
                                                f"{e_s} edge visits, F={FEAT}, in destination-row blocks of ~4M edges",
                                      "seconds": t_cpu}
            del cpu
        except Exception as ex:
            extras["cpu_baseline"] = {"error": repr(ex)[:300]}

    if rank == 0 and world == 1 and not args.no_extras and os.environ.get("STG_BENCH_EPOCHS", "1") != "0":
        # ---- the other BASELINE.json configs (scripts/bench_configs.py: the reference's training loops on synthetic
        # inputs of its datasets' shapes); secondary figures, run in a separate process with a time limit
        try:
            import tempfile

            with tempfile.TemporaryDirectory() as tmp:
                path = os.path.join(tmp, "configs.json")
                env = dict(os.environ, STG_CONFIGS_OUT=path, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank)))
                del x, gout, out_f, out_b
                torch.cuda.empty_cache()
                subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "bench_configs.py"), "1", "2", "3", "4", "ref"], env=env,
                               cwd=ROOT, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=420, check=True)
                res = json.load(open(path))
            extras["other_configs"] = res
        except Exception as ex:      # secondary figures only
            extras["other_configs"] = {"error": repr(ex)[:300]}

    if rank == 0:
        peak, peak_src = peaks()
        packed = world > 1 or bool(graph._forward_graph._meta_cache)
        # per GPU: one rank's share of the algorithmic bytes over the slowest rank's forward aggregation
        achieved = b_alg_one / world / (ms_fwd_kernel * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "num_nodes": n, "num_edges": e, "feat": FEAT, "locality": args.locality,
                       "window": args.window,
                       "l2_policy": "inputs (980 MB features + 500 MB structure) exceed the 126 MB L2; no flush needed"
                                    if world == 1 else "per-rank inputs (rows + halo + structure) exceed the 126 MB L2 up to 8 ranks; no flush",
                       "parallelism": f"cost-balanced contiguous vertex partition x{world}, halo exchange" if world > 1 else "single GPU",
                       "halo": halo_info, "partitioned_result_matches_single_gpu": parity,
                       "edge_metadata": ("{col, norm[col]} packed per CSR slot once per graph (8 B/edge, read coalesced); "
                                         "algorithmic bytes still count 4 B/edge") if packed else "column_indices + norm gather",
                       "row_schedule": "global row queue (StgCsrView.work_queue): warps draw chunks of rows from one device counter",
                       "scale": args.scale},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": UNIT, "frac": achieved / peak,
                         "per_gpu": True,
                         "traffic": ncu_traffic() if world == 1 else None,
                         "kernel": ("agg_rows_pipe_kernel<4,32,1,4,8,kPacked,pair,queue> + agg_hub_kernel<4,32,1,kPacked> overlapped "
                                    "(forward, in-edge CSR)") if world == 1 else
                                   "one rank's forward aggregation: own-source pass (agg_rows_pipe_kernel) || halo exchange, flag wait, "
                                   "halo-source pass; slowest rank",
                         "kernel_ms": ms_fwd_kernel, "algorithmic_bytes": b_alg_one // world, "peak_source": peak_src,
                         "gather_model_gbs": 4.0 * (e * FEAT + n * FEAT + e) / world / (ms_fwd_kernel * 1e-3) / 1e9},
            "gpu_launches": launches, "clocks": clocks,
        }
        if segments is not None:
            line["segments"] = segments
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
