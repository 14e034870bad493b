"""The one-op TGCN cell in fp32 and under bf16 / fp16 autocast, against the reference-structured path autocast ran before.

Three measurements, arms run alternately in one process after a warm-up, medians (and min..max) of ``--reps`` windows:

  * config 2 (``synthetic.wikimaths_shaped``, STGraphTGCN(lags, 16, 1) + Adam, one epoch of 723 steps per window):
    fp32 ``TGCN()`` (fused cell), ``TGCN()`` under bf16 / fp16 autocast (16-bit cell) and ``TGCN(fused=False)`` under
    bf16 / fp16 autocast (three GCNConv through the executor); plus kernels per step from one profiled epoch per arm;
  * config-4 shape: one 20-snapshot BPTT window of TGCN(32, 64) on a GPMAGraph (N = 10^6, 10^7 live edges), same arms;
  * the cell alone at N = 10^6, H = 64 (snapshot 0 of that graph): forward and backward per step, and the gate passes'
    device time from a profiled run with their algorithmic bytes and GB/s.

Prints one JSON line and writes it to ``--out``.

    python scripts/bench_tgcn_h16.py [--reps 5] [--out profiles/r05_tgcn_h16.json]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

DT = {"bf16": torch.bfloat16, "fp16": torch.float16}
ARMS = ("fp32", "bf16", "fp16", "bf16_unfused", "fp16_unfused")


def gpu_card():
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True, check=True)
    name, power = [s.strip() for s in res.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def amp(arm):
    dt = DT.get(arm.split("_")[0])
    return torch.autocast("cuda", dtype=dt or torch.bfloat16, enabled=dt is not None)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def alternate(fns, reps, warmup=1):
    for fn in fns.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            ts[k].append(timed(fn))
    return {k: {"ms": sorted(v)[len(v) // 2], "min": min(v), "max": max(v), "windows": len(v)} for k, v in ts.items()}


def kernels_of(fn, steps):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return len(evs) / steps, evs


def config2(reps):
    from stgraph_b200.graph import StaticGraph
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN
    from stgraph_b200.utils import synthetic

    dev = torch.device("cuda")
    d = synthetic.wikimaths_shaped(seed=0, device=dev)
    n, lags, T = d["num_nodes"], d["lags"], d["num_timestamps"]
    steps = T - lags
    g = StaticGraph(torch.stack([d["src"], d["dst"]], 1), None, n)
    g.set_ndata("norm", g.degree_norm())
    w = d["edge_weight"].reshape(-1, 1).contiguous()
    targets = d["targets"]

    class Model(torch.nn.Module):
        def __init__(self, fused):
            super().__init__()
            self.temporal = TGCN(lags, 16, fused=fused)
            self.linear = torch.nn.Linear(16, lags)
            self.linear2 = torch.nn.Linear(lags, 1)

        def forward(self, x, h):
            h = self.temporal(g, x, w, h)
            y = self.linear(F.relu(h))
            return self.linear2(y), y, h

    y0 = torch.randn(n, lags, device=dev)
    fns = {}
    for arm in ARMS:
        torch.manual_seed(0)
        model = Model(False if arm.endswith("unfused") else None).to(dev)
        opt = torch.optim.Adam(model.parameters(), lr=1e-2)

        def epoch(model=model, opt=opt, arm=arm):
            opt.zero_grad()
            cost, h, y_hat = 0, None, y0
            with amp(arm):
                for t in range(steps):
                    y_out, y_hat, h = model(y_hat, h)
                    cost = cost + torch.mean((y_out.float().reshape(-1) - targets[t]) ** 2)
            (cost / (steps + 1)).backward()
            opt.step()
        fns[arm] = epoch
    res = {"epoch_ms": alternate(fns, reps), "steps": steps, "num_nodes": n, "num_edges": g.get_num_edges()}
    res["kernels_per_step"] = {arm: kernels_of(fn, steps)[0] for arm, fn in fns.items()}
    return res


def config4_shape(reps, T=20):
    from stgraph_b200.graph import GPMAGraph
    from stgraph_b200.nn.pytorch.temporal.tgcn import TGCN
    from stgraph_b200.utils import synthetic

    dev = torch.device("cuda")
    n, base, slide = 1_000_000, 10_000_000, 100_000
    src, dst = synthetic.temporal_stream(n, base + slide * (T - 1), alpha=1.8, seed=0, device=dev, distinct=True,
                                         max_frac=2e-4)
    snaps = [torch.stack([s, d_], 1) for s, d_ in synthetic.sliding_window_snapshots(src, dst, base, slide, T)]
    G = GPMAGraph(snaps, n)
    del snaps, src, dst
    xs = torch.randn(T, n, 32, device=dev)
    gouts = torch.randn(T, n, 64, device=dev)
    fns, models = {}, {}
    for arm in ARMS:
        torch.manual_seed(0)
        models[arm] = model = TGCN(32, 64, fused=False if arm.endswith("unfused") else None).to(dev)

        def window(model=model, arm=arm):
            G.reset_graph()
            h, cost = None, 0
            for t in range(T):
                G.get_graph(t)
                G.set_ndata("norm", G.degree_norm())
                with amp(arm):
                    h = model(G, xs[t], H=h)
                cost = cost + (h.float() * gouts[t]).sum()
            cost.backward()
        fns[arm] = window
    res = {"window_ms": alternate(fns, reps), "snapshots": T, "num_nodes": n}
    G.reset_graph()
    G.get_graph(0)
    G.set_ndata("norm", G.degree_norm())
    res["edges_t0"] = G.get_num_edges()
    res["cell"] = cell_alone(G, models["fp32"], xs[0], gouts[0], reps)
    return res


GATE_BYTES = {   # algorithmic bytes per N*H of each gate pass: fp32 elements 4 bytes, 16-bit elements 2
    "fp32": {"bias_clamp": 24, "reset_fwd": 12, "update_fwd": 16, "update_bwd": 28, "reset_bwd": 24, "clamp_bwd": 36},
    "h16": {"bias_clamp": 12, "reset_fwd": 10, "update_fwd": 16, "update_bwd": 32, "reset_bwd": 26, "clamp_bwd": 18},
}
GATE_NAMES = {"bias_clamp": ("bias_clamp4_kernel", "bias_clamp_kernel", "cell_bias_clamp16_kernel"),
              "reset_fwd": ("cell_reset_fwd_kernel", "cell_reset_fwd16_kernel"),
              "update_fwd": ("cell_update_fwd_kernel",),
              "update_bwd": ("cell_update_bwd_kernel", "cell_update_bwd16_kernel"),
              "reset_bwd": ("cell_reset_bwd_kernel", "cell_reset_bwd16_kernel"),
              "clamp_bwd": ("clamp_bwd_kernel", "cell_clamp_bwd16_kernel")}


def kernel_name(name):
    """``cell_reset_fwd16_kernel`` of ``void stg::(anonymous namespace)::cell_reset_fwd16_kernel<__half, 4>(...)``."""
    m = re.search(r"(\w+_kernel)\b", name)
    return m.group(1) if m else name


def cell_alone(G, model, x, gout, reps, iters=10):
    n, hid = x.shape[0], 64
    H0 = torch.randn(n, hid, device=x.device)
    res = {}
    fwd, bwd = {}, {}
    for arm in ("fp32", "bf16", "fp16"):
        def f(arm=arm):
            with amp(arm):
                return model(G, x, H=H0)

        def step_fwd(f=f):
            for _ in range(iters):
                f()

        def step_bwd(f=f):
            outs = [f() for _ in range(iters)]
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for o in outs:
                o.backward(gout)
            b.record()
            b.synchronize()
            return a.elapsed_time(b)
        fwd[arm], bwd[arm] = step_fwd, step_bwd
    res["forward_ms"] = {k: {kk: vv / iters if kk != "windows" else vv for kk, vv in v.items()}
                         for k, v in alternate(fwd, reps).items()}
    bt = {k: [] for k in bwd}
    for _ in range(reps):
        for k, fn in bwd.items():
            bt[k].append(fn() / iters)
    res["backward_ms"] = {k: {"ms": sorted(v)[len(v) // 2], "min": min(v), "max": max(v)} for k, v in bt.items()}
    gates = {}
    for arm in ("fp32", "bf16", "fp16"):
        def one(arm=arm):
            with amp(arm):
                out = model(G, x, H=H0)
            out.backward(gout)
        one()
        _, evs = kernels_of(one, 1)
        per = {}
        for key, names in GATE_NAMES.items():
            us = sum(e.device_time for e in evs if kernel_name(e.name) in names)
            nbytes = GATE_BYTES["fp32" if arm == "fp32" else "h16"][key] * n * hid
            per[key] = {"us": us, "alg_bytes": nbytes, "GBps": nbytes / (us * 1e-6) / 1e9 if us else None}
        gates[arm] = per
    res["gate_passes"] = gates
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_tgcn_h16.json"))
    ap.add_argument("--skip-config4", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tgcn_h16.py measures on the GPU; no CUDA device found")
    line = {"card": gpu_card(), "torch": torch.__version__, "config2": config2(args.reps)}
    if not args.skip_config4:
        line["config4_shape"] = config4_shape(args.reps)
    text = json.dumps(line)
    print(text)
    with open(args.out, "w") as fh:
        fh.write(text + "\n")


if __name__ == "__main__":
    main()
