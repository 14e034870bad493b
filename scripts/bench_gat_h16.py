"""Config-3 fused edge softmax and GATConv training step in fp32, bf16 and fp16 (16-bit rows of ``csrc/gat.cu``).

The workload is ``scripts/bench_gat.py``'s (``synthetic.arxiv_shaped(seed=0)``: N=169,343, E=1,166,243, H=8, D=16, 128
input features).  Arms run alternately in one process after a warm-up; each timed window is ``--iters`` calls between
CUDA events (``--stock-steps`` for the slow stock layer), repeated ``--reps`` times, so the spread is the min..max of the
window means.  The GATConv arms:

  * native: the layer under autocast as it is, the 16-bit projection goes to the 16-bit kernels;
  * upcast: the same layer with the op given ``proj.float()`` (the path before 16-bit rows: an fp32 copy, fp32 kernels);
  * stock: the default layer (VM kernel on the widened projection) under autocast, and in fp32.

Prints one JSON line.

    python scripts/bench_gat_h16.py [--iters 100] [--reps 5] [--stock-steps 20] [--out /tmp/gat_h16.json]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

DT = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
SLOPE = 0.2


def gpu_card():
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True, check=True)
    name, power = [s.strip() for s in res.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def timed(fn, iters):
    """ms per call of one window of ``iters`` calls."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def summary(ts):
    return {"ms": sorted(ts)[len(ts) // 2], "min": min(ts), "max": max(ts), "windows": len(ts)}


def alternate(arms, iters, reps, warmup=3):
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    windows = {name: [] for name in arms}
    for _ in range(reps):              # each round times one window of every arm
        for name, fn in arms.items():
            windows[name].append(timed(fn, iters if not isinstance(iters, dict) else iters[name]))
    return {name: summary(ts) for name, ts in windows.items()}


def algorithmic_bytes(n, e, h, d, elem):
    """Bytes the two passes must move at least: feat rows of ``elem`` bytes, everything else fp32."""
    nhd = n * h * d
    return {"fwd": elem * nhd + 4 * nhd + 4 * (4 * n * h + e + n + 1),
            "bwd": (elem + 4 + 4 + elem) * nhd + 4 * (6 * n * h + 2 * (e + n + 1))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--stock-steps", type=int, default=20)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    from stgraph_b200 import _lib, kernels, ops_gat
    from stgraph_b200.graph import StaticGraph
    from stgraph_b200.nn.pytorch import GATConv
    from stgraph_b200.ops_gat import gat_edge_softmax_aggregate
    from stgraph_b200.utils import synthetic

    dev = torch.device("cuda", 0)
    card = gpu_card()
    d = synthetic.arxiv_shaped(seed=0, device=dev, scale=args.scale)
    n, e = d["num_nodes"], int(d["src"].shape[0])
    H, D, FIN = d["heads"], d["out_feats"], d["in_feats"]
    g = StaticGraph(torch.stack([d["src"], d["dst"]], 1), None, n)
    del d
    vf, vb = ops_gat._views(g)
    st = _lib.current_stream_ptr()

    # ---- entry points on preallocated buffers
    gen = torch.Generator(device=dev).manual_seed(0)
    feat32 = torch.randn(n, H, D, device=dev, generator=gen)
    el = torch.randn(n, H, device=dev, generator=gen)
    er = torch.randn(n, H, device=dev, generator=gen)
    gout = torch.randn(n, H, D, device=dev, generator=gen)
    feats = {k: feat32.to(t) for k, t in DT.items()}
    dfeats = {k: torch.empty_like(f) for k, f in feats.items()}
    out, rmax, rsum = torch.empty(n, H, D, device=dev), torch.empty(n, H, device=dev), torch.empty(n, H, device=dev)
    d_el, d_er, dot = torch.empty_like(el), torch.empty_like(er), torch.empty_like(el)

    def fwd(k):
        if k == "fp32":
            return _lib.call("stg_gat_softmax_fwd_f32", ctypes.byref(vf), el.data_ptr(), er.data_ptr(), feats[k].data_ptr(),
                             H, D, SLOPE, out.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), st)
        return _lib.call("stg_gat_softmax_fwd_h16", ctypes.byref(vf), el.data_ptr(), er.data_ptr(), feats[k].data_ptr(),
                         H, D, kernels.H16_DTYPES[DT[k]], SLOPE, out.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), st)

    def bwd(k):
        a = (ctypes.byref(vf), ctypes.byref(vb), el.data_ptr(), er.data_ptr(), feats[k].data_ptr(), out.data_ptr(),
             gout.data_ptr(), rmax.data_ptr(), rsum.data_ptr(), H, D)
        t = (SLOPE, dfeats[k].data_ptr(), d_el.data_ptr(), d_er.data_ptr(), dot.data_ptr(), st)
        if k == "fp32":
            return _lib.call("stg_gat_softmax_bwd_f32", *a, *t)
        return _lib.call("stg_gat_softmax_bwd_h16", *a, kernels.H16_DTYPES[DT[k]], *t)

    fwd("fp32")
    torch.cuda.synchronize()
    kernel_arms = {}
    for k in DT:
        kernel_arms[f"fwd_{k}"] = lambda k=k: fwd(k)
        kernel_arms[f"bwd_{k}"] = lambda k=k: bwd(k)
    kernel_ms = alternate(kernel_arms, args.iters, args.reps)

    # result check: every 16-bit launch equals the fp32 one on the widened rows (d_feat rounded once)
    same = {}
    for k in ("bf16", "fp16"):
        save32 = feats["fp32"]
        feats["fp32"] = feats[k].float()
        fwd("fp32"); bwd("fp32")
        ref = [t.clone() for t in (out, rmax, rsum, dfeats["fp32"].to(DT[k]), d_el, d_er)]
        feats["fp32"] = save32
        fwd(k); bwd(k)
        got = (out, rmax, rsum, dfeats[k], d_el, d_er)
        same[k] = all(torch.equal(a.view(torch.int16) if a.element_size() == 2 else a,
                                  b.view(torch.int16) if b.element_size() == 2 else b) for a, b in zip(got, ref))

    # ---- GATConv training steps
    x = torch.randn(n, FIN, device=dev, generator=gen)
    torch.manual_seed(7)
    fused = GATConv(FIN, D, H, softmax="fused").to(dev)
    stock = GATConv(FIN, D, H).to(dev)
    stock.load_state_dict(fused.state_dict())
    opts = {"fused": torch.optim.Adam(fused.parameters(), lr=1e-3), "stock": torch.optim.Adam(stock.parameters(), lr=1e-3)}

    def upcast_forward(layer, xx):
        proj, left, right = layer._scores(xx)
        return gat_edge_softmax_aggregate(g, left, right, proj.float(), layer.negative_slope)

    def autocast(k):
        return torch.autocast("cuda", dtype=DT[k]) if k != "fp32" else torch.autocast("cuda", enabled=False)

    def step(layer, k, upcast=False):
        opt = opts[layer.softmax]
        opt.zero_grad()
        with autocast(k):
            o = upcast_forward(layer, x) if upcast else layer(g, x)
        loss = o.float().square().mean()
        loss.backward()
        opt.step()

    step_arms, iters = {}, {}
    for k in ("bf16", "fp16"):
        step_arms[f"fused_native_{k}"] = lambda k=k: step(fused, k)
        step_arms[f"fused_upcast_{k}"] = lambda k=k: step(fused, k, upcast=True)
    step_arms["fused_fp32"] = lambda: step(fused, "fp32")
    for name in step_arms:
        iters[name] = args.iters
    for k in ("fp32", "bf16", "fp16"):
        step_arms[f"stock_{k}"] = lambda k=k: step(stock, k)
        iters[f"stock_{k}"] = args.stock_steps
    step_ms = alternate(step_arms, iters, args.reps)

    # live memory held for backward after one autocast forward: native against upcast
    live = {}
    for k in ("bf16", "fp16"):
        for mode in ("native", "upcast"):
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            with autocast(k):
                o = upcast_forward(fused, x) if mode == "upcast" else fused(g, x)
            torch.cuda.synchronize()
            live[f"{mode}_{k}"] = torch.cuda.memory_allocated() - base
            del o
        live[f"saved_{k}"] = live[f"upcast_{k}"] - live[f"native_{k}"]

    hd = H * D
    line = {
        "gpu": card, "workload": "config 3: arxiv_shaped(seed=0)", "num_nodes": n, "num_edges": e, "heads": H, "dim": D,
        "in_feats": FIN, "gat_hub_threshold": ops_gat.GAT_HUB_THRESHOLD, "iters_per_window": args.iters,
        "stock_steps_per_window": args.stock_steps,
        "kernel_ms_per_launch": kernel_ms,
        "h16_equals_fp32_on_widened_rows": same,
        "algorithmic_bytes_per_launch": {"fp32": algorithmic_bytes(n, e, H, D, 4), "16bit": algorithmic_bytes(n, e, H, D, 2)},
        "feat_bytes_gathered_per_edge": {"fp32": 4 * hd, "16bit": 2 * hd},
        "gatconv_step_ms": step_ms,
        "live_bytes_after_autocast_forward": live, "n_h_d_4": 4 * n * hd,
    }
    for k in DT:
        b = line["algorithmic_bytes_per_launch"]["fp32" if k == "fp32" else "16bit"]
        line.setdefault("alg_TBps", {})[k] = {p: b[p] / (kernel_ms[f"{p}_{k}"]["ms"] * 1e-3) / 1e12 for p in ("fwd", "bwd")}
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
