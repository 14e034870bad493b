"""Config-5 aggregation and GCN epoch in fp32, bf16 and fp16 (the 16-bit rows of ``csrc/agg_h16.cu``).

The workload is bench.py's (``synthetic.products_shaped(seed=0)``: N=2,449,029, E=61,859,140, F=100).  Arms run
alternately in one process after a warm-up; each timed window is ``--iters`` launches between CUDA events, repeated
``--reps`` times, so the spread is the min..max of the window means.  Prints one JSON line.

    python scripts/bench_agg_h16.py [--iters 200] [--reps 5] [--epochs 5] [--out /tmp/agg_h16.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

FEAT, CLASSES = 100, 47
DT = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def gpu_card():
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True, check=True)
    name, power = [s.strip() for s in res.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def timed(fn, iters, reps):
    """ms per call of each of ``reps`` windows of ``iters`` calls."""
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / iters)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--epochs", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    from stgraph_b200 import kernels
    from stgraph_b200.graph import StaticGraph
    from stgraph_b200.nn.pytorch import GCNConv
    from stgraph_b200.utils import synthetic

    dev = torch.device("cuda", 0)
    card = gpu_card()
    d = synthetic.products_shaped(seed=0, device=dev, scale=args.scale)
    n, e = d["num_nodes"], int(d["src"].shape[0])
    graph = StaticGraph(torch.stack([d["src"], d["dst"]], 1), None, n)
    del d
    norm = graph.degree_norm().reshape(-1)
    fcsr, bcsr = graph._forward_graph, graph._backward_graph
    fv, bv = graph.fwd_view(), graph.bwd_view()
    meta = {"fwd": kernels.pack_edge_meta(fv, norm, None), "bwd": kernels.pack_edge_meta(bv, norm, None)}
    g = torch.Generator(device=dev).manual_seed(0)
    x32 = torch.randn(n, FEAT, device=dev, generator=g)
    gy32 = torch.randn(n, FEAT, device=dev, generator=g)
    xs = {k: x32.to(t) for k, t in DT.items()}
    gys = {k: gy32.to(t) for k, t in DT.items()}
    outs = {k: torch.empty(n, FEAT, device=dev, dtype=t) for k, t in DT.items()}

    arms = {}
    for k in DT:
        arms[f"fwd_plain_{k}"] = lambda k=k: kernels.agg_scaled_sum(fv, xs[k], norm, None, norm, out=outs[k])
        arms[f"fwd_packed_{k}"] = lambda k=k: kernels.agg_packed_sum(fv, meta["fwd"], xs[k], norm, out=outs[k])
        arms[f"bwd_plain_{k}"] = lambda k=k: kernels.agg_scaled_sum(bv, gys[k], norm, None, norm, out=outs[k])
        arms[f"bwd_packed_{k}"] = lambda k=k: kernels.agg_packed_sum(bv, meta["bwd"], gys[k], norm, out=outs[k])
    for fn in arms.values():          # warm-up
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    windows = {name: [] for name in arms}
    for _ in range(args.reps):        # arms alternate: each round times one window of every arm
        for name, fn in arms.items():
            windows[name] += timed(fn, args.iters, 1)

    # result check: the 16-bit forward against the fp32 forward of the same (rounded) input
    ref = kernels.agg_scaled_sum(fv, xs["bf16"].float(), norm, None, norm)
    h = kernels.agg_scaled_sum(fv, xs["bf16"], norm, None, norm).float()
    rel_err_bf16 = float(((h - ref).abs() / ref.abs().clamp_min(1e-3)).median())

    # one 2-layer GCNConv training epoch (bench.py's gcn_2layer_epoch) with autocast off / bf16 / fp16
    graph.set_ndata("norm", norm.reshape(-1, 1))
    torch.manual_seed(7)
    l1, l2 = GCNConv(FEAT, 100, activation=torch.relu).to(dev), GCNConv(100, CLASSES).to(dev)
    params = list(l1.parameters()) + list(l2.parameters())
    labels = torch.randint(0, CLASSES, (n,), device=dev)
    opt = torch.optim.Adam(params, lr=1e-2)

    def epoch(kind):
        opt.zero_grad()
        ac = (torch.autocast("cuda", dtype=DT[kind]) if kind != "fp32" else torch.autocast("cuda", enabled=False))
        with ac:
            logits = l2(graph, l1(graph, x32))
        loss = torch.nn.functional.cross_entropy(logits.float(), labels, reduction="none").sum() / n
        loss.backward()
        opt.step()
        return loss

    epochs = {k: [] for k in DT}
    loss = {}
    for k in DT:
        for _ in range(2):
            epoch(k)
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for k in DT:
            epochs[k] += timed(lambda k=k: loss.__setitem__(k, epoch(k)), args.epochs, 1)

    def summary(ts):
        return {"ms": sorted(ts)[len(ts) // 2], "min": min(ts), "max": max(ts), "windows": len(ts)}

    line = {
        "gpu": card, "workload": "config 5: products_shaped(seed=0)", "num_nodes": n, "num_edges": e, "feat": FEAT,
        "iters_per_window": args.iters, "hub_threshold": fv.hub_threshold,
        "agg_ms_per_launch": {name: summary(ts) for name, ts in windows.items()},
        "algorithmic_bytes_per_launch": {"fp32": synthetic.gcn_algorithmic_bytes(n, e, FEAT),
                                         "16bit": synthetic.gcn_algorithmic_bytes(n, e, FEAT, elem_bytes=2)},
        "gcn_2layer_epoch_ms": {k: summary(ts) for k, ts in epochs.items()},
        "epoch_loss": {k: float(v) for k, v in loss.items()},
        "median_rel_err_bf16_fwd_vs_fp32": rel_err_bf16,
    }
    for k in DT:
        b = line["algorithmic_bytes_per_launch"]["fp32" if k == "fp32" else "16bit"]
        line.setdefault("agg_TBps", {})[f"fwd_packed_{k}"] = b / (line["agg_ms_per_launch"][f"fwd_packed_{k}"]["ms"] * 1e-3) / 1e12
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
