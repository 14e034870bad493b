"""Config-3 stock GATConv training step under autocast: 16-bit projection rows read by the VM kernel (``stg_vm_run_mixed``)
against the same layer with the program given ``proj.float()`` (the path before the VM read 16-bit tensors).

The workload is ``scripts/bench_gat_h16.py``'s (``synthetic.arxiv_shaped(seed=0)``: N=169,343, E=1,166,243, H=8, D=16,
128 input features).  A step is forward, backward and Adam.  Arms run alternately in one process after a warm-up; each
timed window is ``--steps`` steps between CUDA events, repeated ``--reps`` times, so the spread is the min..max of the
window means.  The arms:

  * native_{bf16,fp16}: the layer under autocast as it is (the VM reads the 16-bit projection);
  * upcast_{bf16,fp16}: the same layer with the program given ``proj.float()`` (one cast, fp32 VM launches);
  * fp32: the layer outside autocast.

A separate ``torch.profiler`` run then records the VM kernels of each arm, split into forward and backward launches.
The outputs and all gradients of one step of the two autocast arms are compared bit for bit at this size.
Prints one JSON line.

    python scripts/bench_vm_h16.py [--steps 30] [--reps 7] [--out /tmp/vm_h16.json]
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

DT = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


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
            windows[name].append(timed(fn, iters))
    return {name: summary(ts) for name, ts in windows.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--profile-steps", type=int, default=10)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    from torch.profiler import ProfilerActivity, profile

    from stgraph_b200.graph import StaticGraph
    from stgraph_b200.nn.pytorch import GATConv
    from stgraph_b200.utils import synthetic

    dev = torch.device("cuda", 0)
    card = gpu_card()
    d = synthetic.arxiv_shaped(seed=0, device=dev, scale=args.scale)
    n, e = d["num_nodes"], int(d["src"].shape[0])
    H, D, FIN = d["heads"], d["out_feats"], d["in_feats"]
    g = StaticGraph(torch.stack([d["src"], d["dst"]], 1), None, n)
    del d
    x = torch.randn(n, FIN, device=dev, generator=torch.Generator(device=dev).manual_seed(0))

    torch.manual_seed(7)
    native = GATConv(FIN, D, H).to(dev)
    upcast = GATConv(FIN, D, H).to(dev)
    upcast.load_state_dict(native.state_dict())

    def upcast_forward(layer, xx):
        proj, left, right = layer._scores(xx)
        return layer._stock_program()(g=g, n_feats={"el": left, "er": right, "feat_src": proj.float()})

    def autocast(k):
        return torch.autocast("cuda", dtype=DT[k]) if k != "fp32" else torch.autocast("cuda", enabled=False)

    def forward(layer, k):
        with autocast(k):
            return upcast_forward(layer, x) if layer is upcast else layer(g, x)

    # result check before any optimizer step: same weights, one forward + backward per arm
    same = {}
    gout = torch.randn(n, H, D, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    for k in ("bf16", "fp16"):
        res = []
        for layer in (native, upcast):
            layer.zero_grad()
            o = forward(layer, k)
            o.backward(gout)
            res.append([o.detach().clone()] + [p.grad.clone() for p in layer.parameters()])
        same[k] = all(a.dtype == b.dtype and torch.equal(a.view(torch.int32), b.view(torch.int32))
                      for a, b in zip(*res))

    opts = {id(native): torch.optim.Adam(native.parameters(), lr=1e-3),
            id(upcast): torch.optim.Adam(upcast.parameters(), lr=1e-3)}

    def step(layer, k):
        opt = opts[id(layer)]
        opt.zero_grad()
        loss = forward(layer, k).float().square().mean()
        loss.backward()
        opt.step()

    arms = {}
    for k in ("bf16", "fp16"):
        arms[f"native_{k}"] = lambda k=k: step(native, k)
        arms[f"upcast_{k}"] = lambda k=k: step(upcast, k)
    arms["fp32"] = lambda: step(native, "fp32")
    step_ms = alternate(arms, args.steps, args.reps)

    # per-launch VM kernel times (separate profiler run): forward launches are the first ones of each step
    def vm_events(fn, steps):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
        evs = [ev for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
        evs.sort(key=lambda ev: ev.time_range.start)
        return [ev for ev in evs if "vm_kernel" in ev.name], len(evs)

    def name_of(ev):
        return re.search(r"vm_kernel<[^>]*>", ev.name).group(0).replace(" ", "")

    kernels = {}
    for name, layer, k in (("native_bf16", native, "bf16"), ("native_fp16", native, "fp16"), ("upcast_bf16", upcast, "bf16"),
                           ("upcast_fp16", upcast, "fp16"), ("fp32", native, "fp32")):
        with torch.no_grad():
            fwd_only, fwd_all = vm_events(lambda: forward(layer, k), args.profile_steps)
        both, both_all = vm_events(lambda: forward(layer, k).float().square().mean().backward(), args.profile_steps)
        nf = len(fwd_only) // args.profile_steps
        per = len(both) // args.profile_steps
        fwd_us, bwd_us = [], []
        for s in range(args.profile_steps):
            evs = both[s * per:(s + 1) * per]
            fwd_us.append(sum(ev.time_range.elapsed_us() for ev in evs[:nf]))
            bwd_us.append(sum(ev.time_range.elapsed_us() for ev in evs[nf:]))
        kernels[name] = {
            "vm_fwd_ms_per_step": sorted(fwd_us)[len(fwd_us) // 2] / 1e3, "vm_bwd_ms_per_step": sorted(bwd_us)[len(bwd_us) // 2] / 1e3,
            "vm_launches_fwd": nf, "vm_launches_bwd": per - nf,
            "vm_kernel_us_per_launch": {
                kn: sum(ev.time_range.elapsed_us() for ev in both if name_of(ev) == kn) / sum(name_of(ev) == kn for ev in both)
                for kn in sorted({name_of(ev) for ev in both})},
            "cuda_events_per_forward": fwd_all // args.profile_steps,
        }
        native.zero_grad()
        upcast.zero_grad()

    line = {
        "gpu": card, "workload": "config 3: arxiv_shaped(seed=0), stock GATConv", "num_nodes": n, "num_edges": e, "heads": H,
        "dim": D, "in_feats": FIN, "steps_per_window": args.steps,
        "step_ms": step_ms,
        "vm_kernels_profiled": kernels,
        "native_equals_upcast_bitwise": same,
        "proj_cast_bytes": {"read_16bit": 2 * n * H * D, "write_fp32": 4 * n * H * D},
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
