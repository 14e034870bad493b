"""CPU check of the bench.py contract on the arm that runs without a GPU (``--impl reference``): one JSON line
with the keys the driver reads; the CUDA arm refuses to run without a device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT,
                          timeout=600, env=env)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--scale", "0.005")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["steps"] == 2 and line["warmup"] == 1
    assert line["unit"] == "GB/s" and line["value"] > 0 and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_is_rank0_only_under_torchrun():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = _run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--scale", "0.005", env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_rows_are_fixed_and_bounded():
    """--dump-outputs writes every row of a small graph and the same seeded sample of a config-5-sized one, under 64 MB."""
    import importlib.util

    import torch

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert torch.equal(bench.dump_rows(1000, 400, 2), torch.arange(1000))
    rows = bench.dump_rows(2449029, 400, 2)
    assert torch.equal(rows, bench.dump_rows(2449029, 400, 2))
    assert 0 < rows.numel() * 400 * 2 <= 64 * 10**6 - 4096
    assert bool((rows[1:] > rows[:-1]).all()) and int(rows[-1]) < 2449029


def test_bench_rejects_zero_steps_and_dump_on_reference_arm(tmp_path):
    r = _run("--impl", "reference", "--steps", "0", "--warmup", "0", "--scale", "0.005")
    assert r.returncode == 2 and "--steps" in r.stderr
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--scale", "0.005", "--dump-outputs", str(tmp_path))
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not any(tmp_path.iterdir())


@pytest.mark.gpu
def test_cuda_arm_times_steps_and_dumps_what_they_computed(cuda, tmp_path):
    """--steps sets the timed steps (kernel launches in the timed window scale with it); --dump-outputs holds the last
    step's aggregations of the seeded inputs (oracle)."""
    import numpy as np
    import torch

    from oracle import aggregate as A
    from oracle import structure as S
    from stgraph_b200.utils import synthetic

    launches = {}
    for steps in (2, 5):
        dump = ["--dump-outputs", str(tmp_path)] if steps == 5 else []
        r = _run("--steps", str(steps), "--warmup", "1", "--scale", "0.002", "--no-extras", *dump)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        launches[steps] = line["gpu_launches"]
    assert launches[2] > 0 and launches[5] * 2 == launches[2] * 5, launches
    d = synthetic.products_shaped(seed=0, device=cuda, scale=0.002)
    n, src, dst = d["num_nodes"], d["src"].cpu().numpy(), d["dst"].cpu().numpy()
    gen = torch.Generator(device=cuda).manual_seed(1)
    x = torch.randn(n, 100, device=cuda, generator=gen).cpu()
    gout = torch.randn(n, 100, device=cuda, generator=gen).cpu()
    f, b = S.forward_csr(src, dst, n), S.backward_csr(src, dst, n)
    deg = torch.from_numpy(f.row_degrees.astype(np.float32))
    norm = torch.where(deg > 0, deg.pow(-0.5), torch.zeros_like(deg))
    for name, run, csr, h in (("fwd_aggregate", A.gcn_forward, f, x), ("bwd_aggregate", A.gcn_backward, b, gout)):
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float32 and got.shape == (n, 100)
        A.assert_close_rel(torch.from_numpy(got), run(csr, h, norm), rel=1e-5, abs_terms=run(csr, h.abs(), norm) + 1e-6,
                           what=name)


def test_cuda_arm_has_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        return
    r = _run("--steps", "1", "--warmup", "0", "--scale", "0.005")
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
