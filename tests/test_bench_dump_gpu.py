"""bench.py --dump-outputs: the last timed step's outputs land in DIR as float32 .npy files; they are what the step computes on
the benchmark's inputs (recomputed here through the public API), and two runs with the same arguments dump the same outputs
(the inputs, the parameters and the Philox noise of the timed steps do not depend on the run).  Both step paths are covered:
the one-piece step (cfg1: loss, gradient and the per-date / per-stock outputs) and the micro-batched step (cfg4: loss and
gradient)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu
STEPS = 3


def _bench(out_dir, workload, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", str(steps), "--warmup", "3",
           "--no-cpu-baseline", "--no-e2e", "--no-eager", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return line, {n[:-4]: np.load(os.path.join(out_dir, n)) for n in os.listdir(out_dir)}


def _close(a, b, tol, name):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (name, a.shape, b.shape)
    scale = max(1.0, float(np.abs(b).max()))
    assert float(np.abs(a - b).max()) <= tol * scale, name


def _cfg1_last_step(steps, dev):
    """The last timed step of `bench.py --workload cfg1 --steps <steps>`: the benchmark's parameters and batch, Philox step
    <steps> (the timed steps are steps 1..K of the noise stream)."""
    import bench
    from factorvae_b200 import engine
    from factorvae_b200.batched import DateShardedStep
    wl = bench.WORKLOADS["cfg1"]
    N, T, H, K, M = (wl[k] for k in "NTHKM")
    C = bench.C_FEATURES
    layout = engine.ParamLayout(C, H, K, M)
    flat = layout.pack(bench.build_params(H, K, M), dev)
    gen = torch.Generator(device=dev).manual_seed(1234)
    store = torch.zeros(N, T, 160, dtype=torch.bfloat16, device=dev)           # the benchmark's 16-byte row pitch
    x = store[:, :, :C]
    x[:] = torch.randn(N, T, C, generator=gen, device=dev).clamp_(-3, 3).to(torch.bfloat16)
    y = torch.randn(N, generator=gen, device=dev)
    stepper = DateShardedStep(layout, flat, precision="bf16" if engine.tc_supported(C, H) else "fp32", seed=42)
    stepper.step_index = steps - 1
    out, _ = stepper.step(x, y, engine.uniform_date_ptr(1, N, dev), global_dates=1)
    torch.cuda.synchronize()
    res = {k: v.detach().float().cpu().numpy() for k, v in out.items()}
    res["grad"] = stepper.grad.cpu().numpy()
    return res


def test_dump_outputs_one_piece_step(tmp_path, cuda_device):
    (line0, d0), (line1, d1) = (_bench(tmp_path / f"run{i}", "cfg1", STEPS) for i in range(2))
    assert {"loss", "grad", "date_loss", "yhat", "mu_y", "sigma_y", "mu_post", "sigma_post", "mu_prior", "sigma_prior"} == set(d0)
    assert set(d1) == set(d0)
    for name, a in d0.items():
        assert a.dtype == np.float32 and np.isfinite(a).all(), name
        _close(a, d1[name], 1e-6, name)                                            # run to run
    assert float(d0["loss"][0]) == pytest.approx(line0["loss"], rel=1e-6)
    ref = _cfg1_last_step(STEPS, cuda_device)
    for name, a in d0.items():
        _close(a, ref[name], 1e-5, name)                                           # what the step computes on these inputs


def test_dump_outputs_micro_batched_step(tmp_path, cuda_device):
    import bench
    from factorvae_b200 import engine
    wl = bench.WORKLOADS["cfg4"]
    line, d = _bench(tmp_path / "run", "cfg4", 1)
    assert set(d) == {"loss", "grad"}
    total = engine.ParamLayout(bench.C_FEATURES, wl["H"], wl["K"], wl["M"]).total
    assert d["grad"].dtype == np.float32 and d["grad"].shape == (total,) and np.isfinite(d["grad"]).all()
    assert float(np.abs(d["grad"]).max()) > 0
    assert float(d["loss"][0]) == pytest.approx(line["loss"], rel=1e-6)
