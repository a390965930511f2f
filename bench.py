"""bench.py -- dates x stocks / second per ELBO step (forward + backward [+ gradient all-reduce]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path (FactorVAE.forward + backward, reference module.py:250-270 +
train_model.py:29) over one batch of synthetic dates.

Workloads (BASELINE.json configs; H = K, M = 128):
  cfg1  1 date x 64 stocks, T=20, K=20                    per GPU, weak scaling
  cfg2  256 dates x 300, T=20, K=20   (DEFAULT, N=1..8)    per GPU, weak scaling: every rank processes 256 dates
  cfg3  256 dates x 500, T=60, K=60                        per GPU, weak scaling
  cfg4  512 dates x 1000, T=20, K=48  GLOBAL batch         strong scaling: 512 / N dates per GPU, micro-batches of 64 dates
  cfg5  1024 dates x 3000, T=60, K=60 GLOBAL batch         strong scaling: 1024 / N dates per GPU, micro-batches of 128 dates
`--gpus N` without `--workload` runs cfg2 (the configuration BASELINE.json's metric is quoted on for one GPU).

Prints ONE JSON line (rank 0).  `value` = whole-job units/s with the panel resident in HBM; `e2e` = the same through the
host-buffer entry of the resident row table: per step the batch's NEW (date, instrument) rows cross PCIe from pinned host
memory (each row once, not T times inside T overlapping windows), one kernel builds the look-back index, the step runs, the
loss is read back on the host; `roofline` / `cpu_baseline` as specified in the task statement.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # per-GPU batches (weak scaling)
    "cfg1": dict(B=1, N=64, T=20, H=20, K=20, M=128, scaling="weak", micro=1),
    "cfg2": dict(B=256, N=300, T=20, H=20, K=20, M=128, scaling="weak", micro=256),
    "cfg3": dict(B=256, N=500, T=60, H=60, K=60, M=128, scaling="weak", micro=256),
    # global batches split over the ranks (strong scaling), processed in micro-batches of `micro` dates
    "cfg4": dict(B=512, N=1000, T=20, H=48, K=48, M=128, scaling="strong", micro=64),
    # micro = 128: the fp32 CUDA-core heads (H, K > 32) run one CTA per date -- 32-date micro-batches left 116 of 148 SMs idle there
    "cfg5": dict(B=1024, N=3000, T=60, H=60, K=60, M=128, scaling="strong", micro=128),
}
C_FEATURES = 158
METRIC = "dates x stocks / sec per ELBO step (fwd+bwd), K=20 C=158"
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def f_fe(T, H, C=C_FEATURES):
    """Algorithmic FLOPs per date x stock per step: FeatureExtractor contractions, fwd + 2x bwd (SURVEY 8d)."""
    return 3 * 2 * T * (C * C + 3 * H * C + 3 * H * H)


def workload_desc(name, world):
    wl = WORKLOADS[name]
    if wl["scaling"] == "weak":
        return (f"{name}: B={wl['B']} dates/GPU x N={wl['N']} stocks x T={wl['T']} x C={C_FEATURES}, K=H={wl['K']}, M={wl['M']}; "
                f"{world} GPU(s), dates sharded, weak scaling")
    return (f"{name}: GLOBAL B={wl['B']} dates x N={wl['N']} stocks x T={wl['T']} x C={C_FEATURES}, K=H={wl['K']}, M={wl['M']}; "
            f"{world} GPU(s), {wl['B'] // world} dates/GPU in micro-batches of {wl['micro']}, strong scaling")


def build_params(H, K, M, seed=42):
    import torch
    import factorvae_b200 as fb
    torch.manual_seed(seed)
    model = fb.FactorVAE(fb.FeatureExtractor(C_FEATURES, H), fb.FactorEncoder(K, M, H),
                         fb.FactorDecoder(fb.AlphaLayer(H), fb.BetaLayer(H, K)), fb.FactorPredictor(H, K))
    return {k: v.detach().clone() for k, v in model.state_dict().items()}


def load_reference_module():
    """The unmodified reference module.py, byte-compiled into oracle/_ref by __graft_entry__.build() (oracle/stage_reference.py)
    where the original project is present, or None."""
    path = os.path.join(REF_DIR, "module.pyc")
    if not os.path.exists(path):
        return None
    spec = importlib.util.spec_from_file_location("fvae_reference_module", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def build_reference_model(ref, H, K, M, seed=42):
    """Built exactly as main.py:27-33 under torch.manual_seed(42) (main.py:109)."""
    import torch
    torch.manual_seed(seed)
    return ref.FactorVAE(ref.FeatureExtractor(num_latent=C_FEATURES, hidden_size=H), ref.FactorEncoder(num_factors=K, num_portfolio=M, hidden_size=H),
                         ref.FactorDecoder(ref.AlphaLayer(H), ref.BetaLayer(H, K)), ref.FactorPredictor(H, K))


class ReferenceStepper:
    """One reference training step per date, as train_model.py:26-29: zero_grad -> forward -> loss.item() -> backward.
    (optimizer.step() of train_model.py:30 is NOT timed on either arm: the metric is per ELBO step, forward + backward.)"""

    def __init__(self, wl, device="cpu"):
        import torch
        self.kind = "port"
        ref = load_reference_module()
        if ref is not None:
            self.kind = "reference"
            self.model = build_reference_model(ref, wl["H"], wl["K"], wl["M"]).to(device).train()
        else:
            from oracle.cpu_port import CpuPort
            assert device == "cpu", "the port is a CPU baseline"
            self.port = CpuPort(build_params(wl["H"], wl["K"], wl["M"]))
        self.device = device

    def train_step(self, x, y):
        if self.kind == "port":
            return self.port.train_step(x, y)
        self.model.zero_grad(set_to_none=True)
        loss = self.model(x, y)[0]
        v = loss.item()
        loss.backward()
        return v


def pick_threads(stepper, x, y):
    """Intra-op thread count at which the reference step is fastest on this host ("all the host threads it can use": these
    are small ATen ops; on a 128-core host the full-width pool is far SLOWER than a few threads -- probing keeps the baseline
    the reference at its best, not a strawman).  Returns (picked, host_cpus)."""
    import torch
    ncpu = os.cpu_count() or 1
    best = (float("inf"), 1)
    for cand in sorted({1, 4, 8, 16, 32, min(64, ncpu), ncpu}):
        if cand > ncpu:
            continue
        torch.set_num_threads(cand)
        stepper.train_step(x, y)
        t0 = time.perf_counter()
        stepper.train_step(x, y)
        dt = time.perf_counter() - t0
        if dt < best[0]:
            best = (dt, cand)
        if dt > 2.0:
            break
    torch.set_num_threads(best[1])
    return best[1], ncpu


def time_reference_cpu(wl, budget_s=10.0, warmup=2, min_steps=3):
    """Per-date reference steps of the workload's (N, T, K) on the host cores for ~budget_s seconds."""
    import torch
    st = ReferenceStepper(wl, "cpu")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(wl["N"], wl["T"], C_FEATURES, generator=g).clamp_(-3, 3)
    y = torch.randn(wl["N"], 1, generator=g)
    threads, ncpu = pick_threads(st, x, y)
    for _ in range(warmup):
        st.train_step(x, y)
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < min_steps or (time.perf_counter() < t_end and len(times) < 2000):
        t0 = time.perf_counter()
        st.train_step(x, y)
        times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return dict(value=wl["N"] / med, ms_per_date=med * 1e3, steps=len(times), cores=threads, host_cpus=ncpu, kind=st.kind)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING warm-up + the timed region (one `nvidia-smi -lms 100`
    child process; stopped by its exact PID)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.proc = gpu_index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            try:
                self.proc.terminate()
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            rows = [[c.strip() for c in ln.split(",")] for ln in out.strip().splitlines() if ln.count(",") >= 8]
        busy = [r for r in rows if r[3].replace(".", "").isdigit() and float(r[3]) > 250.0] or rows      # samples under load
        sm = sorted(float(r[1]) for r in busy if r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(rows), "samples_under_load": len(busy)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, stepper, out):
    """--dump-outputs: what a caller of the timed step holds after its last call, one float32 DIR/<name>.npy per array: the
    global-batch loss and flat gradient (DateShardedStep.loss / .grad) and, when the step runs in one piece rather than in
    micro-batches, the per-date and per-stock outputs of this rank's dates (the dict DateShardedStep.step returns)."""
    import numpy as np
    arrays = {"loss": stepper.loss, "grad": stepper.grad}
    arrays.update((k, v) for k, v in (out or {}).items() if k != "loss")        # out["loss"] is stepper.loss
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_reference(args, wl, rank, world):
    """Reference arm: the reference's own CPU implementation of the path -- the unmodified module.py from oracle/_ref
    (kind "reference"; oracle/cpu_port.py, kind "port", only if that copy is absent) -- on the host cores, one date per step as
    train_model.py does; each bench step = a bounded sample of `dates_per_step` dates of the workload's per-date shape."""
    if rank != 0:
        return
    import torch
    st = ReferenceStepper(wl, "cpu")
    g = torch.Generator().manual_seed(1234)
    dates_per_step = 4
    xs = [torch.randn(wl["N"], wl["T"], C_FEATURES, generator=g).clamp_(-3, 3) for _ in range(dates_per_step)]
    ys = [torch.randn(wl["N"], 1, generator=g) for _ in range(dates_per_step)]
    cores, ncpu = pick_threads(st, xs[0], ys[0])
    for _ in range(args.warmup):
        for x, y in zip(xs, ys):
            st.train_step(x, y)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for x, y in zip(xs, ys):
            st.train_step(x, y)
    dt = time.perf_counter() - t0
    value = args.steps * dates_per_step * wl["N"] / dt
    what = "the unmodified reference module.py (oracle/_ref)" if st.kind == "reference" else "oracle/cpu_port.py (oracle/_ref absent)"
    sample = (f"{dates_per_step} dates/step of the workload's per-date shape (N={wl['N']},T={wl['T']},K=H={wl['K']}), one date per "
              f"reference step (zero_grad, forward, loss.item(), backward; optimizer.step() not timed on either arm), fp32 torch CPU, "
              f"{what}, {cores} intra-op threads (fastest of 1..{ncpu} probed; host has {ncpu} CPUs)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "date*stocks/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload_desc},
            "cpu_baseline": {"value": value, "unit": "date*stocks/s", "cores": cores, "host_cpus": ncpu, "kind": st.kind, "sample": sample},
            "e2e": {"value": value, "unit": "date*stocks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def time_eager_b200(wl, dev, budget_s=4.0):
    """Secondary comparator (SURVEY 2.2 / 8d): the unmodified reference module.py through PyTorch eager on this B200 (cuDNN
    GRU + cuBLAS + ATen, fp32, one date per step) -- the only pre-existing Blackwell-capable implementation of the path."""
    import torch
    if load_reference_module() is None:
        return None
    st = ReferenceStepper(wl, dev)
    g = torch.Generator(device=dev).manual_seed(5)
    x = torch.randn(wl["N"], wl["T"], C_FEATURES, generator=g, device=dev).clamp_(-3, 3)
    y = torch.randn(wl["N"], 1, generator=g, device=dev)
    for _ in range(3):
        st.train_step(x, y)
    torch.cuda.synchronize()
    n, t0 = 0, time.perf_counter()
    while n < 5 or (time.perf_counter() - t0 < budget_s and n < 1000):
        st.train_step(x, y)
        n += 1
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) / n * 1e3
    return {"value": wl["N"] / (ms * 1e-3), "unit": "date*stocks/s", "ms_per_date": ms, "dates_timed": n,
            "what": "unmodified reference module.py (oracle/_ref), PyTorch eager on this GPU, fp32, one date per step "
                    "(zero_grad, forward, loss.item(), backward)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "bf16"])
    ap.add_argument("--panel", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the PyTorch-eager-on-B200 comparator")
    ap.add_argument("--collective", default="auto", choices=["auto", "p2p", "nccl"], help="gradient exchange: the one-kernel NVLink all-reduce or ncclAllReduce")
    ap.add_argument("--windows-e2e", action="store_true", help="also time the legacy variant that ships every window over PCIe")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.workload_desc = workload_desc(args.workload, world)
    if args.impl == "reference":
        return run_reference(args, wl, rank, world)

    import torch
    import torch.distributed as dist
    from factorvae_b200 import _cabi, engine
    from factorvae_b200.batched import DateShardedStep, shard_dates

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        # a stuck rendezvous / collective must end as an error within minutes, never as a hung box
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))
    N, T, H, K, M = (wl[k] for k in "NTHKM")
    strong = wl["scaling"] == "strong"
    if strong:
        B_global = wl["B"]
        d0, d1 = shard_dates(B_global, world, rank)
    else:
        B_global = wl["B"] * world
        d0, d1 = rank * wl["B"], (rank + 1) * wl["B"]
    B = d1 - d0                                   # dates of this rank
    S = B * N
    S_global = B_global * N
    precision = args.precision
    if precision == "auto":
        precision = "bf16" if engine.tc_supported(C_FEATURES, H) else "fp32"
    params = build_params(H, K, M)
    layout = engine.ParamLayout(C_FEATURES, H, K, M)
    flat = layout.pack(params, dev)

    # synthetic panel: N(0,1) clipped to +-3 per GLOBAL date id (identical global batch for any sharding)
    pdt = torch.bfloat16 if args.panel == "bf16" else torch.float32
    # rows padded to a 16-byte pitch ([S][T][160], 158 features used): every row is then a legal TMA box row (+1.3 % bytes)
    x_store = torch.zeros(S, T, 160 if pdt == torch.bfloat16 else C_FEATURES, dtype=pdt, device=dev)
    x = x_store[:, :, :C_FEATURES]
    y = torch.empty(S, dtype=torch.float32, device=dev)
    gen = torch.Generator(device=dev)
    for d in range(B):
        gen.manual_seed(1234 + d0 + d)
        x[d * N:(d + 1) * N] = torch.randn(N, T, C_FEATURES, generator=gen, device=dev).clamp_(-3, 3).to(pdt)
        y[d * N:(d + 1) * N] = torch.randn(N, generator=gen, device=dev)
    stepper = DateShardedStep(layout, flat, precision=precision, seed=42, collective=args.collective)
    unit_base = d0 * N
    lib = _cabi.lib()
    micro = min(wl["micro"], B)
    if micro >= B:
        date_ptr = engine.uniform_date_ptr(B, N, dev)

        def one_step():
            return stepper.step(x, y, date_ptr, global_dates=B_global, unit_base=unit_base, train=True)[0]
    else:
        mbs = []
        for m0 in range(0, B, micro):
            m1 = min(B, m0 + micro)
            mbs.append((x[m0 * N:m1 * N], y[m0 * N:m1 * N], engine.uniform_date_ptr(m1 - m0, N, dev), unit_base + m0 * N))

        def one_step():
            stepper.step_accumulate(mbs, global_dates=B_global, train=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    t_warm = time.perf_counter()
    for _ in range(args.warmup):
        one_step()
    # keep the GPU under load for ~0.5 s so the clock sampler sees a few samples.  The number of extra steps must be the
    # SAME on every rank (each step carries an all-reduce): agree on it with one collective instead of a per-rank clock.
    torch.cuda.synchronize()
    t_probe = time.perf_counter()
    nprobe = 10 if not strong else 2
    for _ in range(nprobe):                                        # fixed count: identical on every rank
        one_step()
    torch.cuda.synchronize()
    per_step = max((time.perf_counter() - t_probe) / nprobe, 1e-5)
    extra = torch.tensor([int(min(5000, max(0.0, 0.5 - (time.perf_counter() - t_warm)) / per_step))], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(extra, op=dist.ReduceOp.MAX)
    for _ in range(int(extra.item())):
        one_step()
    barrier()
    # the number of load steps above follows the clock: restart the Philox step counter so that the timed steps are always
    # steps 1..K of the noise stream, and runs with the same arguments compute the same outputs
    stepper.step_index = 0
    l0 = lib.fvae_debug_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        last_out = one_step()
    ev1.record()
    barrier()
    launches = lib.fvae_debug_launch_count() - l0
    clocks = sampler.stop() if sampler else None
    ms = ev0.elapsed_time(ev1)
    loss_val = float(stepper.loss.item())
    if args.dump_outputs and rank == 0:                 # before the sections below reuse the step's buffers
        dump_outputs(args.dump_outputs, stepper, last_out)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = S_global / (ms_per_step * 1e-3)

    # ---- launch-bound workloads (the reference's own per-date step, configs[0]): the same step captured in a CUDA graph
    graph_detail = None
    if world == 1 and micro >= B and S <= 8192:
        try:
            g = stepper.capture(x, y, date_ptr, unit_base=unit_base, train=True)
            for _ in range(max(3, args.warmup)):
                g.replay()
            torch.cuda.synchronize()
            nrep = args.steps
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(nrep):
                g.replay()
            g1.record()
            torch.cuda.synchronize()
            gms = g0.elapsed_time(g1) / nrep
            graph_detail = {"ms_per_step": gms, "value": S_global / (gms * 1e-3), "replays": nrep, "loss": float(stepper.loss.item()),
                            "note": "DateShardedStep.capture: forward + backward of this batch shape replayed as ONE CUDA graph launch; "
                                    "Philox step counter in device memory (fvae_noise.step_dev), advanced by the graph"}
        except Exception as exc:                        # diagnostics only: never take the bench line down
            graph_detail = {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}

    # ---- roofline of the dominant kernel, timed ALONE with CUDA events on the launching stream
    # dominant kernel = the front forward (K1: LayerNorm -> GEMM 128x160x160 -> LeakyReLU -> GEMM 128xNCx160 per item);
    # algorithmic work per launch: FLOPs = S*T*2*(C^2 + 3HC); bytes = one read of the bf16 panel (S*T*C*2).
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_burst = float(peaks.get("bf16_tflops", 1590.0))
    peak_sust = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_hbm = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md: 1.59 PFLOP/s burst, 6.65 TB/s)"
    flops_step = S_global * f_fe(T, H)
    step_tf = flops_step / (ms_per_step * 1e-3) / 1e12 / world         # per GPU
    roofline = None
    Sk = min(S, micro * N)                                              # sequences of one launch of the kernel
    if rank == 0 and precision == "bf16":
        xk, yk = x[:Sk], y[:Sk]
        out_k, st_k = engine.elbo_forward(layout, flat, xk, yk, engine.uniform_date_ptr(Sk // N, N, dev), train=True,
                                          precision="bf16", philox=(42, 1, unit_base))
        torch.cuda.synchronize()
        reps = args.steps
        for _ in range(3):
            engine.rerun_front_forward(st_k)
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(reps):
            engine.rerun_front_forward(st_k)
        k1.record()
        torch.cuda.synchronize()
        k_ms = k0.elapsed_time(k1) / reps
        k_flops = Sk * T * 2.0 * (C_FEATURES * C_FEATURES + 3 * H * C_FEATURES)
        k_bytes = Sk * T * C_FEATURES * (2 if args.panel == "bf16" else 4)
        traffic, traffic_src = None, None
        try:       # DRAM bytes of this kernel from the committed `ncu --set full` capture (ncu cannot run inside the timed bench)
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_step_traffic.json")))
            if args.workload == tj.get("workload"):
                traffic, traffic_src = tj.get("front_forward_dram_bytes_per_launch"), "profiles/r02_step_traffic.json (ncu --set full, one step)"
        except Exception:
            pass
        ach = k_flops / (k_ms * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": "front forward (K1): LayerNorm + GEMM1 + LeakyReLU + GEMM2 per 128-row item", "achieved": ach,
                    "peak": peak_burst, "unit": "TFLOP/s",
                    "frac": ach / peak_burst, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peak_src + ", burst figure (kernel timed alone)",
                    "kernel_ms": k_ms, "algorithmic_flops_per_launch": k_flops, "algorithmic_bytes_per_launch": k_bytes,
                    "hbm_algorithmic_gbs": k_bytes / (k_ms * 1e-3) / 1e9, "hbm_frac_algorithmic": k_bytes / (k_ms * 1e-3) / 1e9 / peak_hbm,
                    "step": {"achieved": step_tf, "peak": peak_sust, "frac": step_tf / peak_sust,
                             "note": "whole ELBO step (all kernels), per GPU: S*3*2T(C^2+3HC+3H^2) algorithmic FLOPs / step time vs sustained bf16 peak"}}
        del out_k, st_k
    elif rank == 0:
        roofline = {"bound": "tensor", "kernel": "whole step (fp32 CUDA-core mode)", "achieved": step_tf, "peak": peak_sust,
                    "unit": "TFLOP/s", "frac": step_tf / peak_sust, "traffic": None, "peak_source": peak_src}

    # ---- end to end through the host-buffer entry of the RESIDENT row table (SURVEY 8 f-1; replaces dataset.py:139-181,207-249
    # and train_model.py:17-24).  Per step, inside the timed region: the batch's NEW rows (B*N rows x 160 bf16 + labels) and its
    # date ids are copied from pinned host memory (copy stream, into the table the NEXT step reads, under the current step's
    # compute), fvae_window_index builds the look-back index, the ELBO kernels read the rows in place, the loss is copied to
    # pinned host memory and read there (the read of step i happens while step i+1 is queued: one-step-deferred logging).
    e2e = None
    n_e2e = args.steps
    if not args.no_e2e and not strong:
        import numpy as np
        from factorvae_b200.panel import PanelIndex, ResidentPanel
        Dn = B + T - 1
        idx_mat = np.arange(Dn * N, dtype=np.int32).reshape(Dn, N)
        sd = np.repeat(np.arange(T - 1, Dn, dtype=np.int32), N)
        sj = np.tile(np.arange(N, dtype=np.int32), B)
        pidx = PanelIndex(idx_mat, sd, sj, np.arange(0, (B + 1) * N, N), Dn * N)
        grow = torch.Generator(device="cpu").manual_seed(99 + rank)
        vals = torch.randn(Dn * N, C_FEATURES + 1, generator=grow).clamp_(-3, 3).numpy()
        tables = [ResidentPanel(vals, pidx, C_FEATURES, dev, dtype=pdt) for _ in range(2)]     # double-buffered row table
        pitch = tables[0].table.shape[1]
        first_new = (T - 1) * N                                             # rows of the batch's B dates (the history is resident)
        rows_h = tables[0].table[first_new:first_new + B * N].to("cpu").pin_memory()
        lab_h = tables[0].label[first_new:first_new + B * N].to("cpu").pin_memory()
        dates_h = torch.arange(B, dtype=torch.int32).pin_memory()
        dates_d = torch.empty(B, dtype=torch.int32, device=dev)
        loss_h = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        compute = torch.cuda.current_stream(dev)
        copy_stream = torch.cuda.Stream(dev)
        uploaded = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]
        done = [torch.cuda.Event(), torch.cuda.Event()]
        losses = []

        def upload(slot):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])                      # the step that last read this table has finished
                tables[slot].upload_rows(first_new, rows_h, lab_h)
                dates_d.copy_(dates_h, non_blocking=True)                   # which dates the step trains on (same copy stream: a small H2D
                uploaded[slot].record(copy_stream)                          # on the compute stream would queue behind the 25 MB upload)

        host = {"issue": 0.0, "wait": 0.0}
        def run_resident(nsteps, stream_rows):
            """stream_rows False: the table is resident (uploaded once, untimed -- the reference's one-time pickle load); the
            step's host input is WHICH dates to train on.  True: additionally the batch's new rows are (re)uploaded every step."""
            t_a = time.perf_counter()
            consumed[0].record(compute); consumed[1].record(compute)
            if stream_rows:
                upload(0)
            for i in range(nsteps):
                slot = i & 1 if stream_rows else 0
                if stream_rows:
                    if i + 1 < nsteps:
                        upload(slot ^ 1)                                    # next step's rows, under this step's compute
                    compute.wait_event(uploaded[slot])
                else:
                    dates_d.copy_(dates_h, non_blocking=True)               # the step's host input: the date ids of the batch
                xw, yw, pw = tables[slot].batch(range(B), T)                # window-index kernel (+ labels)
                stepper.step(xw, yw, pw, global_dates=B_global, unit_base=unit_base, train=True)
                consumed[slot].record(compute)
                b = i & 1
                loss_h[b].copy_(stepper.loss.reshape(1), non_blocking=True)         # D2H of the loss
                done[b].record(compute)
                if i >= 1:                                                  # host read of the previous step's loss
                    t_b = time.perf_counter()
                    done[b ^ 1].synchronize()
                    t_c = time.perf_counter()
                    host["issue"] += t_b - t_a; host["wait"] += t_c - t_b; t_a = t_c
                    losses.append(float(loss_h[b ^ 1][0]))
            done[(nsteps - 1) & 1].synchronize()
            losses.append(float(loss_h[(nsteps - 1) & 1][0]))

        def time_resident(stream_rows):
            run_resident(8, stream_rows)          # warm-up: both table slots, every allocation size seen by the caching allocator
            # the host-side set-up of this section (numpy panel, table uploads) left the GPU idle long enough to drop its clocks:
            # keep it under load for ~0.4 s before timing, like the main loop does.  Same count on every rank (each step carries
            # the gradient exchange).
            torch.cuda.synchronize()
            t_p = time.perf_counter()
            run_resident(8, stream_rows)
            torch.cuda.synchronize()
            per = max((time.perf_counter() - t_p) / 8, 1e-5)
            nload = torch.tensor([int(min(2000, 0.4 / per))], dtype=torch.int64, device=dev)
            if world > 1:
                dist.all_reduce(nload, op=dist.ReduceOp.MAX)
            run_resident(max(2, int(nload.item())), stream_rows)
            barrier()
            host["issue"] = host["wait"] = 0.0
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            run_resident(n_e2e, stream_rows)
            r1.record()
            barrier()
            t3 = torch.tensor([r0.elapsed_time(r1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t3, op=dist.ReduceOp.MAX)
            return float(t3.item()) / n_e2e, {"issuing": host["issue"] / n_e2e * 1e3, "blocked_on_gpu": host["wait"] / n_e2e * 1e3}

        msr, host_res = time_resident(False)
        mss, host_str = time_resident(True)
        h2d_rows = rows_h.numel() * rows_h.element_size() + lab_h.numel() * 4 + dates_h.numel() * 4
        pname = str(pdt).replace("torch.", "")
        e2e = {"value": S_global / (msr * 1e-3), "unit": "date*stocks/s", "ms_per_step": msr, "h2d_bytes_per_step": dates_h.numel() * 4,
               "d2h_bytes_per_step": 4, "host_panel_dtype": pname,
               "entry": "ResidentPanel.batch + DateShardedStep.step (date ids in, loss out)",
               "note": "the (date, instrument) row table (%.1f MB %s, pitch %d) is uploaded ONCE, untimed, like the reference's one-time "
                       "pickle load (main.py:36); per step, inside the timed region: the batch's date ids H2D from pinned memory, "
                       "fvae_window_index (TSDataSampler._get_indices), the ELBO step reading rows through fvae_panel.row_index, the loss D2H "
                       "and its host read (deferred by one step).  The reference's loader instead rebuilds every window on the host "
                       "and ships each row T times as fp32" % (tables[0].table.numel() * tables[0].table.element_size() / 1e6, pname, pitch),
               "host_ms_per_step": host_res, "last_loss": losses[-1],
               "stream_new_rows": {"value": S_global / (mss * 1e-3), "ms_per_step": mss, "h2d_bytes_per_step": h2d_rows,
                                   "h2d_gbs": h2d_rows / (mss * 1e-3) / 1e9, "host_ms_per_step": host_str,
                                   "note": "streaming variant: additionally the batch's B*N new rows (+ labels) are uploaded every step from pinned "
                                           "memory into a double-buffered table on a copy stream under the previous step's compute (each row "
                                           "crosses PCIe once); bounded by the host's PCIe share on a busy box"}}
        if args.windows_e2e:       # legacy variant: the (S, T, C) fp32 window tensor crosses PCIe every step (what the reference's loader yields)
            ph = engine.uniform_date_ptr(B, N, dev).to("cpu").pin_memory()
            yh = y.to("cpu").pin_memory()
            xh32 = x.float().to("cpu").pin_memory()
            kw = dict(global_dates=B_global, unit_base=unit_base, train=True)
            for _ in stepper.run_from_host([(xh32, yh, ph)] * 3, **kw):
                pass
            barrier()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in stepper.run_from_host([(xh32, yh, ph)] * n_e2e, **kw):
                pass
            b1.record()
            barrier()
            msw = b0.elapsed_time(b1) / n_e2e
            e2e["windows_over_pcie"] = {"value": S_global / (msw * 1e-3), "ms_per_step": msw,
                                        "h2d_bytes_per_step": xh32.numel() * 4 + yh.numel() * 4 + ph.numel() * 4,
                                        "note": "legacy: the fp32 (S,T,C) window tensor is shipped every step (20x redundant rows)"}
            del xh32
        del tables

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        r = time_reference_cpu(wl, budget_s=10.0)
        what = "the unmodified reference module.py (oracle/_ref)" if r["kind"] == "reference" else "oracle/cpu_port.py"
        cpu_baseline = {"value": r["value"], "unit": "date*stocks/s", "cores": r["cores"], "host_cpus": r["host_cpus"], "kind": r["kind"],
                        "sample": f"{r['steps']} per-date reference steps (N={N},T={T},K=H={K}; zero_grad, forward, loss.item(), backward; "
                                  f"no optimizer) in ~10 s, median {r['ms_per_date']:.2f} ms/date, fp32 torch CPU, {what}, "
                                  f"{r['cores']} intra-op threads (fastest probed) of {r['host_cpus']} host CPUs"}
    eager = None
    if rank == 0 and world == 1 and not args.no_eager:
        try:
            eager = time_eager_b200(wl, dev)
        except Exception as exc:                       # a comparator must never take the bench line down
            eager = {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}
    if roofline is not None:
        roofline["eager_b200"] = eager

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "date*stocks/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": wl["scaling"],
                "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
                "config": {"workload": args.workload_desc},
                "detail": {"panel_dtype": args.panel, "precision": precision,
                           "l2": "inputs larger than L2 (panel %.0f MB per GPU)" % (x_store.numel() * x_store.element_size() / 1e6),
                           "panel_layout": "x[S][T][%d] %s, %d features per row used (row pitch padded to 16 bytes)" % (x_store.shape[2], args.panel, C_FEATURES),
                           "noise": "in-kernel Philox (eps + dropout masks), keyed by global unit id",
                           "parallelism": f"dp{world} over dates", "dates_per_gpu": B, "micro_batch_dates": micro,
                           "collective": ("one all-reduce of the flat fp32 gradient (+ loss) per step: " +
                                          ("one kernel over NVLink peer memory (fvae_p2p_allreduce)" if stepper.p2p is not None else "ncclAllReduce"))
                                         if world > 1 else "none"},
                "cuda_graph": graph_detail,
                "loss": loss_val, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
                "cpu_baseline": cpu_baseline, "e2e": e2e}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
