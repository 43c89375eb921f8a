#!/usr/bin/env python
"""bench.py -- filtered observation-steps/s (N x K per second) of the batched CD-EKF hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): CD-EKF on stochastic Lorenz-63,
d_x = 3, d_y = 1 (observe x), N = 65,536 trajectories, K = 1,000 irregular observation times, classical RK4 moment ODE
with dt0 = mean gap / 4.  One "step" = one filter pass over the whole batch (update + predict for all N x K
observation-steps, writing the four moment arrays the reference returns by default) followed by the sum of the
per-trajectory log-likelihoods and, at N > 1 GPUs, one all-reduce of that scalar (cdk_ll_allreduce on a raw NCCL
communicator).  Trajectories are independent and shard with no data-path collective.

`--scaling strong` (default): the north star's FIXED N = 65,536 is split over the ranks (parallel.shard_bounds), so the
            value at 8 GPUs is the 8-GPU time of the SAME job; `--scaling weak`: 65,536 trajectories PER GPU.  At N > 1 the
            other mode is measured too and reported beside the headline (`weak_scaling` / `strong_scaling` object).

`value`   : inputs resident in HBM, CUDA-event timed, max over ranks.
`e2e`     : the same metric through the public drop-in API with HOST (pinned) buffers: every step copies emissions and
            time stamps host->device and reads the log-likelihoods device->host.
`--impl reference`: the CPU restatement of the reference algorithm (oracle/, C + OpenMP, all host cores) on a bounded
            sample of the same workload.  The reference's own JAX path cannot run here (jax/diffrax are not
            installable in this image; BASELINE.md section 2) -- this is a "CPU restatement (not JAX)".
`--dump-outputs DIR`: after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64): the
            per-trajectory outputs of the posterior (marginal_loglik, filtered/predicted means and covariances) for a
            fixed, seeded sample of rank 0's trajectories, at most 60 MB in all, and ll_sum, the summed log-likelihood
            of the whole batch.  The inputs depend on the arguments only, so two builds run with the same arguments can
            be compared output for output.

The benchmark writes nothing into the source tree, which may be read-only.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ in the source tree

METRIC = "filtered observation-steps/sec (N x K per second)"
UNIT = "obs-steps/s"
CFG = dict(N=65536, K=1000, n=3, m=1, mean_gap=0.01, dt0=0.0025, solver="rk4", seed=1237)
# flop model (1 FMA = 2 flop).  SURVEY 8(d) ALGORITHMIC count: 496*q + 107 per observation-step for n=3, m=1 (dense
# 3x3 products, loop-invariant L Qc L^T hoisted) -- this is the figure `roofline.achieved` is computed from.
# The kernel stores P symmetric (6 entries), uses the sparsity of the Lorenz-63 Jacobian and folds dt into the RK
# coefficients, so it EXECUTES fewer: per RK4 substep 4 stages * (f 8 + J.P 33 + dP 12 + stage/accumulate FMAs 36) - 18
# = 324 (SASS: 143 DFMA + 25 DADD + 13 DMUL per substep; 338 = 127 + 51 + 25 before the leaner covariance RHS); scalar-emission update 60.  Both are reported (`achieved` /
# `achieved_executed`).
FLOP_SUBSTEP_SURVEY, FLOP_UPDATE_SURVEY = 496.0, 107.0
FLOP_SUBSTEP_EXEC, FLOP_UPDATE_EXEC = 324.0, 60.0
BYTES_PER_OBS_STEP = 16 + 192  # y,t in (16 B) + filtered/predicted mean+cov out (24 doubles)
TRAFFIC_NCU_BYTES = 15.15e9  # dram read 1.95 GB + write 13.19 GB: profiles/r02_ekf_small_lw_time_sliced_N65536.txt


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: --n-traj is the TOTAL batch, split over the GPUs (north star); weak: --n-traj per GPU")
    ap.add_argument("--n-traj", type=int, default=CFG["N"], help="trajectories (default = BASELINE config 3: 65,536)")
    ap.add_argument("--no-other-mode", action="store_true", help="at N > 1 GPUs skip the second (other scaling mode) measurement")
    ap.add_argument("--k-obs", type=int, default=CFG["K"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg (profiling runs)")
    ap.add_argument("--cpu-sample-traj", type=int, default=0, help="trajectories in the CPU sample (0 = auto)")
    ap.add_argument("--simple-data", action="store_true",
                    help="emissions = 8*randn instead of a simulated Lorenz-63 truth (profiling runs: skips the "
                         "~100k setup launches that would otherwise sit in front of the profiled kernel)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def l63(x, s=10.0, r=28.0, b=8.0 / 3.0):
    import torch
    return torch.stack([s * (x[:, 1] - x[:, 0]), x[:, 0] * (r - x[:, 2]) - x[:, 1], x[:, 0] * x[:, 1] - b * x[:, 2]], 1)


def make_emissions(t, seed, first_traj, device):
    """Synthetic data from the library's own batched sampler (cdk_sample_path, ONE launch; SURVEY 8f rank 2): the stochastic
    Lorenz-63 truth started near the attractor (x_0 ~ N([1, 1, 20], I)), Euler-Maruyama with 8 substeps per mean gap,
    Qc = I, observe x with unit noise.  The Philox counter is the GLOBAL trajectory index (rng_offset = first_traj), so a
    shard of the strong-scaling run sees the same data whatever the number of GPUs.  Setup only, never timed."""
    import torch

    import cd_dynamax_b200 as cd
    f64 = dict(dtype=torch.float64, device=device)
    truth = cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(torch.tensor([1.0, 1.0, 20.0], **f64)),
                                      cov=cd.LearnableMatrix(torch.eye(3, **f64))),
        dynamics=cd.ParamsCDNLGSSMDynamics(
            drift=cd.LearnableLorenz63(sigma=torch.tensor(10.0, **f64), rho=torch.tensor(28.0, **f64),
                                       beta=torch.tensor(8.0 / 3.0, **f64)),
            diffusion_coefficient=cd.LearnableMatrix(torch.eye(3, **f64)), diffusion_cov=cd.LearnableMatrix(torch.eye(3, **f64))),
        emissions=cd.ParamsCDNLGSSMEmissions(
            emission_function=cd.LearnableLinear(weights=torch.tensor([[1.0, 0.0, 0.0]], **f64), bias=torch.zeros(1, **f64)),
            emission_cov=cd.LearnableMatrix(torch.eye(1, **f64))))
    if t.shape[0] == 0:
        return torch.empty(0, t.shape[1], 1, **f64)
    _, y = cd.cdnlgssm_path_sample(truth, seed, t.shape[1], t[..., None],
                                   diffeqsolve_settings={"solver": "euler", "dt0": CFG["mean_gap"] / 8},
                                   rng_offset=first_traj, device_resident=True)
    return y


def make_emissions_torch(t, seed, device):
    """Synthetic data: simulate the stochastic Lorenz-63 truth (Euler-Maruyama, 8 substeps per gap, Qc = I) and
    observe x with unit noise.  Runs in torch on `device` (setup only, never timed)."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    N, K = t.shape
    x = torch.tensor([1.0, 1.0, 20.0], dtype=torch.float64, device=device).repeat(N, 1)
    x = x + torch.randn(N, 3, generator=g, device=device, dtype=torch.float64)
    y = torch.empty(N, K, 1, dtype=torch.float64, device=device)
    sub = 8
    for k in range(K):
        if k > 0:
            h = ((t[:, k] - t[:, k - 1]) / sub)[:, None]
            for _ in range(sub):
                x = x + h * l63(x) + torch.sqrt(h) * torch.randn(N, 3, generator=g, device=device, dtype=torch.float64)
        y[:, k, 0] = x[:, 0] + torch.randn(N, generator=g, device=device, dtype=torch.float64)
    return y


def substeps_total(t, dt0, dt_final=1e-10):
    """Sum over all gaps of the solver substep count q_k (diffrax clipping rule), vectorised closed form checked
    against oracle.substep_counts in tests."""
    from oracle.cd_oracle import substep_counts
    t1 = np.concatenate([t[:, 1:], t[:, -1:] + dt_final], axis=1)
    # bounded memory: process in row blocks
    tot = 0
    for i in range(0, t.shape[0], 8192):
        tot += int(substep_counts(t[i:i + 8192], t1[i:i + 8192], dt0).sum())
    return tot


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            p = [c.strip() for c in r.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def cpu_reference_leg(n_traj, K, steps, warmup):
    """Time the CPU restatement (oracle/, C + OpenMP when built, else NumPy) on a bounded sample of the workload."""
    from oracle import cpu_baseline
    return cpu_baseline.time_ekf_l63(n_traj, K, CFG, steps=steps, warmup=warmup)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_traj = args.cpu_sample_traj or 512 * cores
    res = cpu_reference_leg(n_traj, args.k_obs, steps=args.steps, warmup=min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.gpus, extra={"cpu_sample": res["sample"]}),
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"],
                         "sample": res["sample"], "value_ll_only": res.get("value_ll_only")},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of the reference algorithm (C + OpenMP port, naive dense runtime-n loops; NOT the "
                "reference's JAX path: jax/diffrax are not installable in this image)",
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world, extra=None):
    strong = args.scaling == "strong"
    c = {"workload": "CD-EKF stochastic Lorenz-63 (BASELINE configs[2])",
         "n_traj_total": args.n_traj if strong else args.n_traj * world,
         "n_traj_per_gpu": (args.n_traj + world - 1) // world if strong else args.n_traj,
         "k_obs": args.k_obs, "d_x": 3, "d_y": 1, "state_order": "second", "solver": "rk4", "dt0": CFG["dt0"],
         "mean_gap": CFG["mean_gap"], "outputs": "filtered+predicted means and covariances, log-likelihood",
         "parallelism": f"trajectory-sharded x{world} (no data-path collective; 1 all-reduce of sum ll)",
         "l2": "inputs+outputs per step (>= 1 GB per 65,536 trajectories) exceed the 126 MB L2; no explicit flush"}
    if extra:
        c.update(extra)
    return c


class Job:
    """One rank's share of the workload, resident on its GPU, plus the pre-marshalled direct C-ABI launch used to time
    the kernel alone."""

    def __init__(self, n_local, first_traj, K, rank, dev, simple_data):
        import torch

        import cd_dynamax_b200 as cd
        self.N, self.K, self.dev = n_local, K, dev
        # time grids: rows [first_traj, first_traj + n_local) of ONE global generator stream per 8,192-row block, so a
        # shard of the strong-scaling run filters the same grids whatever the number of GPUs
        self.t_np = make_times_rows(first_traj, n_local, K, CFG["seed"])
        self.t_dev = torch.as_tensor(self.t_np, device=dev)
        if simple_data:
            gen = torch.Generator(device=dev)
            gen.manual_seed(CFG["seed"] + first_traj)
            self.y_dev = 8.0 * torch.randn(n_local, K, 1, generator=gen, device=dev, dtype=torch.float64)
        else:
            self.y_dev = make_emissions(self.t_dev, CFG["seed"], first_traj, dev)
        self.sum_q = substeps_total(self.t_np, CFG["dt0"]) if n_local else 0
        f64 = dict(dtype=torch.float64, device=dev)
        self.params = cd.ParamsCDNLGSSM(
            initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(torch.zeros(3, **f64)),
                                          cov=cd.LearnableMatrix(5.0 * torch.eye(3, **f64))),
            dynamics=cd.ParamsCDNLGSSMDynamics(
                drift=cd.LearnableLorenz63(sigma=torch.tensor(10.0, **f64), rho=torch.tensor(28.0, **f64),
                                           beta=torch.tensor(8.0 / 3.0, **f64)),
                diffusion_coefficient=cd.LearnableMatrix(torch.eye(3, **f64)),
                diffusion_cov=cd.LearnableMatrix(torch.eye(3, **f64))),
            emissions=cd.ParamsCDNLGSSMEmissions(
                emission_function=cd.LearnableLinear(weights=torch.tensor([[1.0, 0.0, 0.0]], **f64),
                                                     bias=torch.zeros(1, **f64)),
                emission_cov=cd.LearnableMatrix(torch.eye(1, **f64))))
        self.hp = cd.EKFHyperParams(state_order="second",
                                    diffeqsolve_settings={"solver": cd.solvers.RK4(), "dt0": CFG["dt0"]})

    def direct_launch(self, lib, L):
        """cdk_ekf_filter_f64 with every pointer marshalled ONCE: calling the returned function enqueues exactly one
        ekf_small_lw launch (all four moment outputs) on the given stream and nothing else."""
        import torch
        N, K, dev = self.N, self.K, self.dev
        f64 = dict(dtype=torch.float64, device=dev)
        d = L.new_desc()
        d.N, d.K, d.n, d.m = N, K, 3, 1
        d.solver, d.dt0, d.state_order, d.num_iter = L.SOLVERS["rk4"], CFG["dt0"], 2, 1
        d.drift_id, d.n_theta, d.emission_id = L.DRIFT_LORENZ63, 3, 0
        d.batched_mask = (1 << L.IN_Y) | (1 << L.IN_T)
        ins = {L.IN_Y: self.y_dev, L.IN_T: self.t_dev, L.IN_M0: torch.zeros(3, **f64), L.IN_P0: 5.0 * torch.eye(3, **f64),
               L.IN_F: torch.tensor([10.0, 28.0, 8.0 / 3.0], **f64), L.IN_L: torch.eye(3, **f64),
               L.IN_QC: torch.eye(3, **f64), L.IN_H: torch.tensor([[1.0, 0.0, 0.0]], **f64), L.IN_D: torch.zeros(1, **f64),
               L.IN_R: torch.eye(1, **f64)}
        outs = {L.OUT_LL: torch.empty(N, **f64), L.OUT_FM: torch.empty(N, K, 3, **f64),
                L.OUT_FP: torch.empty(N, K, 3, 3, **f64), L.OUT_PM: torch.empty(N, K, 3, **f64),
                L.OUT_PP: torch.empty(N, K, 3, 3, **f64), L.OUT_STATUS: torch.zeros(N, dtype=torch.int32, device=dev)}
        in_ptrs = (ctypes.c_void_p * L.NUM_IN)()
        out_ptrs = (ctypes.c_void_p * L.NUM_OUT)()
        for slot, t in ins.items():
            in_ptrs[slot] = t.data_ptr()
        for slot, t in outs.items():
            out_ptrs[slot] = t.data_ptr()
        keep = (d, ins, outs, in_ptrs, out_ptrs)

        def launch(stream):
            L.check(lib.cdk_ekf_filter_f64(ctypes.byref(d), in_ptrs, out_ptrs, ctypes.c_void_p(stream.cuda_stream)),
                    "cdk_ekf_filter_f64")
        launch.keep = keep
        return launch


def make_times_rows(first, count, K, seed, block=8192):
    """Rows [first, first + count) of the global time-grid array: block b of 8,192 trajectories comes from
    PCG64(seed + b), so any shard can be generated without the others."""
    out = np.empty((count, K))
    r = 0
    while r < count:
        g = first + r
        b, off = divmod(g, block)
        take = min(block - off, count - r)
        rng = np.random.Generator(np.random.PCG64(seed + b))
        gaps = CFG["mean_gap"] * rng.uniform(0.5, 1.5, size=(block, K))[off:off + take]
        gaps[:, 0] = 0.0
        out[r:r + take] = np.cumsum(gaps, axis=1)
        r += take
    return out


def time_resident(job, args, steps, ctx):
    """W warm-up passes, then `steps` passes through the public API with resident inputs, bracketed by barrier + sync;
    CUDA events on the launching stream, max over ranks.  Returns (ms total, launches, ll_total, non-finite count, clocks,
    (posterior, summed log-likelihood) of the last timed pass)."""
    import torch
    import cd_dynamax_b200 as cd
    from cd_dynamax_b200 import _engine as E
    dist, world, rank, dev, lib = ctx["dist"], ctx["world"], ctx["rank"], ctx["dev"], ctx["lib"]

    def step():
        if job.N > 0:
            post = cd.cdnlgssm_filter(job.params, job.y_dev, job.t_dev[..., None], job.hp)
            s = E.ll_sum(post.marginal_loglik)
        else:
            post, s = None, torch.zeros(1, dtype=torch.float64, device=dev)
        ctx["allreduce"](s)  # one all-reduce of 8 bytes when world > 1
        return post, s

    for _ in range(max(args.warmup, 3)):
        post, s = step()
    ctx["barrier"]()
    ll_total = float(s.item())
    n_bad = int((post.marginal_loglik != post.marginal_loglik).sum().item()) if post is not None else 0
    del post
    sampler = ClockSampler(ctx["local_rank"])
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = lib.cdk_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx["barrier"]()
    e0.record()
    for _ in range(steps):
        post = None  # the previous pass's outputs are freed before this pass allocates its own
        post, s = step()
    e1.record()
    ctx["barrier"]()
    launches = lib.cdk_launch_count() - launches0
    tmax = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    return float(tmax.item()), int(launches), ll_total, n_bad, clocks, (post, s)


DUMP_BYTES = 60_000_000


def dump_outputs(out_dir, post, ll_sum, seed=CFG["seed"]):
    """Write the outputs of one timed pass as out_dir/<name>.npy: ll_sum, and every per-trajectory field of the posterior
    for the same sample of trajectories (all of them when they fit in DUMP_BYTES, else a sorted sample drawn with a fixed
    seed, so that it depends on the batch size only)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    fields = {k: v for k, v in post._asdict().items() if v is not None}
    n = fields["marginal_loglik"].shape[0]
    row_bytes = sum(v[:1].numel() * v.element_size() for v in fields.values())
    rows = min(n, DUMP_BYTES // row_bytes)
    idx = np.sort(np.random.default_rng(seed).choice(n, size=rows, replace=False)) if rows < n else np.arange(n)
    sel = torch.as_tensor(idx, device=fields["marginal_loglik"].device)
    for name, v in fields.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.index_select(0, sel).cpu().numpy())
    np.save(os.path.join(out_dir, "ll_sum.npy"), ll_sum.cpu().numpy())


def time_kernel(job, ctx, reps=7):
    """Average duration of ONE ekf_small_lw launch: the kernel is enqueued back to back through the pre-marshalled C-ABI
    call and the events sit between two launches on the launching stream, so neither Python marshalling nor launch
    latency is inside the interval (the GPU is still busy with the previous launch when the next is enqueued)."""
    import torch
    if job.N == 0:
        return None
    stream = torch.cuda.current_stream(ctx["dev"])
    launch = job.direct_launch(ctx["lib"], ctx["L"])
    launch(stream)
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    launch(stream)  # keeps the GPU busy while the timed launches are enqueued
    for i in range(reps):
        evs[i].record(stream)
        launch(stream)
    evs[reps].record(stream)
    torch.cuda.synchronize()
    ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(reps)]
    del launch
    return float(np.mean(ms))


def time_e2e(job, args, ctx, all_outputs=False, n_limit=None):
    """The same metric through the public drop-in API with HOST (pinned) buffers: every step copies emissions and time
    stamps host->device and reads the result device->host (the [N] log-likelihoods, or -- all_outputs -- the four moment
    arrays as well, the work the CPU arm does).  Returns (ms total, steps, h2d bytes, d2h bytes, N used, ll host)."""
    import torch
    import cd_dynamax_b200 as cd
    dist, world, dev = ctx["dist"], ctx["world"], ctx["dev"]
    N = job.N if n_limit is None else min(job.N, n_limit)
    if N > 0:
        y_host = job.y_dev[:N].cpu().pin_memory()
        t_host = job.t_dev[:N].cpu().pin_memory()[..., None]
    p_host = cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(np.zeros(3)), cov=cd.LearnableMatrix(5.0 * np.eye(3))),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableLorenz63(sigma=10.0, rho=28.0, beta=8.0 / 3.0),
                                           diffusion_coefficient=cd.LearnableMatrix(np.eye(3)),
                                           diffusion_cov=cd.LearnableMatrix(np.eye(3))),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=np.array([[1.0, 0, 0]]),
                                                                                  bias=np.zeros(1)),
                                             emission_cov=cd.LearnableMatrix(np.eye(1))))

    def step():
        if N == 0:
            return None
        if all_outputs:
            return cd.cdnlgssm_filter(p_host, y_host, t_host, job.hp)
        return cd.cdnlgssm_filter(p_host, y_host, t_host, job.hp, output_fields=[])

    for _ in range(2):
        post = step()
    ctx["barrier"]()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = max(3, min(args.steps, 10)) if not all_outputs else 3
    e0.record()
    for _ in range(steps):
        post = step()
    e1.record()
    ctx["barrier"]()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    h2d = int(N * job.K * 16)
    d2h = int(N * 8 + (N * job.K * 24 * 8 if all_outputs else 0))
    ll_host = post.marginal_loglik if post is not None else None
    return float(ms.item()), steps, h2d, d2h, N, ll_host


def probe_fp64_peaks(ctx):
    """FP64 FMA peak probes (roofline denominators; MEASURED_PEAKS.json has no FP64 entry)."""
    import torch
    lib, L, dev = ctx["lib"], ctx["L"], ctx["dev"]
    stream = torch.cuda.current_stream(dev)
    blocks, iters = 148 * 8, 20000
    sink = torch.empty(blocks * 256, dtype=torch.float64, device=dev)
    seed = torch.rand(256, dtype=torch.float64, device=dev)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = best3 = 0.0
    for _ in range(5):
        p0.record()
        L.check(lib.cdk_fma_probe_f64(blocks, iters, ctypes.c_void_p(sink.data_ptr()), ctypes.c_void_p(stream.cuda_stream)),
                "fma_probe")
        p1.record()
        torch.cuda.synchronize()
        best = max(best, 2.0 * 16 * iters * blocks * 256 / (p0.elapsed_time(p1) * 1e-3) / 1e12)
    for _ in range(5):  # three distinct register operands per DFMA (what filter arithmetic looks like)
        p0.record()
        L.check(lib.cdk_fma3_probe_f64(blocks, iters, ctypes.c_void_p(sink.data_ptr()), ctypes.c_void_p(seed.data_ptr()),
                                       ctypes.c_void_p(stream.cuda_stream)), "fma3_probe")
        p1.record()
        torch.cuda.synchronize()
        best3 = max(best3, 2.0 * 16 * iters * blocks * 256 / (p0.elapsed_time(p1) * 1e-3) / 1e12)
    return best, best3


def run_ours(args):
    import torch
    import torch.distributed as dist

    from cd_dynamax_b200 import _lib as L
    from cd_dynamax_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.lib()
    K = args.k_obs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the one collective of the path: cdk_ll_allreduce (C ABI) on a raw ncclComm_t created outside torch.distributed, as a
    # non-torch host would; cross-checked once against torch.distributed's all-reduce, which is also the fallback
    comm, allreduce_kind = None, "none (1 GPU)"
    if world > 1:
        try:
            comm = parallel.RawNcclComm(rank=rank, world_size=world, device=dev)
            probe = torch.tensor([float(rank + 1)], dtype=torch.float64, device=dev)
            parallel.allreduce_loglik_nccl(probe, comm)
            torch.cuda.synchronize()
            assert abs(probe.item() - world * (world + 1) / 2) < 1e-12, probe.item()
            allreduce_kind = "cdk_ll_allreduce (C ABI) on a raw ncclComm_t, checked against sum(1..world)"
        except Exception as e:  # noqa: BLE001 -- keep the bench alive, say what happened
            comm, allreduce_kind = None, f"torch.distributed all_reduce (raw communicator unavailable: {e!r})"
        ok = torch.tensor([1.0 if comm is not None else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() == 0.0 and comm is not None:
            comm, allreduce_kind = None, "torch.distributed all_reduce (raw communicator failed on another rank)"

    def allreduce(sv):
        if world == 1:
            return sv
        if comm is not None:
            return parallel.allreduce_loglik_nccl(sv, comm)
        return parallel.allreduce_loglik(sv)

    ctx = dict(dist=dist, world=world, rank=rank, local_rank=local_rank, dev=dev, lib=lib, L=L, barrier=barrier,
               allreduce=allreduce)

    def make_job(mode):
        if mode == "strong":
            lo, hi = parallel.shard_bounds(args.n_traj, rank, world)
        else:
            lo, hi = rank * args.n_traj, (rank + 1) * args.n_traj
        return Job(hi - lo, lo, K, rank, dev, args.simple_data), (args.n_traj if mode == "strong" else args.n_traj * world)

    # ---- headline mode ----
    job, n_total = make_job(args.scaling)
    total_ms, launches, ll_total, n_bad, clocks, (post, s) = time_resident(job, args, args.steps, ctx)
    if args.dump_outputs and rank == 0 and post is not None:
        dump_outputs(args.dump_outputs, post, s)
    del post, s
    kernel_ms = time_kernel(job, ctx)
    e2e_ms, e2e_steps, h2d, d2h, _, ll_host = time_e2e(job, args, ctx)
    e2e_ok = None
    if world == 1 and ll_host is not None:
        e2e_ok = bool(abs(float(np.sum(np.asarray(ll_host, dtype=np.float64))) - ll_total) <= 1e-9 * abs(ll_total))
    # the same through the API with ALL FOUR moment arrays returned to pinned host memory (the work the CPU arm does), on a
    # bounded slice of the batch: the device->host copy of 192 B per observation-step dominates (PCIe), it is a rate
    n_all = min(job.N, 16384)
    ea_ms, ea_steps, ea_h2d, ea_d2h, ea_n, _ = time_e2e(job, args, ctx, all_outputs=True, n_limit=n_all)
    n_all_total = torch.tensor([float(ea_n)], dtype=torch.float64, device=dev)
    sumq_total = torch.tensor([float(job.sum_q)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(n_all_total)
        dist.all_reduce(sumq_total)
    fp64_peak, fp64_peak3 = probe_fp64_peaks(ctx) if rank == 0 else (None, None)

    # ---- the other scaling mode, beside the headline (N > 1 only; at one GPU the two coincide) ----
    other = None
    if world > 1 and not args.no_other_mode:
        other_mode = "weak" if args.scaling == "strong" else "strong"
        del job.y_dev, job.t_dev
        torch.cuda.empty_cache()
        job2, n_total2 = make_job(other_mode)
        o_ms, o_launches, o_ll, o_bad = time_resident(job2, args, args.steps, ctx)[:4]
        o_kernel_ms = time_kernel(job2, ctx)
        other = {"scaling": other_mode, "n_traj_total": n_total2, "n_traj_per_gpu": job2.N,
                 "value": n_total2 * K * args.steps / (o_ms * 1e-3), "unit": UNIT, "ms_per_step": o_ms / args.steps,
                 "kernel_ms_rank0": o_kernel_ms, "gpu_launches": o_launches, "ll_sum": o_ll,
                 "non_finite_trajectories_rank0": o_bad}
    if comm is not None:
        comm.destroy()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    units_per_step = n_total * K
    value = units_per_step * args.steps / (total_ms * 1e-3)
    peaks, peak_src = measured_peaks()
    N0 = job.N  # the roofline describes rank 0's launch
    flops_exec = FLOP_SUBSTEP_EXEC * job.sum_q + FLOP_UPDATE_EXEC * N0 * K
    flops_survey = FLOP_SUBSTEP_SURVEY * job.sum_q + FLOP_UPDATE_SURVEY * N0 * K
    ach = flops_exec / (kernel_ms * 1e-3) / 1e12
    ach_survey = flops_survey / (kernel_ms * 1e-3) / 1e12
    hbm_ach = BYTES_PER_OBS_STEP * N0 * K / (kernel_ms * 1e-3) / 1e9
    warps = (N0 + 31) // 32
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world, extra={"mean_substeps_per_gap": float(sumq_total.item()) / (n_total * K)}),
        "clocks": clocks,
        "e2e": {"value": units_per_step * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps, "result": "per-trajectory log-likelihoods (the loss)",
                "result_matches_resident": e2e_ok, "bytes_are": "per GPU"},
        "e2e_all_outputs": {"value": float(n_all_total.item()) * K * ea_steps / (ea_ms * 1e-3), "unit": UNIT,
                            "h2d_bytes_per_step": ea_h2d, "d2h_bytes_per_step": ea_d2h, "steps": ea_steps,
                            "n_traj_per_gpu": ea_n,
                            "result": "log-likelihoods + filtered/predicted means and covariances in pinned host memory "
                                      "(what the CPU arm produces); bounded slice of the batch, PCIe-bound"},
        "gpu_launches": int(launches),
        "allreduce": allreduce_kind,
        "roofline": {
            "bound": "fp64", "kernel": f"ekf_small_lw<double, DriftL63, 1, RK4> on rank 0: {warps} groups of 32 trajectories "
                                        "(state and drift parameters in registers, TMA tensor stores); up to one balanced "
                                        "wave each group keeps one warp, warps per CTA chosen from N so that they spread over "
                                        "all SMs and sub-partitions; above it (this config at 1 GPU) the groups of an SM are "
                                        "time-sliced over 8 resident warps in K-segments through shared memory",
            "achieved": ach_survey, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": ach_survey / fp64_peak if fp64_peak else None,
            "peak_source": "DFMA probe (cdk_fma_probe_f64) measured in this run, burst; MEASURED_PEAKS.json has no FP64 "
                           "entry; nominal 148 SM x 64 FMA/clk x 2 x 1.965 GHz = 37.2",
            "flop_model": "algorithmic (SURVEY 8d): 496*sum_q + 107*N*K of rank 0's shard",
            "achieved_executed": ach, "frac_executed": ach / fp64_peak if fp64_peak else None,
            "peak_3_register_operands": fp64_peak3,
            "peak_3_register_operands_note": "cdk_fma3_probe_f64, measured in this run: a DFMA whose three operands are "
                                             "distinct vector registers issues every 3 cycles per SM sub-partition on "
                                             "B200, not 2 (register-file bandwidth); most of the 143 DFMAs among the kernel's 181 FP64 "
                                             "instructions per substep are such DFMAs; frac_of_3_register_peak divides the ALGORITHMIC rate by it and can exceed 1 "
                                             "(the kernel executes fewer flops than the survey counts: see achieved_executed)",
            "frac_of_3_register_peak": ach_survey / fp64_peak3 if fp64_peak3 else None,
            "flop_model_executed": "324*sum_q + 60*N*K (symmetric P, sparse Lorenz-63 Jacobian, dt folded into RK weights)",
            "kernel_ms": kernel_ms,
            "kernel_ms_how": "CUDA events between back-to-back launches of the pre-marshalled C-ABI call on the launching "
                             "stream (mean of 7), GPU kept busy by the previous launch: kernel duration only",
            "traffic": TRAFFIC_NCU_BYTES * (N0 / 65536.0) * (K / 1000.0),
            "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel at "
                            "N = 65,536, K = 1,000 (profiles/), scaled to this launch; algorithmic bytes = 208 * N * K",
            "hbm": {"achieved": hbm_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_ach / peaks["hbm_gbs"],
                    "peak_source": f"MEASURED_PEAKS.json ({peak_src})", "bytes_per_obs_step": BYTES_PER_OBS_STEP},
        },
        "ll_sum": ll_total, "non_finite_trajectories_rank0": n_bad,
    }
    if other is not None:
        line[other["scaling"] + "_scaling"] = other
    if not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        res = cpu_reference_leg(args.cpu_sample_traj or 512 * cores, K, steps=2, warmup=1)
        line["cpu_baseline"] = {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"],
                                "sample": res["sample"], "value_ll_only": res.get("value_ll_only")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
