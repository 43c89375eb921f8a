#!/usr/bin/env python
"""Cost of the CD-EKF log-likelihood gradient for the registry drifts (cdk_ekf_grad_dense_f64) against the filter it
differentiates (cdk_ekf_filter_f64 writing the outputs its forward pass writes: LL, status, filtered and predicted
moments).

    python scripts/ekf_grad_bench.py [--reps R] [--profile] [--scale S]

Shapes:
  (a) Lorenz-96, n = 40, m = 20 (every other component observed), K = 500, N = 1,024 (the C4 model of
      scripts/bench_configs.py, mean gap 0.02), with RK4 at dt0 = 0.005 and with Dopri5 at dt0 = 0.01;
  (b) Lorenz-63 with H = I_3, N = 8,192, K = 1,000, RK4 at dt0 = 0.0025 (the C3 grid, mean gap 0.01);
  (c) Lorenz-63 with a scalar emission at the C3 shape (N = 65,536, K = 1,000), through the Lorenz-63 reverse-mode
      kernel (cdk_ekf_grad_f64 with CDK_GRAD_REVERSE, all 23 columns) and through the dense one.
Inputs and outputs stay on the device; every entry point is called through the C ABI on preallocated buffers, warmed
up, then the variants are alternated over the repeats and timed with CUDA events.  --profile adds a torch.profiler pass
(a separate run) with the time of every kernel of one gradient call.  --scale < 1 shrinks N.  Prints one JSON line,
with the card's name, power limit and max SM clock read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cd_dynamax_b200 import _lib as L  # noqa: E402

dev = torch.device("cuda", 0)
f64 = dict(dtype=torch.float64, device=dev)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def problem(cfg, solver, dt0, scale):
    g = torch.Generator(device=dev)
    g.manual_seed(3)
    if cfg == "l96":
        n, m, K, N, gap = 40, 20, 500, max(148, int(1024 * scale)), 0.02
        theta = np.array([8.0])
        pars = dict(L=np.eye(n), Qc=0.1 * np.eye(n), H=np.eye(n)[::2], d=np.zeros(m), R=np.eye(m),
                    m0=8 + 0.5 * np.random.default_rng(4).standard_normal(n), P0=np.eye(n))
        y = 8 + 2 * torch.randn(max(148, int(1024 * scale)), K, m, generator=g, **f64)
        drift = L.DRIFT_LORENZ96
    else:
        m = 3 if cfg == "l63_h3" else 1
        n, K, N, gap = 3, 1000, max(148, int((8192 if m == 3 else 65536) * scale)), 0.01
        theta = np.array([10.0, 28.0, 8.0 / 3.0])
        pars = dict(L=np.eye(n), Qc=np.eye(n), H=np.eye(3)[:m], d=np.zeros(m), R=np.eye(m), m0=np.zeros(n),
                    P0=5 * np.eye(n))
        y = 8 * torch.randn(N, K, m, generator=g, **f64)
        drift = L.DRIFT_LORENZ63
    gaps = gap * (0.5 + torch.rand(N, K, generator=g, **f64))
    gaps[:, 0] = 0.0
    ins = {L.IN_T: torch.cumsum(gaps, dim=1), L.IN_Y: y, L.IN_F: torch.as_tensor(theta, **f64)}
    slots = dict(L=L.IN_L, Qc=L.IN_QC, H=L.IN_H, d=L.IN_D, R=L.IN_R, m0=L.IN_M0, P0=L.IN_P0)
    for k, s in slots.items():
        ins[s] = torch.as_tensor(pars[k], **f64).contiguous()
    d = L.new_desc()
    d.N, d.K, d.n, d.m = N, K, n, m
    d.solver, d.dt0, d.state_order = L.SOLVERS[solver], dt0, L.ORDERS["second"]
    d.drift_id, d.n_theta, d.emission_id = drift, len(theta), 0
    d.batched_mask = (1 << L.IN_Y) | (1 << L.IN_T)
    return d, ins, (N, K, n, m)


def call(lib, name, d, ins, outs):
    ip = (ctypes.c_void_p * L.NUM_IN)(*[ins[s].data_ptr() if s in ins else None for s in range(L.NUM_IN)])
    op = (ctypes.c_void_p * L.NUM_OUT)(*[outs[s].data_ptr() if s in outs else None for s in range(L.NUM_OUT)])
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    return lambda: L.check(getattr(lib, name)(ctypes.byref(d), ip, op, stream), name)


def measure(cfg, solver, dt0, reps, profile, scale, with_l63_kernel=False):
    lib = L.lib()
    d, ins, (N, K, n, m) = problem(cfg, solver, dt0, scale)
    st = lambda: torch.empty(N, dtype=torch.int32, device=dev)
    outs_f = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(), L.OUT_FM: torch.empty(N, K, n, **f64),
              L.OUT_FP: torch.empty(N, K, n, n, **f64), L.OUT_PM: torch.empty(N, K, n, **f64),
              L.OUT_PP: torch.empty(N, K, n, n, **f64)}
    scratch = int(lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad_dense"))
    outs_g = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(),
              L.OUT_GRAD: torch.empty(N, L.grad_cols_ekf(n, m, d.n_theta), **f64),
              L.OUT_SCRATCH: torch.empty(scratch, dtype=torch.uint8, device=dev)}
    fns = {"filter": call(lib, "cdk_ekf_filter_f64", d, ins, outs_f),
           "grad_dense": call(lib, "cdk_ekf_grad_dense_f64", d, ins, outs_g)}
    if with_l63_kernel:
        d63 = L.CdkDesc.from_buffer_copy(d)
        d63.reserved[3] = 127 | L.GRAD_REVERSE
        s63 = int(lib.cdk_scratch_bytes(ctypes.byref(d63), b"cdk_ekf_grad"))
        outs_r = {L.OUT_LL: torch.empty(N, **f64), L.OUT_GRAD: torch.empty(N, L.GRAD_COLS_L63, **f64),
                  L.OUT_SCRATCH: torch.empty(s63, dtype=torch.uint8, device=dev)}
        fns["grad_l63_reverse"] = call(lib, "cdk_ekf_grad_f64", d63, ins, outs_r)
    for _ in range(2):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    assert torch.equal(outs_f[L.OUT_LL], outs_g[L.OUT_LL]) and int(outs_g[L.OUT_STATUS].abs().sum()) == 0
    assert bool(torch.isfinite(outs_g[L.OUT_GRAD]).all())
    ev = lambda: torch.cuda.Event(enable_timing=True)
    times = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            e0, e1 = ev(), ev()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = dict(config=f"{cfg} n={n} m={m} N={N} K={K}", solver=solver, dt0=dt0,
               **{f"{k}_ms": v for k, v in med.items()},
               **{f"{k}_ms_min": float(min(v)) for k, v in times.items()},
               **{f"{k}_filter_passes": med[k] / med["filter"] for k in med if k != "filter"},
               scratch_bytes=scratch)
    if profile:
        from torch.profiler import ProfilerActivity, profile as prof
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            fns["grad_dense"]()
            torch.cuda.synchronize()
        res["grad_dense_kernels_ms"] = {e.key: e.device_time_total / 1e3 for e in p.key_averages()
                                        if e.device_time_total > 0}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--scale", type=float, default=1.0)
    args = ap.parse_args()
    r = lambda *a, **k: measure(*a, reps=args.reps, profile=args.profile, scale=args.scale, **k)
    out = dict(card=card(), results=[r("l96", "rk4", 0.005), r("l96", "dopri5", 0.01), r("l63_h3", "rk4", 0.0025),
                                     r("l63_m1", "rk4", 0.0025, with_l63_kernel=True)])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
