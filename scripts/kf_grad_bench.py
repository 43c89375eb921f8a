#!/usr/bin/env python
"""Cost of the linear CD-KF log-likelihood gradient (cdk_kf_grad_f64) against the filter it differentiates
(cdk_kf_filter_f64 writing the same outputs its forward pass writes: LL, status, filtered and predicted moments).

    python scripts/kf_grad_bench.py [--reps R] [--profile]

Shapes: the C2 chunk (N = 8,192, n = 16, m = 4, K = 500, the inputs of scripts/bench_configs.py c2) with RK4 at
dt0 = 0.01 and with the reference's default Dopri5, and the C1 latency case (N = 1, n = 4, m = 2, K = 200).  Inputs and
outputs stay on the device; both entry points are called through the C ABI on preallocated buffers, warmed up, then
alternated over the repeats and timed with CUDA events.  --profile adds a torch.profiler pass (a separate run) with the
time of every kernel.  Prints one JSON line, with the card's name and power limit read in the same run.
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


def problem(cfg, solver):
    if cfg == "c2":
        n, m, K, N = 16, 4, 500, 8192
        rng = np.random.default_rng(1235)
        F = -0.5 * np.eye(n) + 0.3 * rng.standard_normal((n, n)) / np.sqrt(n)
        pars = dict(F=F, b=np.zeros(n), L=np.eye(n), Qc=0.1 * np.eye(n), H=np.eye(n)[:m], d=np.zeros(m),
                    R=0.1 * np.eye(m), m0=np.zeros(n), P0=np.eye(n))
        mean_gap, dt0, dt_final = 0.04, 0.01, 1e-10
    else:
        n, m, K, N = 4, 2, 200, 1
        F = np.zeros((n, n))
        F[0, 2] = F[1, 3] = 1.0
        pars = dict(F=F, b=np.zeros(n), L=1e-3 * np.eye(n), Qc=np.eye(n), H=np.eye(m, n), d=np.zeros(m),
                    R=0.5 * np.eye(m), m0=np.array([8.0, 10.0, 1.0, 0.0]), P0=0.1 * np.eye(n))
        mean_gap, dt0, dt_final = 0.05, 0.0125, 1.0
    g = torch.Generator(device=dev)
    g.manual_seed(2)
    gaps = mean_gap * (0.5 + torch.rand(N, K, generator=g, **f64))
    gaps[:, 0] = 0.0
    ins = {L.IN_T: torch.cumsum(gaps, dim=1), L.IN_Y: torch.randn(N, K, m, generator=g, **f64)}
    slots = dict(F=L.IN_F, b=L.IN_B, L=L.IN_L, Qc=L.IN_QC, H=L.IN_H, d=L.IN_D, R=L.IN_R, m0=L.IN_M0, P0=L.IN_P0)
    for k, s in slots.items():
        ins[s] = torch.as_tensor(pars[k], **f64).contiguous()
    d = L.new_desc()
    d.N, d.K, d.n, d.m = N, K, n, m
    d.solver, d.dt0, d.dt_final = L.SOLVERS[solver], dt0, dt_final
    d.batched_mask = (1 << L.IN_Y) | (1 << L.IN_T)
    return d, ins, (N, K, n, m)


def call(lib, name, d, ins, outs):
    ip = (ctypes.c_void_p * L.NUM_IN)(*[ins[s].data_ptr() if s in ins else None for s in range(L.NUM_IN)])
    op = (ctypes.c_void_p * L.NUM_OUT)(*[outs[s].data_ptr() if s in outs else None for s in range(L.NUM_OUT)])
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    return lambda: L.check(getattr(lib, name)(ctypes.byref(d), ip, op, stream), name)


def measure(cfg, solver, reps, profile):
    lib = L.lib()
    d, ins, (N, K, n, m) = problem(cfg, solver)
    outs_f = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: torch.empty(N, dtype=torch.int32, device=dev),
              L.OUT_FM: torch.empty(N, K, n, **f64), L.OUT_FP: torch.empty(N, K, n, n, **f64),
              L.OUT_PM: torch.empty(N, K, n, **f64), L.OUT_PP: torch.empty(N, K, n, n, **f64)}
    scratch = int(lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_kf_grad"))
    outs_g = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: torch.empty(N, dtype=torch.int32, device=dev),
              L.OUT_GRAD: torch.empty(N, L.grad_cols_kf(n, m), **f64),
              L.OUT_SCRATCH: torch.empty(scratch, dtype=torch.uint8, device=dev)}
    filt = call(lib, "cdk_kf_filter_f64", d, ins, outs_f)
    grad = call(lib, "cdk_kf_grad_f64", d, ins, outs_g)
    for _ in range(3):
        filt()
        grad()
    torch.cuda.synchronize()
    assert torch.equal(outs_f[L.OUT_LL], outs_g[L.OUT_LL]) and int(outs_g[L.OUT_STATUS].abs().sum()) == 0
    assert bool(torch.isfinite(outs_g[L.OUT_GRAD]).all())
    ev = lambda: torch.cuda.Event(enable_timing=True)
    tf, tg = [], []
    for _ in range(reps):
        for fn, acc in ((filt, tf), (grad, tg)):
            e0, e1 = ev(), ev()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            acc.append(e0.elapsed_time(e1))
    res = dict(config=f"{cfg.upper()} n={n} m={m} N={N} K={K}", solver=solver, dt0=d.dt0, filter_ms=float(np.median(tf)),
               grad_ms=float(np.median(tg)), ratio=float(np.median(tg) / np.median(tf)),
               filter_ms_min=min(tf), grad_ms_min=min(tg), scratch_bytes=scratch)
    if profile:
        from torch.profiler import ProfilerActivity, profile as prof
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            grad()
            torch.cuda.synchronize()
        res["grad_kernels_ms"] = {e.key: e.device_time_total / 1e3 for e in p.key_averages() if e.device_time_total > 0}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    out = dict(card=card(), results=[measure("c2", "rk4", args.reps, args.profile),
                                     measure("c2", "dopri5", args.reps, args.profile),
                                     measure("c1", "rk4", 4 * args.reps, args.profile)])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
