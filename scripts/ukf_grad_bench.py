#!/usr/bin/env python
"""Cost of the CD-UKF log-likelihood gradient (cdk_ukf_grad_dense_f64) against the filter it differentiates
(cdk_ukf_filter_f64 writing the outputs its forward pass writes: LL, status, filtered and predicted moments).

    python scripts/ukf_grad_bench.py [--reps R] [--scale S]

Shape: the C4 model (Lorenz-96, n = 40, m = 20, every other component observed, K = 500, N = 1,024, mean gap 0.02; the
problem of scripts/ekf_grad_bench.py), with RK4 at dt0 = 0.005 and with Dopri5 at dt0 = 0.01.  Both run the filter's
register-resident moment ODE in the forward pass.  Inputs and outputs stay on the device; both entry points are called
through the C ABI on preallocated buffers, warmed up, then alternated over the repeats and timed with CUDA events.
--scale < 1 shrinks N.  Prints one JSON line, with the card's name, power limit and max SM clock read in the same run.
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cd_dynamax_b200 import _lib as L  # noqa: E402
from ekf_grad_bench import call, card, dev, f64, problem  # noqa: E402


def measure(solver, dt0, reps, scale):
    lib = L.lib()
    d, ins, (N, K, n, m) = problem("l96", solver, dt0, scale)
    st = lambda: torch.empty(N, dtype=torch.int32, device=dev)
    outs_f = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(), L.OUT_FM: torch.empty(N, K, n, **f64),
              L.OUT_FP: torch.empty(N, K, n, n, **f64), L.OUT_PM: torch.empty(N, K, n, **f64),
              L.OUT_PP: torch.empty(N, K, n, n, **f64)}
    scratch = int(lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ukf_grad_dense"))
    outs_g = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(),
              L.OUT_GRAD: torch.empty(N, L.grad_cols_ekf(n, m, d.n_theta), **f64),
              L.OUT_SCRATCH: torch.empty(scratch, dtype=torch.uint8, device=dev)}
    fns = {"filter": call(lib, "cdk_ukf_filter_f64", d, ins, outs_f),
           "grad": call(lib, "cdk_ukf_grad_dense_f64", d, ins, outs_g)}
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
    return dict(config=f"l96 n={n} m={m} N={N} K={K}", solver=solver, dt0=dt0,
                **{f"{k}_ms": v for k, v in med.items()},
                **{f"{k}_ms_min": float(min(v)) for k, v in times.items()},
                grad_filter_passes=med["grad"] / med["filter"], scratch_bytes=scratch)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0)
    args = ap.parse_args()
    out = dict(card=card(), results=[measure("rk4", 0.005, args.reps, args.scale),
                                     measure("dopri5", 0.01, args.reps, args.scale)])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
