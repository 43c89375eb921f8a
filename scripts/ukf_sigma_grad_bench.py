#!/usr/bin/env python
"""Cost of the gradient of the CD-UKF with literal sigma points (cdk_ukf_grad_sigma_f64) against the filter it
differentiates (cdk_ukf_filter_f64 with CDK_FLAG_UKF_SIGMA_POINTS, writing the outputs the gradient's forward pass
writes: LL, status, filtered and predicted moments).

    python scripts/ukf_sigma_grad_bench.py [--reps R] [--scale S] [--out FILE]

Shapes:
  (a) the C4 model of scripts/ukf_grad_bench.py (Lorenz-96, n = 40, m = 20, K = 500, N = 1,024, mean gap 0.02), RK4 at
      dt0 = 0.005 and Dopri5 at dt0 = 0.01: the sigma-point gradient, the sigma-point filter and the closed-form gradient
      (cdk_ukf_grad_dense_f64) on the same inputs;
  (b) Van der Pol and the tanh network (examples/, n_theta = 82) with n = 2, m = 1, N = 8,192, K = 500, RK4 at
      dt0 = 0.01 (the problem of scripts/user_drift_grad_bench.py): the gradient against the same variant's sigma-point
      filter (a user drift always runs sigma points).
Inputs and outputs stay on the device; the entry points are called through the C ABI on preallocated buffers, warmed up
once, then alternated over the repeats and timed with CUDA events; the median is reported.  Appends one JSON line, with
the card's name, power limit and max SM clock read in the same run, to --out (default
profiles/r03_ukf_sigma_grad_bench.jsonl) and prints it.
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cd_dynamax_b200 import _lib as L  # noqa: E402
from cd_dynamax_b200 import build as B  # noqa: E402
from scripts.ekf_grad_bench import call, card, dev, f64, problem  # noqa: E402
from scripts.user_drift_grad_bench import example, small_problem  # noqa: E402


def outputs(lib, d, shape, entry):
    N, K, n, m = shape
    st = lambda: torch.empty(N, dtype=torch.int32, device=dev)
    if entry == "filter":
        return {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(), L.OUT_FM: torch.empty(N, K, n, **f64),
                L.OUT_FP: torch.empty(N, K, n, n, **f64), L.OUT_PM: torch.empty(N, K, n, **f64),
                L.OUT_PP: torch.empty(N, K, n, n, **f64)}
    scratch = int(lib.cdk_scratch_bytes(ctypes.byref(d), entry.encode()))
    return {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(),
            L.OUT_GRAD: torch.empty(N, L.grad_cols_ekf(n, m, d.n_theta), **f64),
            L.OUT_SCRATCH: torch.empty(scratch, dtype=torch.uint8, device=dev)}


def timed(fns, reps):
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    return {f"{k}_ms": float(np.median(v)) for k, v in times.items()}


def check(outs_f, outs_g):
    """The gradient's log-likelihood and status are the filter's; -> the number of trajectories whose status is not 0
    (their log-likelihood and gradient row are NaN)."""
    ok = outs_g[L.OUT_STATUS] == 0
    assert torch.equal(outs_f[L.OUT_STATUS], outs_g[L.OUT_STATUS])
    assert torch.equal(outs_f[L.OUT_LL][ok], outs_g[L.OUT_LL][ok])
    assert bool(torch.isfinite(outs_g[L.OUT_GRAD][ok]).all())
    return int((~ok).sum())


def c4(solver, dt0, reps, scale):
    lib = L.lib()
    d, ins, shape = problem("l96", solver, dt0, scale)
    ds = L.CdkDesc.from_buffer_copy(d)
    ds.reserved[2] = L.FLAG_UKF_SIGMA_POINTS
    of, og, oc = outputs(lib, ds, shape, "filter"), outputs(lib, d, shape, "cdk_ukf_grad_sigma"), \
        outputs(lib, d, shape, "cdk_ukf_grad_dense")
    fns = {"sigma_filter": call(lib, "cdk_ukf_filter_f64", ds, ins, of),
           "sigma_grad": call(lib, "cdk_ukf_grad_sigma_f64", d, ins, og),
           "closed_grad": call(lib, "cdk_ukf_grad_dense_f64", d, ins, oc)}
    r = timed(fns, reps)
    failed = check(of, og)
    N, K, n, m = shape
    return dict(config=f"l96 n={n} m={m} N={N} K={K}", solver=solver, dt0=dt0, **r, failed_trajectories=failed,
                sigma_grad_filter_passes=r["sigma_grad_ms"] / r["sigma_filter_ms"],
                sigma_over_closed_grad=r["sigma_grad_ms"] / r["closed_grad_ms"])


def user(name, code, theta, reps, scale):
    lib = L.lib(B.build_user_drift(code, grad=True))
    d, ins, shape = small_problem(theta, "first", scale)
    d.alpha, d.beta, d.kappa = float(np.sqrt(3.0)), 2.0, 1.0
    of, og = outputs(lib, d, shape, "filter"), outputs(lib, d, shape, "cdk_ukf_grad_sigma")
    r = timed({"filter": call(lib, "cdk_ukf_filter_f64", d, ins, of),
               "grad": call(lib, "cdk_ukf_grad_sigma_f64", d, ins, og)}, reps)
    failed = check(of, og)
    N, K, n, m = shape
    return dict(config=f"{name} n={n} m={m} N={N} K={K} n_theta={len(theta)}", solver="rk4", dt0=0.01, **r,
                failed_trajectories=failed,
                grad_filter_passes=r["grad_ms"] / r["filter_ms"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_ukf_sigma_grad_bench.jsonl"))
    args = ap.parse_args()
    results = [c4("rk4", 0.005, args.reps, args.scale), c4("dopri5", 0.01, args.reps, args.scale)]
    mlp_rng = np.random.default_rng(6)
    mlp_theta = np.concatenate([0.8 * mlp_rng.standard_normal(32), 0.3 * mlp_rng.standard_normal(16),
                                0.1 * mlp_rng.standard_normal(32), 0.1 * mlp_rng.standard_normal(2)])
    for name, code, theta in (("vdp", example("vdp_drift.cuh"), np.array([1.3, 0.4])),
                              ("mlp", example("mlp_drift.cuh"), mlp_theta)):
        results.append(user(name, code, theta, args.reps, args.scale))
    line = json.dumps(dict(card=card(), results=results))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
