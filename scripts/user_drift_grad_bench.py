#!/usr/bin/env python
"""Cost of the CD-EKF log-likelihood gradient for USER-DEFINED drifts (cdk_ekf_grad_dense_f64 in a variant library built
with build_user_drift(code, grad=True)) against the filter of the same variant (cdk_ekf_filter_f64 writing the outputs
the gradient's forward pass writes).

    python scripts/user_drift_grad_bench.py [--reps R] [--scale S]

Shapes:
  (a) Van der Pol (examples/vdp_drift.cuh), n = 2, m = 1, N = 8,192, K = 500, RK4 at dt0 = 0.01 (mean gap 0.05),
      state_order first and second;
  (b) the tanh network of examples/mlp_drift.cuh (n_theta = 82) at the same shape and orders;
  (c) a user drift that restates Lorenz-63, H = I_3, N = 8,192, K = 1,000, RK4 at dt0 = 0.0025 (row (b) of
      scripts/ekf_grad_bench.py), next to the registry Lorenz-63 on the same inputs: the cost of the dual-number
      contractions over the registry's.
Inputs and outputs stay on the device; the entry points are called through the C ABI on preallocated buffers, warmed up,
alternated over the repeats and timed with CUDA events.  Prints one JSON line with the card's name, power limit and max
SM clock read in the same run.
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

LORENZ63 = r'''
namespace cdk_user {
template <typename T, class XF> __device__ T f(const T* th, int n, int i, XF x) {
  if (i == 0) return th[0] * (x(1) - x(0));
  if (i == 1) return x(0) * (th[1] - x(2)) - x(1);
  return x(0) * x(1) - th[2] * x(2);
}
template <typename T> __device__ T jac(const T* th, int n, int i, int j, const T* x) {
  if (i == 0) return j == 0 ? -th[0] : (j == 1 ? th[0] : T(0));
  if (i == 1) return j == 0 ? th[1] - x[2] : (j == 1 ? T(-1) : -x[0]);
  return j == 0 ? x[1] : (j == 1 ? x[0] : -th[2]);
}
template <typename T> __device__ T graddiv(const T* th, int n, int k, const T* x) { return T(0); }
}
'''


def example(name):
    return open(os.path.join(ROOT, "cd_dynamax_b200", "examples", name)).read()


def small_problem(theta, order, scale):
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    n, m, K, N = 2, 1, 500, max(148, int(8192 * scale))
    gaps = 0.05 * (0.5 + torch.rand(N, K, generator=g, **f64))
    gaps[:, 0] = 0.0
    pars = dict(L=np.eye(n), Qc=0.1 * np.eye(n), H=np.array([[1.0, 0.2]]), d=np.zeros(m), R=0.1 * np.eye(m),
                m0=np.array([1.0, 0.5]), P0=0.3 * np.eye(n))
    ins = {L.IN_T: torch.cumsum(gaps, dim=1), L.IN_Y: 1.5 * torch.randn(N, K, m, generator=g, **f64),
           L.IN_F: torch.as_tensor(theta, **f64)}
    for k, s in dict(L=L.IN_L, Qc=L.IN_QC, H=L.IN_H, d=L.IN_D, R=L.IN_R, m0=L.IN_M0, P0=L.IN_P0).items():
        ins[s] = torch.as_tensor(pars[k], **f64).contiguous()
    d = L.new_desc()
    d.N, d.K, d.n, d.m = N, K, n, m
    d.solver, d.dt0, d.state_order = L.SOLVERS["rk4"], 0.01, L.ORDERS[order]
    d.drift_id, d.n_theta, d.emission_id = L.DRIFT_USER, len(theta), 0
    d.batched_mask = (1 << L.IN_Y) | (1 << L.IN_T)
    return d, ins, (N, K, n, m)


def entry_points(lib, d, ins, shape, tag):
    N, K, n, m = shape
    st = lambda: torch.empty(N, dtype=torch.int32, device=dev)
    outs_f = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(), L.OUT_FM: torch.empty(N, K, n, **f64),
              L.OUT_FP: torch.empty(N, K, n, n, **f64), L.OUT_PM: torch.empty(N, K, n, **f64),
              L.OUT_PP: torch.empty(N, K, n, n, **f64)}
    scratch = int(lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad_dense"))
    outs_g = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(),
              L.OUT_GRAD: torch.empty(N, L.grad_cols_ekf(n, m, d.n_theta), **f64),
              L.OUT_SCRATCH: torch.empty(scratch, dtype=torch.uint8, device=dev)}
    fns = {f"{tag}filter": call(lib, "cdk_ekf_filter_f64", d, ins, outs_f),
           f"{tag}grad": call(lib, "cdk_ekf_grad_dense_f64", d, ins, outs_g)}
    return fns, (outs_f, outs_g)


def timed(fns, checks, reps):
    for _ in range(2):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    for outs_f, outs_g in checks:
        assert torch.equal(outs_f[L.OUT_LL], outs_g[L.OUT_LL]) and int(outs_g[L.OUT_STATUS].abs().sum()) == 0
        assert bool(torch.isfinite(outs_g[L.OUT_GRAD]).all())
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0)
    args = ap.parse_args()
    results = []
    mlp_rng = np.random.default_rng(6)
    mlp_theta = np.concatenate([0.8 * mlp_rng.standard_normal(32), 0.3 * mlp_rng.standard_normal(16),
                                0.1 * mlp_rng.standard_normal(32), 0.1 * mlp_rng.standard_normal(2)])
    for name, code, theta in (("vdp", example("vdp_drift.cuh"), np.array([1.3, 0.4])),
                              ("mlp", example("mlp_drift.cuh"), mlp_theta)):
        lib = L.lib(B.build_user_drift(code, grad=True))
        for order in ("first", "second"):
            d, ins, shape = small_problem(theta, order, args.scale)
            fns, outs = entry_points(lib, d, ins, shape, "")
            r = timed(fns, [outs], args.reps)
            results.append(dict(config=f"{name} n=2 m=1 N={shape[0]} K={shape[1]} n_theta={len(theta)}", solver="rk4",
                                dt0=0.01, state_order=order, **r, grad_filter_passes=r["grad_ms"] / r["filter_ms"]))
    d, ins, shape = problem("l63_h3", "rk4", 0.0025, args.scale)
    reg, outs_r = entry_points(L.lib(), d, ins, shape, "registry_")
    du = L.CdkDesc.from_buffer_copy(d)
    du.drift_id = L.DRIFT_USER
    user, outs_u = entry_points(L.lib(B.build_user_drift(LORENZ63, grad=True)), du, ins, shape, "user_")
    r = timed({**reg, **user}, [outs_r, outs_u], args.reps)
    results.append(dict(config=f"lorenz63 user vs registry n=3 m=3 N={shape[0]} K={shape[1]}", solver="rk4", dt0=0.0025,
                        state_order="second", **r, user_grad_filter_passes=r["user_grad_ms"] / r["user_filter_ms"],
                        registry_grad_filter_passes=r["registry_grad_ms"] / r["registry_filter_ms"],
                        user_over_registry_grad=r["user_grad_ms"] / r["registry_grad_ms"]))
    print(json.dumps(dict(card=card(), results=results)))


if __name__ == "__main__":
    main()
