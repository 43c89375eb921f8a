#!/usr/bin/env python
"""Cost of the CD-EKF log-likelihood gradient for USER-DEFINED emissions (cdk_ekf_grad_dense_f64 in a variant library
built with build_variant(..., emission_grad=True)) against the filter of the same library (cdk_ekf_filter_f64 writing
the outputs the gradient's forward pass writes).

    python scripts/user_emission_grad_bench.py [--reps R] [--scale S] [--out FILE]

Cases:
  (a) Lorenz-96, n = 40, m = 20 (every other component observed), N = 1,024, K = 500, RK4 at dt0 = 0.005 (mean gap
      0.05), with the stock linear emission (stock library), the linear emission written as user code
      (examples/linear_emission.cuh, n_phi = 820) and the range emission to 20 beacons (examples/range_emission.cuh,
      n_phi = 801);
  (b) Van der Pol (examples/vdp_drift.cuh) with the range emission to 3 beacons, n = 2, N = 8,192, K = 500, RK4 at
      dt0 = 0.01, in one variant holding both codes with both gradient units.
Inputs and outputs stay on the device; the entry points are called through the C ABI on preallocated buffers, warmed up,
alternated over the repeats (median of R) and timed with CUDA events.  Prints one JSON line with the card's name, power
limit and max SM clock read in the same run, and appends it to FILE (default profiles/r03_user_emission_grad_bench.jsonl).
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
from scripts.ekf_grad_bench import call, card, dev, f64  # noqa: E402


def example(name):
    return open(os.path.join(ROOT, "cd_dynamax_b200", "examples", name)).read()


def make(n, m, N, K, dt0, drift_id, theta, emission, seed):
    """(desc, inputs, shape) of one case; emission: 'stock' (H, d), 'linear' (phi = [H | d]) or 'range' (beacons, eps)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    gaps = 0.05 * (0.5 + torch.rand(N, K, generator=g, **f64))
    gaps[:, 0] = 0.0
    rng = np.random.default_rng(seed)
    H = np.zeros((m, n))
    H[np.arange(m), (np.arange(m) * n) // m] = 1.0
    d_ = np.zeros(m)
    ins = {L.IN_T: torch.cumsum(gaps, dim=1), L.IN_F: torch.as_tensor(theta, **f64),
           L.IN_L: torch.eye(n, **f64), L.IN_QC: 0.1 * torch.eye(n, **f64), L.IN_R: 0.1 * torch.eye(m, **f64),
           L.IN_M0: torch.as_tensor(np.full(n, 1.0) + 0.1 * rng.standard_normal(n), **f64),
           L.IN_P0: 0.3 * torch.eye(n, **f64)}
    if emission == "range":  # beacons around the initial state, ranges observed from it with noise
        B_ = ins[L.IN_M0].cpu().numpy() + 2.0 * rng.standard_normal((m, n))
        r0 = np.sqrt(((ins[L.IN_M0].cpu().numpy() - B_) ** 2).sum(-1) + 0.1)
        ins[L.IN_H] = torch.as_tensor(np.concatenate([B_.reshape(-1), [0.1]]), **f64)
        ins[L.IN_Y] = torch.as_tensor(r0, **f64) + 0.3 * torch.randn(N, K, m, generator=g, **f64)
    else:
        ins[L.IN_Y] = 1.5 * torch.randn(N, K, m, generator=g, **f64)
        if emission == "linear":
            ins[L.IN_H] = torch.as_tensor(np.concatenate([H.reshape(-1), d_]), **f64)
        else:
            ins[L.IN_H], ins[L.IN_D] = torch.as_tensor(H, **f64), torch.as_tensor(d_, **f64)
    d = L.new_desc()
    d.N, d.K, d.n, d.m = N, K, n, m
    d.solver, d.dt0, d.state_order = L.SOLVERS["rk4"], dt0, L.ORDERS["second"]
    d.drift_id, d.n_theta = drift_id, len(theta)
    d.emission_id = L.EMISSION_LINEAR if emission == "stock" else L.EMISSION_USER
    d.batched_mask = (1 << L.IN_Y) | (1 << L.IN_T)
    return d, ins, (N, K, n, m)


def entry_points(lib, d, ins, shape, tag):
    N, K, n, m = shape
    st = lambda: torch.empty(N, dtype=torch.int32, device=dev)
    outs_f = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(), L.OUT_FM: torch.empty(N, K, n, **f64),
              L.OUT_FP: torch.empty(N, K, n, n, **f64), L.OUT_PM: torch.empty(N, K, n, **f64),
              L.OUT_PP: torch.empty(N, K, n, n, **f64)}
    cols = (L.grad_cols_ekf(n, m, d.n_theta) if d.emission_id == L.EMISSION_LINEAR
            else L.grad_cols_ekf_ue(n, m, d.n_theta, int(lib.cdk_user_emission_params(n, m))))
    scratch = int(lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad_dense"))
    outs_g = {L.OUT_LL: torch.empty(N, **f64), L.OUT_STATUS: st(), L.OUT_GRAD: torch.empty(N, cols, **f64),
              L.OUT_SCRATCH: torch.empty(scratch, dtype=torch.uint8, device=dev)}
    fns = {f"{tag}filter": call(lib, "cdk_ekf_filter_f64", d, ins, outs_f),
           f"{tag}grad": call(lib, "cdk_ekf_grad_dense_f64", d, ins, outs_g)}
    return fns, (outs_f, outs_g)


def timed(fns, checks, reps):
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    for outs_f, outs_g in checks:
        bad = int((outs_g[L.OUT_STATUS] != 0).sum())
        ok = outs_g[L.OUT_STATUS] == 0
        assert torch.equal(outs_f[L.OUT_LL][ok], outs_g[L.OUT_LL][ok]), "the gradient's log-likelihood is not the filter's"
        assert bad == 0, f"{bad} trajectories with a non-zero status"
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
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_user_emission_grad_bench.jsonl"))
    args = ap.parse_args()
    results = []
    N = max(148, int(1024 * args.scale))
    for name, lib, emission in (("stock_linear", L.lib(), "stock"),
                                ("linear_as_user", L.lib(B.build_variant(None, example("linear_emission.cuh"),
                                                                         emission_grad=True)), "linear"),
                                ("range", L.lib(B.build_variant(None, example("range_emission.cuh"),
                                                                emission_grad=True)), "range")):
        d, ins, shape = make(40, 20, N, 500, 0.005, L.DRIFT_LORENZ96, [8.0], emission, 7)
        fns, outs = entry_points(lib, d, ins, shape, "")
        r = timed(fns, [outs], args.reps)
        results.append(dict(case="a", config=f"lorenz96 {name} n=40 m=20 N={N} K=500", solver="rk4", dt0=0.005,
                            state_order="second", **r, grad_filter_ratio=r["grad_ms"] / r["filter_ms"]))
    lib = L.lib(B.build_variant(example("vdp_drift.cuh"), example("range_emission.cuh"), True, emission_grad=True))
    N = max(148, int(8192 * args.scale))
    d, ins, shape = make(2, 3, N, 500, 0.01, L.DRIFT_USER, [1.3, 0.4], "range", 8)
    fns, outs = entry_points(lib, d, ins, shape, "")
    r = timed(fns, [outs], args.reps)
    results.append(dict(case="b", config=f"vdp range(3 beacons) n=2 m=3 N={N} K=500", solver="rk4", dt0=0.01,
                        state_order="second", **r, grad_filter_ratio=r["grad_ms"] / r["filter_ms"]))
    line = json.dumps(dict(card=card(), results=results))
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
