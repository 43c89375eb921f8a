#!/usr/bin/env python
"""What a user-defined emission costs: filter time with the stock linear emission (LearnableLinear), with the SAME linear
emission written as user device code (examples/linear_emission.cuh: the user-emission update paths doing the stock
arithmetic), and with the range emission (examples/range_emission.cuh), for

  * the EKF and the UKF (closed-form predict, literal sigma-point update with a user emission) at BASELINE config 4:
    Lorenz-96 n = 40, m = 20, N = 8,192, K = 500, RK4 dt0 = 0.005;
  * the EnKF at BASELINE config 5: the same model, E = 1,024, N = 1,024, K = 500, Euler-Maruyama dt0 = 0.005.

Each case is warmed up, then timed `--reps` times with CUDA events around the filter call (inputs resident on the device,
log-likelihood only: output_fields=[]), the cases of one filter interleaved so that drift of a shared machine hits them
alike; the median is reported.  The GPU's name, power limit and clocks are read before and after.  One JSON line goes to
profiles/r03_user_emission_bench.jsonl (or --out).

    python scripts/user_emission_bench.py [--reps R] [--scale S] [--out PATH]
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cd_dynamax_b200 as cd  # noqa: E402

dev = torch.device("cuda", 0)
f64 = dict(dtype=torch.float64, device=dev)
EX = os.path.join(ROOT, "cd_dynamax_b200", "examples")
LINEAR_CODE, RANGE_CODE = (open(os.path.join(EX, f)).read() for f in ("linear_emission.cuh", "range_emission.cuh"))


def gpu_state():
    q = "name,power.limit,power.draw,clocks.sm,clocks.max.sm,temperature.gpu"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else r.stderr


def problem(N, K, seed):
    n, m = 40, 20
    rng = np.random.default_rng(seed)
    T = lambda x: torch.as_tensor(np.asarray(x, dtype=np.float64), device=dev)
    m0 = 8 + 0.5 * rng.standard_normal(n)
    H = np.eye(n)[:: n // m][:m]
    B = 8 + 4 * rng.standard_normal((m, n))
    emissions = {
        "stock_linear": cd.LearnableLinear(weights=T(H), bias=T(np.zeros(m))),
        "user_linear": cd.LearnableUserEmission(LINEAR_CODE, T(np.concatenate([H.reshape(-1), np.zeros(m)]))),
        "user_range": cd.LearnableUserEmission(RANGE_CODE, T(np.concatenate([B.reshape(-1), [0.1]]))),
    }
    params = {k: cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(T(m0)), cov=cd.LearnableMatrix(T(np.eye(n)))),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableLorenz96(forcing=torch.tensor(8.0, **f64)),
                                           diffusion_coefficient=cd.LearnableMatrix(T(np.eye(n))),
                                           diffusion_cov=cd.LearnableMatrix(T(0.1 * np.eye(n)))),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=e, emission_cov=cd.LearnableMatrix(T(np.eye(m)))))
        for k, e in emissions.items()}
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    gaps = 0.02 * (0.5 + torch.rand(N, K, generator=g, **f64))
    gaps[:, 0] = 0.0
    t = torch.cumsum(gaps, dim=1)[..., None]
    ylin = 8 + 2 * torch.randn(N, K, m, generator=g, **f64)
    yrange = torch.as_tensor(np.sqrt(((m0 - B) ** 2).sum(-1) + 0.1), **f64) + torch.randn(N, K, m, generator=g, **f64)
    ys = {"stock_linear": ylin, "user_linear": ylin, "user_range": yrange}
    return params, ys, t


def run_cases(params, ys, t, hp, reps):
    calls = {k: (lambda k=k: cd.cdnlgssm_filter(params[k], ys[k], t, hp, output_fields=[])) for k in params}
    for fn in calls.values():  # warm-up: module load, variant load, first-touch allocations
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for k, fn in calls.items():
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
            assert bool(torch.isfinite(out.marginal_loglik).all()), k
    return {k: dict(median_ms=float(np.median(v)), min_ms=float(np.min(v)), max_ms=float(np.max(v)), reps=len(v))
            for k, v in times.items()}


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 5
    scale = float(sys.argv[sys.argv.index("--scale") + 1]) if "--scale" in sys.argv else 1.0
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(ROOT, "profiles",
                                                                                        "r03_user_emission_bench.jsonl")
    K = 500
    N4, N5 = max(148, int(8192 * scale)), max(37, int(1024 * scale))
    rec = dict(bench="user_emission", gpu_before=gpu_state(), K=K)
    st = {"solver": "rk4", "dt0": 0.005}
    params, ys, t = problem(N4, K, 4)
    rec["ekf_config4"] = dict(N=N4, **run_cases(params, ys, t, cd.EKFHyperParams(state_order="first",
                                                                                  diffeqsolve_settings=st), reps))
    rec["ukf_config4"] = dict(N=N4, **run_cases(params, ys, t, cd.UKFHyperParams(diffeqsolve_settings=st), reps))
    params, ys, t = problem(N5, K, 5)
    hp = cd.EnKFHyperParams(N_particles=1024, key=1234, diffeqsolve_settings={"solver": "euler", "dt0": 0.005})
    rec["enkf_config5"] = dict(N=N5, E=1024, **run_cases(params, ys, t, hp, reps))
    rec["gpu_after"] = gpu_state()
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
