"""GPU: per-trajectory (batched) model parameters on every kernel, one parameter slot at a time.

A leaf with a leading N sets bit `slot` of `cdk_desc.batched_mask`.  The warp kernels (kf_warp_filter / _smooth / _grad,
ekf_small_lw) load the model ONCE per CTA or warp unless the mask intersects their model mask; a slot missing from that
mask would make every trajectory of a CTA use warp 0's values.  Batching all slots at once hides such an omission (the
other slots set the mask), and so does a batch smaller than one CTA.  So every row of TARGETS below (one per dispatch
target) is run with each slot it reads batched ALONE, plus all of them together, at an N that spans several CTAs / warps
with a ragged last one, and checked for
  (a) parity with the NumPy oracle, which takes the same batched parameters, at the suite's existing gates;
  (b) path identity: the shared value expanded to N identical rows gives the shared call's result bit for bit;
  (c) chunked host streaming of the batched slot (the `lo * row` offset of `_engine.run`) = one device-resident launch;
  (d) the broadcast rule: a leading axis of 1 is the unbatched call, bit for bit;
  (e) dispatch: the launched kernel (and its template arguments) is the one the row is meant to reach."""
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _engine as E
from cd_dynamax_b200 import _lib as L
from oracle import cd_oracle as o
from tests.helpers import make_drift, max_rel_err, moment_err, record, scaled_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["filtered_means", "filtered_covariances", "predicted_means", "predicted_covariances"]
TOL = 1e-9


def _kernel_const(name, fname="cdk_kfwarp.cu"):
    """A launch-geometry constant of the CUDA source (trajectories per CTA of the warp kernels)."""
    with open(os.path.join(ROOT, "cd_dynamax_b200", "csrc", fname)) as f:
        return int(re.search(rf"constexpr int {name} = (\d+);", f.read()).group(1))


KW_WPC, KS_WPC, KG_WPC_MAX = (_kernel_const(k) for k in ("KW_WPC", "KS_WPC", "KG_WPC_MAX"))
# kf_warp_*: one trajectory per warp, KW_WPC / KS_WPC / (up to) KG_WPC_MAX per CTA -> two full rounds of every CTA size
# plus a ragged last CTA for each of them (53 for 4 / 6 / 8: 13 + 1, 8 + 1 and 6 + 1 CTAs)
_LCM = math.lcm(KW_WPC, KS_WPC, KG_WPC_MAX)
N_WARP = 2 * _LCM + min(KW_WPC, KS_WPC, KG_WPC_MAX) + 1
# ekf_small_lw / eks_small_lw: one trajectory per LANE; below 148 SMs x 32 trajectories lw_warps_per_cta gives one warp
# per CTA, so 71 = three CTAs, the last one ragged (7 live lanes)
N_LW = 2 * 32 + 7
N_CTA = 5  # one CTA per trajectory (generic kernels, EnKF)
K = 12


def fac(i):
    return 1.0 + 0.04 * ((7 * i) % 11)


F_N = lambda N: np.array([fac(i) for i in range(N)])  # noqa: E731

VEC = ("m0", "b", "d")


def batch_slot(g, slot, N):
    """g with g[slot] replaced by N distinct, well-conditioned per-trajectory values (SPD stays SPD)."""
    f = F_N(N)
    v = np.asarray(g[slot], np.float64)
    fb = f.reshape((N,) + (1,) * v.ndim)
    if slot in VEC:
        return dict(g, **{slot: v[None] * fb + 0.3 * (fb - 1.0)})
    return dict(g, **{slot: v[None] * fb})


def expand_slot(g, slot, N):
    return dict(g, **{slot: np.broadcast_to(np.asarray(g[slot]), (N,) + np.shape(g[slot])).copy()})


def lead1_all(g, slots):
    return dict(g, **{s: np.asarray(g[s])[None] for s in slots})


# ---- problems ---------------------------------------------------------------------------------------------------------
def l63_model(m, seed=1):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((3, 3))
    H = np.eye(3)[:m] + 0.1 * rng.standard_normal((m, 3))
    B = rng.standard_normal((m, m))
    return dict(m0=np.array([1.0, 1.0, 20.0]), P0=2 * np.eye(3) + 0.1 * (A + A.T), theta=np.array([10.0, 28.0, 8.0 / 3.0]),
                L=np.eye(3) + 0.1 * rng.standard_normal((3, 3)), Qc=np.eye(3) + 0.05 * (A @ A.T), H=H,
                d=0.1 * rng.standard_normal(m), R=0.5 * np.eye(m) + 0.05 * B @ B.T)


def nl_model(kind, n, m, seed=2):
    if kind == "lorenz63":
        return l63_model(m, seed)
    rng = np.random.default_rng(seed)
    if kind == "linear":
        theta = np.concatenate([(-0.5 * np.eye(n) + 0.3 * rng.standard_normal((n, n)) / np.sqrt(n)).ravel(),
                                0.1 * rng.standard_normal(n)])
    elif kind == "quadratic":
        theta = np.concatenate([0.2 * rng.standard_normal(n), (-0.8 * np.eye(n) + 0.1 * rng.standard_normal((n, n))).ravel(),
                                0.05 * rng.standard_normal(n ** 3)])
    elif kind == "lorenz96":
        theta = np.array([8.0])
    A = rng.standard_normal((m, m))
    x0 = 8.0 + rng.standard_normal(n) if kind == "lorenz96" else rng.standard_normal(n)
    return dict(m0=x0, P0=0.7 * np.eye(n), theta=theta, L=np.eye(n) + 0.1 * rng.standard_normal((n, n)),
                Qc=0.1 * np.eye(n) + 0.01, H=rng.standard_normal((m, n)) / np.sqrt(n), d=0.2 * rng.standard_normal(m),
                R=0.1 * (A @ A.T + np.eye(m)))


def kf_model(n, m, d_u=0, diag_r=False, seed=3):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((m, m))
    g = dict(m0=rng.standard_normal(n), P0=0.7 * np.eye(n), F=-0.5 * np.eye(n) + 0.3 * rng.standard_normal((n, n)) / np.sqrt(n),
             b=0.1 * rng.standard_normal(n), L=np.eye(n) + 0.1 * rng.standard_normal((n, n)), Qc=0.1 * np.eye(n) + 0.01,
             H=rng.standard_normal((m, n)), d=0.2 * rng.standard_normal(m),
             R=0.1 + 0.2 * rng.uniform(size=m) if diag_r else 0.1 * (A @ A.T + np.eye(m)))
    if d_u:
        g.update(BU=0.3 * rng.standard_normal((n, d_u)), DU=0.3 * rng.standard_normal((m, d_u)))
    return g


def data(N, m, gap, seed, d_u=0, scale=1.0):
    rng = np.random.default_rng(seed)
    gaps = gap * rng.uniform(0.5, 1.5, size=(N, K))
    gaps[:, 0] = 0.0
    t = np.cumsum(gaps, axis=1)
    y = scale * rng.standard_normal((N, K, m))
    u = rng.standard_normal((N, K, d_u)) if d_u else None
    return t, y, u


# One row per dispatch target: how the dispatch rules in code (launch_ekf_small, launch_eks_small, kf_warp_eligible, the
# reg_ode condition of launch_generic, launch_enkf) route this model / solver / dtype / entry point.
def _row(name, family, entry, kernel, N, n, m, solver, dt0, **kw):
    r = dict(name=name, family=family, entry=entry, kernel=kernel, N=N, n=n, m=m, solver=solver, dt0=dt0, dtype=np.float64,
             order="second", num_iter=1, drift="lorenz63", cov_rescaling=1.0, d_u=0, diag_r=False, smoother_type=1,
             cache=True, env={}, E=0, cluster=0)
    r.update(kw)
    return r


SID = o.SOLVER_IDS
TARGETS = [
    # ekf_small_lw<T, DriftL63, NY = m, SOLVER, WPC>: Lorenz-63, n = 3, m <= 3, first / second order, every dtype
    _row("lw_m1_f64_rk4_second", "nl", "ekf", r"ekf_small_lw<double,[^,]*DriftL63,\s*1,\s*5,", N_LW, 3, 1, "rk4", 0.0025),
    _row("lw_m2_f64_dopri5_first_iter2", "nl", "ekf", r"ekf_small_lw<double,[^,]*DriftL63,\s*2,\s*6,", N_LW, 3, 2, "dopri5",
         0.01, order="first", num_iter=2),
    _row("lw_m3_f64_rk4_first", "nl", "ekf", r"ekf_small_lw<double,[^,]*DriftL63,\s*3,\s*5,", N_LW, 3, 3, "rk4", 0.0025,
         order="first"),
    _row("lw_m1_f32_dopri5_second", "nl", "ekf", r"ekf_small_lw<float,[^,]*DriftL63,\s*1,\s*6,", N_LW, 3, 1, "dopri5", 0.01,
         dtype=np.float32),
    _row("lw_m3_f32_rk4_second_iter2", "nl", "ekf", r"ekf_small_lw<float,[^,]*DriftL63,\s*3,\s*5,", N_LW, 3, 3, "rk4", 0.0025,
         dtype=np.float32, num_iter=2),
    _row("lw_forecast", "nl", "forecast", r"ekf_small_lw<double,[^,]*DriftL63,\s*1,\s*5,", N_LW, 3, 1, "rk4", 0.0025),
    _row("eks_lw", "nl", "eks", r"eks_small_lw<double,[^,]*DriftL63,\s*5>", N_LW, 3, 1, "rk4", 0.0025),
    # generic_filter_kernel<T, 0>: every drift but Lorenz-63, Lorenz-63 at zeroth order or with a solver ekf_small_lw lacks
    _row("generic_ekf_linear", "nl", "ekf", r"generic_filter_kernel<double,\s*0>", N_CTA, 4, 2, "rk4", 0.01, drift="linear"),
    _row("generic_ekf_quadratic", "nl", "ekf", r"generic_filter_kernel<double,\s*0>", N_CTA, 3, 2, "rk4", 0.01,
         drift="quadratic"),
    _row("generic_ekf_l63_zeroth", "nl", "ekf", r"generic_filter_kernel<double,\s*0>", N_CTA, 3, 1, "rk4", 0.0025,
         order="zeroth", cov_rescaling=0.7),
    _row("generic_ekf_l63_bosh3_iter2", "nl", "ekf", r"generic_filter_kernel<double,\s*0>", N_CTA, 3, 1, "bosh3", 0.0025,
         num_iter=2),
    # generic_filter_kernel<T, 1>: the register-resident Lorenz-96 moment ODE (chain tableau)
    _row("l96_stencil_ekf", "nl", "ekf", r"generic_filter_kernel<double,\s*1>", N_CTA, 8, 4, "rk4", 0.005, drift="lorenz96"),
    _row("l96_stencil_ukf", "nl", "ukf", r"generic_filter_kernel<double,\s*1>", N_CTA, 8, 4, "rk4", 0.005, drift="lorenz96"),
    # the literal sigma-point UKF
    _row("ukf_sigma_l63", "nl", "ukf", r"generic_filter_kernel<double,\s*0>", N_CTA, 3, 1, "rk4", 0.0025,
         env={"CDK_UKF_SIGMA_POINTS": "1"}),
    _row("ukf_sigma_linear", "nl", "ukf", r"generic_filter_kernel<double,\s*0>", N_CTA, 4, 2, "rk4", 0.01, drift="linear",
         env={"CDK_UKF_SIGMA_POINTS": "1"}),
    # kf_warp_filter / kf_warp_smooth<POLY>: fp64, n <= 16, m <= 8, no inputs; chain tableaux (rk4) and Dopri5's polynomial
    _row("kfw_filter_rk4", "kf", "kf_filter", r"kf_warp_filter<false>", N_WARP, 5, 2, "rk4", 0.01),
    _row("kfw_filter_dopri5", "kf", "kf_filter", r"kf_warp_filter<true>", N_WARP, 5, 2, "dopri5", 0.01),
    _row("kfw_smooth_cached_dopri5", "kf", "kf_smoother", r"kf_warp_smooth<true>", N_WARP, 5, 2, "dopri5", 0.01),
    _row("kfw_smooth_uncached_rk4", "kf", "kf_smoother", r"kf_warp_smooth<false>", N_WARP, 5, 2, "rk4", 0.01, cache=False),
    # the generic KF: inputs, a diagonal R, n > 16, the type-2 smoother
    _row("generic_kf_inputs", "kf", "kf_filter", r"generic_filter_kernel<double,\s*0>", N_CTA, 4, 2, "rk4", 0.01, d_u=2),
    _row("generic_kf_diag_r", "kf", "kf_filter", r"generic_filter_kernel<double,\s*0>", N_CTA, 4, 2, "dopri5", 0.01,
         diag_r=True),
    _row("generic_kf_n20", "kf", "kf_smoother", r"generic_smooth_kernel<double>", N_CTA, 20, 3, "rk4", 0.01),
    _row("generic_kf_smoother2", "kf", "kf_smoother", r"generic_smooth_kernel<double>", N_CTA, 5, 2, "heun", 0.01,
         smoother_type=2),
    # enkf_kernel: the linear drift, with and without a thread-block cluster
    _row("enkf_linear", "nl", "enkf", r"enkf_kernel<double", N_CTA, 4, 2, "euler", 0.0125, drift="linear", E=48),
    _row("enkf_linear_cluster", "nl", "enkf", r"enkf_kernel<double", N_CTA, 4, 2, "heun", 0.0125, drift="linear", E=40,
         env={"CDK_ENKF_CLUSTER": "2"}),
]
ROWS = {r["name"]: r for r in TARGETS}


def slots_of(row):
    if row["family"] == "kf":
        s = ["m0", "P0", "F", "b", "L", "Qc", "H", "d", "R"]
        return s + (["BU", "DU"] if row["d_u"] else [])
    if row["entry"] == "forecast":
        return ["m0", "P0", "theta", "L", "Qc"]  # a forecast reads no emission model
    return ["m0", "P0", "theta", "L", "Qc", "H", "d", "R"]


def cases():
    for r in TARGETS:
        for s in slots_of(r) + ["all"]:
            yield pytest.param(r["name"], s, id=f"{r['name']}-{s}")


def base_problem(row):
    N, n, m = row["N"], row["n"], row["m"]
    if row["family"] == "kf":
        g = kf_model(n, m, row["d_u"], row["diag_r"])
        t, y, u = data(N, m, 0.04, 11 + n, row["d_u"])
    else:
        g = nl_model(row["drift"], n, m)
        l63 = row["drift"] == "lorenz63"
        t, y, u = data(N, m, 0.01 if l63 else 0.04, 7 + n + m, scale=8.0 if l63 else 1.0)
        if row["entry"] == "forecast":
            t = np.concatenate([np.zeros((N, 1)), 0.01 + t], axis=1)  # t_init = 0 first
    if row["dtype"] == np.float32:  # the oracle sees exactly the fp32-rounded numbers the kernel reads
        r32 = lambda a: None if a is None else np.asarray(a, np.float32).astype(np.float64)  # noqa: E731
        g = {k: r32(v) for k, v in g.items()}
        t, y, u = r32(t), r32(y), r32(u)
    return g, t, y, u


def problem(row, slot):
    g, t, y, u = base_problem(row)
    for s in (slots_of(row) if slot == "all" else [slot] if slot else []):
        g = batch_slot(g, s, row["N"])
    return g, t, y, u


# ---- the API call of a row ------------------------------------------------------------------------------------------
def drift_api(kind, theta, n):
    theta = theta if isinstance(theta, torch.Tensor) else np.asarray(theta)
    if kind == "lorenz63":
        return cd.LearnableLorenz63(sigma=theta[..., 0], rho=theta[..., 1], beta=theta[..., 2])
    if kind == "lorenz96":
        return cd.LearnableLorenz96(forcing=theta[..., 0])
    lead = tuple(theta.shape[:-1])
    if kind == "linear":
        return cd.LearnableLinear(weights=theta[..., :n * n].reshape(lead + (n, n)), bias=theta[..., n * n:])
    return cd.LearnableQuadratic(a=theta[..., :n], B=theta[..., n:n + n * n].reshape(lead + (n, n)),
                                 C=theta[..., n + n * n:].reshape(lead + (n, n, n)))


def api_params(row, g):
    if row["family"] == "kf":
        return cd.make_cdlgssm_params(g["m0"], g["P0"], g["F"], g["L"], g["Qc"], g["H"], g["R"], dynamics_bias=g["b"],
                                      dynamics_input_weights=g.get("BU"), emissions_bias=g["d"],
                                      emissions_input_weights=g.get("DU"))
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(g["m0"]), cov=cd.LearnableMatrix(g["P0"])),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=drift_api(row["drift"], g["theta"], row["n"]),
                                           diffusion_coefficient=cd.LearnableMatrix(g["L"]),
                                           diffusion_cov=cd.LearnableMatrix(g["Qc"])),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=g["H"], bias=g["d"]),
                                             emission_cov=cd.LearnableMatrix(g["R"])))


OUT_FIELDS = {"ekf": ["marginal_loglik"] + FIELDS, "ukf": ["marginal_loglik"] + FIELDS, "enkf": ["marginal_loglik"] + FIELDS,
              "kf_filter": ["marginal_loglik"] + FIELDS,
              "eks": ["marginal_loglik", "filtered_means", "filtered_covariances", "smoothed_means", "smoothed_covariances"],
              "kf_smoother": ["marginal_loglik", "filtered_means", "filtered_covariances", "smoothed_means",
                              "smoothed_covariances", "smoothed_cross_covariances"],
              "forecast": ["forecasted_state_means", "forecasted_state_covariances"]}


def run_api(row, g, t, y, u, dev=None):
    """-> {field: numpy array} of the row's entry point.  `dev`: hand every array in as a CUDA tensor instead."""
    T = (lambda a: a) if dev is None else (lambda a: None if a is None else torch.as_tensor(np.asarray(a), device=dev))
    if dev is not None:
        g = {k: T(v) for k, v in g.items()}
    dt = row["dtype"]
    y, t = T(np.asarray(y, dt)), T(np.asarray(t, dt))
    u = None if u is None else T(np.asarray(u, dt))
    p = api_params(row, g)
    settings = {"solver": row["solver"], "dt0": row["dt0"]}
    e = row["entry"]
    if e in ("ekf", "eks", "forecast"):
        hp = cd.EKFHyperParams(state_order=row["order"], cov_rescaling=row["cov_rescaling"], diffeqsolve_settings=settings)
    elif e == "ukf":
        hp = cd.UKFHyperParams(diffeqsolve_settings=settings)
    elif e == "enkf":
        hp = cd.EnKFHyperParams(N_particles=row["E"], key=4321, diffeqsolve_settings=settings)
    else:
        hp = cd.KFHyperParams(dt_final=0.03, diffeqsolve_settings=settings)
    if e in ("ekf", "ukf", "enkf"):
        post = cd.cdnlgssm_filter(p, y, t[..., None], hp, num_iter=row["num_iter"])
    elif e == "eks":
        post = cd.cdnlgssm_smoother(p, y, t[..., None], hp)
    elif e == "forecast":
        post = cd.cdnlgssm_forecast(p, (g["m0"], g["P0"]), t[:, 0], t[:, 1:, None], hyperparams=hp)
    elif e == "kf_filter":
        post = cd.cdlgssm_filter(p, y, t[..., None], hp, u)
    else:
        post = cd.cdlgssm_smoother(p, y, t[..., None], hp, u, smoother_type=f"cd_smoother_{row['smoother_type']}")
    c = lambda x: x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)  # noqa: E731
    return {f: c(getattr(post, f)) for f in OUT_FIELDS[e]}


def call(row, g, t, y, u, monkeypatch, dev=None):
    for k, v in row["env"].items():
        monkeypatch.setenv(k, v)
    if not row["cache"]:
        # no room for the pushforward cache: the type-1 smoother re-integrates every gap
        free, total = torch.cuda.mem_get_info()
        monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a, **k: (0, total))
    try:
        return run_api(row, g, t, y, u, dev)
    finally:
        monkeypatch.undo()


# ---- the oracle run of a row ----------------------------------------------------------------------------------------
def run_oracle(row, g, t, y, u):
    e, n = row["entry"], row["n"]
    s = o.SolverSettings(row["solver"], float(np.float32(row["dt0"])) if row["dtype"] == np.float32 else row["dt0"],
                         time_dtype=np.float32 if row["dtype"] == np.float32 else None)
    if row["family"] == "kf":
        p = o.LinearParams(m0=g["m0"], P0=g["P0"], F=g["F"], L=g["L"], Qc=g["Qc"], H=g["H"], R=g["R"], b=g["b"], d=g["d"],
                           B=g.get("BU"), D=g.get("DU"))
        if e == "kf_filter":
            return o.cdlgssm_filter(p, y, t, dt_final=0.03, settings=s, inputs=u)
        return o.cdlgssm_smoother(p, y, t, dt_final=0.03, settings=s, inputs=u, smoother_type=row["smoother_type"])
    p = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift(row["drift"], g["theta"], n), L=g["L"], Qc=g["Qc"],
                          H=g["H"], R=g["R"], d=g["d"])
    if e == "ekf":
        return o.extended_kalman_filter(p, y, t, state_order=row["order"], settings=s, num_iter=row["num_iter"],
                                        cov_rescaling=row["cov_rescaling"])
    if e == "forecast":
        r = o.extended_kalman_filter(p, y, t, state_order=row["order"], settings=s, forecast=True)
        return dict(forecasted_state_means=r["predicted_means"], forecasted_state_covariances=r["predicted_covariances"])
    if e == "eks":
        return o.extended_kalman_smoother(p, y, t, state_order=row["order"], settings=s)
    if e == "ukf":
        return o.unscented_kalman_filter(p, y, t, settings=s)
    return o.ensemble_kalman_filter(p, y, t, E=row["E"], seed=4321, settings=s)


def check_parity(row, got, ref, tag):
    """The gates of the existing tests of each kernel family."""
    e = row["entry"]
    if row["dtype"] == np.float32:  # test_ekf_l63_fp32_variant_bound
        err = max_rel_err(got["marginal_loglik"], ref["marginal_loglik"])
        record(f"batched:{tag}:marginal_loglik", err)
        assert err < 2e-4, (tag, err)
        for f in FIELDS:
            err = scaled_err(got[f], ref[f])
            record(f"batched:{tag}:{f}", err)
            assert err < 2e-3, (tag, f, err)
        return
    if e == "forecast":  # test_gpu_forecast_sample
        for f in got:
            err = scaled_err(got[f], ref[f])
            record(f"batched:{tag}:{f}", err)
            assert err < 1e-8, (tag, f, err)
        return
    if e == "enkf":  # test_enkf_vs_oracle
        for f in got:
            err = max_rel_err(got[f], ref[f]) if f == "marginal_loglik" else scaled_err(got[f], ref[f])
            record(f"batched:{tag}:{f}", err)
            assert err < 1e-8, (tag, f, err)
        return
    err = max_rel_err(got["marginal_loglik"], ref["marginal_loglik"])
    record(f"batched:{tag}:marginal_loglik", err)
    assert err < TOL, (tag, err)
    for f in got:
        if f == "marginal_loglik":
            continue
        if f.startswith("smoothed"):
            if ref[f].size == 0 or np.isnan(ref[f]).all():
                assert np.isnan(got[f]).all() == np.isnan(ref[f]).all(), (tag, f)
                continue
            err = scaled_err(got[f], ref[f])
            record(f"batched:{tag}:{f}", err)
            assert err < 1e-8, (tag, f, err)
            continue
        post = type("P", (), {f: got[f]})
        ge, en = moment_err(post, ref, f)
        record(f"batched:{tag}:{f}:gate", ge)
        record(f"batched:{tag}:{f}:own_norm", en)
        assert ge < TOL and en < 0.1 * TOL, (tag, f, ge, en)


@pytest.mark.parametrize("name,slot", list(cases()))
def test_batched_slot_matches_oracle(name, slot, monkeypatch):
    """(a) Each slot batched alone (and all together) against the oracle given the same per-trajectory parameters."""
    row = ROWS[name]
    g, t, y, u = problem(row, slot)
    got = call(row, g, t, y, u, monkeypatch)
    ref = run_oracle(row, g, t, y, u)
    check_parity(row, got, ref, f"{name}:{slot}")


# ---- (b) path identity ------------------------------------------------------------------------------------------------
def lw_batched_wpc(row):
    """Warps per CTA of ekf_small_lw when a parameter block is batched (launch_one, cdk_small.cu): 7 when fourteen warps'
    per-lane fp64 blocks exceed the 227 KB of a CTA; the fp32 blocks are half as large and keep the 14-warp variant."""
    return 7 if row["dtype"] == np.float64 else 14


LW_ROWS = [r["name"] for r in TARGETS if "_small_lw" in r["kernel"] and lw_batched_wpc(r) == 7]
# the slots ekf_small_lw reads per lane when any of them is batched (par_mask, cdk_small.cu); the 7-warp variant serves them
LW_PAR_SLOTS = ("theta", "L", "Qc", "H", "d", "R")


def _assert_same(a, b, tag):
    for f in a:
        assert a[f].shape == b[f].shape, (tag, f)
        same = np.array_equal(a[f], b[f], equal_nan=True)
        if not same:
            d = np.nanmax(np.abs(a[f] - b[f]))
            raise AssertionError(f"{tag}: {f} is not bit-identical (max |difference| {d:.3e})")


@pytest.fixture(scope="module")
def lw_shared_wpc7(tmp_path_factory):
    """The shared-parameter results of the register rows under CDK_LW_WPC=7, the instantiation a batched parameter block
    runs on.  CDK_LW_WPC is read once per process (a static initialiser), so they come from a child process."""
    out = tmp_path_factory.mktemp("lw_wpc7")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-c", "import sys; from tests.test_gpu_batched_parameters import _child_main; _child_main(sys.argv[1])", str(out)]
    env = dict(os.environ, CDK_LW_WPC="7", PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    res = {}
    for name in LW_ROWS:
        with np.load(out / f"{name}.npz") as z:
            res[name] = {k: z[k] for k in z.files}
    return res


def _child_main(out_dir):
    for name in LW_ROWS:
        row = ROWS[name]
        g, t, y, u = problem(row, None)
        np.savez(os.path.join(out_dir, f"{name}.npz"), **run_api(row, g, t, y, u))


@pytest.mark.parametrize("name,slot", list(cases()))
def test_expanded_shared_value_is_bit_identical(name, slot, monkeypatch, request):
    """(b) The shared value expanded to N identical rows sets the mask bit without changing a value: the result must be
    the shared call's, bit for bit."""
    row = ROWS[name]
    g, t, y, u = base_problem(row)
    ge = g
    for s in (slots_of(row) if slot == "all" else [slot]):
        ge = expand_slot(ge, s, row["N"])
    got = call(row, ge, t, y, u, monkeypatch)
    if name in LW_ROWS and (slot == "all" or slot in LW_PAR_SLOTS) and lw_batched_wpc(row) == 7:
        ref = request.getfixturevalue("lw_shared_wpc7")[name]
    else:
        ref = call(row, g, t, y, u, monkeypatch)
    _assert_same(got, ref, f"{name}:{slot}")


# ---- (c) chunked host streaming ---------------------------------------------------------------------------------------
STREAM_ROWS = {"generic_ekf_quadratic": 21, "kfw_smooth_cached_dopri5": N_WARP}


@pytest.mark.parametrize("name,slot", [(nm, s) for nm in STREAM_ROWS for s in slots_of(ROWS[nm])])
def test_chunked_streaming_of_a_batched_slot(name, slot, monkeypatch):
    """(c) Host-resident batched parameters staged in N-chunks (each chunk offsets every batched slot by lo * row) give
    the device-resident single launch bit for bit."""
    row = dict(ROWS[name], N=STREAM_ROWS[name])
    g, t, y, u = problem(row, slot)
    assert row["N"] >= 2 * E.STREAM_CHUNKS
    once = call(row, g, t, y, u, monkeypatch, dev=torch.device("cuda", 0))
    monkeypatch.setattr(E, "STREAM_MIN_BYTES", 1)
    chunked = run_api(row, g, t, y, u)
    monkeypatch.undo()
    _assert_same(chunked, once, f"{name}:{slot}:chunked")


# ---- (d) broadcast rule -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(ROWS))
def test_leading_axis_of_one_is_shared(name, monkeypatch):
    """(d) Every slot with a leading axis of length 1 is the unbatched call, bit for bit."""
    row = ROWS[name]
    g, t, y, u = base_problem(row)
    got = call(row, lead1_all(g, slots_of(row)), t, y, u, monkeypatch)
    _assert_same(got, call(row, g, t, y, u, monkeypatch), f"{name}:lead1")


# ---- (e) dispatch -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(ROWS))
def test_row_reaches_its_kernel(name, monkeypatch):
    """(e) The kernel (and template arguments) each row is meant to reach, from the CUDA activity of a profiled call with
    every slot batched."""
    from torch.profiler import ProfilerActivity, profile
    row = ROWS[name]
    g, t, y, u = problem(row, "all")
    call(row, g, t, y, u, monkeypatch)  # warm (module load, tensor maps) outside the profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call(row, g, t, y, u, monkeypatch)
        torch.cuda.synchronize()
    names = sorted({ev.key for ev in prof.key_averages()})
    assert any(re.search(row["kernel"], k) for k in names), (name, row["kernel"], names)
    if "ekf_small_lw" in row["kernel"]:  # every lane carries its own parameter block
        wpc = lw_batched_wpc(row)
        assert any(re.search(row["kernel"] + rf"\s*{wpc}\b", k) for k in names), (name, wpc, names)


# ---- the gradients ----------------------------------------------------------------------------------------------------
KF_GRAD_SLOTS = ["F", "b", "L", "Qc", "H", "d", "R", "m0", "P0"]


@pytest.mark.parametrize("slot", KF_GRAD_SLOTS)
def test_kf_warp_grad_one_slot_batched(slot):
    """kf_warp_grad with ONE slot batched (the existing arbiter cases batch every slot at once, which sets the model mask
    through the others), N over several CTAs of up to KG_WPC_MAX warps, against torch autograd of the arbiter."""
    from tests.test_gpu_kf_grad import compare
    from tests.test_kf_grad_host import random_grid, random_model
    N, n, m = N_WARP, 5, 2
    p = batch_slot(random_model(n, m, seed=17), slot, N)
    y = np.random.default_rng(3).standard_normal((N, K, m))
    compare(f"batched_one_slot:{slot}", p, y, random_grid(N, K, 6), "rk4", 0.02)


L63_GRAD_SLOTS = ["L", "Qc", "H", "d", "R", "m0", "P0"]
N_GRAD = 128 + 5  # ekf_l63_grad_kernel: one trajectory per thread, 128 per CTA -> a second, ragged CTA


@pytest.mark.parametrize("slot", L63_GRAD_SLOTS)
def test_ekf_l63_grad_one_slot_batched(slot, monkeypatch):
    """The Lorenz-63 CD-EKF gradient with one slot batched: reverse mode against forward mode (both exact derivatives of
    the same discrete filter), and row i of the batch against a shared-parameter call with sample i's values."""
    N = N_GRAD
    g0 = l63_model(1)
    g = batch_slot(g0, slot, N)
    t, y, _ = data(N, 1, 0.01, 5, scale=8.0)
    row = dict(ROWS["lw_m1_f64_rk4_second"], N=N)
    hp = cd.EKFHyperParams(dt_final=0.004, diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    monkeypatch.setenv("CDK_GRAD_MODE", "forward")
    ll_f, gf = cd.ekf_marginal_log_prob_and_grad(api_params(row, g), y, t[..., None], hp, wrt="all")
    monkeypatch.setenv("CDK_GRAD_MODE", "reverse")
    ll_r, gr = cd.ekf_marginal_log_prob_and_grad(api_params(row, g), y, t[..., None], hp, wrt="all")
    assert max_rel_err(ll_r, ll_f) < 1e-12
    for k in sorted(gf):
        err = np.max(np.abs(gr[k] - gf[k])) / np.max(np.abs(gf[k]))
        record(f"batched:ekf_l63_grad:{slot}:{k}", err)
        assert err < 1e-9, (slot, k, err)
    for i in (0, 64, N - 1):
        gi = dict(g0, **{slot: np.asarray(g[slot])[i]})
        ll_i, g_i = cd.ekf_marginal_log_prob_and_grad(api_params(row, gi), y, t[..., None], hp, wrt="all")
        assert max_rel_err(ll_r[i], ll_i[i]) < 1e-13, (slot, i)
        for k in gr:
            assert np.max(np.abs(gr[k][i] - g_i[k][i])) <= 1e-12 * max(1.0, np.max(np.abs(g_i[k][i]))), (slot, i, k)


# ---- sampler and emission moments: batched m0 only / nothing batched -------------------------------------------------
def test_sampler_batched_m0_and_loud_refusal_of_model_slots():
    N, m = 37, 1
    g = l63_model(m)
    gm = batch_slot(g, "m0", N)
    row = dict(ROWS["lw_m1_f64_rk4_second"], N=N)
    t = np.cumsum(np.full((1, K), 0.01), axis=1)
    settings = {"solver": "heun", "dt0": 0.0025}
    xs, ys = cd.cdnlgssm_path_sample(api_params(row, gm), 99, K, t[0][:, None], diffeqsolve_settings=settings,
                                     num_sequences=N)
    po = o.NonlinearParams(m0=gm["m0"], P0=g["P0"], drift=make_drift("lorenz63", g["theta"], 3), L=g["L"], Qc=g["Qc"],
                           H=g["H"], R=g["R"], d=g["d"])
    rx, ry = o.sample_paths(po, np.repeat(t, N, 0), seed=99, settings=o.SolverSettings("heun", 0.0025))
    for tag, a, b in (("states", xs, rx), ("emissions", ys, ry)):
        err = scaled_err(a, b)
        record(f"batched:sampler:m0:{tag}", err)
        assert err < 1e-8, (tag, err)
    for slot in ("P0", "theta", "L", "Qc", "H", "d", "R"):
        with pytest.raises(L.CdkError, match="must not be batched"):
            cd.cdnlgssm_path_sample(api_params(row, batch_slot(g, slot, N)), 99, K, t[0][:, None],
                                    diffeqsolve_settings=settings, num_sequences=N)


@pytest.mark.parametrize("slot", ["H", "d", "R"])
def test_emission_moments_refuse_batched_emission_model(slot):
    N, m = 6, 2
    g = nl_model("linear", 4, m)
    row = dict(ROWS["generic_ekf_linear"], N=N)
    sm = np.random.default_rng(1).standard_normal((N, K, 4))
    sp = np.broadcast_to(np.eye(4), (N, K, 4, 4)).copy()
    t = np.cumsum(np.full((N, K), 0.01), axis=1)[..., None]
    em, ec = cd.cdnlgssm_emissions(api_params(row, g), t, sm, sp, hyperparams=cd.EKFHyperParams())
    assert np.isfinite(em).all() and np.isfinite(ec).all()
    with pytest.raises(L.CdkError, match="must not be batched"):
        cd.cdnlgssm_emissions(api_params(row, batch_slot(g, slot, N)), t, sm, sp, hyperparams=cd.EKFHyperParams())
