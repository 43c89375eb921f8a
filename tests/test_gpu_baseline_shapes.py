"""GPU parity at the shapes BASELINE.json benchmarks (VERDICT r01 "no parity test at BASELINE sizes"):

  C3  CD-EKF Lorenz-63, K = 1,000 chaotic steps, N = 2,048 and every launch geometry the occupancy-aware launcher picks
      (1 .. 14 warps per CTA), against the C restatement (oracle/cd_oracle_c.c, itself pinned to the NumPy oracle in
      tests/test_oracle_golden.py);
  C4  CD-UKF Lorenz-96 n = 40, m = 20 (5 Cholesky panels, the aliased 108 KB layout) against the NumPy oracle;
  C5  CD-EnKF E = 1,024 members on a 4-CTA cluster (256 members per CTA, the benchmarked shape);
  C2  CD-KF n = 16, m = 4, K = 500 (filter, both smoother types);
and one stated-bound test for every fp32 entry point of include/cdk.h.

Gates: log-likelihood rel 1e-9; filtered / predicted moments: SURVEY 8(d)'s element-wise gate at 1e-9 and 1e-10 of every
moment's own norm (tests/helpers.gate_err, moment_norm_err); smoothed moments and the EnKF 1e-8 (see test_gpu_parity.py);
fp32 bounds are written in each test, about 10x the error measured on B200 (gpurun_out/parity_errors.json)."""
import ctypes

import numpy as np
import pytest

from oracle import cd_oracle as o
from tests.helpers import gate_err, max_rel_err, moment_err, record, scaled_err
from tests.test_gpu_parity import FIELDS, TOL, api, c3_problem, check_moments, linear_params_api, nonlinear_params_api

pytestmark = pytest.mark.gpu

L63 = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]), L=np.eye(3),
           Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))


def _c_oracle_ekf(y, t, solver="rk4", dt0=0.0025, dt_final=1e-10):
    from oracle import cpu_baseline as cb
    g = L63
    return cb.filter_c("ekf", y, t, g["m0"], g["P0"], g["theta"], g["L"], g["Qc"], g["H"], g["d"], g["R"], drift_id=1,
                       solver=solver, dt0=dt0, dt_final=dt_final)


def test_c3_ekf_l63_k1000_multi_cta_vs_c_oracle():
    """BASELINE config 3 at full K: 2,048 trajectories (64 warps, several CTAs), 1,000 irregular gaps with 3..6 RK4
    substeps each, the every-8-steps log folding of the scalar-emission update, TMA tensor stores of all four moments."""
    cd = api()
    N, K = 2048, 1000
    t, y = c3_problem(N, K)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    f = cd.cdnlgssm_filter(nonlinear_params_api(L63), y, t[..., None], hp)
    r = _c_oracle_ekf(y, t)
    assert np.isfinite(r["marginal_loglik"]).all()
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record("c3_k1000:marginal_loglik", e)
    assert e < TOL
    check_moments(f, r, "c3_k1000")
    # log-likelihood-only call (no staging, no stores) and the cumulative form take different code paths in the kernel
    f0 = cd.cdnlgssm_filter(nonlinear_params_api(L63), y, t[..., None], hp, output_fields=[])
    assert max_rel_err(f0.marginal_loglik, r["marginal_loglik"]) < TOL
    fc = cd.cdnlgssm_filter(nonlinear_params_api(L63), y[:300], t[:300, :, None], hp, output_fields=["marginal_loglik"])
    assert max_rel_err(fc.marginal_loglik[:, -1], r["marginal_loglik"][:300]) < TOL


def test_c3_full_size_sharding_invariance_and_oracle_sample():
    """BASELINE config 3 at FULL size (N = 65,536, K = 1,000; the time-sliced launch) through size-independent properties:
    the full batch equals its eight 8,192-trajectory shards bit for bit (what trajectory sharding over 8 GPUs relies on: a
    trajectory's arithmetic does not depend on the batch it travels in, nor on the launch geometry), a permuted batch gives the
    permuted result, and a sample of trajectories matches the C oracle."""
    import torch
    cd = api()
    N, K = 65536, 1000
    t, y = c3_problem(N, K, seed=3)
    dev = torch.device("cuda", 0)
    td, yd = torch.as_tensor(t, device=dev), torch.as_tensor(y, device=dev)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    p = nonlinear_params_api(L63)
    full = cd.cdnlgssm_filter(p, yd, td[..., None], hp, output_fields=["filtered_means", "predicted_covariances"])
    assert bool(torch.isfinite(full.marginal_loglik).all())
    for sh in range(8):
        lo, hi = sh * 8192, (sh + 1) * 8192
        part = cd.cdnlgssm_filter(p, yd[lo:hi], td[lo:hi, :, None], hp, output_fields=["filtered_means", "predicted_covariances"])
        assert torch.equal(part.marginal_loglik, full.marginal_loglik[lo:hi]), sh
        assert torch.equal(part.filtered_means, full.filtered_means[lo:hi]), sh
        assert torch.equal(part.predicted_covariances, full.predicted_covariances[lo:hi]), sh
    perm = torch.randperm(N, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    pf = cd.cdnlgssm_filter(p, yd[perm].contiguous(), td[perm].contiguous()[..., None], hp, output_fields=["filtered_means"])
    assert torch.equal(pf.marginal_loglik, full.marginal_loglik[perm])
    assert torch.equal(pf.filtered_means, full.filtered_means[perm])
    sel = np.r_[0:96, 30000:30096, N - 64:N]
    r = _c_oracle_ekf(y[sel], t[sel])
    e = max_rel_err(full.marginal_loglik[sel].cpu().numpy(), r["marginal_loglik"])
    record("c3_full_size_sample:marginal_loglik", e)
    assert e < TOL
    assert gate_err(full.filtered_means[sel].cpu().numpy(), r["filtered_means"]) < TOL


@pytest.mark.parametrize("N", [4736, 4737, 8192, 16384, 20000, 41000])
def test_c3_occupancy_aware_launch_geometries(N):
    """The launcher picks 1, 2, 4, 5, 9 ... warps per CTA from N (148 SMs): N = 8,192 is the 8-GPU shard of config 3 and
    N = 16,384 the 4-GPU one.  Every geometry must give the oracle's numbers, the ragged last warp / CTA included."""
    cd = api()
    K = 24
    t, y = c3_problem(N, K, seed=N)
    hp = cd.EKFHyperParams(dt_final=0.003, diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    s = cd.cdnlgssm_smoother(nonlinear_params_api(L63), y, t[..., None], hp)  # filter + EKS backward pass
    r = _c_oracle_ekf(y, t, dt_final=0.003)
    assert max_rel_err(s.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(s, r, f"c3_geometry_N{N}", fields=("filtered_means", "filtered_covariances"))
    sel = np.r_[0:40, N - 40:N]  # the NumPy oracle smooths the first and the last trajectories
    po = o.NonlinearParams(m0=L63["m0"], P0=L63["P0"], drift=o.Lorenz63Drift(*L63["theta"]), L=L63["L"], Qc=L63["Qc"],
                           H=L63["H"], R=L63["R"], d=L63["d"])
    rs = o.extended_kalman_smoother(po, y[sel], t[sel], dt_final=0.003, settings=o.SolverSettings("rk4", 0.0025))
    for fld in ("smoothed_means", "smoothed_covariances"):
        assert scaled_err(getattr(s, fld)[sel], rs[fld]) < 1e-8, fld


def _l96_case(N, K, seed, n=40, m=20):
    rng = np.random.default_rng(seed)
    x0 = 8.0 + rng.standard_normal(n)
    g = dict(m0=x0, P0=np.eye(n), drift="lorenz96", theta=np.array([8.0]), L=np.eye(n), Qc=0.1 * np.eye(n),
             H=np.eye(n)[::2][:m], R=np.eye(m), d=np.zeros(m))
    gaps = 0.02 * rng.uniform(0.5, 1.5, size=(N, K))
    gaps[:, 0] = 0.0
    t = np.cumsum(gaps, axis=1)
    y = (g["H"] @ x0)[None, None, :] + 2.0 * rng.standard_normal((N, K, m))
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=o.Lorenz96Drift(8.0), L=g["L"], Qc=g["Qc"], H=g["H"], R=g["R"],
                           d=g["d"])
    return g, po, t, y


@pytest.mark.parametrize("sigma_points", [False, True])
@pytest.mark.parametrize("solver,dt0", [("rk4", 0.005), ("dopri5", 0.01)])
def test_c4_ukf_l96_n40_m20_vs_oracle(solver, dt0, sigma_points, monkeypatch):
    """BASELINE config 4 shape: n = 40, m = 20, against the oracle's literal sigma points.  Closed-form kernel (default):
    stencil Jacobian, RK4 takes the aliased 84 KB layout.  Sigma-point kernel: the blocked Cholesky runs 5 panels, RK4 (a
    chain tableau with m <= n) takes the aliased two-CTAs-per-SM layout, Dopri5 the six-stage one."""
    cd = api()
    monkeypatch.setenv("CDK_UKF_SIGMA_POINTS", "1" if sigma_points else "0")
    solver_tag = solver + ("_sigma" if sigma_points else "_closed")
    g, po, t, y = _l96_case(N=6, K=40, seed=40)
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": solver, "dt0": dt0})
    f = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], hp)
    r = o.unscented_kalman_filter(po, y, t, settings=o.SolverSettings(solver, dt0))
    assert np.isfinite(r["marginal_loglik"]).all()
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record(f"c4_ukf_n40_{solver_tag}:marginal_loglik", e)
    assert e < TOL
    check_moments(f, r, f"c4_ukf_n40_{solver_tag}")


@pytest.mark.parametrize("algo", ["ekf", "ukf"])
@pytest.mark.parametrize("solver,dt0", [("euler", 0.004), ("heun", 0.005), ("midpoint", 0.005), ("bosh3", 0.006), ("dopri5", 0.01)])
def test_l96_register_ode_every_solver_vs_oracle(algo, solver, dt0):
    """The register-resident Lorenz-96 moment ODE at n = 40 for every tableau: odd stage counts (euler 1, bosh3 3: the stage
    buffers alternate over all stages of a solve), b_1 = 0 (midpoint) and the six-stage Dopri5 variant (stage increments in
    registers), EKF (compact two-CTA layout) and closed-form UKF."""
    cd = api()
    g, po, t, y = _l96_case(N=4, K=25, seed=60 + len(solver))
    p = nonlinear_params_api(g)
    st = {"solver": solver, "dt0": dt0}
    if algo == "ekf":
        f = cd.cdnlgssm_filter(p, y, t[..., None], cd.EKFHyperParams(diffeqsolve_settings=st))
        r = o.extended_kalman_filter(po, y, t, settings=o.SolverSettings(solver, dt0))
    else:
        f = cd.cdnlgssm_filter(p, y, t[..., None], cd.UKFHyperParams(diffeqsolve_settings=st))
        r = o.unscented_kalman_filter(po, y, t, settings=o.SolverSettings(solver, dt0))
    assert np.isfinite(r["marginal_loglik"]).all()
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record(f"l96_reg_{algo}_{solver}:marginal_loglik", e)
    assert e < TOL
    check_moments(f, r, f"l96_reg_{algo}_{solver}")


@pytest.mark.parametrize("solver", ["euler", "heun"])
def test_c5_enkf_l96_e1024_cluster4_vs_oracle(solver):
    """BASELINE config 5 shape: 1,024 members = a cluster of 4 CTAs x 256 members (the launcher's own choice for E = 1,024,
    no CDK_ENKF_CLUSTER override), n = 40, m = 20, shared Philox stream."""
    cd = api()
    g, po, t, y = _l96_case(N=3, K=10, seed=50)
    hp = cd.EnKFHyperParams(N_particles=1024, key=1234, diffeqsolve_settings={"solver": solver, "dt0": 0.005})
    f = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], hp)
    r = o.ensemble_kalman_filter(po, y, t, E=1024, seed=1234, settings=o.SolverSettings(solver, 0.005))
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record(f"c5_enkf_e1024_{solver}:marginal_loglik", e)
    assert e < 1e-8
    for fld in FIELDS:
        record(f"c5_enkf_e1024_{solver}:{fld}:own_norm", moment_err(f, r, fld)[1])
        assert scaled_err(getattr(f, fld), r[fld]) < 1e-8, fld


def _c2_case(N, K, seed=1235, n=16, m=4):
    rng = np.random.default_rng(seed)
    F = -0.5 * np.eye(n) + 0.3 * rng.standard_normal((n, n)) / np.sqrt(n)
    g = dict(m0=np.zeros(n), P0=np.eye(n), F=F, b=np.zeros(n), B=None, L=np.eye(n), Qc=0.1 * np.eye(n), H=np.eye(n)[:m],
             d=np.zeros(m), D=None, R=0.1 * np.eye(m))
    gaps = 0.04 * rng.uniform(0.5, 1.5, size=(N, K))
    gaps[:, 0] = 0.0
    t = np.cumsum(gaps, axis=1)
    y = rng.standard_normal((N, K, m))
    po = o.LinearParams(m0=g["m0"], P0=g["P0"], F=F, L=g["L"], Qc=g["Qc"], H=g["H"], R=g["R"], b=g["b"], d=g["d"])
    return g, po, t, y


@pytest.mark.parametrize("solver,dt0", [("rk4", 0.01), ("dopri5", 0.01)])
def test_c2_kf_n16_k500_vs_oracle(solver, dt0):
    """BASELINE config 2 at full K: n = 16, m = 4, K = 500, N = 64 -- filter on the C oracle, both smoother types on the
    NumPy oracle (first trajectories).  dopri5 is the reference's default solver (diffrax_utils.py:121-124)."""
    from oracle import cpu_baseline as cb
    cd = api()
    N, K = 64, 500
    g, po, t, y = _c2_case(N, K)
    hp = cd.KFHyperParams(diffeqsolve_settings={"solver": solver, "dt0": dt0})
    f = cd.cdlgssm_filter(linear_params_api(g), y, t[..., None], hp)
    r = cb.filter_c("kf", y, t, g["m0"], g["P0"], g["F"], g["L"], g["Qc"], g["H"], g["d"], g["R"], bias=g["b"],
                    solver=solver, dt0=dt0)
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record(f"c2_kf_k500_{solver}:marginal_loglik", e)
    assert e < TOL
    check_moments(f, r, f"c2_kf_k500_{solver}")
    ns = 3
    for stype in ("cd_smoother_1", "cd_smoother_2"):
        s = cd.cdlgssm_smoother(linear_params_api(g), y[:ns], t[:ns, :, None], hp, smoother_type=stype)
        rs = o.cdlgssm_smoother(po, y[:ns], t[:ns], settings=o.SolverSettings(solver, dt0), smoother_type=int(stype[-1]))
        for fld in ("smoothed_means", "smoothed_covariances"):
            record(f"c2_kf_k500_{solver}_{stype}:{fld}:own_norm", moment_err(s, rs, fld)[1])
            assert scaled_err(getattr(s, fld), rs[fld]) < 1e-8, (stype, fld)


@pytest.mark.parametrize("E,cluster", [(1024, 4), (600, 4), (1000, 8), (200, 1)])
def test_c5_enkf_light_mapping_is_bit_identical(E, cluster, monkeypatch):
    """The two-threads-per-member mapping (ensemble swept in place in shared memory, 512 threads) against the
    one-thread-per-member register mapping: same counters, same operation order -> identical bits (ragged last CTA at E = 600)."""
    cd = api()
    g, po, t, y = _l96_case(N=2, K=12, seed=51)
    hp = cd.EnKFHyperParams(N_particles=E, key=77, diffeqsolve_settings={"solver": "euler", "dt0": 0.005})
    monkeypatch.setenv("CDK_ENKF_CLUSTER", str(cluster))  # members per CTA: 256, 150, 125 (ragged), 200
    monkeypatch.setenv("CDK_ENKF_LIGHT", "0")
    f0 = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], hp)
    monkeypatch.setenv("CDK_ENKF_LIGHT", "1")
    f1 = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], hp)
    assert np.array_equal(np.asarray(f0.marginal_loglik), np.asarray(f1.marginal_loglik))
    for fld in FIELDS:
        assert np.array_equal(np.asarray(getattr(f0, fld)), np.asarray(getattr(f1, fld))), fld


@pytest.mark.parametrize("n,m", [(36, 36), (32, 40), (12, 33)])
def test_kf_maximum_sizes_vs_oracle(n, m):
    """The largest KF the 227 KB of a CTA hold (n = m = 36; cdk.h) and emission dimensions above 32 (two rows per lane in the single-warp Cholesky, the
    chunked triangular solves and the warp log-density; m > n exercises the scratch sizing) -- generic kernel, filter and
    type-1 smoother against the NumPy oracle."""
    cd = api()
    N, K = 3, 12
    rng = np.random.default_rng(n * 100 + m)
    g, _, t, _ = _c2_case(N, K, seed=n + m, n=n, m=min(m, n))
    H = rng.standard_normal((m, n)) / np.sqrt(n)
    A = rng.standard_normal((m, m)) / np.sqrt(m)
    g.update(H=H, d=0.1 * rng.standard_normal(m), R=0.2 * np.eye(m) + 0.1 * A @ A.T)
    y = rng.standard_normal((N, K, m))
    po = o.LinearParams(m0=g["m0"], P0=g["P0"], F=g["F"], L=g["L"], Qc=g["Qc"], H=g["H"], R=g["R"], b=g["b"], d=g["d"])
    hp = cd.KFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    f = cd.cdlgssm_filter(linear_params_api(g), y, t[..., None], hp)
    r = o.cdlgssm_filter(po, y, t, settings=o.SolverSettings("rk4", 0.01))
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record(f"kf_max_n{n}_m{m}:marginal_loglik", e)
    assert e < TOL
    check_moments(f, r, f"kf_max_n{n}_m{m}")
    s = cd.cdlgssm_smoother(linear_params_api(g), y, t[..., None], hp, smoother_type="cd_smoother_1")
    rs = o.cdlgssm_smoother(po, y, t, settings=o.SolverSettings("rk4", 0.01), smoother_type=1)
    for fld in ("smoothed_means", "smoothed_covariances"):
        assert scaled_err(getattr(s, fld), rs[fld]) < 1e-8, fld


def test_oversized_request_fails_loudly():
    """n = m = 64 is inside the ABI bounds but its working set exceeds one CTA's shared memory: CDK_E_SIZE with a message."""
    from cd_dynamax_b200._lib import CdkError
    cd = api()
    g, _, t, y = _c2_case(2, 4, n=64, m=64)
    with pytest.raises(CdkError, match="227 KB"):
        cd.cdlgssm_filter(linear_params_api(g), y, t[..., None], cd.KFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01}))


def test_ukf_and_enkf_wide_emission_vs_oracle():
    """m = 36 > 32 on the nonlinear kernels: closed-form UKF (Lorenz-96 n = 40) and EnKF (cluster path, tensor-core gain)."""
    cd = api()
    n, m, N, K = 40, 36, 2, 8
    g, po, t, y = _l96_case(N, K, seed=21, n=n, m=20)
    rng = np.random.default_rng(7)
    H = rng.standard_normal((m, n)) / np.sqrt(n)
    g.update(H=H, d=np.zeros(m), R=0.5 * np.eye(m))
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=o.Lorenz96Drift(g["theta"][0]), L=g["L"], Qc=g["Qc"], H=H, R=g["R"], d=g["d"])
    y = (H @ g["m0"])[None, None, :] + rng.standard_normal((N, K, m))
    p = nonlinear_params_api(g)
    f = cd.cdnlgssm_filter(p, y, t[..., None], cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.005}))
    r = o.unscented_kalman_filter(po, y, t, settings=o.SolverSettings("rk4", 0.005))
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, "ukf_wide_m36")
    E = 128
    hp = cd.EnKFHyperParams(N_particles=E, key=99, diffeqsolve_settings={"solver": "euler", "dt0": 0.005})
    fe = cd.cdnlgssm_filter(p, y, t[..., None], hp)
    re = o.ensemble_kalman_filter(po, y, t, E=E, seed=99, settings=o.SolverSettings("euler", 0.005))
    assert max_rel_err(fe.marginal_loglik, re["marginal_loglik"]) < 1e-8
    for fld in ("filtered_means", "filtered_covariances", "predicted_means", "predicted_covariances"):
        assert scaled_err(getattr(fe, fld), re[fld]) < 1e-8, fld


def test_c4_full_size_sharding_invariance_and_oracle_sample():
    """BASELINE config 4 at FULL size (UKF, Lorenz-96 n = 40, m = 20, N = 8,192, K = 500; log-likelihood + filtered means --
    all four moment arrays would be 105 GB): shards reproduce the batch bit for bit; three trajectories against the NumPy
    oracle's literal sigma points over all 500 steps (t = 10, ~17 Lyapunov times of the unobserved system: the filter's
    contraction keeps the two roundings together)."""
    import torch
    cd = api()
    N, K = 8192, 500
    g, po, t, y = _l96_case(N=N, K=K, seed=4)
    dev = torch.device("cuda", 0)
    td, yd = torch.as_tensor(t, device=dev), torch.as_tensor(y, device=dev)
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.005})
    p = nonlinear_params_api(g)
    full = cd.cdnlgssm_filter(p, yd, td[..., None], hp, output_fields=["filtered_means", "marginal_loglik"])  # cumulative ll
    assert bool(torch.isfinite(full.marginal_loglik).all()) and bool(torch.isfinite(full.filtered_means).all())
    for lo, hi in ((0, 1000), (5000, 8192)):
        part = cd.cdnlgssm_filter(p, yd[lo:hi], td[lo:hi, :, None], hp, output_fields=["filtered_means", "marginal_loglik"])
        assert torch.equal(part.marginal_loglik, full.marginal_loglik[lo:hi])
        assert torch.equal(part.filtered_means, full.filtered_means[lo:hi])
    sel = np.array([0, 4097, N - 1])
    r = o.unscented_kalman_filter(po, y[sel], t[sel], settings=o.SolverSettings("rk4", 0.005))
    llc = full.marginal_loglik[sel].cpu().numpy()
    fm = full.filtered_means[sel].cpu().numpy()
    # the first 100 steps at the parity gate; the whole chaotic run (two roundings of the same algorithm drift apart at the
    # system's Lyapunov rate between the corrections of the filter) at 1e-6 of the log-likelihood / 1e-3 of the mean scale
    k0 = 100
    ref_cum = r["marginal_loglik_cumulative"]
    e100 = scaled_err(fm[:, :k0], r["filtered_means"][:, :k0])
    eall = scaled_err(fm, r["filtered_means"])
    ell = max_rel_err(llc[:, -1], r["marginal_loglik"])
    record("c4_full_size_sample:filtered_means_first100:scaled", e100)
    record("c4_full_size_sample:filtered_means_all500:scaled", eall)
    record("c4_full_size_sample:marginal_loglik_all500", ell)
    assert e100 < 1e-8 and eall < 1e-3 and ell < 1e-6, (e100, eall, ell)
    assert max_rel_err(llc[:, k0 - 1], ref_cum[:, k0 - 1]) < TOL


def test_c5_full_size_subset_invariance_and_oracle_sample():
    """BASELINE config 5 at FULL size (EnKF, n = 40, m = 20, E = 1,024, N = 1,024, K = 500): a subset of the batch reproduces
    its rows bit for bit (the Philox counters are per trajectory index); the first 60 steps of two trajectories against the
    oracle on the shared stream (the filter is causal)."""
    import torch
    cd = api()
    N, K = 1024, 500
    g, po, t, y = _l96_case(N=N, K=K, seed=5)
    dev = torch.device("cuda", 0)
    td, yd = torch.as_tensor(t, device=dev), torch.as_tensor(y, device=dev)
    hp = cd.EnKFHyperParams(N_particles=1024, key=1234, diffeqsolve_settings={"solver": "euler", "dt0": 0.005})
    p = nonlinear_params_api(g)
    full = cd.cdnlgssm_filter(p, yd, td[..., None], hp, output_fields=["filtered_means"])
    assert bool(torch.isfinite(full.marginal_loglik).all())
    part = cd.cdnlgssm_filter(p, yd[:96], td[:96, :, None], hp, output_fields=["filtered_means"])
    assert torch.equal(part.marginal_loglik, full.marginal_loglik[:96])
    assert torch.equal(part.filtered_means, full.filtered_means[:96])
    Ks = 60
    r = o.ensemble_kalman_filter(po, y[:2, :Ks], t[:2, :Ks], E=1024, seed=1234, settings=o.SolverSettings("euler", 0.005))
    em = scaled_err(full.filtered_means[:2, :Ks].cpu().numpy(), r["filtered_means"])
    record("c5_full_size_sample:filtered_means:scaled", em)
    assert em < 1e-8, em


def test_c2_full_size_sharding_invariance_and_oracle_sample():
    """BASELINE config 2 at FULL size (KF n = 16, m = 4, N = 262,144, K = 500, log-likelihood only: 5 GB of inputs resident):
    a slice of the batch reproduces its rows bit for bit; 64 trajectories against the C oracle."""
    import torch
    from oracle import cpu_baseline as cb
    cd = api()
    N, K = 262144, 500
    g, _, t, y = _c2_case(N, K, seed=22)
    dev = torch.device("cuda", 0)
    td, yd = torch.as_tensor(t, device=dev), torch.as_tensor(y, device=dev)
    from cd_dynamax_b200 import _lib as L
    from cd_dynamax_b200.continuous_discrete_linear_gaussian_ssm.inference import _filter_device
    hp = cd.KFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    p = linear_params_api(g)
    # the reference's linear filter has no output_fields: the moments of this batch would be 570 GB, so the test asks the
    # shim's device-level driver for the log-likelihoods only (what marginal_log_prob does)
    ll = lambda yy, tt: _filter_device(p, yy, tt[..., None], hp, None, (L.OUT_LL,))[0][L.OUT_LL]
    full = ll(yd, td)
    assert bool(torch.isfinite(full).all())
    lo, hi = 100000, 108192
    assert torch.equal(ll(yd[lo:hi], td[lo:hi]), full[lo:hi])
    sel = np.r_[0:32, N - 32:N]
    r = cb.filter_c("kf", y[sel], t[sel], g["m0"], g["P0"], g["F"], g["L"], g["Qc"], g["H"], g["d"], g["R"], bias=g["b"],
                    solver="rk4", dt0=0.01)
    e = max_rel_err(full[sel].cpu().numpy(), r["marginal_loglik"])
    record("c2_full_size_sample:marginal_loglik", e)
    assert e < TOL


# ---- fp32 entry points: one stated bound each (oracle in fp64 on the fp32-rounded inputs, stepping on fp32 times with the
# ---- fp32 tolerance -- the substeps the fp32 kernels take -- so the comparison isolates the arithmetic precision).  The reference's own fp32 "match" ladder is 1e-5 .. 1e-4 on well-conditioned linear models
# ---- (test_utils.py:160-180); chaotic drifts amplify rounding by e^{lambda t}.
def _f32(*arrs):
    return [np.asarray(a, np.float32) for a in arrs]


def _as64(a):
    return np.asarray(a, np.float32).astype(np.float64)


def test_fp32_kf_filter_and_smoothers_bound():
    """cdk_kf_filter_f32 / cdk_kf_smooth_f32 (generic kernels; the DMMA warp kernels are fp64-only): n = 8, m = 3, K = 100.
    Bound: 2e-4 relative on the log-likelihood, 2e-4 scaled on the moments."""
    cd = api()
    N, K = 9, 100
    g, po, t, y = _c2_case(N, K, seed=8, n=8, m=3)
    y32, t32 = _f32(y, t)
    hp = cd.KFHyperParams(dt_final=0.01, diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    g32 = {k: (v if v is None else np.asarray(v, np.float32)) for k, v in g.items()}
    r = o.cdlgssm_smoother(po, _as64(y32), _as64(t32), dt_final=float(np.float32(0.01)),
                           settings=o.SolverSettings("rk4", float(np.float32(0.01)), time_dtype=np.float32))
    for stype in ("cd_smoother_1", "cd_smoother_2"):
        s = cd.cdlgssm_smoother(linear_params_api(g32), y32, t32[..., None], hp, smoother_type=stype)
        assert s.smoothed_means.dtype == np.float32
        e = max_rel_err(s.marginal_loglik, r["marginal_loglik"])
        record(f"fp32_kf_{stype}:marginal_loglik", e)
        assert e < 2e-4
        r2 = r if stype == "cd_smoother_1" else o.cdlgssm_smoother(
            po, _as64(y32), _as64(t32), dt_final=float(np.float32(0.01)),
            settings=o.SolverSettings("rk4", float(np.float32(0.01)), time_dtype=np.float32), smoother_type=2)
        for fld in ("filtered_means", "filtered_covariances", "smoothed_means", "smoothed_covariances"):
            e = scaled_err(getattr(s, fld), r2[fld])
            record(f"fp32_kf_{stype}:{fld}", e)
            assert e < 2e-4, (stype, fld, e)


def test_fp32_ukf_bound():
    """cdk_ukf_filter_f32: Lorenz-63, K = 100.  Bound: 5e-4 relative on the log-likelihood, 5e-3 scaled on the moments."""
    cd = api()
    N, K = 16, 100
    t, y = c3_problem(N, K, seed=9)
    y32, t32 = _f32(y, t)
    g = dict(L63, m0=np.array([1.0, 1.0, 20.0]), P0=2 * np.eye(3))
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    f = cd.cdnlgssm_filter(nonlinear_params_api(g), y32, t32[..., None], hp)
    assert f.filtered_means.dtype == np.float32
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=o.Lorenz63Drift(*g["theta"]), L=g["L"], Qc=g["Qc"], H=g["H"],
                           R=g["R"], d=g["d"])
    r = o.unscented_kalman_filter(po, _as64(y32), _as64(t32), settings=o.SolverSettings("rk4", float(np.float32(0.0025)), time_dtype=np.float32))
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record("fp32_ukf:marginal_loglik", e)
    assert e < 5e-4
    for fld in FIELDS:
        e = scaled_err(getattr(f, fld), r[fld])
        record(f"fp32_ukf:{fld}", e)
        assert e < 5e-3, (fld, e)


@pytest.mark.parametrize("algo", ["ekf", "ukf"])
@pytest.mark.parametrize("solver,dt0", [("rk4", 0.005), ("dopri5", 0.01)])
def test_fp32_l96_register_ode_bound(algo, solver, dt0):
    """The fp32 instantiations of the register-resident Lorenz-96 moment ODE (chain tableau and Dopri5) at n = 40, short
    horizon (K = 8).  Bound: 2e-3 relative on the log-likelihood, 5e-3 scaled on the moments."""
    cd = api()
    g, po, t, y = _l96_case(N=3, K=8, seed=71)
    y32, t32 = _f32(y, t)
    st = {"solver": solver, "dt0": dt0}
    so = o.SolverSettings(solver, float(np.float32(dt0)), time_dtype=np.float32)
    if algo == "ekf":
        f = cd.cdnlgssm_filter(nonlinear_params_api(g), y32, t32[..., None], cd.EKFHyperParams(diffeqsolve_settings=st))
        r = o.extended_kalman_filter(po, _as64(y32), _as64(t32), settings=so)
    else:
        f = cd.cdnlgssm_filter(nonlinear_params_api(g), y32, t32[..., None], cd.UKFHyperParams(diffeqsolve_settings=st))
        r = o.unscented_kalman_filter(po, _as64(y32), _as64(t32), settings=so)
    assert f.filtered_means.dtype == np.float32
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < 2e-3
    for fld in FIELDS:
        assert scaled_err(getattr(f, fld), r[fld]) < 5e-3, fld


def test_fp32_enkf_bound():
    """cdk_enkf_filter_f32: linear drift (no chaotic amplification of the fp32 normal deviates), E = 256, K = 40, same
    Philox counters as the fp64 oracle.  Bound: 1e-3 relative on the log-likelihood, 2e-3 scaled on the moments."""
    from tests.test_gpu_parity import _enkf_case
    cd = api()
    g, t, y, dt0 = _enkf_case("lin", 4, 40, 256, seed=12)
    y32, t32 = _f32(y, t)
    hp = cd.EnKFHyperParams(N_particles=256, key=77, diffeqsolve_settings={"solver": "euler", "dt0": dt0})
    f = cd.cdnlgssm_filter(nonlinear_params_api(g), y32, t32[..., None], hp)
    assert f.filtered_means.dtype == np.float32
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=o.LinearDrift(g["theta"][:16].reshape(4, 4), g["theta"][16:]),
                           L=g["L"], Qc=g["Qc"], H=g["H"], R=g["R"], d=g["d"])
    r = o.ensemble_kalman_filter(po, _as64(y32), _as64(t32), E=256, seed=77,
                                 settings=o.SolverSettings("euler", float(np.float32(dt0)), time_dtype=np.float32))
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record("fp32_enkf:marginal_loglik", e)
    assert e < 1e-3
    for fld in FIELDS:
        e = scaled_err(getattr(f, fld), r[fld])
        record(f"fp32_enkf:{fld}", e)
        assert e < 2e-3, (fld, e)


def test_fp32_enkf_l96_light_mapping(monkeypatch):
    """cdk_enkf_filter_f32 on Lorenz-96 n = 40 (the fp32 instantiation of the two-threads-per-member mapping): against the fp32
    register mapping to fp32 rounding (separate template instantiations may contract a * b + c differently in fp32), and, over
    a short horizon (K = 6: chaos amplifies fp32 rounding by e^{lambda t}), against the fp64 oracle."""
    cd = api()
    g, po, t, y = _l96_case(N=2, K=6, seed=52)
    y32, t32 = _f32(y, t)
    hp = cd.EnKFHyperParams(N_particles=512, key=5, diffeqsolve_settings={"solver": "euler", "dt0": 0.005})
    monkeypatch.setenv("CDK_ENKF_CLUSTER", "2")
    monkeypatch.setenv("CDK_ENKF_LIGHT", "0")
    f0 = cd.cdnlgssm_filter(nonlinear_params_api(g), y32, t32[..., None], hp)
    monkeypatch.setenv("CDK_ENKF_LIGHT", "1")
    f1 = cd.cdnlgssm_filter(nonlinear_params_api(g), y32, t32[..., None], hp)
    assert f1.filtered_means.dtype == np.float32
    for fld in FIELDS:
        assert scaled_err(getattr(f1, fld), np.asarray(getattr(f0, fld), np.float64)) < 2e-4, fld
    r = o.ensemble_kalman_filter(po, _as64(y32), _as64(t32), E=512, seed=5, settings=o.SolverSettings("euler", float(np.float32(0.005)), time_dtype=np.float32))
    assert max_rel_err(f1.marginal_loglik, r["marginal_loglik"]) < 5e-3
    for fld in FIELDS:
        assert scaled_err(getattr(f1, fld), r[fld]) < 5e-3, fld


def test_fp32_eks_bound():
    """cdk_ekf_smooth_f32 (register kernel, Lorenz-63), K = 100.  Bound: 5e-3 scaled on the smoothed moments."""
    cd = api()
    N, K = 40, 100
    t, y = c3_problem(N, K, seed=10)
    y32, t32 = _f32(y, t)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    s = cd.cdnlgssm_smoother(nonlinear_params_api(L63), y32, t32[..., None], hp)
    assert s.smoothed_means.dtype == np.float32
    po = o.NonlinearParams(m0=L63["m0"], P0=L63["P0"], drift=o.Lorenz63Drift(*L63["theta"]), L=L63["L"], Qc=L63["Qc"],
                           H=L63["H"], R=L63["R"], d=L63["d"])
    r = o.extended_kalman_smoother(po, _as64(y32), _as64(t32), settings=o.SolverSettings("rk4", float(np.float32(0.0025)), time_dtype=np.float32))
    for fld in ("smoothed_means", "smoothed_covariances"):
        e = scaled_err(getattr(s, fld), r[fld])
        record(f"fp32_eks:{fld}", e)
        assert e < 5e-3, (fld, e)


# ---- the XLA custom-call adaptor and the NCCL hook of include/cdk.h, executed ------------------------------------------
def test_xla_custom_call_adaptor_matches_direct_entry_point():
    """cdk_xla_custom_call(stream, buffers, opaque, opaque_len) -- the legacy XLA GPU custom-call signature jax 0.4.13
    registers (INTEGRATION.md) -- called through ctypes with a packed cdk_xla_opaque and torch device buffers: inputs
    then outputs, absent slots passed as dummies and flagged in desc.reserved[0] / [1].  Same bits as the direct call."""
    import torch
    from cd_dynamax_b200 import _lib as L
    cd = api()
    lib = L.lib()
    N, K = 300, 40
    t, y = c3_problem(N, K, seed=3)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    ref = cd.cdnlgssm_filter(nonlinear_params_api(L63), y, t[..., None], hp)
    dev = torch.device("cuda", 0)
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=dev)
    ins = {L.IN_Y: T(y), L.IN_T: T(t), L.IN_M0: T(L63["m0"]), L.IN_P0: T(L63["P0"]), L.IN_F: T(L63["theta"]),
           L.IN_L: T(L63["L"]), L.IN_QC: T(L63["Qc"]), L.IN_H: T(L63["H"]), L.IN_D: T(L63["d"]), L.IN_R: T(L63["R"])}
    outs = {L.OUT_LL: torch.empty(N, dtype=torch.float64, device=dev),
            L.OUT_FM: torch.empty(N, K, 3, dtype=torch.float64, device=dev),
            L.OUT_PP: torch.empty(N, K, 3, 3, dtype=torch.float64, device=dev),
            L.OUT_STATUS: torch.zeros(N, dtype=torch.int32, device=dev)}
    dummy = torch.zeros(1, dtype=torch.float64, device=dev)  # XLA passes a (zero-size) buffer for every operand
    d = L.new_desc()
    d.N, d.K, d.n, d.m = N, K, 3, 1
    d.solver, d.dt0, d.drift_id, d.n_theta, d.state_order = L.SOLVERS["rk4"], 0.0025, L.DRIFT_LORENZ63, 3, 2
    d.batched_mask = (1 << L.IN_Y) | (1 << L.IN_T)
    absent_in = sum(1 << s for s in range(L.NUM_IN) if s not in ins)
    absent_out = sum(1 << s for s in range(L.NUM_OUT) if s not in outs)
    d.reserved[0], d.reserved[1] = absent_in, absent_out

    class Opaque(ctypes.Structure):
        _fields_ = [("entry_point", ctypes.c_char * 32), ("desc", L.CdkDesc)]

    op = Opaque()
    op.entry_point = b"cdk_ekf_filter_f64"
    op.desc = d
    bufs = (ctypes.c_void_p * (L.NUM_IN + L.NUM_OUT))()
    for s in range(L.NUM_IN):
        bufs[s] = ins[s].data_ptr() if s in ins else dummy.data_ptr()
    for s in range(L.NUM_OUT):
        bufs[L.NUM_IN + s] = outs[s].data_ptr() if s in outs else dummy.data_ptr()
    blob = ctypes.string_at(ctypes.byref(op), ctypes.sizeof(op))
    stream = torch.cuda.current_stream(dev).cuda_stream
    lib.cdk_xla_custom_call(ctypes.c_void_p(stream), bufs, blob, len(blob))
    torch.cuda.synchronize()
    assert np.array_equal(outs[L.OUT_LL].cpu().numpy(), ref.marginal_loglik)
    assert np.array_equal(outs[L.OUT_FM].cpu().numpy(), ref.filtered_means)
    assert np.array_equal(outs[L.OUT_PP].cpu().numpy(), ref.predicted_covariances)
    assert (outs[L.OUT_STATUS].cpu().numpy() == 0).all()
    assert lib.cdk_xla_last_rc() == 0
    # status-returning signature, same buffers: a NULL status is allowed; an invalid descriptor is reported, nothing runs
    outs[L.OUT_LL].zero_()
    lib.cdk_xla_custom_call_status(ctypes.c_void_p(stream), bufs, blob, len(blob), None)
    torch.cuda.synchronize()
    assert np.array_equal(outs[L.OUT_LL].cpu().numpy(), ref.marginal_loglik)
    op.desc.dt0 = -1.0
    blob = ctypes.string_at(ctypes.byref(op), ctypes.sizeof(op))
    lib.cdk_xla_custom_call_status(ctypes.c_void_p(stream), bufs, blob, len(blob), None)
    assert lib.cdk_xla_last_rc() == -2 and b"dt0" in lib.cdk_last_error()


def test_ll_allreduce_with_a_raw_nccl_communicator():
    """cdk_ll_allreduce(ncclComm_t, double*, stream) with a communicator created outside torch.distributed (ctypes on the
    libnccl that torch bundles): one rank here (the multi-rank run is bench.py --gpus N, which cross-checks it against
    torch.distributed's all-reduce on every rank)."""
    import torch
    from cd_dynamax_b200 import _engine as E
    from cd_dynamax_b200 import parallel
    dev = torch.device("cuda", 0)
    comm = parallel.RawNcclComm(rank=0, world_size=1, device=dev)
    ll = torch.arange(1000, dtype=torch.float64, device=dev) * -0.37
    s = E.ll_sum(ll)
    before = s.item()
    parallel.allreduce_loglik_nccl(s, comm)
    torch.cuda.synchronize()
    assert s.item() == before == float(np.sum(np.arange(1000) * -0.37)) or abs(s.item() - before) == 0.0
    comm.destroy()


@pytest.mark.parametrize("sigma_points", [False, True])
def test_ukf_l63_k1000_long_run_vs_oracle(sigma_points, monkeypatch):
    """A LONG unscented run (K = 1,000, config 3's data) through the shared-memory UKF kernels: the UKF never symmetrises its
    covariance, so anything that amplified the rounding asymmetry of the update would show here (it did, on the Lorenz-96
    register path, after ~240 steps: DESIGN 4.2)."""
    cd = api()
    monkeypatch.setenv("CDK_UKF_SIGMA_POINTS", "1" if sigma_points else "0")
    N, K = 6, 1000
    t, y = c3_problem(N, K, seed=12)
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    f = cd.cdnlgssm_filter(nonlinear_params_api(L63), y, t[..., None], hp)
    po = o.NonlinearParams(m0=L63["m0"], P0=L63["P0"], drift=o.Lorenz63Drift(*L63["theta"]), L=L63["L"], Qc=L63["Qc"],
                           H=L63["H"], R=L63["R"], d=L63["d"])
    r = o.unscented_kalman_filter(po, y, t, settings=o.SolverSettings("rk4", 0.0025))
    assert np.isfinite(r["marginal_loglik"]).all()
    P = np.asarray(f.filtered_covariances)
    assert np.abs(P - np.swapaxes(P, -1, -2)).max() < 1e-12 * np.abs(P).max()
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record(f"ukf_l63_k1000_{'sigma' if sigma_points else 'closed'}:marginal_loglik", e)
    assert e < 1e-8
    for fld in FIELDS:
        assert scaled_err(getattr(f, fld), r[fld]) < 1e-6, fld


@pytest.mark.parametrize("algo,solver,dt0", [("ekf", "rk4", 0.005), ("ekf", "dopri5", 0.01), ("ukf", "dopri5", 0.01), ("ukf", "heun", 0.005)])
def test_l96_n40_long_runs_vs_oracle(algo, solver, dt0):
    """K = 300 observation steps on Lorenz-96 n = 40 through the register-resident ODE variants (chain tableau, Dopri5; EKF,
    UKF): finite and symmetric to the end, the first 100 steps at the parity gate, the whole run at 1e-3 of the scale (two
    roundings of a chaotic filter separate at the Lyapunov rate between corrections)."""
    cd = api()
    g, po, t, y = _l96_case(N=2, K=300, seed=31)
    st = {"solver": solver, "dt0": dt0}
    if algo == "ekf":
        f = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], cd.EKFHyperParams(diffeqsolve_settings=st))
        r = o.extended_kalman_filter(po, y, t, settings=o.SolverSettings(solver, dt0))
    else:
        f = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], cd.UKFHyperParams(diffeqsolve_settings=st))
        r = o.unscented_kalman_filter(po, y, t, settings=o.SolverSettings(solver, dt0))
    P = np.asarray(f.filtered_covariances)
    assert np.isfinite(P).all() and np.isfinite(np.asarray(f.marginal_loglik)).all()
    assert np.abs(P - np.swapaxes(P, -1, -2)).max() < 1e-12 * np.abs(P).max()
    e100 = scaled_err(np.asarray(f.filtered_means)[:, :100], r["filtered_means"][:, :100])
    eall = scaled_err(f.filtered_means, r["filtered_means"])
    record(f"l96_long_{algo}_{solver}:filtered_means_first100", e100)
    record(f"l96_long_{algo}_{solver}:filtered_means_all300", eall)
    assert e100 < 1e-8 and eall < 1e-3, (e100, eall)
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < 1e-6


def test_c3_eks_k1000_long_run_vs_oracle():
    """Config 3's smoother at full K: filter + EKS backward pass over 1,000 steps (register kernels) against the NumPy oracle."""
    cd = api()
    N, K = 5, 1000
    t, y = c3_problem(N, K, seed=14)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    s = cd.cdnlgssm_smoother(nonlinear_params_api(L63), y, t[..., None], hp)
    po = o.NonlinearParams(m0=L63["m0"], P0=L63["P0"], drift=o.Lorenz63Drift(*L63["theta"]), L=L63["L"], Qc=L63["Qc"],
                           H=L63["H"], R=L63["R"], d=L63["d"])
    rs = o.extended_kalman_smoother(po, y, t, settings=o.SolverSettings("rk4", 0.0025))
    assert np.isfinite(np.asarray(s.smoothed_covariances)).all()
    assert max_rel_err(s.marginal_loglik, rs["marginal_loglik"]) < TOL
    for fld in ("smoothed_means", "smoothed_covariances"):
        e = scaled_err(getattr(s, fld), rs[fld])
        record(f"c3_eks_k1000:{fld}", e)
        assert e < 1e-8, (fld, e)


def test_c5_enkf_heun_full_length_finite_and_causal_sample():
    """EnKF with the reference's default SDE solver (Heun) over config 5's full K = 500 on a few trajectories: finite to the
    end; the first 40 steps against the oracle on the shared stream."""
    cd = api()
    g, po, t, y = _l96_case(N=3, K=500, seed=53)
    hp = cd.EnKFHyperParams(N_particles=1024, key=9, diffeqsolve_settings={"solver": "heun", "dt0": 0.005})
    f = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], hp)
    assert np.isfinite(np.asarray(f.filtered_covariances)).all() and np.isfinite(np.asarray(f.marginal_loglik)).all()
    Ks = 40
    r = o.ensemble_kalman_filter(po, y[:2, :Ks], t[:2, :Ks], E=1024, seed=9, settings=o.SolverSettings("heun", 0.005))
    assert scaled_err(np.asarray(f.filtered_means)[:2, :Ks], r["filtered_means"]) < 1e-8


def test_eks_l96_n40_generic_smoother_vs_oracle():
    """Filter (register ODE, compact layout) + EKS backward pass (generic_smooth_kernel) at n = 40, m = 20."""
    cd = api()
    g, po, t, y = _l96_case(N=2, K=30, seed=33)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.005})
    s = cd.cdnlgssm_smoother(nonlinear_params_api(g), y, t[..., None], hp)
    rs = o.extended_kalman_smoother(po, y, t, settings=o.SolverSettings("rk4", 0.005))
    assert max_rel_err(s.marginal_loglik, rs["marginal_loglik"]) < TOL
    for fld in ("smoothed_means", "smoothed_covariances"):
        e = scaled_err(getattr(s, fld), rs[fld])
        record(f"eks_l96_n40:{fld}", e)
        assert e < 1e-8, (fld, e)


def test_kf_generic_n32_long_run_vs_oracle():
    """The shared-memory linear kernel beyond the warp kernel's n <= 16: n = 32, m = 8, K = 300 against the C oracle, both
    smoother types against the NumPy oracle on a shorter slice."""
    from oracle import cpu_baseline as cb
    cd = api()
    N, K = 6, 300
    g, po, t, y = _c2_case(N, K, seed=41, n=32, m=8)
    hp = cd.KFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    f = cd.cdlgssm_filter(linear_params_api(g), y, t[..., None], hp)
    r = cb.filter_c("kf", y, t, g["m0"], g["P0"], g["F"], g["L"], g["Qc"], g["H"], g["d"], g["R"], bias=g["b"], solver="rk4", dt0=0.01)
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record("kf_generic_n32_k300:marginal_loglik", e)
    assert e < TOL
    check_moments(f, r, "kf_generic_n32_k300")
    Ks = 40
    for stype in ("cd_smoother_1", "cd_smoother_2"):
        s = cd.cdlgssm_smoother(linear_params_api(g), y[:2, :Ks], t[:2, :Ks, None], hp, smoother_type=stype)
        rs = o.cdlgssm_smoother(po, y[:2, :Ks], t[:2, :Ks], settings=o.SolverSettings("rk4", 0.01), smoother_type=int(stype[-1]))
        for fld in ("smoothed_means", "smoothed_covariances"):
            assert scaled_err(getattr(s, fld), rs[fld]) < 1e-8, (stype, fld)
