"""GPU: the CUDA path, called through the reference-shaped Python API (-> C ABI), against
 (a) golden vectors produced by the reference's own code (tests/golden/make_golden.py) and
 (b) the NumPy oracle on seeded random inputs.
Tolerance: fp64 rel 1e-9 (north star); smoothed moments 1e-8 on the scaled error (RTS recursion amplifies rounding by
cond(P_pred)); fp32 bounds are stated per test."""
import numpy as np
import pytest

from oracle import cd_oracle as o
from tests.helpers import golden_cases, load_golden, make_drift, max_rel_err, moment_err, record, scaled_err

pytestmark = pytest.mark.gpu
TOL = 1e-9
FIELDS = ["filtered_means", "filtered_covariances", "predicted_means", "predicted_covariances"]


def api():
    import cd_dynamax_b200 as cd
    return cd


def check_moments(post, ref, tag, prefix="", tol=TOL, fields=FIELDS):
    """Filtered / predicted moments against the oracle or a golden case: SURVEY 8(d)'s element-wise gate
    (tests/helpers.gate_err: |a - b| <= max(1e-9 |b|, 1e-12 scale)) AND every mean vector / covariance matrix to 1e-10 of
    its own norm (tests/helpers.moment_norm_err)."""
    for fld in fields:
        e, en = moment_err(post, ref, fld, prefix)
        record(f"{tag}:{fld}:gate", e)
        record(f"{tag}:{fld}:own_norm", en)
        assert e < tol, (tag, fld, e)
        assert en < 0.1 * tol, (tag, fld, en)


def linear_params_api(g):
    cd = api()
    return cd.ParamsCDLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=g["m0"], cov=g["P0"]),
        dynamics=cd.ParamsCDLGSSMDynamics(weights=g["F"], bias=g["b"], input_weights=g["B"],
                                          diffusion_coefficient=g["L"], diffusion_cov=g["Qc"]),
        emissions=cd.ParamsLGSSMEmissions(weights=g["H"], bias=g["d"], input_weights=g["D"], cov=g["R"]))


def drift_api(kind, theta, n):
    cd = api()
    kind = str(kind)
    if kind == "lorenz63":
        return cd.LearnableLorenz63(sigma=theta[0], rho=theta[1], beta=theta[2])
    if kind == "lorenz96":
        return cd.LearnableLorenz96(forcing=theta[0])
    if kind == "linear":
        return cd.LearnableLinear(weights=theta[: n * n].reshape(n, n), bias=theta[n * n:])
    if kind == "quadratic":
        return cd.LearnableQuadratic(a=theta[:n], B=theta[n:n + n * n].reshape(n, n),
                                     C=theta[n + n * n:].reshape(n, n, n))
    raise ValueError(kind)


def nonlinear_params_api(g):
    cd = api()
    n = g["m0"].shape[-1]
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(g["m0"]), cov=cd.LearnableMatrix(g["P0"])),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=drift_api(g["drift"], g["theta"], n),
                                           diffusion_coefficient=cd.LearnableMatrix(g["L"]),
                                           diffusion_cov=cd.LearnableMatrix(g["Qc"])),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=g["H"], bias=g["d"]),
                                             emission_cov=cd.LearnableMatrix(g["R"])))


def settings_api(g):
    return {"solver": str(g["solver"]), "dt0": float(g["dt0"])}


@pytest.mark.parametrize("name", golden_cases("kf_"))
def test_kf_filter_and_smoothers_vs_reference_golden(name):
    cd = api()
    g = load_golden(name)
    p = linear_params_api(g)
    hp = cd.KFHyperParams(dt_final=float(g["dt_final"]), diffeqsolve_settings=settings_api(g))
    u = g.get("u")
    f = cd.cdlgssm_filter(p, g["y"], g["t"][..., None], hp, u)
    assert max_rel_err(f.marginal_loglik, g["filt_marginal_loglik"]) < TOL
    check_moments(f, g, name, prefix="filt_")
    s1 = cd.cdlgssm_smoother(p, g["y"], g["t"][..., None], hp, u, smoother_type="cd_smoother_1")
    for fld in ("smoothed_means", "smoothed_covariances", "smoothed_cross_covariances"):
        assert scaled_err(getattr(s1, fld), g["s1_" + fld]) < 1e-8, fld
    if "s2_smoothed_means" in g:
        s2 = cd.cdlgssm_smoother(p, g["y"], g["t"][..., None], hp, u, smoother_type="cd_smoother_2")
        for fld in ("smoothed_means", "smoothed_covariances"):
            assert scaled_err(getattr(s2, fld), g["s2_" + fld]) < 1e-8, fld
        assert np.isnan(s2.smoothed_cross_covariances).all()
    # single-trajectory call keeps the reference's unbatched shapes
    f0 = cd.cdlgssm_filter(p, g["y"][0], g["t"][0][:, None], hp, None if u is None else u[0])
    assert f0.filtered_means.shape == g["filt_filtered_means"].shape[1:]
    assert np.ndim(f0.marginal_loglik) == 0
    assert scaled_err(f0.filtered_covariances, g["filt_filtered_covariances"][0]) < TOL


@pytest.mark.parametrize("name", golden_cases("ekf_"))
def test_ekf_and_eks_vs_reference_golden(name):
    cd = api()
    g = load_golden(name)
    p = nonlinear_params_api(g)
    hp = cd.EKFHyperParams(dt_final=float(g["dt_final"]), state_order=str(g["state_order"]),
                           cov_rescaling=float(g["cov_rescaling"]), diffeqsolve_settings=settings_api(g))
    f = cd.cdnlgssm_filter(p, g["y"], g["t"][..., None], hp, num_iter=int(g["num_iter"]))
    assert max_rel_err(f.marginal_loglik, g["filt_marginal_loglik"]) < TOL
    check_moments(f, g, name, prefix="filt_")
    c = cd.cdnlgssm_filter(p, g["y"], g["t"][..., None], hp, num_iter=int(g["num_iter"]),
                           output_fields=["marginal_loglik"])
    assert c.filtered_means is None
    assert max_rel_err(c.marginal_loglik, g["filt_marginal_loglik_cumulative"]) < TOL
    if "smooth_smoothed_means" in g:
        s = cd.cdnlgssm_smoother(p, g["y"], g["t"][..., None], hp)
        for fld in ("smoothed_means", "smoothed_covariances"):
            assert scaled_err(getattr(s, fld), g["smooth_" + fld]) < 1e-8, fld


@pytest.mark.parametrize("sigma_points", [False, True])
@pytest.mark.parametrize("name", golden_cases("ukf_"))
def test_ukf_vs_reference_golden(name, sigma_points, monkeypatch):
    """Both UKF kernels against the reference's output: the closed-form unscented predict (default) and the literal
    sigma-point evaluation (CDK_UKF_SIGMA_POINTS=1)."""
    cd = api()
    monkeypatch.setenv("CDK_UKF_SIGMA_POINTS", "1" if sigma_points else "0")
    g = load_golden(name)
    p = nonlinear_params_api(g)
    hp = cd.UKFHyperParams(dt_final=float(g["dt_final"]), diffeqsolve_settings=settings_api(g))
    f = cd.cdnlgssm_filter(p, g["y"], g["t"][..., None], hp)
    assert max_rel_err(f.marginal_loglik, g["filt_marginal_loglik"]) < TOL
    check_moments(f, g, name + ("_sigma" if sigma_points else "_closed"), prefix="filt_")


def _tag():
    import os
    return os.environ.get("PYTEST_CURRENT_TEST", "?").split("::")[-1].split(" ")[0]


def c3_problem(N, K, seed=1237, dtype=np.float64):
    """BASELINE config 3 at reduced N, K: Lorenz-63, observe x, R = 1, Qc = I, P0 = 5 I, gaps 0.01*U(0.5,1.5)."""
    rng = np.random.default_rng(seed)
    gaps = 0.01 * rng.uniform(0.5, 1.5, size=(N, K))
    gaps[:, 0] = 0.0
    t = np.cumsum(gaps, axis=1)
    y = 8.0 * rng.standard_normal((N, K, 1))
    return t.astype(dtype), y.astype(dtype)


@pytest.mark.parametrize("solver,dt0", [("rk4", 0.0025), ("dopri5", 0.01), ("euler", 0.002), ("heun", 0.005)])
def test_ekf_l63_fast_path_vs_oracle(solver, dt0):
    cd = api()
    N, K = 257, 120  # ragged: not a multiple of the CTA size
    t, y = c3_problem(N, K)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": solver, "dt0": dt0})
    f = cd.cdnlgssm_filter(p, y, t[..., None], hp)
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift("lorenz63", g["theta"], 3), L=g["L"], Qc=g["Qc"],
                           H=g["H"], R=g["R"], d=g["d"])
    r = o.extended_kalman_filter(po, y, t, settings=o.SolverSettings(solver, dt0))
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, _tag())


@pytest.mark.parametrize("fields", [None, [], ["filtered_means", "marginal_loglik"]])
@pytest.mark.parametrize("wres,sms,N,K,dtype", [(3, 2, 437, 260, np.float64), (2, 3, 1000, 206, np.float64), (12, 1, 600, 300, np.float64),
                                               (4, 2, 500, 220, np.float32)])
def test_ekf_l63_time_sliced_launch_is_bit_identical(wres, sms, N, K, dtype, fields, monkeypatch):
    """The time-sliced launch of the Lorenz-63 kernel (groups of 32 trajectories handed from warp to warp between
    K-segments of 50 steps through shared memory; taken by default above one balanced wave, forced here on a pretended
    2-3 SM GPU) must reproduce the one-warp-per-group launch BIT FOR BIT -- same arithmetic, different schedule -- for every
    output, ragged last groups and a last segment shorter than 50 steps included; and both match the oracle."""
    cd = api()
    t, y = c3_problem(N, K, seed=77, dtype=dtype)  # fp32: the cooperative-copy flush instead of the TMA stores
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    monkeypatch.setenv("CDK_LW_SLICE", "0")
    f0 = cd.cdnlgssm_filter(p, y, t[..., None], hp, output_fields=fields)
    monkeypatch.setenv("CDK_LW_SLICE", str(wres))
    monkeypatch.setenv("CDK_LW_SLICE_SMS", str(sms))
    f1 = cd.cdnlgssm_filter(p, y, t[..., None], hp, output_fields=fields)
    for fld in ("marginal_loglik",) + tuple(FIELDS):
        a, b = getattr(f0, fld), getattr(f1, fld)
        assert (a is None) == (b is None), fld
        if a is not None:
            a, b = np.asarray(a), np.asarray(b)
            if dtype == np.float64:
                assert np.array_equal(a, b), fld
            else:
                # the sliced launch is its own template instantiation (12 warps, 170 registers): in fp32 the compiler contracts
                # a few plain a * b + c expressions differently there, so agreement is to fp32 rounding, not to the bit
                assert np.abs(a - b).max() <= 2e-5 * max(1.0, np.abs(a).max()), (fld, np.abs(a - b).max())
    if fields is None and dtype == np.float64:
        po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift("lorenz63", g["theta"], 3), L=g["L"], Qc=g["Qc"],
                               H=g["H"], R=g["R"], d=g["d"])
        r = o.extended_kalman_filter(po, y[:64], t[:64], settings=o.SolverSettings("rk4", 0.0025))
        assert max_rel_err(f1.marginal_loglik[:64], r["marginal_loglik"]) < TOL


def test_ekf_l63_default_launch_slices_large_batches_identically(monkeypatch):
    """N = 40,007 x K = 200 is more than one balanced wave of a B200 (1,251 groups > 148 SMs x 8 warps), so the DEFAULT launch
    is the time-sliced one on the real SM count; it must equal the unsliced launch bit for bit (all four moment arrays)."""
    cd = api()
    N, K = 40007, 200
    t, y = c3_problem(N, K, seed=5)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    f1 = cd.cdnlgssm_filter(p, y, t[..., None], hp)
    monkeypatch.setenv("CDK_LW_SLICE", "0")
    f0 = cd.cdnlgssm_filter(p, y, t[..., None], hp)
    assert np.isfinite(np.asarray(f1.marginal_loglik)).all()
    for fld in ("marginal_loglik",) + tuple(FIELDS):
        assert np.array_equal(np.asarray(getattr(f0, fld)), np.asarray(getattr(f1, fld))), fld


@pytest.mark.parametrize("N,K", [(1, 1), (3, 7), (225, 33), (500, 64)])
def test_ekf_l63_fast_path_ragged_shapes(N, K):
    """Odd / tiny K and N around the 224-slot CTA size: the TMA store path needs even K, the cooperative flush covers
    the rest; both must give the oracle's numbers."""
    cd = api()
    t, y = c3_problem(N, K, seed=7 + N + K)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    f = cd.cdnlgssm_filter(p, y, t[..., None], hp)
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift("lorenz63", g["theta"], 3), L=g["L"], Qc=g["Qc"],
                           H=g["H"], R=g["R"], d=g["d"])
    r = o.extended_kalman_filter(po, y, t, settings=o.SolverSettings("rk4", 0.0025))
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, _tag())
    # a subset of outputs (NULL output pointers) must not change the others
    f2 = cd.cdnlgssm_filter(p, y, t[..., None], hp, output_fields=["predicted_covariances"])
    assert f2.filtered_means is None and np.array_equal(f2.predicted_covariances, f.predicted_covariances)


def test_ekf_l63_fp32_variant_bound():
    """fp32 variant vs the fp64 oracle: stated bound 2e-3 on the scaled error of the moments and 2e-4 relative on the
    log-likelihood over K = 200 steps (the reference's own fp32 'match' ladder tops out at 1e-4, test_utils.py:160-180;
    the Lorenz-63 tangent dynamics amplify rounding by ~e^{0.9 t})."""
    cd = api()
    N, K = 128, 200
    t, y = c3_problem(N, K)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    f32 = cd.cdnlgssm_filter(p, y.astype(np.float32), t.astype(np.float32)[..., None], hp)
    assert f32.filtered_means.dtype == np.float32
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift("lorenz63", g["theta"], 3), L=g["L"], Qc=g["Qc"],
                           H=g["H"], R=g["R"], d=g["d"])
    # oracle in fp64 on the SAME (fp32-rounded) times, stepping in fp32 (fp32 times and tolerance: the kernel's substeps),
    # so the comparison isolates arithmetic precision
    r = o.extended_kalman_filter(po, y.astype(np.float32), t.astype(np.float32).astype(np.float64),
                                 settings=o.SolverSettings("rk4", float(np.float32(0.0025)), time_dtype=np.float32))
    assert max_rel_err(f32.marginal_loglik, r["marginal_loglik"]) < 2e-4
    for fld in FIELDS:
        assert scaled_err(getattr(f32, fld), r[fld]) < 2e-3, fld


def test_batched_parameters_and_shared_data():
    """vmap over parameter samples with shared data (cdlgssm_learnParams_oscillator notebook idiom, SURVEY 2.1)."""
    cd = api()
    N, K = 33, 40
    t, y = c3_problem(1, K)
    rng = np.random.default_rng(5)
    sig, rho, beta = 10 + rng.standard_normal(N), 28 + rng.standard_normal(N), 8 / 3 + 0.1 * rng.standard_normal(N)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1),
             d=np.zeros(1))
    p = cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(g["m0"]), cov=cd.LearnableMatrix(g["P0"])),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableLorenz63(sigma=sig, rho=rho, beta=beta),
                                           diffusion_coefficient=cd.LearnableMatrix(g["L"]),
                                           diffusion_cov=cd.LearnableMatrix(g["Qc"])),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=g["H"], bias=g["d"]),
                                             emission_cov=cd.LearnableMatrix(g["R"])))
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    Y, T = np.repeat(y, N, axis=0), np.repeat(t, N, axis=0)
    f = cd.cdnlgssm_filter(p, Y, T[..., None], hp)
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=o.Lorenz63Drift(sig, rho, beta), L=g["L"], Qc=g["Qc"],
                           H=g["H"], R=g["R"], d=g["d"])
    r = o.extended_kalman_filter(po, Y, T, settings=o.SolverSettings("rk4", 0.0025))
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    assert scaled_err(f.predicted_covariances, r["predicted_covariances"]) < TOL


def test_nonfinite_and_max_steps_status(monkeypatch):
    """Numerical failure is not an error at the C ABI: NaN outputs + status (SURVEY 8b 'Errors').  The Python shim turns
    status 2 into an exception for host callers, as diffrax does when max_steps is reached."""
    import torch
    from cd_dynamax_b200 import _engine as E
    from cd_dynamax_b200 import _lib as L
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm._common import run_filter
    cd = api()
    t0, y0 = c3_problem(4, 6)
    with pytest.raises(E.MaxStepsReached):
        cd.cdnlgssm_filter(nonlinear_params_api(dict(
            m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]), L=np.eye(3),
            Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))), y0, t0[..., None],
            cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025, "max_steps": 2}))
    # device-resident callers stay asynchronous: no exception, the status tensor is there to inspect
    fdev = cd.cdnlgssm_filter(nonlinear_params_api(dict(
        m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]), L=np.eye(3),
        Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))), torch.as_tensor(y0).cuda(),
        torch.as_tensor(t0).cuda()[..., None],
        cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025, "max_steps": 2}))
    assert fdev.marginal_loglik.is_cuda and (E.last_status().cpu().numpy() == 2).all()
    monkeypatch.setattr(E, "RAISE_ON_MAX_STEPS", False)
    N, K = 8, 10
    t, y = c3_problem(N, K)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    fields = dict(dt_final=1e-10, state_order=2, num_iter=1, cov_rescaling=1.0)
    # max_steps = 2 < 3..6 substeps per gap -> status 2, NaN moments (diffrax raises; we flag)
    post, out, _ = run_filter("cdk_ekf_filter", p, y, t[..., None], None, None, fields,
                              diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025, "max_steps": 2})
    assert (out[L.OUT_STATUS].cpu().numpy() == 2).all()
    assert np.isnan(post.predicted_means).all() and np.isnan(post.marginal_loglik).all()
    # non-PD prior covariance -> NaN log-likelihood, status 1
    g2 = dict(g, P0=-np.eye(3))
    post, out, _ = run_filter("cdk_ekf_filter", nonlinear_params_api(g2), y, t[..., None], None, None, fields,
                              diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    assert (out[L.OUT_STATUS].cpu().numpy() == 1).all() and np.isnan(post.marginal_loglik).all()
    assert torch.cuda.is_available()


def test_ll_sum_and_device_resident_inputs():
    import torch
    from cd_dynamax_b200 import _engine as E
    cd = api()
    N, K = 1000, 30
    t, y = c3_problem(N, K)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    yd, td = torch.as_tensor(y).cuda(), torch.as_tensor(t).cuda()
    f = cd.cdnlgssm_filter(p, yd, td[..., None], hp, output_fields=[])
    assert f.marginal_loglik.is_cuda and f.filtered_means is None
    s = E.ll_sum(f.marginal_loglik)
    ref = np.sum(f.marginal_loglik.cpu().numpy().astype(np.float64))
    assert abs(s.item() - ref) <= 1e-12 * abs(ref)
    f_np = cd.cdnlgssm_filter(p, y, t[..., None], hp, output_fields=[])
    assert np.array_equal(f_np.marginal_loglik, f.marginal_loglik.cpu().numpy())  # bit-identical across call styles


# ---- CD-EnKF (a12): shared Philox stream => parity with the oracle to rounding ----------------------------------------
def _enkf_case(kind, N, K, E, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "l63":
        n, m = 3, 1
        g = dict(m0=np.array([1.0, 1.0, 20.0]), P0=2.0 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
                 L=np.eye(3), Qc=0.5 * np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
        mean_gap, dt0 = 0.01, 0.0025
    elif kind == "l96":
        n, m = 40, 20
        x0 = 8.0 + rng.standard_normal(n)
        g = dict(m0=x0, P0=np.eye(n), drift="lorenz96", theta=np.array([8.0]), L=np.eye(n), Qc=0.1 * np.eye(n),
                 H=np.eye(n)[::2], R=np.eye(m), d=np.zeros(m))
        mean_gap, dt0 = 0.02, 0.005
    else:  # generic path: linear drift, dense diffusion, correlated emission noise, emission bias
        n, m = 4, 2
        F = -0.5 * np.eye(n) + 0.3 * rng.standard_normal((n, n)) / 2
        Lm = np.eye(n) + 0.2 * rng.standard_normal((n, n))
        A = rng.standard_normal((m, m))
        g = dict(m0=rng.standard_normal(n), P0=np.eye(n), drift="linear", theta=np.concatenate([F.ravel(), 0.1 * rng.standard_normal(n)]),
                 L=Lm, Qc=0.3 * np.eye(n) + 0.05, H=rng.standard_normal((m, n)), R=A @ A.T + np.eye(m), d=np.array([0.3, -0.2]))
        mean_gap, dt0 = 0.05, 0.0125
    gaps = mean_gap * rng.uniform(0.5, 1.5, size=(N, K))
    gaps[:, 0] = 0.0
    t = np.cumsum(gaps, axis=1)
    y = (g["H"] @ g["m0"])[None, None, :] + 2.0 * rng.standard_normal((N, K, m))
    return g, t, y, dt0


@pytest.mark.parametrize("kind,N,K,E,solver,cluster", [
    ("l63", 5, 40, 64, "euler", 0), ("l63", 3, 25, 100, "heun", 2), ("l96", 3, 12, 96, "euler", 0),
    ("l96", 2, 10, 200, "euler", 4), ("lin", 4, 30, 50, "euler", 0), ("lin", 3, 20, 37, "heun", 2)])
def test_enkf_vs_oracle(kind, N, K, E, solver, cluster, monkeypatch):
    cd = api()
    if cluster:
        monkeypatch.setenv("CDK_ENKF_CLUSTER", str(cluster))
    g, t, y, dt0 = _enkf_case(kind, N, K, E)
    p = nonlinear_params_api(g)
    hp = cd.EnKFHyperParams(N_particles=E, key=12345, diffeqsolve_settings={"solver": solver, "dt0": dt0})
    f = cd.cdnlgssm_filter(p, y, t[..., None], hp)
    n = g["m0"].shape[0]
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift(g["drift"], g["theta"], n), L=g["L"], Qc=g["Qc"],
                           H=g["H"], R=g["R"], d=g["d"])
    r = o.ensemble_kalman_filter(po, y, t, E=E, seed=12345, settings=o.SolverSettings(solver, dt0))
    # 1e-8: libm (NumPy) and CUDA log / sincos differ in the last ulp of every normal deviate, and the chaotic drifts
    # amplify that over the K steps
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < 1e-8
    for fld in FIELDS:
        assert scaled_err(getattr(f, fld), r[fld]) < 1e-8, fld


def test_normal_deviates_bit_identical_to_oracle():
    """The library's deviate stream (Philox4x32-10 + fp32 Box-Muller out of correctly rounded operations only) against the
    oracle's restatement: every bit of 4 x 200,000 deviates."""
    import ctypes
    import torch
    from cd_dynamax_b200 import _lib as L
    lib = L.lib()
    count, traj, step, c3b, seed = 200_000, 77, 5, (2 << 28) | (3 << 8), 0x1234567887654321
    out = torch.empty(4 * count, dtype=torch.float64, device="cuda")
    L.check(lib.cdk_rng_probe_f64(count, traj, step, c3b, seed, ctypes.c_void_p(out.data_ptr()), None), "rng_probe")
    torch.cuda.synchronize()
    z = out.cpu().numpy().reshape(count, 4)
    i = np.arange(count, dtype=np.uint32)
    ref = np.stack(o.philox_normal_quad(i, np.uint32(traj), np.uint32(step), np.uint32(c3b) + (i & np.uint32(0xFF)), seed), axis=1)
    assert np.array_equal(z.view(np.uint64), ref.view(np.uint64))
    assert abs(z.mean()) < 5e-3 and abs(z.var() - 1.0) < 5e-3 and np.abs(z).max() < 6.77


def test_enkf_matches_kalman_filter_in_distribution():
    """The reference's own EnKF check (cdnlgssm_test_filter_linear_TRegular.py:434-470): on a linear model the EnKF
    moments approach the CD-KF's as E grows.  E = 4096 members: Monte-Carlo error ~ 1/sqrt(E)."""
    cd = api()
    g, t, y, dt0 = _enkf_case("lin", 2, 25, 0, seed=11)
    n = 4
    F, b = g["theta"][:16].reshape(4, 4), g["theta"][16:]
    p = nonlinear_params_api(dict(g, theta=np.concatenate([F.ravel(), np.zeros(4)])))
    hp = cd.EnKFHyperParams(N_particles=4096, key=7, diffeqsolve_settings={"solver": "euler", "dt0": dt0 / 4})
    f = cd.cdnlgssm_filter(p, y, t[..., None], hp)
    lp = cd.ParamsCDLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=g["m0"], cov=g["P0"]),
        dynamics=cd.ParamsCDLGSSMDynamics(weights=F, bias=np.zeros(4), input_weights=None, diffusion_coefficient=g["L"],
                                          diffusion_cov=g["Qc"]),
        emissions=cd.ParamsLGSSMEmissions(weights=g["H"], bias=g["d"], input_weights=None, cov=g["R"]))
    kf = cd.cdlgssm_filter(lp, y, t[..., None], cd.KFHyperParams(diffeqsolve_settings={"solver": "dopri5", "dt0": dt0}))
    assert scaled_err(f.filtered_means, kf.filtered_means) < 0.06
    assert scaled_err(f.filtered_covariances, kf.filtered_covariances) < 0.12
    assert max_rel_err(f.marginal_loglik, kf.marginal_loglik) < 0.03


# ---- host-resident inputs streamed in N-chunks (copy / compute / copy-back overlap) must not change a single bit ------
def test_chunked_host_streaming_is_bit_identical(monkeypatch):
    import torch
    from cd_dynamax_b200 import _engine as E
    cd = api()
    N, K = 203, 24  # N not divisible by the chunk count
    t, y = c3_problem(N, K)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    # one batched parameter (vmap over parameter samples): per-trajectory initial means
    m0 = np.random.default_rng(5).standard_normal((N, 3))
    p = nonlinear_params_api(dict(g, m0=m0))
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    dev = lambda a: torch.as_tensor(a).cuda()
    p_dev = nonlinear_params_api(dict(g, m0=dev(m0)))
    ref = cd.cdnlgssm_filter(p_dev, dev(y), dev(t)[..., None], hp)  # resident: one launch
    monkeypatch.setattr(E, "STREAM_MIN_BYTES", 1)
    for yy, tt in ((y, t[..., None]), (torch.as_tensor(y).pin_memory(), torch.as_tensor(t).pin_memory()[..., None])):
        f = cd.cdnlgssm_filter(p, yy, tt, hp)
        for fld in ["marginal_loglik"] + FIELDS:
            a = getattr(f, fld)
            a = a.numpy() if isinstance(a, torch.Tensor) else a
            assert np.array_equal(a, getattr(ref, fld).cpu().numpy()), fld
    # EnKF: the random stream is indexed by the global trajectory number, so chunking must not change it either
    ge, te, ye, dt0 = _enkf_case("l63", 37, 12, 64)
    pe = nonlinear_params_api(ge)
    hpe = cd.EnKFHyperParams(N_particles=64, key=99, diffeqsolve_settings={"solver": "euler", "dt0": dt0})
    f_chunked = cd.cdnlgssm_filter(pe, ye, te[..., None], hpe)
    monkeypatch.setattr(E, "STREAM_MIN_BYTES", 1 << 60)
    f_once = cd.cdnlgssm_filter(pe, ye, te[..., None], hpe)
    for fld in ["marginal_loglik"] + FIELDS:
        assert np.array_equal(getattr(f_chunked, fld), getattr(f_once, fld)), fld
    # linear smoother from host arrays: filter inputs staged once, reused by the backward pass
    gl = load_golden("kf_tracking_c1")
    monkeypatch.setattr(E, "STREAM_MIN_BYTES", 1)
    y1, t1 = gl["y"][0], gl["t"][0]
    Yb, Tb = np.repeat(y1[None], 20, 0), np.repeat(t1[None], 20, 0)
    kh = cd.KFHyperParams(dt_final=float(gl["dt_final"]), diffeqsolve_settings=settings_api(gl))
    s_chunked = cd.cdlgssm_smoother(linear_params_api(gl), Yb, Tb[..., None], kh)
    s_one = cd.cdlgssm_smoother(linear_params_api(gl), y1, t1[:, None], kh)
    assert np.array_equal(s_chunked.smoothed_means[7], s_one.smoothed_means)
    assert np.array_equal(s_chunked.smoothed_covariances[19], s_one.smoothed_covariances)


# ---- CD-KF warp kernels (DMMA, one warp per trajectory): seeded oracle parity at ragged shapes ----------------------
@pytest.mark.parametrize("N,K,n,m,solver,batched_model", [
    (1, 1, 16, 4, "rk4", False), (7, 2, 16, 4, "rk4", False), (13, 9, 5, 2, "heun", False),
    (25, 12, 16, 8, "bosh3", True), (6, 5, 3, 1, "euler", False)])
def test_kf_warp_filter_and_smoother_vs_oracle(N, K, n, m, solver, batched_model):
    cd = api()
    rng = np.random.default_rng(100 + N + K)
    lead = (N,) if batched_model else ()
    F = -0.5 * np.eye(n) + 0.3 * rng.standard_normal(lead + (n, n)) / np.sqrt(n)
    Lm = np.eye(n) + 0.1 * rng.standard_normal((n, n))
    A = rng.standard_normal((m, m))
    g = dict(m0=rng.standard_normal(n), P0=np.eye(n) * 0.7, F=F, b=0.1 * rng.standard_normal(n), B=None, L=Lm,
             Qc=0.1 * np.eye(n) + 0.01, H=rng.standard_normal((m, n)), d=0.2 * rng.standard_normal(m), D=None,
             R=0.1 * (A @ A.T + np.eye(m)))
    gaps = 0.04 * rng.uniform(0.5, 1.5, size=(N, K))
    gaps[:, 0] = 0.0
    t = np.cumsum(gaps, axis=1)
    y = rng.standard_normal((N, K, m))
    hp = cd.KFHyperParams(dt_final=0.03, diffeqsolve_settings={"solver": solver, "dt0": 0.01})
    s = cd.cdlgssm_smoother(linear_params_api(g), y, t[..., None], hp)
    f = cd.cdlgssm_filter(linear_params_api(g), y, t[..., None], hp)
    po = o.LinearParams(m0=g["m0"], P0=g["P0"], F=F, L=Lm, Qc=g["Qc"], H=g["H"], R=g["R"], b=g["b"], d=g["d"])
    r = o.cdlgssm_smoother(po, y, t, dt_final=0.03, settings=o.SolverSettings(solver, 0.01))
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, _tag())
    for fld in ("smoothed_means", "smoothed_covariances", "smoothed_cross_covariances"):
        if r[fld].size:
            record(f"{_tag()}:{fld}:own_norm", moment_err(s, r, fld)[1])
            assert scaled_err(getattr(s, fld), r[fld]) < 1e-8, fld
    assert s.smoothed_cross_covariances.shape == (N, K - 1, n, n)


# ---- EKS fast path (register kernel, Lorenz-63): seeded oracle parity at ragged shapes, all four solvers --------------
@pytest.mark.parametrize("N,K,solver,dt0", [(1, 1, "rk4", 0.0025), (3, 2, "rk4", 0.0025), (45, 7, "heun", 0.005),
                                            (100, 30, "rk4", 0.0025), (33, 16, "dopri5", 0.01), (450, 12, "euler", 0.002)])
def test_eks_l63_fast_path_vs_oracle(N, K, solver, dt0):
    cd = api()
    t, y = c3_problem(N, K, seed=77 + N)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3) + 0.1 * np.arange(9).reshape(3, 3) / 9, Qc=np.eye(3) + 0.05, H=np.array([[1.0, 0.0, 0.0]]),
             R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    hp = cd.EKFHyperParams(dt_final=0.004, diffeqsolve_settings={"solver": solver, "dt0": dt0})
    s = cd.cdnlgssm_smoother(p, y, t[..., None], hp)
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift("lorenz63", g["theta"], 3), L=g["L"], Qc=g["Qc"],
                           H=g["H"], R=g["R"], d=g["d"])
    r = o.extended_kalman_smoother(po, y, t, dt_final=0.004, settings=o.SolverSettings(solver, dt0))
    assert max_rel_err(s.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(s, r, _tag(), fields=("filtered_means", "filtered_covariances"))
    for fld in ("smoothed_means", "smoothed_covariances"):
        record(f"{_tag()}:{fld}:own_norm", moment_err(s, r, fld)[1])
        assert scaled_err(getattr(s, fld), r[fld]) < 1e-8, fld
    # the last smoothed step is the filtered one, verbatim
    assert np.array_equal(s.smoothed_means[:, -1], s.filtered_means[:, -1])
    assert np.array_equal(s.smoothed_covariances[:, -1], s.filtered_covariances[:, -1])


def test_eks_fast_path_matches_generic_kernel(monkeypatch):
    """Same inputs through the register kernel and through generic_smooth_kernel (CDK_EKS_FAST=0 is read once per
    process, so the generic result comes from the golden test above; here: per-trajectory drift parameters)."""
    cd = api()
    N, K = 70, 20
    t, y = c3_problem(N, K, seed=5)
    rng = np.random.default_rng(8)
    theta = np.array([10.0, 28.0, 8.0 / 3.0])[None] * (1 + 0.05 * rng.standard_normal((N, 3)))
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=theta[0], L=np.eye(3), Qc=np.eye(3),
             H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    p = nonlinear_params_api(g)
    p = p._replace(dynamics=p.dynamics._replace(drift=cd.LearnableLorenz63(sigma=theta[:, 0], rho=theta[:, 1], beta=theta[:, 2])))
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    s = cd.cdnlgssm_smoother(p, y, t[..., None], hp)
    for n in (0, 13, 69):
        gi = dict(g, theta=theta[n])
        po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift("lorenz63", theta[n], 3), L=g["L"], Qc=g["Qc"],
                               H=g["H"], R=g["R"], d=g["d"])
        r = o.extended_kalman_smoother(po, y[n:n + 1], t[n:n + 1], settings=o.SolverSettings("rk4", 0.0025))
        assert scaled_err(s.smoothed_means[n], r["smoothed_means"][0]) < 1e-8
        assert scaled_err(s.smoothed_covariances[n], r["smoothed_covariances"][0]) < 1e-8


# ---- d log-likelihood / d drift parameters (SURVEY 8f rank 1, first step): forward-mode kernel vs central differences of
# ---- the oracle's log-likelihood ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("solver,dt0", [("rk4", 0.0025), ("dopri5", 0.01), ("heun", 0.002)])
def test_ekf_loglik_gradient_vs_oracle_finite_differences(solver, dt0):
    cd = api()
    N, K = 6, 40
    t, y = c3_problem(N, K, seed=21)
    theta = np.array([10.0, 28.0, 8.0 / 3.0])
    g = dict(m0=np.array([1.0, 1.0, 20.0]), P0=2 * np.eye(3), drift="lorenz63", theta=theta,
             L=np.eye(3) + 0.1 * np.arange(9).reshape(3, 3) / 9, Qc=np.eye(3) + 0.05, H=np.array([[1.0, 0.3, -0.2]]),
             R=0.7 * np.eye(1), d=np.array([0.1]))
    hp = cd.EKFHyperParams(dt_final=0.004, diffeqsolve_settings={"solver": solver, "dt0": dt0})
    ll, grad = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(g), y, t[..., None], hp)
    f = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], hp, output_fields=[])
    assert max_rel_err(ll, f.marginal_loglik) < 1e-12  # the value is the filter's own

    def oracle_ll(th):
        po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift("lorenz63", th, 3), L=g["L"], Qc=g["Qc"],
                               H=g["H"], R=g["R"], d=g["d"])
        return o.extended_kalman_filter(po, y, t, dt_final=0.004, settings=o.SolverSettings(solver, dt0))["marginal_loglik"]

    for p, name in enumerate(("sigma", "rho", "beta")):
        h = 1e-5 * theta[p]
        tp, tm = theta.copy(), theta.copy()
        tp[p] += h
        tm[p] -= h
        fd = (oracle_ll(tp) - oracle_ll(tm)) / (2 * h)
        # central differences at h = 1e-5 |theta|: truncation ~1e-10 relative, round-off ~1e-9 absolute
        np.testing.assert_allclose(grad[name], fd, rtol=2e-6, atol=2e-7, err_msg=name)
    # unbatched call keeps scalar shapes; unsupported requests fail loudly
    ll1, g1 = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(g), y[0], t[0][:, None], hp)
    assert np.ndim(ll1) == 0 and np.ndim(g1["rho"]) == 0 and g1["rho"] == grad["rho"][0]
    with pytest.raises(NotImplementedError):
        cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(dict(g, H=np.eye(3)[:2], R=np.eye(2), d=np.zeros(2))),
                                          np.zeros((K, 2)), t[0][:, None], hp)


def test_ekf_loglik_gradient_all_parameter_groups():
    """Every leaf of the Lorenz-63 CD-EKF model: directional derivatives of the oracle's log-likelihood (central
    differences) against <gradient, direction>.  Symmetric matrices are probed along symmetric directions."""
    cd = api()
    N, K = 4, 30
    t, y = c3_problem(N, K, seed=33)
    rng = np.random.default_rng(4)
    A = rng.standard_normal((3, 3))
    g = dict(m0=np.array([1.0, 1.0, 20.0]), P0=2 * np.eye(3) + 0.1 * (A + A.T), drift="lorenz63",
             theta=np.array([10.0, 28.0, 8.0 / 3.0]), L=np.eye(3) + 0.2 * rng.standard_normal((3, 3)),
             Qc=np.eye(3) + 0.05 * (A @ A.T), H=np.array([[1.0, 0.3, -0.2]]), R=0.7 * np.eye(1), d=np.array([0.1]))
    hp = cd.EKFHyperParams(dt_final=0.004, diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    ll, grads = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(g), y, t[..., None], hp, wrt="all")
    assert set(grads) == {"sigma", "rho", "beta", "diffusion_coefficient", "diffusion_cov", "emission_cov", "emission_bias",
                          "emission_weights", "initial_mean", "initial_cov"}

    def oracle_ll(**over):
        q = dict(g, **over)
        po = o.NonlinearParams(m0=q["m0"], P0=q["P0"], drift=make_drift("lorenz63", q["theta"], 3), L=q["L"], Qc=q["Qc"],
                               H=q["H"], R=q["R"], d=q["d"])
        return o.extended_kalman_filter(po, y, t, dt_final=0.004, settings=o.SolverSettings("rk4", 0.0025))["marginal_loglik"]

    def check(key, name, direction, h=1e-6):
        base = g[key]
        fd = (oracle_ll(**{key: base + h * direction}) - oracle_ll(**{key: base - h * direction})) / (2 * h)
        got = np.sum(grads[name].reshape(N, -1) * direction.reshape(1, -1), axis=1)
        np.testing.assert_allclose(got, fd, rtol=5e-6, atol=5e-7, err_msg=f"{name} along {direction.ravel()}")

    E = lambda i, j: np.eye(3)[:, [i]] @ np.eye(3)[[j], :]
    for i in range(3):
        check("m0", "initial_mean", np.eye(3)[i])
        check("H", "emission_weights", np.eye(3)[[i]])
        for j in range(3):
            check("L", "diffusion_coefficient", E(i, j))  # exact entry-wise gradient
        for j in range(i, 3):
            D = E(i, j) + E(j, i) if i != j else E(i, i)  # symmetric directions
            check("Qc", "diffusion_cov", D)
            check("P0", "initial_cov", D)
    check("R", "emission_cov", np.ones((1, 1)))
    check("d", "emission_bias", np.ones(1))
    # the gradient matrices of symmetric parameters are symmetric; the default group is the drift alone
    assert np.allclose(grads["diffusion_cov"], np.swapaxes(grads["diffusion_cov"], 1, 2))
    ll2, g2 = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(g), y, t[..., None], hp)
    # (the drift-only default runs the forward-mode kernels, wrt="all" the reverse-mode one: equal to rounding)
    assert set(g2) == {"sigma", "rho", "beta"} and np.allclose(g2["rho"], grads["rho"], rtol=1e-10, atol=0)
    assert np.allclose(ll2, ll, rtol=1e-13, atol=0)


def test_streaming_filter_in_chunks_matches_one_call():
    """cd_dynamax_b200.streaming.filter_in_chunks (how BASELINE config 2's 285 GB of moments are produced and consumed
    chunk by chunk): double-buffered host->device staging must give bit-identical results to one resident call."""
    import torch
    from cd_dynamax_b200 import streaming
    cd = api()
    gl = load_golden("kf_n16_rk4")
    rng = np.random.default_rng(0)
    N, K = 53, 20
    y = torch.as_tensor(rng.standard_normal((N, K, 4))).pin_memory()
    t = torch.as_tensor(np.cumsum(0.04 * rng.uniform(0.5, 1.5, (N, K)), axis=1)[..., None]).pin_memory()
    p = linear_params_api({k: (torch.as_tensor(v).cuda() if isinstance(v, np.ndarray) and v.dtype == np.float64 and v.size else v)
                           for k, v in gl.items() if k in ("m0", "P0", "F", "b", "B", "L", "Qc", "H", "d", "D", "R")})
    p = p._replace(dynamics=p.dynamics._replace(input_weights=None), emissions=p.emissions._replace(input_weights=None))
    hp = cd.KFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    ref = cd.cdlgssm_filter(p, y.cuda(), t.cuda(), hp)
    got_ll = torch.empty(N, dtype=torch.float64, device="cuda")
    got_pp = torch.empty_like(ref.predicted_covariances)
    seen = []

    def consume(post, lo, hi):
        got_ll[lo:hi] = post.marginal_loglik
        got_pp[lo:hi] = post.predicted_covariances
        seen.append((lo, hi))

    streaming.filter_in_chunks(lambda yy, tt: cd.cdlgssm_filter(p, yy, tt, hp), y, t, 16, consume)
    assert seen == [(0, 16), (16, 32), (32, 48), (48, 53)]
    assert torch.equal(got_ll, ref.marginal_loglik) and torch.equal(got_pp, ref.predicted_covariances)


@pytest.mark.parametrize("solver,dt0", [("rk4", 0.0025), ("rk4", 0.0006), ("heun", 0.002), ("euler", 0.002), ("dopri5", 0.01)])
def test_ekf_loglik_gradient_reverse_mode_matches_forward_mode(solver, dt0, monkeypatch):
    """SURVEY 8f rank 1: the reverse-mode kernel (forward filter + ONE backward launch for all 23 columns) against the
    forward-mode kernels (one launch per column, themselves checked against central differences of the oracle above): both
    are exact derivatives of the same discrete filter, so they agree to rounding.  dt0 = 0.0006 gives ~17 substeps per gap:
    more than the 8 substep checkpoints, i.e. the re-integration path."""
    cd = api()
    N, K = 7, 40
    t, y = c3_problem(N, K, seed=33)
    rng = np.random.default_rng(4)
    A = rng.standard_normal((3, 3))
    g = dict(m0=np.array([1.0, 1.0, 20.0]), P0=2 * np.eye(3) + 0.1 * (A + A.T), drift="lorenz63",
             theta=np.array([10.0, 28.0, 8.0 / 3.0]), L=np.eye(3) + 0.2 * rng.standard_normal((3, 3)),
             Qc=np.eye(3) + 0.05 * (A @ A.T), H=np.array([[1.0, 0.3, -0.2]]), R=0.7 * np.eye(1), d=np.array([0.1]))
    hp = cd.EKFHyperParams(dt_final=0.004, diffeqsolve_settings={"solver": solver, "dt0": dt0})
    monkeypatch.setenv("CDK_GRAD_MODE", "forward")
    ll_f, gf = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(g), y, t[..., None], hp, wrt="all")
    monkeypatch.setenv("CDK_GRAD_MODE", "reverse")
    ll_r, gr = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(g), y, t[..., None], hp, wrt="all")
    assert set(gf) == set(gr) and max_rel_err(ll_r, ll_f) < 1e-12
    for name in sorted(gf):
        scale = np.max(np.abs(gf[name]))
        err = np.max(np.abs(gr[name] - gf[name])) / scale
        record(f"grad_reverse_vs_forward_{solver}_{dt0}:{name}", err)
        assert err < 1e-9, (name, err)
    # the default ("auto") picks reverse mode as soon as more than the drift group is requested; per-trajectory parameters
    monkeypatch.setenv("CDK_GRAD_MODE", "auto")
    th = np.array([10.0, 28.0, 8.0 / 3.0])[None] * (1 + 0.03 * rng.standard_normal((N, 3)))
    p = nonlinear_params_api(g)
    p = p._replace(dynamics=p.dynamics._replace(drift=cd.LearnableLorenz63(sigma=th[:, 0], rho=th[:, 1], beta=th[:, 2])))
    _, ga = cd.ekf_marginal_log_prob_and_grad(p, y, t[..., None], hp, wrt=("drift", "initial_mean"))
    monkeypatch.setenv("CDK_GRAD_MODE", "forward")
    _, gb = cd.ekf_marginal_log_prob_and_grad(p, y, t[..., None], hp, wrt=("drift", "initial_mean"))
    for name in ("sigma", "rho", "beta", "initial_mean"):
        assert np.max(np.abs(ga[name] - gb[name])) < 1e-9 * np.max(np.abs(gb[name])), name


def test_ekf_loglik_gradient_long_run_reverse_vs_forward(monkeypatch):
    """The two independent derivative kernels over config 3's full K = 1,000 (the reverse pass walks 1,000 stored steps and
    ~4,500 re-integrated substeps backwards): they must still agree to rounding relative to each gradient's scale, and the
    reverse-mode log-likelihood must be the filter's."""
    cd = api()
    N, K = 40, 1000
    t, y = c3_problem(N, K, seed=35)
    g = dict(m0=np.zeros(3), P0=5 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
             L=np.eye(3), Qc=np.eye(3), H=np.array([[1.0, 0.0, 0.0]]), R=np.eye(1), d=np.zeros(1))
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    p = nonlinear_params_api(g)
    monkeypatch.setenv("CDK_GRAD_MODE", "forward")
    ll_f, gf = cd.ekf_marginal_log_prob_and_grad(p, y, t[..., None], hp, wrt=("drift", "emission_cov", "initial_mean"))
    monkeypatch.setenv("CDK_GRAD_MODE", "reverse")
    ll_r, gr = cd.ekf_marginal_log_prob_and_grad(p, y, t[..., None], hp, wrt=("drift", "emission_cov", "initial_mean"))
    f = cd.cdnlgssm_filter(p, y, t[..., None], hp, output_fields=[])
    assert max_rel_err(ll_r, np.asarray(f.marginal_loglik)) < 1e-12 and max_rel_err(ll_f, ll_r) < 1e-12
    for name in sorted(gf):
        scale = np.max(np.abs(gf[name]))
        err = np.max(np.abs(gr[name] - gf[name])) / scale
        record(f"grad_long_run_reverse_vs_forward:{name}", err)
        assert np.isfinite(gr[name]).all() and err < 1e-8, (name, err)


def test_torch_autograd_wrapper_around_the_reverse_mode_kernel():
    """cd_dynamax_b200.autograd.ekf_marginal_log_prob: the custom_vjp-shaped wrapper (forward = CUDA filter, backward = the
    reverse-mode kernel).  `(-ll.sum()).backward()` -- fit_sgd's loss -- must put the summed gradients on shared leaves."""
    import torch
    from cd_dynamax_b200 import autograd
    cd = api()
    N, K = 5, 30
    t, y = c3_problem(N, K, seed=3)
    dev = torch.device("cuda")
    T = lambda a, rg=True: torch.tensor(np.asarray(a, dtype=np.float64), device=dev, requires_grad=rg)
    leaves = dict(sigma=T(10.0), rho=T(28.0), beta=T(8.0 / 3.0), L=T(np.eye(3)), Qc=T(np.eye(3) + 0.05), R=T([[0.7]]), d=T([0.1]),
                  H=T([[1.0, 0.3, -0.2]]), m0=T([1.0, 1.0, 20.0]), P0=T(2 * np.eye(3)))
    p = cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(leaves["m0"]), cov=cd.LearnableMatrix(leaves["P0"])),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableLorenz63(sigma=leaves["sigma"], rho=leaves["rho"], beta=leaves["beta"]),
                                           diffusion_coefficient=cd.LearnableMatrix(leaves["L"]),
                                           diffusion_cov=cd.LearnableMatrix(leaves["Qc"])),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=leaves["H"], bias=leaves["d"]),
                                             emission_cov=cd.LearnableMatrix(leaves["R"])))
    hp = cd.EKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    yd, td = torch.as_tensor(y, device=dev), torch.as_tensor(t, device=dev)[..., None]
    ll = autograd.ekf_marginal_log_prob(p, yd, td, hp)
    assert ll.shape == (N,) and ll.requires_grad
    (-ll.sum()).backward()
    with torch.no_grad():
        pd = jax_like_detach(p)
        ll0, g = cd.ekf_marginal_log_prob_and_grad(pd, yd, td, hp, wrt="all")
    assert torch.allclose(ll.detach(), ll0, rtol=1e-13, atol=0)
    for leaf, name in (("sigma", "sigma"), ("rho", "rho"), ("Qc", "diffusion_cov"), ("L", "diffusion_coefficient"), ("R", "emission_cov"),
                       ("H", "emission_weights"), ("m0", "initial_mean"), ("P0", "initial_cov"), ("d", "emission_bias")):
        want = -g[name].sum(0)
        assert torch.allclose(leaves[leaf].grad, want.reshape(leaves[leaf].shape), rtol=1e-10, atol=1e-12), name


def jax_like_detach(p):
    """The same parameter tuple with every torch leaf detached."""
    import torch
    det = lambda x: x.detach() if isinstance(x, torch.Tensor) else x
    cd = api()
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(det(p.initial.mean.params)), cov=cd.LearnableMatrix(det(p.initial.cov.params))),
        dynamics=cd.ParamsCDNLGSSMDynamics(
            drift=cd.LearnableLorenz63(sigma=det(p.dynamics.drift.sigma), rho=det(p.dynamics.drift.rho), beta=det(p.dynamics.drift.beta)),
            diffusion_coefficient=cd.LearnableMatrix(det(p.dynamics.diffusion_coefficient.params)),
            diffusion_cov=cd.LearnableMatrix(det(p.dynamics.diffusion_cov.params))),
        emissions=cd.ParamsCDNLGSSMEmissions(
            emission_function=cd.LearnableLinear(weights=det(p.emissions.emission_function.weights), bias=det(p.emissions.emission_function.bias)),
            emission_cov=cd.LearnableMatrix(det(p.emissions.emission_cov.params))))
