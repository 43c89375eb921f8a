"""GPU: a USER-DEFINED emission function compiled into a variant of libcdk.so (cd_dynamax_b200.build.build_variant) --
the range to m beacons of examples/range_emission.cuh -- through the EKF (first / second order, iterated), the EKS, the UKF
(literal sigma-point update), the EnKF and the path sampler, against the oracle's filters restated with the same emission
in NumPy (tests/user_emission_oracle.py); with a user drift in the same variant and with registry drifts (Lorenz-63, whose fast paths must be bypassed, and Lorenz-96 at
BASELINE config 4 / 5 sizes); the linear emission written as user code against the stock LearnableLinear runs; per-trajectory
phi; fp32; and the entry points that must refuse the id."""
import ctypes
import os

import numpy as np
import pytest

from oracle import cd_oracle as o
from tests.helpers import make_drift, max_rel_err, record, scaled_err
from tests.test_gpu_parity import FIELDS, TOL, api, check_moments
from tests.test_gpu_user_drift import VDP_CODE, VdpDrift
from tests import user_emission_oracle as uo

pytestmark = pytest.mark.gpu

_EX = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cd_dynamax_b200", "examples")
RANGE_CODE = open(os.path.join(_EX, "range_emission.cuh")).read()
LINEAR_CODE = open(os.path.join(_EX, "linear_emission.cuh")).read()


class RangeEmission:
    """examples/range_emission.cuh for the oracle: h_a(x) = sqrt(|x - b_a|^2 + eps)."""

    def __init__(self, B, eps):
        self.B, self.eps = np.asarray(B, np.float64), float(eps)

    def phi(self):
        return np.concatenate([self.B.reshape(-1), [self.eps]])

    def h(self, x):
        r = x[..., None, :] - self.B
        return np.sqrt(np.sum(r * r, axis=-1) + self.eps)

    def jac(self, x):
        return (x[..., None, :] - self.B) / self.h(x)[..., None]


def _params(cd, drift_api, em_code, phi, g):
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(g["m0"]), cov=cd.LearnableMatrix(g["P0"])),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=drift_api, diffusion_coefficient=cd.LearnableMatrix(g["L"]),
                                           diffusion_cov=cd.LearnableMatrix(g["Qc"])),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableUserEmission(device_code=em_code, phi=phi),
                                             emission_cov=cd.LearnableMatrix(g["R"])))


def _vdp_range(N=7, K=30, seed=0):
    """VdP drift (user code) + range to m = 2 beacons (user code): one variant holding both."""
    cd = api()
    rng = np.random.default_rng(seed)
    theta = np.array([1.3, 0.4])
    em = RangeEmission([[2.0, 0.0], [-1.0, 2.5]], 0.01)
    g = dict(m0=np.array([1.0, 0.5]), P0=0.3 * np.eye(2), L=np.eye(2) + 0.1 * rng.standard_normal((2, 2)),
             Qc=0.2 * np.eye(2) + 0.02, R=0.05 * np.eye(2) + 0.01)
    p = _params(cd, cd.LearnableUserDrift(device_code=VDP_CODE, theta=theta), RANGE_CODE, em.phi(), g)
    po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=VdpDrift(*theta), L=g["L"], Qc=g["Qc"], H=None, R=g["R"])
    t = np.cumsum(0.05 * rng.uniform(0.5, 1.5, (N, K)), axis=1)
    x = np.stack([np.cos(2 * t), np.sin(2 * t)], axis=-1)
    y = em.h(x) + 0.2 * rng.standard_normal((N, K, 2))
    return cd, p, po, t, y, em


ST = {"solver": "rk4", "dt0": 0.0125}
OST = o.SolverSettings("rk4", 0.0125)


@pytest.mark.parametrize("order,num_iter", [("first", 1), ("second", 1), ("first", 2)])
def test_user_drift_and_emission_ekf_eks(order, num_iter):
    cd, p, po, t, y, em = _vdp_range()
    hp = cd.EKFHyperParams(state_order=order, dt_final=0.02, diffeqsolve_settings=ST)
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm import extended_kalman_filter
    f = extended_kalman_filter(p, y, t[..., None], hp, num_iter=num_iter)
    r = uo.extended_kalman_filter(po, em, y, t, dt_final=0.02, state_order=order, settings=OST, num_iter=num_iter)
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, f"user_emission_ekf_{order}_{num_iter}")
    if num_iter == 1:
        s = cd.cdnlgssm_smoother(p, y, t[..., None], hp)
        rs = uo.extended_kalman_smoother(po, em, y, t, dt_final=0.02, state_order=order, settings=OST)
        for fld in ("smoothed_means", "smoothed_covariances"):
            assert scaled_err(getattr(s, fld), rs[fld]) < 1e-8, fld


def test_user_drift_and_emission_ukf_enkf_sampler():
    cd, p, po, t, y, em = _vdp_range(N=5, K=25, seed=1)
    f = cd.cdnlgssm_filter(p, y, t[..., None], cd.UKFHyperParams(diffeqsolve_settings=ST))
    r = uo.unscented_kalman_filter(po, em, y, t, settings=OST)
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, "user_emission_ukf")
    fe = cd.cdnlgssm_filter(p, y, t[..., None], cd.EnKFHyperParams(N_particles=80, key=3, diffeqsolve_settings={"dt0": 0.0125}))
    re = uo.ensemble_kalman_filter(po, em, y, t, E=80, seed=3, settings=o.SolverSettings("heun", 0.0125))
    assert max_rel_err(fe.marginal_loglik, re["marginal_loglik"]) < 1e-8
    for fld in FIELDS:
        assert scaled_err(getattr(fe, fld), re[fld]) < 1e-8, fld
    xs, ys = cd.cdnlgssm_path_sample(p, 11, t.shape[1], t[..., None], diffeqsolve_settings={"dt0": 0.0125})
    rx, ry = uo.sample_paths(po, em, t, seed=11, settings=o.SolverSettings("heun", 0.0125))
    assert scaled_err(xs, rx) < 1e-8 and scaled_err(ys, ry) < 1e-8
    record("user_emission_sampler:emissions", scaled_err(ys, ry))


def _registry(kind, n, m, seed):
    cd = api()
    rng = np.random.default_rng(seed)
    theta = np.array([10.0, 28.0, 8.0 / 3.0]) if kind == "lorenz63" else np.array([8.0])
    em = RangeEmission(4.0 * rng.standard_normal((m, n)), 0.1)
    m0 = np.full(n, 1.0) + 0.5 * rng.standard_normal(n)
    g = dict(m0=m0, P0=0.5 * np.eye(n), L=np.eye(n), Qc=0.5 * np.eye(n), R=0.2 * np.eye(m))
    drift = cd.LearnableLorenz63(*theta) if kind == "lorenz63" else cd.LearnableLorenz96(forcing=theta[0])
    p = _params(cd, drift, RANGE_CODE, em.phi(), g)
    po = o.NonlinearParams(m0=m0, P0=g["P0"], drift=make_drift(kind, theta, n), L=g["L"], Qc=g["Qc"], H=None, R=g["R"])
    return cd, p, po, em


def test_lorenz63_range_bypasses_the_fast_paths():
    cd, p, po, em = _registry("lorenz63", 3, 2, 4)
    N, K = 6, 40
    rng = np.random.default_rng(5)
    t = np.cumsum(0.01 * rng.uniform(0.5, 1.5, (N, K)), axis=1)
    y = em.h(np.zeros((N, K, 3)) + np.array([1.0, 1.0, 20.0])) + rng.standard_normal((N, K, 2))
    hp = cd.EKFHyperParams(state_order="first", diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    f = cd.cdnlgssm_filter(p, y, t[..., None], hp)
    r = uo.extended_kalman_filter(po, em, y, t, state_order="first", settings=o.SolverSettings("rk4", 0.0025))
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, "user_emission_l63_ekf")
    s = cd.cdnlgssm_smoother(p, y, t[..., None], hp)
    rs = uo.extended_kalman_smoother(po, em, y, t, state_order="first", settings=o.SolverSettings("rk4", 0.0025))
    for fld in ("smoothed_means", "smoothed_covariances"):
        assert scaled_err(getattr(s, fld), rs[fld]) < 1e-8, fld


def test_lorenz96_n40_m20_ekf_ukf_enkf():
    """BASELINE config 4 / 5 shapes (n = 40, m = 20; EnKF with E = 1,024 on its cluster path) at small N and K."""
    cd, p, po, em = _registry("lorenz96", 40, 20, 6)
    N, K = 2, 6
    rng = np.random.default_rng(7)
    t = np.cumsum(0.02 * rng.uniform(0.5, 1.5, (N, K)), axis=1)
    y = em.h(np.broadcast_to(po.m0, (N, K, 40))) + 0.5 * rng.standard_normal((N, K, 20))
    st, ost = {"solver": "rk4", "dt0": 0.005}, o.SolverSettings("rk4", 0.005)
    f = cd.cdnlgssm_filter(p, y, t[..., None], cd.EKFHyperParams(state_order="first", diffeqsolve_settings=st))
    r = uo.extended_kalman_filter(po, em, y, t, state_order="first", settings=ost)
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, "user_emission_l96_ekf")
    f = cd.cdnlgssm_filter(p, y, t[..., None], cd.UKFHyperParams(diffeqsolve_settings=st))  # closed-form predict
    r = uo.unscented_kalman_filter(po, em, y, t, settings=ost)
    assert max_rel_err(f.marginal_loglik, r["marginal_loglik"]) < TOL
    check_moments(f, r, "user_emission_l96_ukf")
    fe = cd.cdnlgssm_filter(p, y, t[..., None], cd.EnKFHyperParams(N_particles=1024, key=2,
                                                                    diffeqsolve_settings={"solver": "euler", "dt0": 0.005}))
    re = uo.ensemble_kalman_filter(po, em, y, t, E=1024, seed=2, settings=o.SolverSettings("euler", 0.005))
    assert max_rel_err(fe.marginal_loglik, re["marginal_loglik"]) < 1e-8
    for fld in FIELDS:
        assert scaled_err(getattr(fe, fld), re[fld]) < 1e-8, fld


def test_linear_emission_as_user_code_matches_the_stock_runs():
    """h = H x + d as device code through the user-emission update paths vs LearnableLinear through the stock ones."""
    cd = api()
    n, m, N, K = 6, 3, 4, 30
    rng = np.random.default_rng(8)
    H, d = rng.standard_normal((m, n)), rng.standard_normal(m)
    g = dict(m0=np.ones(n), P0=0.5 * np.eye(n), L=np.eye(n), Qc=0.3 * np.eye(n), R=0.2 * np.eye(m) + 0.05)
    drift = cd.LearnableLorenz96(forcing=8.0)
    pu = _params(cd, drift, LINEAR_CODE, np.concatenate([H.reshape(-1), d]), g)
    pl = pu._replace(emissions=pu.emissions._replace(emission_function=cd.LearnableLinear(weights=H, bias=d)))
    t = np.cumsum(0.02 * rng.uniform(0.5, 1.5, (N, K)), axis=1)
    y = 2.0 * rng.standard_normal((N, K, m))
    st = {"solver": "rk4", "dt0": 0.005}
    for hp in (cd.EKFHyperParams(state_order="first", diffeqsolve_settings=st), cd.UKFHyperParams(diffeqsolve_settings=st)):
        fu, fl = (cd.cdnlgssm_filter(p, y, t[..., None], hp) for p in (pu, pl))
        assert max_rel_err(fu.marginal_loglik, fl.marginal_loglik) < TOL
        check_moments(fu, {k: getattr(fl, k) for k in FIELDS}, f"user_linear_{type(hp).__name__}")
    hp = cd.EnKFHyperParams(N_particles=200, key=1, diffeqsolve_settings={"dt0": 0.005})
    fu, fl = (cd.cdnlgssm_filter(p, y, t[..., None], hp) for p in (pu, pl))
    assert max_rel_err(fu.marginal_loglik, fl.marginal_loglik) < 1e-8
    for fld in FIELDS:
        assert scaled_err(getattr(fu, fld), getattr(fl, fld)) < 1e-8, fld


def test_per_trajectory_phi_equals_separate_runs():
    cd, p, po, t, y, em = _vdp_range(N=4, K=20, seed=2)
    phis = np.stack([em.phi() + 0.3 * i for i in range(4)])
    pb = p._replace(emissions=p.emissions._replace(emission_function=cd.LearnableUserEmission(RANGE_CODE, phis)))
    for hp in (cd.EKFHyperParams(state_order="first", diffeqsolve_settings=ST), cd.UKFHyperParams(diffeqsolve_settings=ST),
               cd.EnKFHyperParams(N_particles=64, key=5, diffeqsolve_settings={"dt0": 0.0125})):
        fb = cd.cdnlgssm_filter(pb, y, t[..., None], hp)
        for i in range(4):  # the whole batch with phi_i shared: same trajectory index, so the EnKF draws the same deviates
            pi = p._replace(emissions=p.emissions._replace(emission_function=cd.LearnableUserEmission(RANGE_CODE, phis[i])))
            fi = cd.cdnlgssm_filter(pi, y, t[..., None], hp)
            assert np.array_equal(fb.marginal_loglik[i], fi.marginal_loglik[i]), (type(hp).__name__, i)
            assert np.array_equal(fb.filtered_means[i], fi.filtered_means[i]), (type(hp).__name__, i)


def test_fp32_ekf_user_emission():
    """cdk_ekf_filter_f32 with the user emission, within the fp32 bound of the parity suite (2e-4 relative on the
    log-likelihood, 2e-3 scaled on the moments)."""
    cd, p, po, t, y, em = _vdp_range(N=16, K=30, seed=3)
    f32 = cd.cdnlgssm_filter(p, y.astype(np.float32), t.astype(np.float32)[..., None],
                             cd.EKFHyperParams(state_order="first", diffeqsolve_settings=ST))
    assert f32.filtered_means.dtype == np.float32
    r = uo.extended_kalman_filter(po, em, y.astype(np.float32), t.astype(np.float32).astype(np.float64), state_order="first",
                                 settings=o.SolverSettings("rk4", float(np.float32(0.0125)), time_dtype=np.float32))
    assert max_rel_err(f32.marginal_loglik, r["marginal_loglik"]) < 2e-4
    for fld in FIELDS:
        assert scaled_err(getattr(f32, fld), r[fld]) < 2e-3, fld


def _call(lib, name, emission_id, n=2, m=2, n_theta=3, drift_id=1):
    from cd_dynamax_b200 import _lib as L
    d = L.new_desc()
    d.N, d.K, d.n, d.m, d.drift_id, d.n_theta, d.emission_id = 2, 3, n, m, drift_id, n_theta, emission_id
    if drift_id == L.DRIFT_LORENZ63:
        d.n = 3
    ins = (ctypes.c_void_p * L.NUM_IN)()
    outs = (ctypes.c_void_p * L.NUM_OUT)()
    return getattr(lib, name)(ctypes.byref(d), ins, outs, None)


def test_libraries_without_the_emission_and_every_gradient_entry_refuse_the_id():
    from cd_dynamax_b200 import _lib as L
    from cd_dynamax_b200 import build as B
    stock = L.lib()
    drift_only = L.lib(B.build_user_drift(VDP_CODE))
    for lib in (stock, drift_only):
        assert lib.cdk_has_user_emission() == 0 and lib.cdk_user_emission_params(2, 2) == -1
        for name in ("cdk_ekf_filter_f64", "cdk_ukf_filter_f64", "cdk_enkf_filter_f64", "cdk_sample_path_f64"):
            assert _call(lib, name, L.EMISSION_USER) == -4, name  # CDK_E_UNSUPPORTED
        assert _call(lib, "cdk_ekf_filter_f64", 7) == -3  # CDK_E_ENUM
    var = L.lib(B.build_variant(None, RANGE_CODE))
    assert var.cdk_has_user_emission() == 1 and var.cdk_user_emission_params(3, 2) == 7
    for name in ("cdk_ekf_grad_f64", "cdk_ekf_grad_dense_f64", "cdk_ukf_grad_dense_f64", "cdk_ukf_grad_sigma_f64",
                 "cdk_emission_moments_f64"):
        assert _call(var, name, L.EMISSION_USER) == -4, name
    assert _call(var, "cdk_ekf_filter_f64", 7) == -3
