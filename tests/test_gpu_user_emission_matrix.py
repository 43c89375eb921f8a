"""GPU: the user-emission (CDK_EMISSION_USER) branches of every filter kernel against tests/user_emission_oracle.py, at the
shapes, layouts, dtypes and edges that the linear emission is tested on.  Three test emissions, each a CUDA code string
with a NumPy twin (h and an analytic jac):

  * range   -- examples/range_emission.cuh, n_phi = m n + 1;
  * wide    -- a one-hidden-layer tanh network, n_phi = 24 (n + 1) + 25 m: at every shape used here n_phi > m (n + 1), so a
               region or a copy sized from m and n instead of n_phi loses weights;
  * square  -- h_a(x) = x_{a mod n}^2, n_phi = 0 (phi is [0]: its device pointer is NULL), in a variant whose user drift
               takes no parameters either (n_theta = 0).

Gates: the parity suite's (log-likelihood relative TOL, check_moments) for the deterministic filters in fp64, 1e-8 for
smoothed moments, the EnKF and sampled paths, and the stated fp32 bounds of tests/test_gpu_baseline_shapes.py."""
import concurrent.futures
import dataclasses
import zlib

import numpy as np
import pytest

from oracle import cd_oracle as o
from tests.helpers import make_drift, max_rel_err, record, scaled_err
from tests.test_gpu_parity import FIELDS, TOL, api, check_moments
from tests.test_gpu_user_drift import VDP_CODE, VdpDrift
from tests.test_gpu_user_emission import RANGE_CODE, RangeEmission
from tests import user_emission_oracle as uo

pytestmark = pytest.mark.gpu

WIDTH = 24
WIDE_CODE = r"""
// h(x) = W2 tanh(W1 x + b1) + b2 with a hidden width of 24; phi = [W1 (24 x n, row-major) | b1 (24) | W2 (m x 24) | b2 (m)]
namespace cdk_user_emission {
__host__ __device__ inline int num_params(int n, int m) { return 24 * (n + 1) + 25 * m; }
template <typename T, class XF> __device__ __forceinline__ T h(const T* phi, int n, int m, int a, XF x) {
  const T* b1 = phi + 24 * n;
  const T* W2 = b1 + 24;
  T s = W2[24 * m + a];
  for (int k = 0; k < 24; ++k) {
    T z = b1[k];
    for (int j = 0; j < n; ++j) z += phi[k * n + j] * x(j);
    s += W2[a * 24 + k] * tanh(z);
  }
  return s;
}
template <typename T> __device__ __forceinline__ T jac(const T* phi, int n, int m, int a, int j, const T* x) {
  const T* b1 = phi + 24 * n;
  const T* W2 = b1 + 24;
  T s = T(0);
  for (int k = 0; k < 24; ++k) {
    T z = b1[k];
    for (int q = 0; q < n; ++q) z += phi[k * n + q] * x[q];
    const T th = tanh(z);
    s += W2[a * 24 + k] * (T(1) - th * th) * phi[k * n + j];
  }
  return s;
}
}
"""

SQUARE_CODE = r"""
// h_a(x) = x_{a mod n}^2: no parameters (num_params = 0)
namespace cdk_user_emission {
__host__ __device__ inline int num_params(int n, int m) { return 0; }
template <typename T, class XF> __device__ __forceinline__ T h(const T* phi, int n, int m, int a, XF x) {
  const T v = x(a % n);
  return v * v;
}
template <typename T> __device__ __forceinline__ T jac(const T* phi, int n, int m, int a, int j, const T* x) {
  return j == a % n ? T(2) * x[j] : T(0);
}
}
"""

ZERO_DRIFT_CODE = r"""
// f_i(x) = -x_i + sin(x_{(i + 1) mod n}): no parameters (n_theta = 0)
namespace cdk_user {
template <typename T, class XF> __device__ __forceinline__ T f(const T* th, int n, int i, XF x) {
  return -x(i) + sin(x(i + 1 == n ? 0 : i + 1));
}
template <typename T> __device__ __forceinline__ T jac(const T* th, int n, int i, int j, const T* x) {
  return (j == i ? T(-1) : T(0)) + (j == (i + 1 == n ? 0 : i + 1) ? cos(x[j]) : T(0));
}
template <typename T> __device__ __forceinline__ T graddiv(const T* th, int n, int k, const T* x) {
  return n == 1 ? -sin(x[0]) : T(0);
}
}
"""


class WideEmission:
    """WIDE_CODE for the oracle."""
    code = WIDE_CODE

    def __init__(self, n, m, rng):
        self.W1 = rng.standard_normal((WIDTH, n)) / np.sqrt(n)
        self.b1 = 0.3 * rng.standard_normal(WIDTH)
        self.W2 = 2.0 * rng.standard_normal((m, WIDTH)) / np.sqrt(WIDTH)
        self.b2 = rng.standard_normal(m)

    def phi(self):
        return np.concatenate([self.W1.reshape(-1), self.b1, self.W2.reshape(-1), self.b2])

    def h(self, x):
        return np.tanh(x @ self.W1.T + self.b1) @ self.W2.T + self.b2

    def jac(self, x):
        th = np.tanh(x @ self.W1.T + self.b1)
        return (self.W2 * (1.0 - th * th)[..., None, :]) @ self.W1


class SquareEmission:
    """SQUARE_CODE for the oracle."""
    code = SQUARE_CODE

    def __init__(self, n, m):
        self.idx = np.arange(m) % n

    def phi(self):
        return np.zeros(0)

    def h(self, x):
        return x[..., self.idx] ** 2

    def jac(self, x):
        J = np.zeros(x.shape[:-1] + (len(self.idx), x.shape[-1]))
        for a, j in enumerate(self.idx):
            J[..., a, j] = 2.0 * x[..., j]
        return J


class ZeroDrift:
    """ZERO_DRIFT_CODE for the oracle."""

    def f(self, x):
        return -x + np.sin(np.roll(x, -1, axis=-1))

    def jac(self, x):
        n = x.shape[-1]
        J = np.broadcast_to(-np.eye(n), x.shape + (n,)).copy()
        c = np.cos(np.roll(x, -1, axis=-1))
        for i in range(n):
            J[..., i, (i + 1) % n] += c[..., i]
        return J

    def grad_div(self, x):
        return np.zeros_like(x)


def _range(n, m, rng, eps=0.1):
    em = RangeEmission(4.0 * rng.standard_normal((m, n)), eps)
    em.code = RANGE_CODE
    return em


def _emission(kind, n, m, rng):
    return {"range": lambda: _range(n, m, rng), "wide": lambda: WideEmission(n, m, rng),
            "square": lambda: SquareEmission(n, m)}[kind]()


@pytest.fixture(scope="module", autouse=True)
def variants():
    """The new variants of this file (each cached by content hash), built side by side before the first case."""
    from cd_dynamax_b200 import build as B
    B.build()
    with concurrent.futures.ThreadPoolExecutor(2) as ex:
        list(ex.map(lambda a: B.build_variant(*a), [(None, WIDE_CODE), (ZERO_DRIFT_CODE, SQUARE_CODE)]))


class Case:
    """One model: API params `p`, oracle params `po`, emission twin `em`, times `t` [N, K] and emissions `y`."""

    def __init__(self, drift, n, m, emission="range", N=4, K=20, seed=0, gap=0.02, noise=0.3, phi=None):
        cd = api()
        rng = np.random.default_rng(seed)
        self.em = em = _emission(emission, n, m, rng)
        m0 = np.ones(n) + 0.5 * rng.standard_normal(n)
        if drift == "vdp":
            theta = np.array([1.3, 0.4])
            d_api, d_or = cd.LearnableUserDrift(device_code=VDP_CODE, theta=theta), VdpDrift(*theta)
            m0 = np.array([1.0, 0.5])
        elif drift == "zero":
            d_api, d_or = cd.LearnableUserDrift(device_code=ZERO_DRIFT_CODE, theta=np.zeros(0)), ZeroDrift()
        elif drift == "lorenz63":
            theta = np.array([10.0, 28.0, 8.0 / 3.0])
            d_api, d_or = cd.LearnableLorenz63(*theta), make_drift("lorenz63", theta, 3)
            m0 = np.array([1.0, 1.0, 20.0]) + rng.standard_normal(3)
        elif drift == "lorenz96":
            d_api, d_or = cd.LearnableLorenz96(forcing=8.0), make_drift("lorenz96", [8.0], n)
        elif drift == "linear":
            A = -0.5 * np.eye(n) + 0.3 * rng.standard_normal((n, n)) / np.sqrt(n)
            b = 0.1 * rng.standard_normal(n)
            d_api, d_or = cd.LearnableLinear(weights=A, bias=b), o.LinearDrift(A, b)
        else:
            raise ValueError(drift)
        Lm = np.eye(n) + 0.05 * rng.standard_normal((n, n))
        g = dict(m0=m0, P0=0.3 * np.eye(n), L=Lm, Qc=0.3 * np.eye(n), R=0.2 * np.eye(m) + 0.02)
        self.phi = em.phi() if phi is None else phi
        self.p = cd.ParamsCDNLGSSM(
            initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(g["m0"]), cov=cd.LearnableMatrix(g["P0"])),
            dynamics=cd.ParamsCDNLGSSMDynamics(drift=d_api, diffusion_coefficient=cd.LearnableMatrix(g["L"]),
                                               diffusion_cov=cd.LearnableMatrix(g["Qc"])),
            emissions=cd.ParamsCDNLGSSMEmissions(
                emission_function=cd.LearnableUserEmission(device_code=em.code, phi=self.phi),
                emission_cov=cd.LearnableMatrix(g["R"])))
        self.po = o.NonlinearParams(m0=m0, P0=g["P0"], drift=d_or, L=g["L"], Qc=g["Qc"], H=None, R=g["R"])
        self.t = np.cumsum(gap * rng.uniform(0.5, 1.5, (N, K)), axis=1)
        self.y = em.h(np.broadcast_to(m0, (N, K, n))) + noise * rng.standard_normal((N, K, m))
        self.N, self.K, self.n, self.m = N, K, n, m

    def with_phi(self, phi):
        cd = api()
        return self.p._replace(emissions=self.p.emissions._replace(
            emission_function=cd.LearnableUserEmission(device_code=self.em.code, phi=phi)))


def _seed(name):
    return zlib.crc32(name.encode()) % 1000


def _st(solver, dt0):
    return {"solver": solver, "dt0": dt0}, o.SolverSettings(solver, dt0)


def _check_filter(f, r, tag, ll_tol=TOL, moments=True):
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record(f"{tag}:marginal_loglik", e)
    assert e < ll_tol, (tag, e)
    if moments:
        check_moments(f, r, tag)


def _check_sampled(f, r, tag, fields=tuple(FIELDS), tol=1e-8):
    if "marginal_loglik" in r and getattr(f, "marginal_loglik", None) is not None:
        e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
        record(f"{tag}:marginal_loglik", e)
        assert e < tol, (tag, e)
    for fld in fields:
        e = scaled_err(getattr(f, fld), r[fld])
        record(f"{tag}:{fld}", e)
        assert e < tol, (tag, fld, e)


# ---- EKF / EKS ------------------------------------------------------------------------------------------------------------
EKF_CASES = [
    # name: (drift, n, m, emission, order, num_iter, solver, dt0, eks)
    ("vdp_first", ("vdp", 2, 2, "range", "first", 1, "rk4", 0.0125, True)),        # first-order linearisation + EKS
    ("vdp_second", ("vdp", 2, 2, "range", "second", 1, "rk4", 0.0125, True)),      # second-order predict + EKS
    ("vdp_zeroth", ("vdp", 2, 2, "range", "zeroth", 1, "rk4", 0.0125, False)),     # zeroth-order predict
    ("vdp_iter3", ("vdp", 2, 2, "range", "first", 3, "rk4", 0.0125, False)),       # condition_on iterated 3 times
    ("linear_m1", ("linear", 3, 1, "range", "first", 1, "rk4", 0.01, False)),      # m = 1
    ("vdp_m9", ("vdp", 2, 9, "range", "first", 1, "rk4", 0.0125, True)),           # m > n (9 beacons, n = 2)
    ("l96_n6_m40", ("lorenz96", 6, 40, "range", "first", 1, "rk4", 0.005, False)),  # m > 32: chol_warp over > 1 warp
    ("l96_n40_m20_dopri5", ("lorenz96", 40, 20, "range", "first", 1, "dopri5", 0.01, False)),  # nslots > 1 layout
    ("l96_n6_wide_second", ("lorenz96", 6, 6, "wide", "second", 1, "rk4", 0.005, True)),  # n_phi >> m (n + 1) + EKS
    ("l63_wide_iter3", ("lorenz63", 3, 2, "wide", "first", 3, "rk4", 0.0025, False)),  # PHI past [H | d], iterated
    ("zero_square", ("zero", 2, 3, "square", "first", 1, "rk4", 0.0125, True)),    # n_phi = 0 and n_theta = 0 (NULL H, F)
]


@pytest.mark.parametrize("name,spec", EKF_CASES, ids=[c[0] for c in EKF_CASES])
def test_ekf_eks_matrix(name, spec):
    drift, n, m, emission, order, num_iter, solver, dt0, eks = spec
    small = n >= 40 or m >= 40
    c = Case(drift, n, m, emission, N=2 if small else 4, K=6 if small else 20, seed=_seed(name),
             gap=0.01 if drift in ("lorenz63", "lorenz96") else 0.02)
    cd = api()
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm import extended_kalman_filter
    st, ost = _st(solver, dt0)
    hp = cd.EKFHyperParams(state_order=order, dt_final=0.02, diffeqsolve_settings=st)
    f = extended_kalman_filter(c.p, c.y, c.t[..., None], hp, num_iter=num_iter)
    r = uo.extended_kalman_filter(c.po, c.em, c.y, c.t, dt_final=0.02, state_order=order, settings=ost, num_iter=num_iter)
    _check_filter(f, r, f"ue_matrix_ekf_{name}")
    if eks:
        s = cd.cdnlgssm_smoother(c.p, c.y, c.t[..., None], hp)
        rs = uo.extended_kalman_smoother(c.po, c.em, c.y, c.t, dt_final=0.02, state_order=order, settings=ost)
        _check_sampled(s, rs, f"ue_matrix_eks_{name}", fields=("smoothed_means", "smoothed_covariances"))


# ---- UKF --------------------------------------------------------------------------------------------------------------------
UKF_CASES = [
    # name: (drift, n, m, emission, solver, dt0, sigma_points)
    ("l63_rk4", ("lorenz63", 3, 2, "range", "rk4", 0.0025, False)),          # closed form, stencil compact layout
    ("l63_dopri5", ("lorenz63", 3, 2, "range", "dopri5", 0.01, False)),      # closed form, nslots > 1
    ("l96_n8_rk4", ("lorenz96", 8, 4, "range", "rk4", 0.005, False)),         # closed form, Lorenz-96 compact layout
    ("l96_n8_dopri5", ("lorenz96", 8, 4, "range", "dopri5", 0.01, False)),    # closed form, Lorenz-96 Dopri5
    ("l63_sigma", ("lorenz63", 3, 2, "range", "rk4", 0.0025, True)),          # literal sigma points, registry drift
    ("l96_n8_sigma_dopri5", ("lorenz96", 8, 4, "range", "dopri5", 0.01, True)),  # sigma points, general layout
    ("vdp_m9", ("vdp", 2, 9, "range", "rk4", 0.0125, False)),                 # m > n: general layout
    ("l96_n6_m40", ("lorenz96", 6, 40, "range", "rk4", 0.005, False)),         # m = 40 > 32
    ("l96_n40_m20_wide", ("lorenz96", 40, 20, "wide", "rk4", 0.005, False)),   # n_phi = 1,484 at the config-4 shape
    ("zero_square", ("zero", 2, 3, "square", "rk4", 0.0125, False)),           # n_phi = 0, n_theta = 0
]


@pytest.mark.parametrize("name,spec", UKF_CASES, ids=[c[0] for c in UKF_CASES])
def test_ukf_matrix(name, spec, monkeypatch):
    drift, n, m, emission, solver, dt0, sigma = spec
    if sigma:
        monkeypatch.setenv("CDK_UKF_SIGMA_POINTS", "1")
    small = n >= 40 or m >= 40
    c = Case(drift, n, m, emission, N=2 if small else 4, K=6 if small else 20, seed=_seed(name),
             gap=0.01 if drift in ("lorenz63", "lorenz96") else 0.02)
    cd = api()
    st, ost = _st(solver, dt0)
    f = cd.cdnlgssm_filter(c.p, c.y, c.t[..., None], cd.UKFHyperParams(diffeqsolve_settings=st))
    r = uo.unscented_kalman_filter(c.po, c.em, c.y, c.t, settings=ost)
    _check_filter(f, r, f"ue_matrix_ukf_{name}")


def _ukf_user_smem_bytes(n):
    """Shared memory of the closed-form UKF (Lorenz-96, chain tableau, m = n, range emission) in fp64: the Lay of
    csrc/cdk_generic.cu for that branch, every region padded to an even element count."""
    ev = lambda x: (x + 1) & ~1
    ldn = n | 1
    nn = n * ldn
    S = ((n + 1) & ~1) + nn
    # TH | LQL H R P SM SL | DV BV YV MU C0 | YS ACC KS | RV | PHI = [m n + 1] | YP = [(2n + 1) x ldm]
    return 8 * (ev(1) + 6 * ev(nn) + 5 * ev(n) + 3 * ev(S) + ev(2 * n) + ev(n * n + 1) + ev((2 * n + 1) * ldn))


def test_ukf_largest_user_emission_size_and_one_beyond():
    """The largest n (m = n) whose closed-form UKF working set with the range emission fits one CTA's 227 KB runs against
    the oracle; n + 1 raises CDK_E_SIZE with the size message."""
    from cd_dynamax_b200 import _lib as L
    limit = 227 * 1024
    n = max(k for k in range(8, 64) if _ukf_user_smem_bytes(k) <= limit)
    assert _ukf_user_smem_bytes(n + 1) > limit
    cd = api()
    st, ost = _st("rk4", 0.005)
    c = Case("lorenz96", n, n, "range", N=2, K=3, seed=17, gap=0.01)
    f = cd.cdnlgssm_filter(c.p, c.y, c.t[..., None], cd.UKFHyperParams(diffeqsolve_settings=st))
    r = uo.unscented_kalman_filter(c.po, c.em, c.y, c.t, settings=ost)
    _check_filter(f, r, f"ue_matrix_ukf_largest_n{n}")
    c1 = Case("lorenz96", n + 1, n + 1, "range", N=2, K=3, seed=17, gap=0.01)
    with pytest.raises(L.CdkError, match="exceeds the 227 KB of one CTA"):
        cd.cdnlgssm_filter(c1.p, c1.y, c1.t[..., None], cd.UKFHyperParams(diffeqsolve_settings=st))


# ---- EnKF -------------------------------------------------------------------------------------------------------------------
ENKF_CASES = [
    # name: (drift, n, m, emission, E, cluster, solver, perturb)
    *[(f"l63_E37_C{C}", ("lorenz63", 3, 2, "range", 37, C, "euler", True)) for C in (1, 2, 4, 8)],  # C * Eloc != E
    ("l63_E1000_C8", ("lorenz63", 3, 2, "range", 1000, 8, "euler", True)),   # 125 members per CTA, padded to 128
    ("l63_E10_C8", ("lorenz63", 3, 2, "range", 10, 8, "heun", True)),        # CTAs 3..7 own no member
    ("l96_n40_E37", ("lorenz96", 40, 20, "range", 37, 0, "euler", True)),    # NX = 40 kernel, ragged
    ("vdp_heun_noperturb", ("vdp", 2, 2, "range", 37, 0, "heun", False)),    # runtime-n kernel, perturb_measurements=False
    ("linear_n5_wide", ("linear", 5, 3, "wide", 37, 2, "heun", True)),       # runtime-n kernel, n_phi >> m (n + 1)
    ("l63_wide_E37_C4", ("lorenz63", 3, 2, "wide", 37, 4, "euler", False)),  # NX = 3 kernel with the wide phi
    ("zero_square", ("zero", 2, 3, "square", 37, 4, "euler", True)),         # n_phi = 0, n_theta = 0
]


@pytest.mark.parametrize("name,spec", ENKF_CASES, ids=[c[0] for c in ENKF_CASES])
def test_enkf_matrix(name, spec, monkeypatch):
    drift, n, m, emission, E, C, solver, perturb = spec
    if C:
        monkeypatch.setenv("CDK_ENKF_CLUSTER", str(C))
    big = n >= 40 or E >= 1000
    c = Case(drift, n, m, emission, N=2 if big else 4, K=6 if big else 15, seed=_seed(name),
             gap=0.01 if drift in ("lorenz63", "lorenz96") else 0.02)
    cd = api()
    dt0 = 0.0025 if drift in ("lorenz63", "lorenz96") else 0.0125
    hp = cd.EnKFHyperParams(N_particles=E, key=4, perturb_measurements=perturb,
                            diffeqsolve_settings={"solver": solver, "dt0": dt0})
    f = cd.cdnlgssm_filter(c.p, c.y, c.t[..., None], hp)
    r = uo.ensemble_kalman_filter(c.po, c.em, c.y, c.t, E=E, seed=4, perturb_measurements=perturb,
                                  settings=o.SolverSettings(solver, dt0))
    _check_sampled(f, r, f"ue_matrix_enkf_{name}")


def test_enkf_user_emission_block_too_large_for_a_cluster():
    """E = 65,536 members of Lorenz-63 with m = 8: the [m x ldE] block of the members' emissions does not fit an 8-CTA
    cluster; the launcher says so in the user-emission wording."""
    from cd_dynamax_b200 import _lib as L
    cd = api()
    c = Case("lorenz63", 3, 8, "range", N=1, K=2, seed=3, gap=0.01)
    hp = cd.EnKFHyperParams(N_particles=65536, key=1, diffeqsolve_settings={"solver": "euler", "dt0": 0.0025})
    with pytest.raises(L.CdkError, match="user-emission outputs and the model do not fit the shared memory of an 8-CTA"):
        cd.cdnlgssm_filter(c.p, c.y, c.t[..., None], hp)


# ---- path sampler and point-estimate forecast -------------------------------------------------------------------------------
SAMPLER_CASES = [
    ("l63_euler", ("lorenz63", 3, 2, "range", "euler", 0.0025)),  # NX = 3 instantiation, Euler-Maruyama
    ("l63_heun", ("lorenz63", 3, 2, "range", "heun", 0.0025)),    # NX = 3 instantiation, Heun
    ("vdp_euler", ("vdp", 2, 2, "range", "euler", 0.0125)),       # runtime-n, Euler-Maruyama
    ("vdp_heun", ("vdp", 2, 2, "range", "heun", 0.0125)),         # runtime-n, Heun
    ("l96_n8_wide", ("lorenz96", 8, 5, "wide", "heun", 0.005)),   # SLay.H sized by n_phi
    ("zero_square", ("zero", 2, 3, "square", "heun", 0.0125)),    # n_phi = 0, n_theta = 0
]


@pytest.mark.parametrize("name,spec", SAMPLER_CASES, ids=[c[0] for c in SAMPLER_CASES])
def test_sampler_matrix(name, spec):
    drift, n, m, emission, solver, dt0 = spec
    c = Case(drift, n, m, emission, N=5, K=20, seed=_seed(name), gap=0.02)
    cd = api()
    xs, ys = cd.cdnlgssm_path_sample(c.p, 11, c.K, c.t[..., None], diffeqsolve_settings={"solver": solver, "dt0": dt0})
    rx, ry = uo.sample_paths(c.po, c.em, c.t, seed=11, settings=o.SolverSettings(solver, dt0))
    ex, ey = scaled_err(xs, rx), scaled_err(ys, ry)
    record(f"ue_matrix_sampler_{name}:states", ex)
    record(f"ue_matrix_sampler_{name}:emissions", ey)
    assert ex < 1e-8 and ey < 1e-8, (ex, ey)


@pytest.mark.parametrize("drift", ["lorenz63", "vdp"])
def test_forecast_from_a_point_estimate(drift):
    """cdnlgssm_forecast of an array: one sample path from that state (CDK_FLAG_FIXED_INIT), emissions through h."""
    c = Case(drift, 3 if drift == "lorenz63" else 2, 2, "range", N=4, K=12, seed=21, gap=0.02)
    cd = api()
    x0 = c.po.m0[None] + np.random.default_rng(2).standard_normal((c.N, c.n))
    dt0 = 0.0025 if drift == "lorenz63" else 0.0125
    fc = cd.cdnlgssm_forecast(c.p, x0, 0.3, c.t[..., None] + 0.3, key=5, diffeqsolve_settings={"solver": "heun", "dt0": dt0})
    T = np.concatenate([np.full((c.N, 1), 0.3), c.t + 0.3], axis=1)
    rx, ry = uo.sample_paths(dataclasses.replace(c.po, m0=x0), c.em, T, seed=5, settings=o.SolverSettings("heun", dt0), fixed_init=True)
    ex, ey = scaled_err(fc.forecasted_state_path, rx), scaled_err(fc.forecasted_emission_path, ry)
    record(f"ue_matrix_forecast_{drift}:states", ex)
    record(f"ue_matrix_forecast_{drift}:emissions", ey)
    assert ex < 1e-8 and ey < 1e-8, (ex, ey)


def test_sampler_refuses_a_per_trajectory_phi():
    from cd_dynamax_b200 import _lib as L
    c = Case("lorenz63", 3, 2, "range", N=3, K=5, seed=1)
    cd = api()
    p = c.with_phi(np.stack([c.phi] * 3))
    with pytest.raises(L.CdkError, match="cdk_sample_path"):
        cd.cdnlgssm_path_sample(p, 1, c.K, c.t[..., None], diffeqsolve_settings={"solver": "heun", "dt0": 0.0025})


# ---- fp32 -------------------------------------------------------------------------------------------------------------------
def _f32_case(c):
    y32, t32 = c.y.astype(np.float32), c.t.astype(np.float32)
    return y32, t32, t32.astype(np.float64)


def test_fp32_ukf_eks_enkf_sampler():
    """The fp32 instantiations with a user emission against the fp64 oracle on the fp32-rounded data, stepping on fp32
    times.  Bounds (tests/test_gpu_baseline_shapes.py): UKF 5e-4 relative on the log-likelihood and 5e-3 scaled on the
    moments; EKF / EKS 2e-4 and 2e-3; EnKF (linear drift: no chaotic amplification of the fp32 deviates) 1e-3 and 2e-3;
    sampled paths 2e-3 scaled (the EKS bound: one fp32 rounding per substep along a path of a non-chaotic drift)."""
    cd = api()
    tdt = dict(time_dtype=np.float32)
    # UKF: Lorenz-63 closed form with the range emission
    c = Case("lorenz63", 3, 2, "range", N=4, K=30, seed=31, gap=0.01)
    y32, t32, t64 = _f32_case(c)
    f = cd.cdnlgssm_filter(c.p, y32, t32[..., None], cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025}))
    assert f.filtered_means.dtype == np.float32
    r = uo.unscented_kalman_filter(c.po, c.em, y32, t64, settings=o.SolverSettings("rk4", float(np.float32(0.0025)), **tdt))
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record("ue_matrix_fp32_ukf:marginal_loglik", e)
    assert e < 5e-4
    for fld in FIELDS:
        e = scaled_err(getattr(f, fld), r[fld])
        record(f"ue_matrix_fp32_ukf:{fld}", e)
        assert e < 5e-3, (fld, e)
    # EKF + EKS: VdP user drift with the range emission
    c = Case("vdp", 2, 2, "range", N=4, K=30, seed=32)
    y32, t32, t64 = _f32_case(c)
    hp = cd.EKFHyperParams(state_order="first", diffeqsolve_settings={"solver": "rk4", "dt0": 0.0125})
    s = cd.cdnlgssm_smoother(c.p, y32, t32[..., None], hp)
    assert s.smoothed_means.dtype == np.float32
    ost = o.SolverSettings("rk4", float(np.float32(0.0125)), **tdt)
    rs = uo.extended_kalman_smoother(c.po, c.em, y32, t64, state_order="first", settings=ost)
    e = max_rel_err(s.marginal_loglik, rs["marginal_loglik"])
    record("ue_matrix_fp32_eks:marginal_loglik", e)
    assert e < 2e-4
    for fld in ("smoothed_means", "smoothed_covariances"):
        e = scaled_err(getattr(s, fld), rs[fld])
        record(f"ue_matrix_fp32_eks:{fld}", e)
        assert e < 2e-3, (fld, e)
    # EnKF: linear drift, wide emission (the runtime-n kernel)
    c = Case("linear", 4, 3, "wide", N=4, K=30, seed=33)
    y32, t32, t64 = _f32_case(c)
    hp = cd.EnKFHyperParams(N_particles=128, key=7, diffeqsolve_settings={"solver": "euler", "dt0": 0.0125})
    f = cd.cdnlgssm_filter(c.p, y32, t32[..., None], hp)
    assert f.filtered_means.dtype == np.float32
    r = uo.ensemble_kalman_filter(c.po, c.em, y32, t64, E=128, seed=7,
                                  settings=o.SolverSettings("euler", float(np.float32(0.0125)), **tdt))
    e = max_rel_err(f.marginal_loglik, r["marginal_loglik"])
    record("ue_matrix_fp32_enkf:marginal_loglik", e)
    assert e < 1e-3
    for fld in FIELDS:
        e = scaled_err(getattr(f, fld), r[fld])
        record(f"ue_matrix_fp32_enkf:{fld}", e)
        assert e < 2e-3, (fld, e)
    # sampler: VdP with the range emission
    c = Case("vdp", 2, 2, "range", N=4, K=30, seed=34)
    _, t32, t64 = _f32_case(c)
    xs, ys = cd.cdnlgssm_path_sample(c.p, 3, c.K, t32[..., None], diffeqsolve_settings={"solver": "heun", "dt0": 0.0125})
    assert xs.dtype == np.float32
    rx, ry = uo.sample_paths(c.po, c.em, t64, seed=3, settings=o.SolverSettings("heun", float(np.float32(0.0125)), **tdt))
    ex, ey = scaled_err(xs, rx), scaled_err(ys, ry)
    record("ue_matrix_fp32_sampler:states", ex)
    record("ue_matrix_fp32_sampler:emissions", ey)
    assert ex < 2e-3 and ey < 2e-3, (ex, ey)


# ---- invariances (per-trajectory phi, bit for bit) --------------------------------------------------------------------------
def _hps(cd):
    return {"ekf": cd.EKFHyperParams(state_order="first", diffeqsolve_settings={"solver": "rk4", "dt0": 0.0125}),
            "ukf": cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0125}),
            "enkf": cd.EnKFHyperParams(N_particles=37, key=9, diffeqsolve_settings={"solver": "heun", "dt0": 0.0125})}


def _same(a, b, tag):
    for fld in ["marginal_loglik"] + FIELDS:
        x, y = getattr(a, fld), getattr(b, fld)
        x = x.cpu().numpy() if hasattr(x, "cpu") else x
        y = y.cpu().numpy() if hasattr(y, "cpu") else y
        assert np.array_equal(x, y, equal_nan=True), (tag, fld)


def test_batch_equals_shards_and_permutation():
    """Per-trajectory phi: the batch equals its two shards and a permuted batch, bit for bit (EKF and UKF: the EnKF's
    deviates follow the trajectory index, so a shard or a permutation draws other ones)."""
    cd = api()
    N = 8
    c = Case("vdp", 2, 2, "range", N=N, K=15, seed=41)
    rng = np.random.default_rng(42)
    phis = c.phi + 0.2 * rng.standard_normal((N, c.phi.size))
    perm = rng.permutation(N)
    for kind in ("ekf", "ukf"):
        hp = _hps(cd)[kind]
        full = cd.cdnlgssm_filter(c.with_phi(phis), c.y, c.t[..., None], hp)
        pm = cd.cdnlgssm_filter(c.with_phi(phis[perm]), c.y[perm], c.t[perm][..., None], hp)
        for fld in ["marginal_loglik"] + FIELDS:
            assert np.array_equal(getattr(pm, fld), getattr(full, fld)[perm]), (kind, fld)
        for lo, hi in ((0, 3), (3, N)):
            sh = cd.cdnlgssm_filter(c.with_phi(phis[lo:hi]), c.y[lo:hi], c.t[lo:hi][..., None], hp)
            for fld in ["marginal_loglik"] + FIELDS:
                assert np.array_equal(getattr(sh, fld), getattr(full, fld)[lo:hi]), (kind, fld, lo)


def test_host_batch_staged_in_chunks_equals_one_launch(monkeypatch):
    """A host-resident [N, n_phi] phi staged in N-chunks: every chunk offsets the phi pointer by lo * n_phi (n_phi = m n + 1
    for the range emission) and gives the single launch bit for bit.  N = 24 >= 2 * STREAM_CHUNKS, so it does chunk."""
    from cd_dynamax_b200 import _engine
    cd = api()
    N = 24
    assert N >= 2 * _engine.STREAM_CHUNKS
    c = Case("lorenz63", 3, 2, "range", N=N, K=10, seed=43, gap=0.01)
    phis = c.phi + 0.3 * np.random.default_rng(44).standard_normal((N, c.phi.size))
    hps = _hps(cd)
    hps["ekf"] = cd.EKFHyperParams(state_order="first", diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    hps["ukf"] = cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025})
    for kind, hp in hps.items():
        monkeypatch.setattr(_engine, "STREAM_MIN_BYTES", 1 << 60)
        once = cd.cdnlgssm_filter(c.with_phi(phis), c.y, c.t[..., None], hp)
        monkeypatch.setattr(_engine, "STREAM_MIN_BYTES", 0)
        chunked = cd.cdnlgssm_filter(c.with_phi(phis), c.y, c.t[..., None], hp)
        _same(chunked, once, f"chunked_{kind}")


def test_loglik_only_and_leading_axis_of_one():
    """output_fields=[] returns the same log-likelihood bits as the all-outputs call, a partial list the same moments, and
    phi with a leading axis of 1 is the shared call."""
    cd = api()
    c = Case("vdp", 2, 2, "range", N=4, K=15, seed=45)
    for kind, hp in _hps(cd).items():
        full = cd.cdnlgssm_filter(c.p, c.y, c.t[..., None], hp)
        ll = cd.cdnlgssm_filter(c.p, c.y, c.t[..., None], hp, output_fields=[])
        assert ll.filtered_means is None and np.array_equal(ll.marginal_loglik, full.marginal_loglik), kind
        part = cd.cdnlgssm_filter(c.p, c.y, c.t[..., None], hp, output_fields=["predicted_covariances"])
        assert part.filtered_means is None and np.array_equal(part.predicted_covariances, full.predicted_covariances)
        assert np.array_equal(part.marginal_loglik, full.marginal_loglik), kind
        lead1 = cd.cdnlgssm_filter(c.with_phi(c.phi[None]), c.y, c.t[..., None], hp)
        _same(lead1, full, f"lead1_{kind}")


# ---- status -----------------------------------------------------------------------------------------------------------------
def test_non_finite_emission_sets_status_1_on_its_row_only():
    """Row 2's range emission gets eps = -1e6, so h = sqrt(negative) = NaN inside valid memory: that row gets status 1 and
    NaN outputs; every other row equals the run without it bit for bit."""
    from cd_dynamax_b200 import _engine
    cd = api()
    N = 5
    c = Case("vdp", 2, 2, "range", N=N, K=12, seed=47)
    good = np.stack([c.phi] * N)
    bad = good.copy()
    bad[2, -1] = -1e6
    keep = [i for i in range(N) if i != 2]
    for kind, hp in _hps(cd).items():
        ref = cd.cdnlgssm_filter(c.with_phi(good), c.y, c.t[..., None], hp)
        assert np.all(np.asarray(_engine.last_status()) == 0), kind
        f = cd.cdnlgssm_filter(c.with_phi(bad), c.y, c.t[..., None], hp)
        st = np.asarray(_engine.last_status())
        assert st[2] == 1 and np.all(st[keep] == 0), (kind, st)
        assert np.isnan(f.marginal_loglik[2]) and np.isnan(f.filtered_means[2, -1]).all(), kind
        for fld in ["marginal_loglik"] + FIELDS:
            assert np.array_equal(getattr(f, fld)[keep], getattr(ref, fld)[keep]), (kind, fld)


def test_tiny_max_steps_raises():
    from cd_dynamax_b200 import _engine
    cd = api()
    c = Case("vdp", 2, 2, "range", N=3, K=8, seed=48)
    with pytest.raises(_engine.MaxStepsReached):
        cd.cdnlgssm_filter(c.p, c.y, c.t[..., None],
                           cd.EKFHyperParams(state_order="first", diffeqsolve_settings={"solver": "rk4", "dt0": 1e-4,
                                                                                        "max_steps": 3}))


# ---- edge time grids --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", ["degenerate:dt_final=1e-10", "edge:rk4"])
@pytest.mark.parametrize("algo", ["ekf", "ukf", "enkf"])
def test_edge_time_grids(grid, algo):
    """The repeated-stamp / sub-tolerance-gap grid and the rounding-edge grid of tests/test_gpu_time_grids.py with the
    range emission (the first 8 rows: every repeated-stamp and edge pattern of the builders)."""
    from tests.test_gpu_time_grids import GRIDS
    t_all, solver, dt0, dt_final = GRIDS[grid]
    t = t_all[:8]
    cd = api()
    c = Case("vdp", 2, 2, "range", N=t.shape[0], K=t.shape[1], seed=51)
    c.t = t
    if algo == "ekf":
        hp = cd.EKFHyperParams(state_order="first", dt_final=dt_final, diffeqsolve_settings={"solver": solver, "dt0": dt0})
        r = uo.extended_kalman_filter(c.po, c.em, c.y, t, dt_final=dt_final, state_order="first",
                                      settings=o.SolverSettings(solver, dt0))
    elif algo == "ukf":
        hp = cd.UKFHyperParams(dt_final=dt_final, diffeqsolve_settings={"solver": solver, "dt0": dt0})
        r = uo.unscented_kalman_filter(c.po, c.em, c.y, t, dt_final=dt_final, settings=o.SolverSettings(solver, dt0))
    else:
        hp = cd.EnKFHyperParams(N_particles=37, key=2, dt_final=dt_final, diffeqsolve_settings={"solver": "heun", "dt0": dt0})
        r = uo.ensemble_kalman_filter(c.po, c.em, c.y, t, dt_final=dt_final, E=37, seed=2,
                                      settings=o.SolverSettings("heun", dt0))
    f = cd.cdnlgssm_filter(c.p, c.y, t[..., None], hp)
    if algo == "enkf":
        _check_sampled(f, r, f"ue_matrix_grid_{grid}_{algo}")
    else:
        _check_filter(f, r, f"ue_matrix_grid_{grid}_{algo}")
