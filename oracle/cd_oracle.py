"""CPU oracle (NumPy, fp64 or fp32) for the cd-dynamax continuous-discrete filtering hot path.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s CPU-baseline legs may import it.  The product path (``cd_dynamax_b200``) never does.

PARITY STATUS: **parity unpinned at rel 1e-9 against real JAX/diffrax** -- jax 0.4.13, diffrax 0.4.0 and
tensorflow-probability 0.20.1 (pinned in ``hduq_cd_dynamax_requirements.txt:21,40-41,117``) are not installable
in this image, so the arithmetic that lives inside them is *restated* here from their published algorithms:

* diffrax 0.4.0 ``diffeqsolve`` with ``ConstantStepSize`` (call site ``src/utils/diffrax_utils.py:150-163``):
  fixed-step explicit Runge-Kutta, ``tnext = tprev + dt0`` accumulated in floating point, last step clipped to
  ``t1`` when ``tnext > t1 - tol`` (tol = 1e-10 for float64 times, 1e-6 for float32), loop ``while tprev < t1``,
  stage increments ``k_i = dt * f(t_i, y_i)``; Dopri5 propagates the 5th-order solution.
* TFP ``MultivariateNormalFullCovariance(mu, S).log_prob(y)``:
  ``-0.5*||L^-1 (y-mu)||^2 - sum(log L_ii) - 0.5*m*log(2*pi)`` with ``L = chol(S)`` (no jitter).
* ``jax.scipy.linalg.cho_factor/cho_solve`` and ``jnp.linalg.cholesky``: plain Cholesky, NaN on non-PD input.
* ``jax.jacfwd`` / ``jacfwd(jacrev(f))``: analytic Jacobians / Hessian contractions of the registry drifts.

What IS pinned: the reference's own orchestration files are executed verbatim (on NumPy shims of the absent
third-party packages) by ``tests/golden/make_golden.py`` and this oracle is checked against those vectors, against
the two golden constants the reference hard-codes (``src/test_scripts/cdlgssm_test_filter_TRegular.py:61-62``) and
against closed forms (matrix exponential / Van Loan, discrete Kalman filter, joint-Gaussian smoother).

Every function is batched over a leading trajectory axis N -- the axis ``jax.vmap`` adds in the reference
(``src/ssm_temissions.py:555-567``).  Under vmap the diffrax while-loop runs to the maximum trip count over the batch
with masked selects; ``rk_solve`` does the same.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence, Tuple

import numpy as np

# --------------------------------------------------------------------------------------------------------------------
# Explicit Runge-Kutta tableaux (diffrax 0.4.0 solver names; "rk4" is the classical tableau named by the north star,
# diffrax has no such solver -- SURVEY.md F4).
# --------------------------------------------------------------------------------------------------------------------
TABLEAUX = {
    "euler": dict(a=[[]], b=[1.0]),
    "heun": dict(a=[[], [1.0]], b=[0.5, 0.5]),
    "midpoint": dict(a=[[], [0.5]], b=[0.0, 1.0]),
    "ralston": dict(a=[[], [0.75]], b=[1.0 / 3.0, 2.0 / 3.0]),
    "bosh3": dict(a=[[], [0.5], [0.0, 0.75]], b=[2.0 / 9.0, 1.0 / 3.0, 4.0 / 9.0]),
    "rk4": dict(a=[[], [0.5], [0.0, 0.5], [0.0, 0.0, 1.0]], b=[1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0]),
    "dopri5": dict(
        a=[
            [],
            [1.0 / 5.0],
            [3.0 / 40.0, 9.0 / 40.0],
            [44.0 / 45.0, -56.0 / 15.0, 32.0 / 9.0],
            [19372.0 / 6561.0, -25360.0 / 2187.0, 64448.0 / 6561.0, -212.0 / 729.0],
            [9017.0 / 3168.0, -355.0 / 33.0, 46732.0 / 5247.0, 49.0 / 176.0, -5103.0 / 18656.0],
        ],
        # 5th-order weights; the 7th (FSAL) stage has weight 0 and is never needed under constant steps.
        b=[35.0 / 384.0, 0.0, 500.0 / 1113.0, 125.0 / 192.0, -2187.0 / 6784.0, 11.0 / 84.0],
    ),
}
SOLVER_IDS = {"euler": 0, "heun": 1, "midpoint": 2, "ralston": 3, "bosh3": 4, "rk4": 5, "dopri5": 6}


@dataclass
class SolverSettings:
    """The subset of ``diffeqsolve_settings`` (``diffrax_utils.py:40-57``) that the hot path supports."""

    solver: str = "dopri5"  # reference default for ODEs (diffrax_utils.py:121-124)
    dt0: float = 0.01  # diffrax_utils.py:50
    max_steps: int = 100000  # diffrax_utils.py:52
    # dtype of the stepping (times, dt0, clip tolerance); None = the dtype of the state.  np.float32 with an fp64 state
    # takes exactly the substeps an fp32 run takes (fp32 times, tol 1e-6) with fp64 arithmetic, so that a comparison
    # with the fp32 kernels measures arithmetic precision alone.
    time_dtype: Optional[type] = None


def _stepping(settings: SolverSettings, dtype):
    """(time dtype, dt0, tol) of the diffrax stepping rule for a state of `dtype`."""
    tdt = np.dtype(settings.time_dtype if settings.time_dtype is not None else dtype)
    return tdt, tdt.type(settings.dt0), tdt.type(_tol_for(tdt))


def _tol_for(dtype) -> float:
    return 1e-10 if np.dtype(dtype) == np.float64 else 1e-6


def substep_counts(t0, t1, dt0, dtype=np.float64):
    """Number of solver steps diffrax takes per gap (batched, any shape)."""
    t0 = np.asarray(t0, dtype)
    t1 = np.asarray(t1, dtype)
    dt0 = dtype(dt0) if not isinstance(dtype, np.dtype) else dtype.type(dt0)
    tol = t0.dtype.type(_tol_for(t0.dtype))
    tprev = t0.copy()
    tnext = np.minimum(t0 + dt0, t1)
    q = np.zeros(t0.shape, np.int64)
    while True:
        active = tprev < t1
        if not active.any():
            return q
        q += active
        tprev = np.where(active, tnext, tprev)
        cand = tprev + dt0
        tnext = np.where(cand > t1 - tol, t1, cand)


def rk_solve(rhs: Callable, t0, t1, y0: Sequence[np.ndarray], settings: SolverSettings):
    """Fixed-step explicit RK from t0 to t1 (restates diffrax ``diffeqsolve`` + ``ConstantStepSize``).

    t0, t1: [N].  y0: tuple of arrays with leading N.  rhs(t[N], y) -> tuple like y.
    Returns (y(t1) tuple, n_steps[N], hit_max_steps[N] bool).
    """
    tab = TABLEAUX[settings.solver]
    a, b = tab["a"], tab["b"]
    dtype = y0[0].dtype
    tdt, dt0, tol = _stepping(settings, dtype)
    t0 = np.asarray(t0, tdt)
    t1 = np.asarray(t1, tdt)
    y = tuple(np.array(c, dtype, copy=True) for c in y0)
    tprev = t0.copy()
    tnext = np.minimum(t0 + dt0, t1)
    nsteps = np.zeros(t0.shape, np.int64)
    hit = np.zeros(t0.shape, bool)

    def bc(v, like):  # broadcast an [N] vector against [N, ...]
        return v.reshape(v.shape + (1,) * (like.ndim - 1))

    while True:
        active = tprev < t1
        over = active & (nsteps >= settings.max_steps)
        if over.any():
            hit |= over
            active &= ~over
            tprev = np.where(over, t1, tprev)  # abandon those lanes
        if not active.any():
            break
        dt = np.where(active, tnext - tprev, tdt.type(0)).astype(dtype)
        tp = tprev.astype(dtype)
        ks = []
        for i in range(len(b)):
            yi = y
            if i > 0:
                yi = tuple(
                    c + sum(dtype.type(a[i][j]) * ks[j][ci] for j in range(i) if a[i][j] != 0.0)
                    for ci, c in enumerate(y)
                )
            ci_t = dtype.type(sum(a[i])) if i > 0 else dtype.type(0)
            fi = rhs(tp + ci_t * dt, yi)
            ks.append(tuple(bc(dt, f) * f for f in fi))
        ynew = tuple(
            c + sum(dtype.type(b[j]) * ks[j][ci] for j in range(len(b)) if b[j] != 0.0) for ci, c in enumerate(y)
        )
        y = tuple(np.where(bc(active, c), cn, c) for c, cn in zip(y, ynew))
        nsteps += active
        tprev = np.where(active, tnext, tprev)
        cand = tprev + dt0
        tnext = np.where(cand > t1 - tol, t1, cand)
    if hit.any():
        y = tuple(np.where(bc(hit, c), dtype.type(np.nan), c) for c in y)
    return y, nsteps, hit


# --------------------------------------------------------------------------------------------------------------------
# Small dense linear algebra, batched over N, NaN-propagating (no exceptions on non-PD input).
# --------------------------------------------------------------------------------------------------------------------
def symmetrize(A):
    """dynamax/utils/utils.py:209-211"""
    return A.dtype.type(0.5) * (A + np.swapaxes(A, -1, -2))


def cholesky(A):
    """Lower Cholesky factor of A[N,n,n] (reads the lower triangle); NaN where not positive definite."""
    A = np.asarray(A)
    n = A.shape[-1]
    L = np.zeros_like(A)
    with np.errstate(invalid="ignore", divide="ignore"):
        for j in range(n):
            d = A[..., j, j] - np.sum(L[..., j, :j] * L[..., j, :j], axis=-1)
            ljj = np.sqrt(d)
            L[..., j, j] = ljj
            if j + 1 < n:
                s = A[..., j + 1 :, j] - np.einsum("...ik,...k->...i", L[..., j + 1 :, :j], L[..., j, :j])
                L[..., j + 1 :, j] = s / ljj[..., None]
    return L


def cho_solve(L, B):
    """Solve (L L^T) X = B for X; L[N,n,n] lower, B[N,n,r]."""
    n = L.shape[-1]
    Y = np.zeros(np.broadcast_shapes(L.shape[:-2], B.shape[:-2]) + B.shape[-2:], dtype=np.result_type(L, B))
    with np.errstate(invalid="ignore", divide="ignore"):
        for i in range(n):
            s = B[..., i, :] - np.einsum("...k,...kr->...r", L[..., i, :i], Y[..., :i, :])
            Y[..., i, :] = s / L[..., i, i][..., None]
        X = np.zeros_like(Y)
        for i in range(n - 1, -1, -1):
            s = Y[..., i, :] - np.einsum("...k,...kr->...r", L[..., i + 1 :, i], X[..., i + 1 :, :])
            X[..., i, :] = s / L[..., i, i][..., None]
    return X


def psd_solve(A, B, diagonal_boost=1e-9):
    """dynamax/utils/utils.py:202-207: symmetrize, add 1e-9*I, Cholesky solve."""
    A = symmetrize(A) + A.dtype.type(diagonal_boost) * np.eye(A.shape[-1], dtype=A.dtype)
    return cho_solve(cholesky(A), B)


def mvn_logpdf(y, mu, S):
    """TFP MultivariateNormalFullCovariance(mu, S).log_prob(y) (call sites: cd_linear/inference.py:613,
    inference_ekf.py:286, inference_ukf.py:197, inference_enkf.py:129). Cholesky of S without jitter."""
    L = cholesky(S)
    m = S.shape[-1]
    r = (y - mu)[..., None]
    z = np.zeros_like(r)
    with np.errstate(invalid="ignore", divide="ignore"):
        for i in range(m):
            s = r[..., i, :] - np.einsum("...k,...kr->...r", L[..., i, :i], z[..., :i, :])
            z[..., i, :] = s / L[..., i, i][..., None]
        logdet_half = np.sum(np.log(np.diagonal(L, axis1=-2, axis2=-1)), axis=-1)
    dt = S.dtype.type
    return dt(-0.5) * np.sum(z[..., 0] ** 2, axis=-1) - logdet_half - dt(0.5 * m * math.log(2.0 * math.pi))


def _mT(A):
    return np.swapaxes(A, -1, -2)


def _mv(A, x):
    return np.einsum("...ij,...j->...i", A, x)


# --------------------------------------------------------------------------------------------------------------------
# Drift / emission registry (cdnlgssm_utils.py:50-83 plus Lorenz-96, which the reference lacks -- SURVEY F5).
# f, jac: batched.  grad_div(x)[k] = sum_i d2 f_i / dx_i dx_k, the only part of the Hessian the reference's
# "second order" term uses: 0.5*jnp.trace(H_t @ P) == 0.5 * einsum('iik,kl->l', H_t, P)  (inference_ekf.py:111-114).
# --------------------------------------------------------------------------------------------------------------------
def lead(v, x, core):
    """A drift parameter `v` with core rank `core`, shaped to broadcast against states x [N, ..., n]: a per-trajectory
    parameter [N, *core] becomes [N, 1, ..., 1, *core] (one 1 per axis between N and n: sigma points, ensemble members),
    a shared one is returned as is."""
    v = np.asarray(v)
    if v.ndim == core:
        return v
    return v.reshape(v.shape[:1] + (1,) * (x.ndim - 2) + v.shape[1:])


class LinearDrift:
    """LearnableLinear: f(x) = W x + bias (cdnlgssm_utils.py:50-61). W [n,n] or [N,n,n], bias [n] or [N,n]."""

    drift_id = 0

    def __init__(self, weights, bias):
        self.W = np.asarray(weights)
        self.bias = np.asarray(bias)

    def f(self, x):
        return _mv(lead(self.W, x, 2), x) + lead(self.bias, x, 1)

    def jac(self, x):
        W = lead(self.W, x, 2)
        return np.broadcast_to(W, x.shape[:-1] + W.shape[-2:])

    def grad_div(self, x):
        return np.zeros_like(x)

    def theta(self):
        W = self.W.reshape(self.W.shape[:-2] + (-1,))
        lead_shape = np.broadcast_shapes(W.shape[:-1], self.bias.shape[:-1])
        return np.concatenate([np.broadcast_to(W, lead_shape + W.shape[-1:]),
                               np.broadcast_to(self.bias, lead_shape + self.bias.shape[-1:])], axis=-1)


class Lorenz63Drift:
    """LearnableLorenz63 (cdnlgssm_utils.py:63-83). sigma/rho/beta scalars or [N]."""

    drift_id = 1

    def __init__(self, sigma=10.0, rho=28.0, beta=8.0 / 3.0):
        self.sigma, self.rho, self.beta = (np.asarray(v) for v in (sigma, rho, beta))

    def f(self, x):
        s, r, b = (lead(v, x, 0).astype(x.dtype) for v in (self.sigma, self.rho, self.beta))
        return np.stack(
            [s * (x[..., 1] - x[..., 0]), x[..., 0] * (r - x[..., 2]) - x[..., 1], x[..., 0] * x[..., 1] - b * x[..., 2]],
            axis=-1,
        )

    def jac(self, x):
        s, r, b = (lead(v, x, 0).astype(x.dtype) for v in (self.sigma, self.rho, self.beta))
        J = np.zeros(x.shape + (3,), x.dtype)
        J[..., 0, 0] = -s
        J[..., 0, 1] = s
        J[..., 1, 0] = r - x[..., 2]
        J[..., 1, 1] = -1.0
        J[..., 1, 2] = -x[..., 0]
        J[..., 2, 0] = x[..., 1]
        J[..., 2, 1] = x[..., 0]
        J[..., 2, 2] = -b
        return J

    def grad_div(self, x):
        return np.zeros_like(x)

    def theta(self):
        return np.stack(np.broadcast_arrays(self.sigma, self.rho, self.beta), axis=-1).astype(np.float64)


class Lorenz96Drift:
    """dx_i = (x_{i+1} - x_{i-2}) x_{i-1} - x_i + F, cyclic (BASELINE configs 4-5; not in the reference)."""

    drift_id = 2

    def __init__(self, forcing=8.0):
        self.F = np.asarray(forcing)

    def f(self, x):
        xp1, xm1, xm2 = np.roll(x, -1, -1), np.roll(x, 1, -1), np.roll(x, 2, -1)
        F = lead(self.F, x, 0).astype(x.dtype)  # a scalar, or [N] forcings
        return (xp1 - xm2) * xm1 - x + (F[..., None] if F.ndim else F)

    def jac(self, x):
        n = x.shape[-1]
        J = np.zeros(x.shape + (n,), x.dtype)
        idx = np.arange(n)
        xp1, xm1, xm2 = np.roll(x, -1, -1), np.roll(x, 1, -1), np.roll(x, 2, -1)
        # accumulate (n < 4 makes index sets collide, so use +=)
        np.add.at(J, (..., idx, (idx + 1) % n), xm1)
        np.add.at(J, (..., idx, (idx - 2) % n), -xm1)
        np.add.at(J, (..., idx, (idx - 1) % n), xp1 - xm2)
        np.add.at(J, (..., idx, idx), -np.ones_like(x))
        return J

    def grad_div(self, x):
        return np.zeros_like(x)

    def theta(self):
        return np.asarray(self.F, np.float64).reshape(self.F.shape + (1,))


@dataclass
class LinearParams:
    """ParamsCDLGSSM as plain arrays (cd_linear/inference.py:57-102). Any field may carry a leading N."""

    m0: np.ndarray
    P0: np.ndarray
    F: np.ndarray
    L: np.ndarray
    Qc: np.ndarray
    H: np.ndarray
    R: np.ndarray
    b: Optional[np.ndarray] = None  # dynamics bias (added after the pushforward, :204)
    B: Optional[np.ndarray] = None  # dynamics input weights
    d: Optional[np.ndarray] = None  # emission bias
    D: Optional[np.ndarray] = None  # emission input weights


@dataclass
class NonlinearParams:
    """ParamsCDNLGSSM with registry drift and linear emission h(x) = H x + d (cdnlgssm_utils.py:191-206)."""

    m0: np.ndarray
    P0: np.ndarray
    drift: object
    L: np.ndarray
    Qc: np.ndarray
    H: np.ndarray
    R: np.ndarray
    d: Optional[np.ndarray] = None


def _gap_times(t, dt_final):
    """t[N,K] -> (t0[N,K], t1[N,K]) as cd_linear/inference.py:578-589 (last gap = dt_final)."""
    t0 = t
    t1 = np.concatenate([t[:, 1:], t[:, -1:] + t.dtype.type(dt_final)], axis=1)
    return t0, t1


def _bN(x, N, core):
    """Give x a leading N (broadcast view) when it only has `core` dims."""
    x = np.asarray(x)
    if x.ndim == core:
        return np.broadcast_to(x, (N,) + x.shape)
    assert x.ndim == core + 1 and x.shape[0] == N, (x.shape, N, core)
    return x


# --------------------------------------------------------------------------------------------------------------------
# Linear CD Kalman filter / smoother  (cd_linear/inference.py)
# --------------------------------------------------------------------------------------------------------------------
def compute_pushforward(F, LQL, t0, t1, settings: SolverSettings):
    """cd_linear/inference.py:105-144: dA = F A, dQ = F Q + Q F^T + L Qc L^T from (I, 0)."""
    N, n = F.shape[0], F.shape[-1]
    A0 = np.broadcast_to(np.eye(n, dtype=F.dtype), (N, n, n)).copy()
    Q0 = np.zeros((N, n, n), F.dtype)

    def rhs(t, y):
        A, Q = y
        return (F @ A, F @ Q + Q @ _mT(F) + LQL)

    (A, Q), nst, hit = rk_solve(rhs, t0, t1, (A0, Q0), settings)
    return A, Q, hit


def _diag(v):
    return v[..., :, None] * np.eye(v.shape[-1], dtype=v.dtype)


def _kf_condition_on(m, P, H, d, Du, R, y):
    """cd_linear/inference.py:209-259: full-R branch :237-239, diagonal-R (R.ndim == 1) Woodbury branch :240-254."""
    if R.ndim == P.ndim:  # [N, m, m]
        S = R + H @ P @ _mT(H)
        K = _mT(psd_solve(S, H @ P))
    else:  # [N, m]: Woodbury with A = diag(R), U = H chol(P), V = U^T, C = I
        n = P.shape[-1]
        I = np.eye(n, dtype=P.dtype)
        U = H @ cholesky(symmetrize(P))  # jnp.linalg.cholesky symmetrises its input
        X = U / R[..., :, None]
        S_inv = _diag(1.0 / R) - X @ psd_solve(I + _mT(U) @ X, _mT(X))
        K = P @ _mT(H) @ S_inv
        S = _diag(R) + H @ P @ _mT(H)
    Sigma = P - K @ S @ _mT(K)
    mu = m + _mv(K, y - Du - d - _mv(H, m))
    return mu, symmetrize(Sigma)


def cdlgssm_filter(p: LinearParams, y, t, dt_final=1e-10, settings=SolverSettings(), inputs=None, dtype=np.float64):
    """cd_linear/inference.py:555-632. y[N,K,m], t[N,K], inputs[N,K,d_u] or None."""
    y = np.asarray(y, dtype)
    t = np.asarray(t, dtype)
    N, K, mdim = y.shape
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    F, L, Qc, H = c(p.F, 2), c(p.L, 2), c(p.Qc, 2), c(p.H, 2)
    # a 1-D emissions.cov (diagonal R) takes the reference's Woodbury update; its log-likelihood adds the vector to
    # H P H^T by BROADCASTING (cd_linear/inference.py:613: entry (i, j) gets R[j]) and TFP's Cholesky then factors the
    # symmetrised matrix, i.e. H P H^T + (R_i + R_j) / 2 -- restated as is (it equals diag(R) only for a constant vector)
    # the diagonal is [m], or [N, m] batched over parameter samples (a 2-D emissions.cov that is not square)
    Rs = np.shape(p.R)
    diag_R = len(Rs) == 1 or (len(Rs) == 2 and Rs[0] != Rs[1])
    R = c(p.R, 1) if diag_R else c(p.R, 2)
    n = F.shape[-1]
    b = c(p.b if p.b is not None else np.zeros(n), 1)
    d = c(p.d if p.d is not None else np.zeros(mdim), 1)
    LQL = L @ Qc @ _mT(L)
    if inputs is not None:
        u = np.asarray(inputs, dtype)
        B, D = c(p.B, 2), c(p.D, 2)
    m, P = c(p.m0, 1).copy(), c(p.P0, 2).copy()
    t0s, t1s = _gap_times(t, dt_final)
    out = dict(
        filtered_means=np.zeros((N, K, n), dtype),
        filtered_covariances=np.zeros((N, K, n, n), dtype),
        predicted_means=np.zeros((N, K, n), dtype),
        predicted_covariances=np.zeros((N, K, n, n), dtype),
        marginal_loglik_cumulative=np.zeros((N, K), dtype),
    )
    ll = np.zeros(N, dtype)
    status = np.zeros(N, np.int32)
    for k in range(K):
        Du = _mv(D, u[:, k]) if inputs is not None else np.zeros((N, mdim), dtype)
        Bu = _mv(B, u[:, k]) if inputs is not None else np.zeros((N, n), dtype)
        S_ll = H @ P @ _mT(H) + (symmetrize(np.broadcast_to(R[:, None, :], (N, mdim, mdim))) if diag_R else R)
        ll = ll + mvn_logpdf(y[:, k], _mv(H, m) + Du + d, symmetrize(S_ll) if diag_R else S_ll)  # :613
        mf, Pf = _kf_condition_on(m, P, H, d, Du, R, y[:, k])  # :616
        A, Q, hit = compute_pushforward(F, LQL, t0s[:, k], t1s[:, k], settings)  # :619
        m = _mv(A, mf) + Bu + b  # :204
        P = A @ Pf @ _mT(A) + Q  # :205
        status[hit] = 2
        out["filtered_means"][:, k], out["filtered_covariances"][:, k] = mf, Pf
        out["predicted_means"][:, k], out["predicted_covariances"][:, k] = m, P
        out["marginal_loglik_cumulative"][:, k] = ll
    out["marginal_loglik"] = ll
    out["status"] = _finalize_status(status, ll)
    return out


def _finalize_status(status, ll):
    status = status.copy()
    status[(status == 0) & ~np.isfinite(ll)] = 1
    return status


def cdlgssm_smoother(
    p: LinearParams, y, t, dt_final=1e-10, settings=SolverSettings(), inputs=None, smoother_type=1, dtype=np.float64
):
    """cd_linear/inference.py:694-823 (type 1 = :746-773, type 2 = :776-794 + _smooth :636-690)."""
    filt = cdlgssm_filter(p, y, t, dt_final, settings, inputs, dtype)
    t = np.asarray(t, dtype)
    N, K = t.shape
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    F, L, Qc = c(p.F, 2), c(p.L, 2), c(p.Qc, 2)
    n = F.shape[-1]
    b = c(p.b if p.b is not None else np.zeros(n), 1)
    LQL = L @ Qc @ _mT(L)
    fm, fP = filt["filtered_means"], filt["filtered_covariances"]
    sm, sP = np.zeros_like(fm), np.zeros_like(fP)
    cross = np.zeros((N, max(K - 1, 0), n, n), dtype)
    sm[:, -1], sP[:, -1] = fm[:, -1], fP[:, -1]  # :813-814
    ms, Ps = fm[:, -1].copy(), fP[:, -1].copy()
    if inputs is not None:
        u = np.asarray(inputs, dtype)
        B = c(p.B, 2)
    for k in range(K - 2, -1, -1):
        t0, t1 = t[:, k], t[:, k + 1]
        mf, Pf = fm[:, k], fP[:, k]
        if smoother_type == 1:
            A, Q, _ = compute_pushforward(F, LQL, t0, t1, settings)  # :753
            Bu = _mv(B, u[:, k]) if inputs is not None else 0.0
            C = _mT(psd_solve(Q + A @ Pf @ _mT(A), A @ Pf))  # :760
            ms_new = mf + _mv(C, ms - _mv(A, mf) - Bu - b)  # :766
            Ps_new = Pf + C @ (Ps - A @ Pf @ _mT(A) - Q) @ _mT(C)  # :767
            cross[:, k] = C @ Ps + ms_new[:, :, None] * ms[:, None, :]  # :771
            ms, Ps = ms_new, Ps_new
        elif smoother_type == 2:
            aux = _mT(psd_solve(Pf, LQL))  # :677 (loop-invariant over the gap)
            G = F + aux

            def rhs(s, yy, mf=mf, G=G, aux=aux):
                m_s, P_s = yy
                dm = _mv(F, m_s) + _mv(aux, m_s - mf)  # :680
                dP = G @ P_s + P_s @ _mT(G) - LQL  # :682
                return (-dm, -dP)  # reverse_rhs, diffrax_utils.py:13-25

            # :688 passes NO diffeqsolve settings -> always the defaults; integrate s in [0, t1-t0] (:131-135)
            (ms, Ps), _, _ = rk_solve(rhs, np.zeros_like(t0), t1 - t0, (ms, Ps), SolverSettings(time_dtype=settings.time_dtype))
            cross[:, k] = np.nan  # :792
        else:
            raise ValueError(smoother_type)
        sm[:, k], sP[:, k] = ms, Ps
    filt.update(smoothed_means=sm, smoothed_covariances=sP, smoothed_cross_covariances=cross)
    return filt


# --------------------------------------------------------------------------------------------------------------------
# CD-EKF / EKS  (cd_nonlinear/inference_ekf.py)
# --------------------------------------------------------------------------------------------------------------------
def _ekf_predict(m, P, drift, LQL, t0, t1, state_order, settings, cov_rescaling, L, Qc):
    """inference_ekf.py:46-148."""
    if state_order == "zeroth":
        (mp,), _, hit = rk_solve(lambda t, y: (drift.f(y[0]),), t0, t1, (m,), settings)
        dt = (t1 - t0)[:, None, None]
        Ls = L * m.dtype.type(cov_rescaling)
        return mp, P + np.sqrt(dt) * (Ls @ Qc @ _mT(Ls)), hit  # :135-138

    def rhs(t, y):
        mm, PP = y
        J = drift.jac(mm)  # :95
        dm = drift.f(mm)
        if state_order == "second":
            dm = dm + mm.dtype.type(0.5) * np.einsum("...k,...kl->...l", drift.grad_div(mm), PP)  # :111-114 quirk
        elif state_order != "first":
            raise ValueError(state_order)
        return (dm, J @ PP + PP @ _mT(J) + LQL)  # :105 / :116

    (mp, Pp), _, hit = rk_solve(rhs, t0, t1, (m, P), settings)
    return mp, Pp, hit


def _ekf_condition_on(m, P, H, d, R, y, num_iter):
    """inference_ekf.py:153-199 with linear emission h(x) = H x + d (Jacobian H)."""
    for _ in range(num_iter):
        S = R + H @ P @ _mT(H)
        K = _mT(psd_solve(S, H @ P))
        P_new = P - K @ S @ _mT(K)
        m = m + _mv(K, y - (_mv(H, m) + d))
        P = P_new
    return m, symmetrize(P)


def extended_kalman_filter(
    p: NonlinearParams,
    y,
    t,
    dt_final=1e-10,
    state_order="second",
    settings=SolverSettings(),
    num_iter=1,
    cov_rescaling=1.0,
    dtype=np.float64,
    forecast=False,
):
    """inference_ekf.py:202-326. y[N,K,m], t[N,K].  forecast=True: forecast_extended_kalman_filter (:679-761) -- the same
    _predict scanned with no updates; y is ignored (only its shape [N,K,m]), t is [N,K+1] with t_init first and
    predicted_* hold the forecasted moments."""
    y = np.asarray(y, dtype)
    t = np.asarray(t, dtype)
    N, K, mdim = y.shape
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    L, Qc, H, R = c(p.L, 2), c(p.Qc, 2), c(p.H, 2), c(p.R, 2)
    n = L.shape[-1]
    d = c(p.d if p.d is not None else np.zeros(mdim), 1)
    LQL = L @ Qc @ _mT(L)
    m, P = c(p.m0, 1).copy(), c(p.P0, 2).copy()
    t0s, t1s = (t[:, :-1], t[:, 1:]) if forecast else _gap_times(t, dt_final)
    out = dict(
        filtered_means=np.zeros((N, K, n), dtype),
        filtered_covariances=np.zeros((N, K, n, n), dtype),
        predicted_means=np.zeros((N, K, n), dtype),
        predicted_covariances=np.zeros((N, K, n, n), dtype),
        marginal_loglik_cumulative=np.zeros((N, K), dtype),
    )
    ll = np.zeros(N, dtype)
    status = np.zeros(N, np.int32)
    for k in range(K):
        if forecast:
            mf, Pf = m, P
        else:
            ll = ll + mvn_logpdf(y[:, k], _mv(H, m) + d, H @ P @ _mT(H) + R)  # :285-286
            mf, Pf = _ekf_condition_on(m, P, H, d, R, y[:, k], num_iter)  # :289
        m, P, hit = _ekf_predict(mf, Pf, p.drift, LQL, t0s[:, k], t1s[:, k], state_order, settings, cov_rescaling, L, Qc)
        status[hit] = 2
        out["filtered_means"][:, k], out["filtered_covariances"][:, k] = mf, Pf
        out["predicted_means"][:, k], out["predicted_covariances"][:, k] = m, P
        out["marginal_loglik_cumulative"][:, k] = ll
    out["marginal_loglik"] = ll
    out["status"] = _finalize_status(status, ll)
    return out


def extended_kalman_smoother(p: NonlinearParams, y, t, dt_final=1e-10, state_order="second", settings=SolverSettings(), dtype=np.float64, filtered=None):
    """inference_ekf.py:450-539 with _smooth :363-448 (Jacobian and drift frozen at the filtered mean)."""
    filt = filtered or extended_kalman_filter(p, y, t, dt_final, state_order, settings, 1, 1.0, dtype)
    t = np.asarray(t, dtype)
    N, K = t.shape
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    L, Qc = c(p.L, 2), c(p.Qc, 2)
    LQL = L @ Qc @ _mT(L)
    fm, fP = filt["filtered_means"], filt["filtered_covariances"]
    sm, sP = np.zeros_like(fm), np.zeros_like(fP)
    sm[:, -1], sP[:, -1] = fm[:, -1], fP[:, -1]
    ms, Ps = fm[:, -1].copy(), fP[:, -1].copy()
    for k in range(K - 2, -1, -1):
        t0, t1 = t[:, k], t[:, k + 1]
        mf, Pf = fm[:, k], fP[:, k]
        J = p.drift.jac(mf)  # :413
        f_mf = p.drift.f(mf)
        aux = _mT(psd_solve(Pf, LQL))  # :433
        G = J + aux

        def rhs(s, yy, mf=mf, G=G, f_mf=f_mf):
            m_s, P_s = yy
            dm = f_mf + _mv(G, m_s - mf)  # :436
            dP = G @ P_s + P_s @ _mT(G) - LQL  # :438
            return (-dm, -dP)

        (ms, Ps), _, _ = rk_solve(rhs, np.zeros_like(t0), t1 - t0, (ms, Ps), settings)  # :447
        sm[:, k], sP[:, k] = ms, Ps
    filt = dict(filt)
    filt.update(smoothed_means=sm, smoothed_covariances=sP)
    return filt


# --------------------------------------------------------------------------------------------------------------------
# CD-UKF  (cd_nonlinear/inference_ukf.py)
# --------------------------------------------------------------------------------------------------------------------
def ukf_weights(n, alpha, beta, kappa, dtype=np.float64):
    """inference_ukf.py:42,63-89."""
    lamb = alpha**2 * (n + kappa) - n
    factor = 1.0 / (2.0 * (n + lamb))
    w_mean = np.concatenate([[lamb / (n + lamb)], np.ones(2 * n) * factor]).astype(dtype)
    w_cov = np.concatenate([[lamb / (n + lamb) + (1 - alpha**2 + beta)], np.ones(2 * n) * factor]).astype(dtype)
    I_w = np.eye(2 * n + 1, dtype=dtype) - w_mean[:, None]
    W = I_w @ np.diag(w_cov) @ I_w.T
    return dtype(lamb) if not isinstance(dtype, np.dtype) else dtype.type(lamb), w_mean, w_cov, W


def _sigmas(m, P, n, lamb):
    """inference_ukf.py:45-60: rows = m, m + c*L[:,i], m - c*L[:,i]."""
    dist = np.sqrt(m.dtype.type(n + lamb)) * cholesky(P)
    cols = _mT(dist)  # [N, i, :] = dist[:, :, i]
    return np.concatenate([m[:, None, :], m[:, None, :] + cols, m[:, None, :] - cols], axis=1)


def unscented_kalman_filter(
    p: NonlinearParams, y, t, dt_final=1e-10, alpha=math.sqrt(3.0), beta=2.0, kappa=1.0, settings=SolverSettings(), dtype=np.float64,
    forecast=False,
):
    """inference_ukf.py:206-308.  forecast=True: forecast_unscented_kalman_filter (no updates; t is [N,K+1], t_init first)."""
    y = np.asarray(y, dtype)
    t = np.asarray(t, dtype)
    N, K, mdim = y.shape
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    L, Qc, H, R = c(p.L, 2), c(p.Qc, 2), c(p.H, 2), c(p.R, 2)
    n = L.shape[-1]
    d = c(p.d if p.d is not None else np.zeros(mdim), 1)
    LQL = L @ Qc @ _mT(L)
    lamb, w_m, w_c, W = ukf_weights(n, alpha, beta, kappa, np.dtype(dtype).type)
    m, P = c(p.m0, 1).copy(), c(p.P0, 2).copy()
    t0s, t1s = (t[:, :-1], t[:, 1:]) if forecast else _gap_times(t, dt_final)
    out = dict(
        filtered_means=np.zeros((N, K, n), dtype),
        filtered_covariances=np.zeros((N, K, n, n), dtype),
        predicted_means=np.zeros((N, K, n), dtype),
        predicted_covariances=np.zeros((N, K, n, n), dtype),
        marginal_loglik_cumulative=np.zeros((N, K), dtype),
    )
    ll = np.zeros(N, dtype)
    status = np.zeros(N, np.int32)

    def rhs(tt, yy):  # :130-152
        m_t, P_t = yy
        X = _sigmas(m_t, P_t, n, lamb)  # [N,p,n]
        fX = p.drift.f(X)
        dm = np.einsum("npi,p->ni", fX, w_m)
        foo = _mT(fX) @ W @ X
        return (dm, foo + _mT(foo) + LQL)

    for k in range(K):
        if forecast:
            mf, Pf = m, P
        else:
            # _condition_on :162-203
            X = _sigmas(m, P, n, lamb)
            Yp = np.einsum("nij,npj->npi", H, X) + d[:, None, :]
            yhat = np.einsum("p,npi->ni", w_m, Yp)
            dY = Yp - yhat[:, None, :]
            S = np.einsum("p,npi,npj->nij", w_c, dY, dY) + R
            C = np.einsum("p,npi,npj->nij", w_c, X - m[:, None, :], dY)
            ll = ll + mvn_logpdf(y[:, k], yhat, S)  # :197
            Kg = _mT(psd_solve(S, _mT(C)))  # :200
            mf = m + _mv(Kg, y[:, k] - yhat)
            Pf = P - Kg @ S @ _mT(Kg)  # :202 (no symmetrize)
        (m, P), _, hit = rk_solve(rhs, t0s[:, k], t1s[:, k], (mf, Pf), settings)
        status[hit] = 2
        out["filtered_means"][:, k], out["filtered_covariances"][:, k] = mf, Pf
        out["predicted_means"][:, k], out["predicted_covariances"][:, k] = m, P
        out["marginal_loglik_cumulative"][:, k] = ll
    out["marginal_loglik"] = ll
    out["status"] = _finalize_status(status, ll)
    return out


# --------------------------------------------------------------------------------------------------------------------
# Counter-based RNG shared bit-for-bit with the CUDA EnKF kernel (Philox4x32-10; Salmon et al. 2011).
# JAX threefry + diffrax VirtualBrownianTree streams cannot be reproduced outside JAX, so EnKF parity against the
# reference is distributional only (as in its own test, cdnlgssm_test_filter_linear_TRegular.py:434-470).
# --------------------------------------------------------------------------------------------------------------------
_PHILOX_M0, _PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_PHILOX_W0, _PHILOX_W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)


def philox4x32(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10. Counters: uint32 arrays (broadcastable); key: two uint32 scalars."""
    c0, c1, c2, c3 = (np.asarray(c, np.uint32) for c in np.broadcast_arrays(c0, c1, c2, c3))
    k0, k1 = np.uint32(k0), np.uint32(k1)
    mask = np.uint64(0xFFFFFFFF)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = _PHILOX_M0 * c0.astype(np.uint64)
            p1 = _PHILOX_M1 * c2.astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), (p0 & mask).astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), (p1 & mask).astype(np.uint32)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0 = np.uint32((int(k0) + int(_PHILOX_W0)) & 0xFFFFFFFF)
            k1 = np.uint32((int(k1) + int(_PHILOX_W1)) & 0xFFFFFFFF)
    return c0, c1, c2, c3


def box_muller_f32(ra, rb):
    """One Box-Muller pair from two uint32 arrays in float32 arithmetic made of correctly rounded add / mul / div / sqrt only
    (no FMA, no libm), operation for operation csrc/cdk_rng.cuh:box_muller_f32 -- so the GPU deviates are reproduced bit for
    bit.  Returns two float32 arrays."""
    f32 = np.float32
    ra, rb = np.asarray(ra, np.uint32), np.asarray(rb, np.uint32)
    uf = ra.astype(f32) + f32(0.5)
    bits = uf.view(np.uint32)
    e = (bits >> np.uint32(23)).astype(np.int32) - np.int32(127)
    m = ((bits & np.uint32(0x007FFFFF)) | np.uint32(0x3F800000)).view(f32)
    big = m > f32(1.41421354)
    m = np.where(big, m * f32(0.5), m)
    e = np.where(big, e + np.int32(1), e)
    s = (m + f32(-1.0)) / (m + f32(1.0))
    s2 = s * s
    p = np.full(s2.shape, f32(0.111111112), f32)
    for c in (0.142857149, 0.2, 0.333333343, 1.0):
        p = p * s2 + f32(c)
    lnm = (f32(2.0) * s) * p
    lnu = lnm + (e - np.int32(32)).astype(f32) * f32(0.693147182)
    radh = np.sqrt(f32(-2.0) * lnu) * f32(0.707106769)
    q = rb >> np.uint32(30)
    g = (((rb >> np.uint32(7)) & np.uint32(0x7FFFFF)).astype(f32) + f32(0.5)) * f32(1.1920929e-07) + f32(-0.5)
    y = g * f32(1.57079637)
    y2 = y * y
    ps = np.full(y2.shape, f32(2.75573188e-06), f32)
    for c in (-1.98412701e-04, 8.33333377e-03, -0.166666672, 1.0):
        ps = ps * y2 + f32(c)
    sy = y * ps
    pc = np.full(y2.shape, f32(2.48015876e-05), f32)
    for c in (-1.38888892e-03, 4.16666679e-02, -0.5):
        pc = pc * y2 + f32(c)
    cy = pc * y2 + f32(1.0)
    c45, s45 = cy + (-sy), cy + sy
    odd = (q & np.uint32(1)) != 0
    cq = np.where(odd, -s45, c45)
    sq = np.where(odd, c45, s45)
    neg = (q & np.uint32(2)) != 0
    cq = np.where(neg, -cq, cq)
    sq = np.where(neg, -sq, sq)
    z0, z1 = radh * cq, radh * sq
    assert z0.dtype == f32 and z1.dtype == f32 and p.dtype == f32 and lnu.dtype == f32 and y.dtype == f32
    return z0, z1


def philox_normal_quad(c0, c1, c2, c3, seed):
    """Four standard normals per counter: two float32 Box-Muller pairs from words (r0, r1) and (r2, r3), widened to fp64
    (csrc/cdk_rng.cuh:normal_quad)."""
    k0, k1 = np.uint32(seed & 0xFFFFFFFF), np.uint32((seed >> 32) & 0xFFFFFFFF)
    r = philox4x32(c0, c1, c2, c3, k0, k1)
    z0, z1 = box_muller_f32(r[0], r[1])
    z2, z3 = box_muller_f32(r[2], r[3])
    return tuple(z.astype(np.float64) for z in (z0, z1, z2, z3))


# stream ids (counter word c3 high byte)
RNG_INIT, RNG_OBS, RNG_DYN = 0, 1, 2


def enkf_normals(stream, traj, step, substep, E, dim, seed, rng_offset=0):
    """z[len(traj), E, dim] standard normals. Counter layout (shared with csrc/cdk_enkf.cu):
    c0 = member e, c1 = trajectory + rng_offset, c2 = observation index k, c3 = stream<<28 | substep<<8 | quad index;
    quad q supplies dimensions 4q .. 4q+3."""
    traj = np.asarray(traj, np.uint64)
    nquad = (dim + 3) // 4
    e = np.arange(E, dtype=np.uint32)[None, :, None]
    c1 = ((traj + np.uint64(rng_offset)) & np.uint64(0xFFFFFFFF)).astype(np.uint32)[:, None, None]
    j = np.arange(nquad, dtype=np.uint32)[None, None, :]
    c3 = np.uint32((stream << 28) | ((substep & 0xFFFFF) << 8)) | j
    zs = philox_normal_quad(e, c1, np.uint32(step), c3, seed)
    z = np.empty((len(traj), E, 4 * nquad))
    for q in range(4):
        z[..., q::4] = zs[q]
    return z[..., :dim]


def ensemble_kalman_filter(
    p: NonlinearParams,
    y,
    t,
    dt_final=1e-10,
    E=64,
    perturb_measurements=True,
    seed=0,
    rng_offset=0,
    settings=SolverSettings(solver="euler"),
    dtype=np.float64,
    forecast=False,
):
    """inference_enkf.py:151-276 with an Euler-Maruyama (or Heun) SDE step and the shared Philox stream.  forecast=True:
    forecast_ensemble_kalman_filter (no updates; t is [N,K+1], t_init first)."""
    y = np.asarray(y, dtype)
    t = np.asarray(t, dtype)
    N, K, mdim = y.shape
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    L, Qc, H, R = c(p.L, 2), c(p.Qc, 2), c(p.H, 2), c(p.R, 2)
    n = L.shape[-1]
    d = c(p.d if p.d is not None else np.zeros(mdim), 1)
    G = L @ cholesky(Qc)  # :74-80
    cholR = cholesky(R)
    traj = np.arange(N)
    m0, P0 = c(p.m0, 1), c(p.P0, 2)
    z = enkf_normals(RNG_INIT, traj, 0, 0, E, n, seed, rng_offset).astype(dtype)
    X = m0[:, None, :] + np.einsum("nij,nej->nei", cholesky(P0), z)  # :260-262 (cholesky method)
    t0s, t1s = (t[:, :-1], t[:, 1:]) if forecast else _gap_times(t, dt_final)
    out = dict(
        filtered_means=np.zeros((N, K, n), dtype),
        filtered_covariances=np.zeros((N, K, n, n), dtype),
        predicted_means=np.zeros((N, K, n), dtype),
        predicted_covariances=np.zeros((N, K, n, n), dtype),
        marginal_loglik_cumulative=np.zeros((N, K), dtype),
    )
    ll = np.zeros(N, dtype)
    status = np.zeros(N, np.int32)
    tdt, dt0, tol = _stepping(settings, dtype)
    Em1 = np.dtype(dtype).type(E - 1)

    def moments(Z):
        mu = np.mean(Z, axis=1)
        A = Z - mu[:, None, :]
        return mu, np.einsum("nei,nej->nij", A, A) / Em1

    def update(X, k, ll):
        # _condition_on :92-148
        Y = np.einsum("nij,nej->nei", H, X) + d[:, None, :]
        ybar = np.mean(Y, axis=1)
        dY = Y - ybar[:, None, :]
        Cyy = np.einsum("nei,nej->nij", dY, dY) / Em1
        S = Cyy + R
        ll = ll + mvn_logpdf(y[:, k], ybar, S)  # :129
        if perturb_measurements:
            zo = enkf_normals(RNG_OBS, traj, k, 0, E, mdim, seed, rng_offset).astype(dtype)
            Yobs = y[:, k][:, None, :] + np.einsum("nij,nej->nei", cholR, zo)  # :135
        else:
            Yobs = np.broadcast_to(y[:, k][:, None, :], Y.shape)
        xbar = np.mean(X, axis=1)
        Cxy = np.einsum("nei,nej->nij", X - xbar[:, None, :], dY) / Em1  # :141
        Kg = _mT(psd_solve(S, _mT(Cxy)))  # :143
        X = X + np.einsum("nij,nej->nei", Kg, Yobs - Y)  # :146
        mf, Pf = moments(X)  # :225-228
        return X, ll, mf, Pf

    for k in range(K):
        if forecast:
            mf, Pf = moments(X)
        else:
            X, ll, mf, Pf = update(X, k, ll)
        # _predict :47-89 -- per-member SDE solve over the gap
        tprev = t0s[:, k].astype(tdt)
        t1 = t1s[:, k].astype(tdt)
        tnext = np.minimum(tprev + dt0, t1)
        sub = 0
        nst = np.zeros(N, np.int64)
        while True:
            active = tprev < t1
            over = active & (nst >= settings.max_steps)
            if over.any():
                status[over] = 2
                X[over] = np.nan
                active &= ~over
                tprev = np.where(over, t1, tprev)
            if not active.any():
                break
            dt = np.where(active, tnext - tprev, 0.0).astype(dtype)
            zd = enkf_normals(RNG_DYN, traj, k, sub, E, n, seed, rng_offset).astype(dtype)
            dW = np.sqrt(dt)[:, None, None] * zd
            noise = np.einsum("nij,nej->nei", G, dW)
            if settings.solver == "euler":
                Xn = X + dt[:, None, None] * p.drift.f(X) + noise
            elif settings.solver == "heun":
                f0 = p.drift.f(X)
                Xe = X + dt[:, None, None] * f0 + noise
                # x + dt/2 (f(x) + f(xe)) + noise, written without the noise term (the CUDA kernel does not keep it)
                Xn = Xe + dt[:, None, None] * np.dtype(dtype).type(0.5) * (p.drift.f(Xe) - f0)
            else:
                raise ValueError("EnKF supports solver 'euler' (Euler-Maruyama) or 'heun'")
            X = np.where(active[:, None, None], Xn, X)
            nst += active
            sub += 1
            tprev = np.where(active, tnext, tprev)
            cand = tprev + dt0
            tnext = np.where(cand > t1 - tol, t1, cand)
        mp, Pp = moments(X)  # :234-238
        out["filtered_means"][:, k], out["filtered_covariances"][:, k] = mf, Pf
        out["predicted_means"][:, k], out["predicted_covariances"][:, k] = mp, Pp
        out["marginal_loglik_cumulative"][:, k] = ll
    out["marginal_loglik"] = ll
    out["status"] = _finalize_status(status, ll)
    return out


# --------------------------------------------------------------------------------------------------------------------
# Forward sample paths (cd_nonlinear/models.py:525-656 cdnlgssm_path_sample; the point-estimate branch of
# cdnlgssm_forecast :840-936) on the shared Philox stream -- restates csrc/cdk_aux.cu:sample_path_kernel.
# --------------------------------------------------------------------------------------------------------------------
def sample_paths(p: NonlinearParams, t, seed=0, rng_offset=0, settings=SolverSettings(solver="heun"), fixed_init=False,
                 dtype=np.float64):
    """States [N,K,n] and emissions [N,K,m].  x_0 ~ N(m0, P0) and y_0 at t[:,0]; then x_k = SDE solve over [t_{k-1}, t_k]
    (Heun = the reference default for SDEs, diffrax_utils.py:121-127, or Euler-Maruyama), y_k ~ N(H x_k + d, R).
    fixed_init: t is [N,K+1] (t_init first), the path starts AT m0 and the K outputs are the forecast times."""
    t = np.asarray(t, dtype)
    N = t.shape[0]
    K = t.shape[1] - 1 if fixed_init else t.shape[1]
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    L, Qc, H, R = c(p.L, 2), c(p.Qc, 2), c(p.H, 2), c(p.R, 2)
    n, mdim = L.shape[-1], H.shape[-2]
    d = c(p.d if p.d is not None else np.zeros(mdim), 1)
    G = L @ cholesky(Qc)
    cholR = cholesky(R)
    traj = np.arange(N)
    m0 = c(p.m0, 1)
    tdt, dt0, tol = _stepping(settings, dtype)
    xs, ys = np.zeros((N, K, n), dtype), np.zeros((N, K, mdim), dtype)

    def emit(x, row, step):
        z = enkf_normals(RNG_OBS, traj, step, 0, 1, mdim, seed, rng_offset)[:, 0].astype(dtype)
        xs[:, row] = x
        ys[:, row] = _mv(H, x) + d + _mv(cholR, z)

    if fixed_init:
        x = m0.copy()
    else:
        z = enkf_normals(RNG_INIT, traj, 0, 0, 1, n, seed, rng_offset)[:, 0].astype(dtype)
        x = m0 + _mv(cholesky(c(p.P0, 2)), z)
        emit(x, 0, 0)
    for k in range(0 if fixed_init else 1, K):
        tprev = (t[:, k] if fixed_init else t[:, k - 1]).astype(tdt)
        t1 = (t[:, k + 1] if fixed_init else t[:, k]).astype(tdt)
        tnext = np.minimum(tprev + dt0, t1)
        sub = 0
        nst = np.zeros(N, np.int64)
        while True:
            active = tprev < t1
            over = active & (nst >= settings.max_steps)
            if over.any():
                x[over] = np.nan
                active &= ~over
                tprev = np.where(over, t1, tprev)
            if not active.any():
                break
            dt = np.where(active, tnext - tprev, 0.0).astype(dtype)
            zd = enkf_normals(RNG_DYN, traj, k, sub, 1, n, seed, rng_offset)[:, 0].astype(dtype)
            noise = _mv(G, np.sqrt(dt)[:, None] * zd)
            f0 = p.drift.f(x)
            xe = x + dt[:, None] * f0 + noise
            if settings.solver == "heun":
                xn = xe + dt[:, None] * np.dtype(dtype).type(0.5) * (p.drift.f(xe) - f0)
            elif settings.solver == "euler":
                xn = xe
            else:
                raise ValueError("the sampler supports solver 'euler' (Euler-Maruyama) or 'heun'")
            x = np.where(active[:, None], xn, x)
            nst += active
            sub += 1
            tprev = np.where(active, tnext, tprev)
            cand = tprev + dt0
            tnext = np.where(cand > t1 - tol, t1, cand)
        emit(x, k, k + 1 if fixed_init else k)
    return xs, ys


def emission_moments(p: NonlinearParams, state_means, state_covs=None):
    """emissions_extended_kalman_filter (inference_ekf.py:762-855) for h(x) = H x + d: (H m + d, H P H^T + R); without
    covariances the model's own (H m + d, R) (cd_nonlinear/models.py:1000-1047)."""
    sm = np.asarray(state_means)
    H, R = np.asarray(p.H), np.asarray(p.R)
    d = np.asarray(p.d) if p.d is not None else np.zeros(H.shape[0])
    em = sm @ H.T + d
    if state_covs is None:
        return em, np.broadcast_to(R, sm.shape[:-1] + R.shape).copy()
    return em, H @ np.asarray(state_covs) @ H.T + R
