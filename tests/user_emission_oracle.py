"""NumPy restatement of the filters and the path sampler with a NONLINEAR emission (any LearnableFunction.f upstream, what
cd_dynamax_b200.LearnableUserEmission runs): oracle/cd_oracle.py's EKF, UKF, EnKF and sampler with y = h(x) + noise in
place of H x + d, built from that module's own pieces (predict, moments, Philox stream, log-density), so only the
emission differs.  `em` is an object with batched h(x) [..., n] -> [..., m] and jac(x) -> [..., m, n]; `p` is an
oracle NonlinearParams whose H and d are not read."""
import math

import numpy as np

from oracle import cd_oracle as o
from oracle.cd_oracle import _bN, _mT, _mv


def _common(p, y, t, dtype):
    y = np.asarray(y, dtype)
    t = np.asarray(t, dtype)
    N, K, mdim = y.shape
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    L, Qc, R = c(p.L, 2), c(p.Qc, 2), c(p.R, 2)
    return y, t, N, K, mdim, c, L, Qc, R, L.shape[-1]


def _outputs(N, K, n, dtype):
    return dict(filtered_means=np.zeros((N, K, n), dtype), filtered_covariances=np.zeros((N, K, n, n), dtype),
                predicted_means=np.zeros((N, K, n), dtype), predicted_covariances=np.zeros((N, K, n, n), dtype),
                marginal_loglik_cumulative=np.zeros((N, K), dtype))


def _ekf_condition_on(m, P, em, R, y, num_iter):
    """inference_ekf.py:153-199 with H = jacfwd(h) at the running mean of every iteration and residual y - h(m)."""
    for _ in range(num_iter):
        H = em.jac(m)
        S = R + H @ P @ _mT(H)
        K = _mT(o.psd_solve(S, H @ P))
        P_new = P - K @ S @ _mT(K)
        m = m + _mv(K, y - em.h(m))
        P = P_new
    return m, o.symmetrize(P)


def extended_kalman_filter(p, em, y, t, dt_final=1e-10, state_order="second", settings=o.SolverSettings(), num_iter=1,
                           dtype=np.float64):
    y, t, N, K, mdim, c, L, Qc, R, n = _common(p, y, t, dtype)
    LQL = L @ Qc @ _mT(L)
    m, P = c(p.m0, 1).copy(), c(p.P0, 2).copy()
    t0s, t1s = o._gap_times(t, dt_final)
    out = _outputs(N, K, n, dtype)
    ll = np.zeros(N, dtype)
    status = np.zeros(N, np.int32)
    for k in range(K):
        H = em.jac(m)  # h and its Jacobian at the predicted mean (iteration 0)
        ll = ll + o.mvn_logpdf(y[:, k], em.h(m), H @ P @ _mT(H) + R)
        mf, Pf = _ekf_condition_on(m, P, em, R, y[:, k], num_iter)
        m, P, hit = o._ekf_predict(mf, Pf, p.drift, LQL, t0s[:, k], t1s[:, k], state_order, settings, 1.0, L, Qc)
        status[hit] = 2
        out["filtered_means"][:, k], out["filtered_covariances"][:, k] = mf, Pf
        out["predicted_means"][:, k], out["predicted_covariances"][:, k] = m, P
        out["marginal_loglik_cumulative"][:, k] = ll
    out["marginal_loglik"] = ll
    out["status"] = o._finalize_status(status, ll)
    return out


def extended_kalman_smoother(p, em, y, t, dt_final=1e-10, state_order="second", settings=o.SolverSettings()):
    """The oracle's smoother (the emission does not enter the backward pass) behind this module's filter."""
    filt = extended_kalman_filter(p, em, y, t, dt_final, state_order, settings)
    return o.extended_kalman_smoother(p, y, t, dt_final, state_order, settings, filtered=filt)


def unscented_kalman_filter(p, em, y, t, dt_final=1e-10, alpha=math.sqrt(3.0), beta=2.0, kappa=1.0,
                            settings=o.SolverSettings(), dtype=np.float64):
    y, t, N, K, mdim, c, L, Qc, R, n = _common(p, y, t, dtype)
    LQL = L @ Qc @ _mT(L)
    lamb, w_m, w_c, W = o.ukf_weights(n, alpha, beta, kappa, np.dtype(dtype).type)
    m, P = c(p.m0, 1).copy(), c(p.P0, 2).copy()
    t0s, t1s = o._gap_times(t, dt_final)
    out = _outputs(N, K, n, dtype)
    ll = np.zeros(N, dtype)
    status = np.zeros(N, np.int32)

    def rhs(tt, yy):  # inference_ukf.py:130-152
        m_t, P_t = yy
        X = o._sigmas(m_t, P_t, n, lamb)
        fX = p.drift.f(X)
        dm = np.einsum("npi,p->ni", fX, w_m)
        foo = _mT(fX) @ W @ X
        return (dm, foo + _mT(foo) + LQL)

    for k in range(K):
        # _condition_on :162-203, the sigma points pushed through h
        X = o._sigmas(m, P, n, lamb)
        Yp = em.h(X)
        yhat = np.einsum("p,npi->ni", w_m, Yp)
        dY = Yp - yhat[:, None, :]
        S = np.einsum("p,npi,npj->nij", w_c, dY, dY) + R
        C = np.einsum("p,npi,npj->nij", w_c, X - m[:, None, :], dY)
        ll = ll + o.mvn_logpdf(y[:, k], yhat, S)
        Kg = _mT(o.psd_solve(S, _mT(C)))
        mf = m + _mv(Kg, y[:, k] - yhat)
        Pf = P - Kg @ S @ _mT(Kg)  # no symmetrize (:202)
        (m, P), _, hit = o.rk_solve(rhs, t0s[:, k], t1s[:, k], (mf, Pf), settings)
        status[hit] = 2
        out["filtered_means"][:, k], out["filtered_covariances"][:, k] = mf, Pf
        out["predicted_means"][:, k], out["predicted_covariances"][:, k] = m, P
        out["marginal_loglik_cumulative"][:, k] = ll
    out["marginal_loglik"] = ll
    out["status"] = o._finalize_status(status, ll)
    return out


def _sde_step(X, drift, G, dt, zd, solver, dtype):
    """One Euler-Maruyama / Heun substep of the oracle's EnKF and sampler (same operation order)."""
    noise = np.einsum("...ij,...ej->...ei", G, np.sqrt(dt)[:, None, None] * zd)
    f0 = drift.f(X)
    Xe = X + dt[:, None, None] * f0 + noise
    if solver == "heun":
        return Xe + dt[:, None, None] * np.dtype(dtype).type(0.5) * (drift.f(Xe) - f0)
    if solver == "euler":
        return Xe
    raise ValueError("solver 'euler' (Euler-Maruyama) or 'heun'")


def ensemble_kalman_filter(p, em, y, t, dt_final=1e-10, E=64, perturb_measurements=True, seed=0, rng_offset=0,
                           settings=o.SolverSettings(solver="euler"), dtype=np.float64):
    y, t, N, K, mdim, c, L, Qc, R, n = _common(p, y, t, dtype)
    G = L @ o.cholesky(Qc)
    cholR = o.cholesky(R)
    traj = np.arange(N)
    m0, P0 = c(p.m0, 1), c(p.P0, 2)
    z = o.enkf_normals(o.RNG_INIT, traj, 0, 0, E, n, seed, rng_offset).astype(dtype)
    X = m0[:, None, :] + np.einsum("nij,nej->nei", o.cholesky(P0), z)
    t0s, t1s = o._gap_times(t, dt_final)
    out = _outputs(N, K, n, dtype)
    ll = np.zeros(N, dtype)
    status = np.zeros(N, np.int32)
    tdt, dt0, tol = o._stepping(settings, dtype)
    Em1 = np.dtype(dtype).type(E - 1)

    def moments(Z):
        mu = np.mean(Z, axis=1)
        A = Z - mu[:, None, :]
        return mu, np.einsum("nei,nej->nij", A, A) / Em1

    for k in range(K):
        # _condition_on :92-148, every member mapped through h
        Y = em.h(X)
        ybar = np.mean(Y, axis=1)
        dY = Y - ybar[:, None, :]
        S = np.einsum("nei,nej->nij", dY, dY) / Em1 + R
        ll = ll + o.mvn_logpdf(y[:, k], ybar, S)
        if perturb_measurements:
            zo = o.enkf_normals(o.RNG_OBS, traj, k, 0, E, mdim, seed, rng_offset).astype(dtype)
            Yobs = y[:, k][:, None, :] + np.einsum("nij,nej->nei", cholR, zo)
        else:
            Yobs = np.broadcast_to(y[:, k][:, None, :], Y.shape)
        xbar = np.mean(X, axis=1)
        Cxy = np.einsum("nei,nej->nij", X - xbar[:, None, :], dY) / Em1
        Kg = _mT(o.psd_solve(S, _mT(Cxy)))
        X = X + np.einsum("nij,nej->nei", Kg, Yobs - Y)
        mf, Pf = moments(X)
        tprev, t1 = t0s[:, k].astype(tdt), t1s[:, k].astype(tdt)
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
            zd = o.enkf_normals(o.RNG_DYN, traj, k, sub, E, n, seed, rng_offset).astype(dtype)
            X = np.where(active[:, None, None], _sde_step(X, p.drift, G, dt, zd, settings.solver, dtype), X)
            nst += active
            sub += 1
            tprev = np.where(active, tnext, tprev)
            cand = tprev + dt0
            tnext = np.where(cand > t1 - tol, t1, cand)
        mp, Pp = moments(X)
        out["filtered_means"][:, k], out["filtered_covariances"][:, k] = mf, Pf
        out["predicted_means"][:, k], out["predicted_covariances"][:, k] = mp, Pp
        out["marginal_loglik_cumulative"][:, k] = ll
    out["marginal_loglik"] = ll
    out["status"] = o._finalize_status(status, ll)
    return out


def sample_paths(p, em, t, seed=0, rng_offset=0, settings=o.SolverSettings(solver="heun"), fixed_init=False,
                 dtype=np.float64):
    """States [N,K,n] and emissions [N,K,m] = h(x_k) + chol(R) z on the oracle's stream (x_0 ~ N(m0, P0)).
    fixed_init (a forecast from a point estimate): t is [N,K+1] (t_init first), the path starts AT m0 and the K outputs
    are the forecast times, as in oracle.cd_oracle.sample_paths."""
    t = np.asarray(t, dtype)
    N = t.shape[0]
    K = t.shape[1] - 1 if fixed_init else t.shape[1]
    c = lambda x, core: _bN(np.asarray(x, dtype), N, core)
    L, Qc, R = c(p.L, 2), c(p.Qc, 2), c(p.R, 2)
    n, mdim = L.shape[-1], R.shape[-1]
    G = L @ o.cholesky(Qc)
    cholR = o.cholesky(R)
    traj = np.arange(N)
    tdt, dt0, tol = o._stepping(settings, dtype)
    xs, ys = np.zeros((N, K, n), dtype), np.zeros((N, K, mdim), dtype)

    def emit(x, row, step):
        z = o.enkf_normals(o.RNG_OBS, traj, step, 0, 1, mdim, seed, rng_offset)[:, 0].astype(dtype)
        xs[:, row] = x
        ys[:, row] = em.h(x) + _mv(cholR, z)

    if fixed_init:
        x = c(p.m0, 1).copy()
    else:
        z = o.enkf_normals(o.RNG_INIT, traj, 0, 0, 1, n, seed, rng_offset)[:, 0].astype(dtype)
        x = c(p.m0, 1) + _mv(o.cholesky(c(p.P0, 2)), z)
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
            zd = o.enkf_normals(o.RNG_DYN, traj, k, sub, 1, n, seed, rng_offset).astype(dtype)  # [N, 1, n]
            x = np.where(active[:, None], _sde_step(x[:, None, :], p.drift, G, dt, zd, settings.solver, dtype)[:, 0], x)
            nst += active
            sub += 1
            tprev = np.where(active, tnext, tprev)
            cand = tprev + dt0
            tnext = np.where(cand > t1 - tol, t1, cand)
        emit(x, k, k + 1 if fixed_init else k)
    return xs, ys
