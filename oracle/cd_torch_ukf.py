"""Torch float64 restatements of ``cd_oracle.unscented_kalman_filter`` (linear emission, full R), batched over N, so that
``torch.autograd`` gives the gradient of the same discrete filter.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE: the reference gradient that ``cdk_ukf_grad_dense_f64`` is checked against.

Two restatements of the unscented predict, with the oracle's substep rule (``cd_torch_kf.substeps``), tableaux and stage
arithmetic, the registry drift formulas of ``cd_torch_ekf.drift_fns``, the un-boosted Cholesky of S for the log-pdf,
``sym(S) + 1e-9 I`` for the gain and -- as the reference's UKF (inference_ukf.py:202) -- no symmetrisation of the
filtered covariance:

- ``closed="closed"``: what the kernels compute.  Every registry drift is a polynomial of degree <= 2, so the sigma-point
  sums are exactly dm = f(m) + 0.5 tr(Hess f . sym P), dP = J sym(P) + sym(P) J^T + Sigma: a symmetric derivative, so
  the antisymmetric part the update leaves in P is carried across the gap unchanged.
- ``closed="sigma"``: the reference literally -- weights from alpha, beta and kappa, a Cholesky factor of P at every
  stage and of the predicted covariance in the update, the W matrix.

The parameters are (theta, Sigma, H, d, R, m0, P0) with Sigma = L Qc L^T and theta in the layout of include/cdk.h, each
[core] or [N, core].
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import cd_oracle as o
from .cd_torch_ekf import drift_fns
from .cd_torch_kf import _mvn_logpdf, _sym, substeps


def drift_hessian(kind: str, n: int):
    """-> hess(theta) [N, n, n, n]: the constant Hessians d2 f_r / dx_j dx_k of the registry drift."""
    if kind == "linear":
        return lambda th: torch.zeros(th.shape[0], n, n, n, dtype=th.dtype)
    if kind == "lorenz63":
        Hs = np.zeros((3, 3, 3))
        Hs[1, 0, 2] = Hs[1, 2, 0] = -1.0  # f1 = x (rho - z) - y
        Hs[2, 0, 1] = Hs[2, 1, 0] = 1.0   # f2 = x y - beta z
        return lambda th: torch.as_tensor(Hs).expand(th.shape[0], 3, 3, 3)
    if kind == "lorenz96":
        Hs = np.zeros((n, n, n))
        for r in range(n):  # f_r = (x_{r+1} - x_{r-2}) x_{r-1} - x_r + F
            p1, m1, m2 = (r + 1) % n, (r - 1) % n, (r - 2) % n
            Hs[r, p1, m1] += 1.0
            Hs[r, m1, p1] += 1.0
            Hs[r, m2, m1] -= 1.0
            Hs[r, m1, m2] -= 1.0
        return lambda th: torch.as_tensor(Hs).expand(th.shape[0], n, n, n)
    if kind == "quadratic":
        def hess(th):
            C = th[:, n + n * n:].reshape(-1, n, n, n)
            return C + C.transpose(-1, -2)
        return hess
    raise ValueError(kind)


def ukf_weights(n, alpha, beta, kappa):
    lamb, w_m, w_c, W = o.ukf_weights(n, alpha, beta, kappa)
    return float(lamb), torch.as_tensor(w_m), torch.as_tensor(w_c), torch.as_tensor(W)


def _sigmas(m, P, n, lamb):
    """Rows m, m + c L[:, i], m - c L[:, i] with L = chol(P) (lower triangle), c = sqrt(n + lambda)."""
    cols = (math.sqrt(n + lamb) * torch.linalg.cholesky(P)).transpose(-1, -2)
    return torch.cat([m[:, None, :], m[:, None, :] + cols, m[:, None, :] - cols], 1)


def _rk(rhs, m, P, t0, t1, settings):
    tab = o.TABLEAUX[settings.solver]
    a, b = tab["a"], tab["b"]
    dts, acts, hit = substeps(t0, t1, settings)
    for dt_np, act_np in zip(dts, acts):
        dtm = torch.as_tensor(dt_np)[:, None]
        dtP = dtm[..., None]
        ks = []
        for i in range(len(b)):
            ym, yP = m, P
            if i > 0:
                ym = m + sum(a[i][j] * ks[j][0] for j in range(i) if a[i][j] != 0.0)
                yP = P + sum(a[i][j] * ks[j][1] for j in range(i) if a[i][j] != 0.0)
            km, kP = rhs(ym, yP)
            ks.append((dtm * km, dtP * kP))
        mn = m + sum(b[j] * ks[j][0] for j in range(len(b)) if b[j] != 0.0)
        Pn = P + sum(b[j] * ks[j][1] for j in range(len(b)) if b[j] != 0.0)
        act = torch.as_tensor(act_np)
        m, P = torch.where(act[:, None], mn, m), torch.where(act[:, None, None], Pn, P)
    if hit.any():
        h = torch.as_tensor(hit)
        m, P = torch.where(h[:, None], torch.nan, m), torch.where(h[:, None, None], torch.nan, P)
    return m, P, hit


def unscented_kalman_filter(kind, theta, Sigma, H, d, R, m0, P0, y, t, dt_final=1e-10, alpha=math.sqrt(3.0), beta=2.0,
                            kappa=1.0, settings=o.SolverSettings(), closed="closed"):
    """-> dict like ``cd_oracle.unscented_kalman_filter`` (torch tensors; status as a NumPy array).  y [N, K, m], t [N, K].
    closed = "closed" (the kernels' closed form) or "sigma" (literal sigma points, as the reference)."""
    y = torch.as_tensor(np.asarray(y, np.float64))
    t = np.asarray(t, np.float64)
    N, K, mdim = y.shape
    c = lambda x, core: x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))
    theta, Sigma, H, R, P0, d, m0 = c(theta, 1), c(Sigma, 2), c(H, 2), c(R, 2), c(P0, 2), c(d, 1), c(m0, 1)
    n = Sigma.shape[-1]
    f, jac, _ = drift_fns(kind, n)
    lamb, w_m, w_c, W = ukf_weights(n, alpha, beta, kappa)
    if closed == "closed":
        Hs = drift_hessian(kind, n)(theta)

        def rhs(mm, PP):
            Ps = _sym(PP)
            J = jac(theta, mm)
            dm = f(theta, mm) + 0.5 * torch.einsum("nrjk,njk->nr", Hs, Ps)
            return dm, J @ Ps + Ps @ J.transpose(-1, -2) + Sigma
    elif closed == "sigma":
        def rhs(mm, PP):  # inference_ukf.py:130-152
            X = _sigmas(mm, PP, n, lamb)
            p = X.shape[1]
            fX = f(theta[:, None, :].expand(N, p, theta.shape[-1]).reshape(N * p, -1), X.reshape(N * p, n)).reshape(N, p, n)
            dm = torch.einsum("npi,p->ni", fX, w_m)
            foo = fX.transpose(-1, -2) @ W @ X
            return dm, foo + foo.transpose(-1, -2) + Sigma
    else:
        raise ValueError(closed)
    t0s, t1s = o._gap_times(t, dt_final)
    m, P = m0, P0
    ll = torch.zeros(N, dtype=torch.float64)
    status = np.zeros(N, np.int32)
    fm, fp, pm, pp = [], [], [], []
    eye = torch.eye(mdim, dtype=torch.float64)
    for k in range(K):
        if closed == "closed":  # h(x) = H x + d: S = H P H^T + R and the cross term P H^T exactly
            yhat = (H @ m[..., None])[..., 0] + d
            S = R + H @ P @ H.transpose(-1, -2)
            Ct = H @ P
        else:  # inference_ukf.py:162-203
            X = _sigmas(m, P, n, lamb)
            Yp = torch.einsum("nij,npj->npi", H, X) + d[:, None, :]
            yhat = torch.einsum("p,npi->ni", w_m, Yp)
            dY = Yp - yhat[:, None, :]
            S = torch.einsum("p,npi,npj->nij", w_c, dY, dY) + R
            Ct = torch.einsum("p,npi,npj->nji", w_c, X - m[:, None, :], dY)
        ll = ll + _mvn_logpdf(y[:, k], yhat, S)
        Kt = torch.cholesky_solve(Ct, torch.linalg.cholesky(_sym(S) + 1e-9 * eye))
        Kg = Kt.transpose(-1, -2)
        mf = m + (Kg @ (y[:, k] - yhat)[..., None])[..., 0]
        Pf = P - Kg @ S @ Kt  # no symmetrisation (inference_ukf.py:202)
        m, P, hit = _rk(rhs, mf, Pf, t0s[:, k], t1s[:, k], settings)
        status[hit] = 2
        fm.append(mf), fp.append(Pf), pm.append(m), pp.append(P)
    out = dict(marginal_loglik=ll, filtered_means=torch.stack(fm, 1), filtered_covariances=torch.stack(fp, 1),
               predicted_means=torch.stack(pm, 1), predicted_covariances=torch.stack(pp, 1))
    out["status"] = o._finalize_status(status, ll.detach().numpy())
    return out


def marginal_log_prob(kind, theta, Sigma, H, d, R, m0, P0, y, t, dt_final=1e-10, alpha=math.sqrt(3.0), beta=2.0, kappa=1.0,
                      settings=o.SolverSettings(), closed="closed"):
    """Per-trajectory log-likelihood [N]; ``torch.autograd.grad(ll.sum(), params)`` is the reference gradient."""
    return unscented_kalman_filter(kind, theta, Sigma, H, d, R, m0, P0, y, t, dt_final, alpha, beta, kappa, settings,
                                   closed)["marginal_loglik"]
