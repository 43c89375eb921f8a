"""Torch float64 restatement of ``cd_oracle.cdlgssm_filter`` (full-R branch, no inputs), batched over N, so that
``torch.autograd`` gives the gradient of the same discrete filter.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE: the reference gradient that ``cdk_kf_grad_f64`` is checked against.

It takes the oracle's steps: substep lengths from the diffrax ConstantStepSize rule computed in NumPy on the time grid
(they do not depend on the parameters), the same tableaux and stage arithmetic as ``cd_oracle.rk_solve``, the un-boosted
Cholesky for the log-pdf, ``sym(S) + 1e-9 I`` for the gain and a symmetrised filtered covariance.  The parameters are
(F, b, Sigma, H, d, R, m0, P0) with Sigma = L Qc L^T, each [core] or [N, core].
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import cd_oracle as o


def substeps(t0, t1, settings: o.SolverSettings):
    """-> (dts, active): lists over substeps of [N] float64 arrays / bool masks, the oracle's rule (``rk_solve``) on one
    gap per trajectory, and hit[N] where max_steps was exceeded."""
    tdt, dt0, tol = o._stepping(settings, np.float64)
    t0, t1 = np.asarray(t0, tdt), np.asarray(t1, tdt)
    tprev, tnext = t0.copy(), np.minimum(t0 + dt0, t1)
    nsteps = np.zeros(t0.shape, np.int64)
    hit = np.zeros(t0.shape, bool)
    dts, acts = [], []
    while True:
        active = tprev < t1
        over = active & (nsteps >= settings.max_steps)
        if over.any():
            hit |= over
            active &= ~over
            tprev = np.where(over, t1, tprev)
        if not active.any():
            return dts, acts, hit
        dts.append(np.where(active, tnext - tprev, 0.0).astype(np.float64))
        acts.append(active)
        nsteps += active
        tprev = np.where(active, tnext, tprev)
        cand = tprev + dt0
        tnext = np.where(cand > t1 - tol, t1, cand)


def _sym(A):
    return 0.5 * (A + A.transpose(-1, -2))


def _pushforward(F, Sigma, t0, t1, settings):
    tab = o.TABLEAUX[settings.solver]
    a, b = tab["a"], tab["b"]
    N, n = F.shape[0], F.shape[-1]
    A = torch.eye(n, dtype=F.dtype).expand(N, n, n)
    Q = torch.zeros(N, n, n, dtype=F.dtype)
    Ft = F.transpose(-1, -2)
    dts, acts, hit = substeps(t0, t1, settings)
    for dt_np, act_np in zip(dts, acts):
        dt = torch.as_tensor(dt_np)[:, None, None]
        act = torch.as_tensor(act_np)[:, None, None]
        ks = []
        for i in range(len(b)):
            yA, yQ = A, Q
            if i > 0:
                yA = A + sum(a[i][j] * ks[j][0] for j in range(i) if a[i][j] != 0.0)
                yQ = Q + sum(a[i][j] * ks[j][1] for j in range(i) if a[i][j] != 0.0)
            ks.append((dt * (F @ yA), dt * (F @ yQ + yQ @ Ft + Sigma)))
        An = A + sum(b[j] * ks[j][0] for j in range(len(b)) if b[j] != 0.0)
        Qn = Q + sum(b[j] * ks[j][1] for j in range(len(b)) if b[j] != 0.0)
        A, Q = torch.where(act, An, A), torch.where(act, Qn, Q)
    if hit.any():
        h = torch.as_tensor(hit)[:, None, None]
        A, Q = torch.where(h, torch.nan, A), torch.where(h, torch.nan, Q)
    return A, Q, hit


def _mvn_logpdf(y, mu, S):
    L = torch.linalg.cholesky(S)
    z = torch.linalg.solve_triangular(L, (y - mu)[..., None], upper=False)[..., 0]
    m = S.shape[-1]
    return -0.5 * (z ** 2).sum(-1) - torch.log(torch.diagonal(L, dim1=-2, dim2=-1)).sum(-1) - 0.5 * m * math.log(2.0 * math.pi)


def cdlgssm_filter(F, b, Sigma, H, d, R, m0, P0, y, t, dt_final=1e-10, settings=o.SolverSettings()):
    """-> dict like ``cd_oracle.cdlgssm_filter`` (torch tensors; status as a NumPy array).  y [N, K, m], t [N, K]."""
    y = torch.as_tensor(np.asarray(y, np.float64))
    t = np.asarray(t, np.float64)
    N, K, mdim = y.shape
    c = lambda x, core: x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))
    F, Sigma, H, R, P0 = c(F, 2), c(Sigma, 2), c(H, 2), c(R, 2), c(P0, 2)
    b, d, m0 = c(b, 1), c(d, 1), c(m0, 1)
    n = F.shape[-1]
    t0s, t1s = o._gap_times(t, dt_final)
    m, P = m0, P0
    ll = torch.zeros(N, dtype=torch.float64)
    status = np.zeros(N, np.int32)
    fm, fp, pm, pp = [], [], [], []
    eye = torch.eye(mdim, dtype=torch.float64)
    for k in range(K):
        Hm = (H @ m[..., None])[..., 0]
        S = H @ P @ H.transpose(-1, -2) + R
        ll = ll + _mvn_logpdf(y[:, k], Hm + d, S)
        S2 = R + H @ P @ H.transpose(-1, -2)
        Kt = torch.cholesky_solve(H @ P, torch.linalg.cholesky(_sym(S2) + 1e-9 * eye))
        Kg = Kt.transpose(-1, -2)
        mf = m + (Kg @ (y[:, k] - d - Hm)[..., None])[..., 0]
        Pf = _sym(P - Kg @ S2 @ Kt)
        A, Q, hit = _pushforward(F, Sigma, t0s[:, k], t1s[:, k], settings)
        m = (A @ mf[..., None])[..., 0] + b
        P = A @ Pf @ A.transpose(-1, -2) + Q
        status[hit] = 2
        fm.append(mf), fp.append(Pf), pm.append(m), pp.append(P)
    out = dict(marginal_loglik=ll, filtered_means=torch.stack(fm, 1), filtered_covariances=torch.stack(fp, 1),
               predicted_means=torch.stack(pm, 1), predicted_covariances=torch.stack(pp, 1))
    out["status"] = o._finalize_status(status, ll.detach().numpy())
    return out


def marginal_log_prob(F, b, Sigma, H, d, R, m0, P0, y, t, dt_final=1e-10, settings=o.SolverSettings()):
    """Per-trajectory log-likelihood [N]; ``torch.autograd.grad(ll.sum(), params)`` is the reference gradient."""
    return cdlgssm_filter(F, b, Sigma, H, d, R, m0, P0, y, t, dt_final, settings)["marginal_loglik"]
