"""Torch float64 restatement of ``cd_oracle.extended_kalman_filter`` (state_order first / second, num_iter = 1, linear
emission, full R), batched over N, so that ``torch.autograd`` gives the gradient of the same discrete filter.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE: the reference gradient that ``cdk_ekf_grad_dense_f64`` is checked against.

It takes the oracle's steps: substep lengths from the diffrax ConstantStepSize rule computed in NumPy on the time grid
(``cd_torch_kf.substeps``), the same tableaux and stage arithmetic as ``cd_oracle.rk_solve``, the registry drift formulas,
the reference's 'second' order term 0.5 g^T P (g = ``grad_div``), the un-boosted Cholesky for the log-pdf,
``sym(S) + 1e-9 I`` for the gain and a symmetrised filtered covariance.  The parameters are (theta, Sigma, H, d, R, m0, P0)
with Sigma = L Qc L^T and theta in the layout of include/cdk.h, each [core] or [N, core].
"""
from __future__ import annotations

import numpy as np
import torch

from . import cd_oracle as o
from .cd_torch_kf import _mvn_logpdf, _sym, substeps


def drift_fns(kind: str, n: int):
    """-> (f(theta, x) [N, n], jac(theta, x) [N, n, n], graddiv(theta) [N, n]) for theta [N, n_theta], x [N, n]."""
    if kind == "linear":
        W = lambda th: th[:, :n * n].reshape(-1, n, n)
        return (lambda th, x: (W(th) @ x[..., None])[..., 0] + th[:, n * n:],
                lambda th, x: W(th),
                lambda th: torch.zeros(th.shape[0], n, dtype=th.dtype))
    if kind == "lorenz63":
        def f(th, x):
            s, r, b = th[:, 0], th[:, 1], th[:, 2]
            return torch.stack([s * (x[:, 1] - x[:, 0]), x[:, 0] * (r - x[:, 2]) - x[:, 1], x[:, 0] * x[:, 1] - b * x[:, 2]], -1)

        def jac(th, x):
            s, r, b = th[:, 0], th[:, 1], th[:, 2]
            z, one = torch.zeros_like(s), torch.ones_like(s)
            return torch.stack([torch.stack([-s, s, z], -1), torch.stack([r - x[:, 2], -one, -x[:, 0]], -1),
                                torch.stack([x[:, 1], x[:, 0], -b], -1)], -2)
        return f, jac, lambda th: torch.zeros(th.shape[0], 3, dtype=th.dtype)
    if kind == "lorenz96":
        idx = np.arange(n)
        E = {}
        for name, off in (("p1", 1), ("m1", -1), ("m2", -2)):
            M = np.zeros((n, n))
            M[idx, (idx + off) % n] = 1.0
            E[name] = torch.as_tensor(M)

        def f(th, x):
            xp1, xm1, xm2 = torch.roll(x, -1, -1), torch.roll(x, 1, -1), torch.roll(x, 2, -1)
            return (xp1 - xm2) * xm1 - x + th[:, :1]

        def jac(th, x):
            xp1, xm1, xm2 = torch.roll(x, -1, -1), torch.roll(x, 1, -1), torch.roll(x, 2, -1)
            return (xm1[..., None] * (E["p1"] - E["m2"]) + (xp1 - xm2)[..., None] * E["m1"]
                    - torch.eye(n, dtype=x.dtype))
        return f, jac, lambda th: torch.zeros(th.shape[0], n, dtype=th.dtype)
    if kind == "quadratic":
        a = lambda th: th[:, :n]
        B = lambda th: th[:, n:n + n * n].reshape(-1, n, n)
        C = lambda th: th[:, n + n * n:].reshape(-1, n, n, n)
        return (lambda th, x: a(th) + (B(th) @ x[..., None])[..., 0] + torch.einsum("nijk,nj,nk->ni", C(th), x, x),
                lambda th, x: B(th) + torch.einsum("nijk,nk->nij", C(th), x) + torch.einsum("nikj,nk->nij", C(th), x),
                lambda th: torch.einsum("niik->nk", C(th)) + torch.einsum("niki->nk", C(th)))
    raise ValueError(kind)


def _predict(fns, theta, Sigma, m, P, t0, t1, state_order, settings):
    f, jac, graddiv = fns
    tab = o.TABLEAUX[settings.solver]
    a, b = tab["a"], tab["b"]

    def rhs(mm, PP):
        J = jac(theta, mm)
        dm = f(theta, mm)
        if state_order == "second":
            dm = dm + 0.5 * torch.einsum("nk,nkl->nl", graddiv(theta), PP)
        return dm, J @ PP + PP @ J.transpose(-1, -2) + Sigma

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


def extended_kalman_filter(kind, theta, Sigma, H, d, R, m0, P0, y, t, dt_final=1e-10, state_order="second",
                           settings=o.SolverSettings()):
    """-> dict like ``cd_oracle.extended_kalman_filter`` (torch tensors; status as a NumPy array).  y [N, K, m], t [N, K]."""
    y = torch.as_tensor(np.asarray(y, np.float64))
    t = np.asarray(t, np.float64)
    N, K, mdim = y.shape
    c = lambda x, core: x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))
    theta, Sigma, H, R, P0, d, m0 = c(theta, 1), c(Sigma, 2), c(H, 2), c(R, 2), c(P0, 2), c(d, 1), c(m0, 1)
    n = Sigma.shape[-1]
    fns = drift_fns(kind, n)
    t0s, t1s = o._gap_times(t, dt_final)
    m, P = m0, P0
    ll = torch.zeros(N, dtype=torch.float64)
    status = np.zeros(N, np.int32)
    fm, fp, pm, pp = [], [], [], []
    eye = torch.eye(mdim, dtype=torch.float64)
    for k in range(K):
        Hm = (H @ m[..., None])[..., 0]
        ll = ll + _mvn_logpdf(y[:, k], Hm + d, H @ P @ H.transpose(-1, -2) + R)
        S = R + H @ P @ H.transpose(-1, -2)
        Kt = torch.cholesky_solve(H @ P, torch.linalg.cholesky(_sym(S) + 1e-9 * eye))
        Kg = Kt.transpose(-1, -2)
        mf = m + (Kg @ (y[:, k] - (Hm + d))[..., None])[..., 0]
        Pf = _sym(P - Kg @ S @ Kt)
        m, P, hit = _predict(fns, theta, Sigma, mf, Pf, t0s[:, k], t1s[:, k], state_order, settings)
        status[hit] = 2
        fm.append(mf), fp.append(Pf), pm.append(m), pp.append(P)
    out = dict(marginal_loglik=ll, filtered_means=torch.stack(fm, 1), filtered_covariances=torch.stack(fp, 1),
               predicted_means=torch.stack(pm, 1), predicted_covariances=torch.stack(pp, 1))
    out["status"] = o._finalize_status(status, ll.detach().numpy())
    return out


def marginal_log_prob(kind, theta, Sigma, H, d, R, m0, P0, y, t, dt_final=1e-10, state_order="second",
                      settings=o.SolverSettings()):
    """Per-trajectory log-likelihood [N]; ``torch.autograd.grad(ll.sum(), params)`` is the reference gradient."""
    return extended_kalman_filter(kind, theta, Sigma, H, d, R, m0, P0, y, t, dt_final, state_order, settings)["marginal_loglik"]
