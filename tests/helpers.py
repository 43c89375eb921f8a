"""Shared test helpers: golden-case loading, oracle invocation, error metrics."""
import glob
import os

import numpy as np

from oracle import cd_oracle as o

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class QuadraticDrift:
    """f_i = a_i + B_ij x_j + C_ijk x_j x_k (test-only drift with a non-zero reference 'second order' term).  Each of a, B,
    C may carry a leading N (one parameter sample per trajectory); states are [N, ..., n]."""

    drift_id = 3

    def __init__(self, a, B, C):
        self.a, self.B, self.C = np.asarray(a), np.asarray(B), np.asarray(C)

    def f(self, x):
        a, B, C = o.lead(self.a, x, 1), o.lead(self.B, x, 2), o.lead(self.C, x, 3)
        return a + np.einsum("...ij,...j->...i", B, x) + np.einsum("...ijk,...j,...k->...i", C, x, x)

    def jac(self, x):
        B, C = o.lead(self.B, x, 2), o.lead(self.C, x, 3)
        return B + np.einsum("...ijk,...k->...ij", C, x) + np.einsum("...ikj,...k->...ij", C, x)

    def grad_div(self, x):
        # sum_i d2 f_i / dx_i dx_k = sum_i (C_iik + C_iki)
        g = np.einsum("...iik->...k", self.C) + np.einsum("...iki->...k", self.C)
        return np.broadcast_to(o.lead(g, x, 1), x.shape)

    def theta(self):
        lead_shape = np.broadcast_shapes(self.a.shape[:-1], self.B.shape[:-2], self.C.shape[:-3])
        flat = [self.a, self.B.reshape(self.B.shape[:-2] + (-1,)), self.C.reshape(self.C.shape[:-3] + (-1,))]
        return np.concatenate([np.broadcast_to(v, lead_shape + v.shape[-1:]) for v in flat], axis=-1)


def golden_cases(prefix):
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, prefix + "*.npz")))


def load_golden(name):
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz")) as z:
        return {k: z[k] for k in z.files}


def make_drift(kind, theta, n):
    """Oracle drift from its parameter vector theta [n_theta], or [N, n_theta] for one parameter sample per trajectory."""
    kind = str(kind)
    theta = np.asarray(theta)
    if kind == "lorenz63":
        return o.Lorenz63Drift(theta[..., 0], theta[..., 1], theta[..., 2])
    if kind == "lorenz96":
        return o.Lorenz96Drift(theta[..., 0])
    lead = theta.shape[:-1]
    if kind == "linear":
        return o.LinearDrift(theta[..., : n * n].reshape(lead + (n, n)), theta[..., n * n:])
    if kind == "quadratic":
        return QuadraticDrift(theta[..., :n], theta[..., n:n + n * n].reshape(lead + (n, n)),
                              theta[..., n + n * n:].reshape(lead + (n, n, n)))
    raise ValueError(kind)


def linear_params(g):
    return o.LinearParams(m0=g["m0"], P0=g["P0"], F=g["F"], L=g["L"], Qc=g["Qc"], H=g["H"], R=g["R"], b=g["b"],
                          d=g["d"], B=g["B"] if g["B"].size else None, D=g["D"] if g["D"].size else None)


def nonlinear_params(g):
    n = g["m0"].shape[-1]
    return o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift(g["drift"], g["theta"], n), L=g["L"],
                             Qc=g["Qc"], H=g["H"], R=g["R"], d=g["d"])


def settings_of(g):
    return o.SolverSettings(str(g["solver"]), float(g["dt0"]))


def max_rel_err(a, b, floor=1e-12):
    """max |a-b| / max(|b|, floor*scale): rel error with an absolute floor for structurally-zero entries
    (SURVEY 8d parity gate)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.size == 0:
        return 0.0
    both_nan = np.isnan(a) & np.isnan(b)
    scale = np.nanmax(np.abs(b)) if np.isfinite(np.nanmax(np.abs(b))) else 1.0
    den = np.maximum(np.abs(b), max(floor * scale, 1e-300))
    err = np.abs(a - b) / den
    err = np.where(both_nan, 0.0, err)
    return float(np.max(np.where(np.isnan(err), np.inf, err)))


def gate_err(a, b, rel_floor=1e-3):
    """SURVEY 8(d) parity gate, verbatim: element-wise relative error abs(a - b) / abs(b), with an ABSOLUTE floor of
    1e-12 * scale for entries that are ~0 (scale = max |b| of the array).  Written as one number to compare with 1e-9:
        max_i |a_i - b_i| / max(|b_i|, rel_floor * scale)  <  1e-9   <=>   |a_i - b_i| <= max(1e-9 |b_i|, 1e-12 scale).
    (Without the absolute floor the gate measures zero crossings, not parity: means and off-diagonal covariances of a
    chaotic system pass through 0, and the NumPy and C restatements of the SAME algorithm already differ by 1.2e-9 on
    such entries of BASELINE config 3 while agreeing to 1.6e-14 of the scale -- tests/test_oracle_golden.py.)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.size == 0:
        return 0.0
    both_nan = np.isnan(a) & np.isnan(b)
    scale = np.nanmax(np.abs(b)) if np.isfinite(np.nanmax(np.abs(b))) else 1.0
    err = np.abs(a - b) / np.maximum(np.abs(b), max(rel_floor * scale, 1e-300))
    err = np.where(both_nan, 0.0, err)
    return float(np.max(np.where(np.isnan(err), np.inf, err)))


def moment_norm_err(a, b, core_ndim=1):
    """max over (trajectory, step) of ||a - b||_inf / ||b||_inf, each mean vector / covariance matrix (the last `core_ndim`
    axes) measured against ITS OWN norm -- a small covariance late in a trajectory is not hidden behind the prior's scale.
    The tests hold this to 1e-10, an order of magnitude inside the north star's 1e-9."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.size == 0:
        return 0.0
    ax = tuple(range(a.ndim - core_ndim, a.ndim))
    both_nan = np.isnan(a) & np.isnan(b)
    d = np.where(both_nan, 0.0, np.abs(a - b))
    d = np.where(np.isnan(d), np.inf, d)
    with np.errstate(invalid="ignore"):
        s = np.nanmax(np.where(np.isnan(b), 0.0, np.abs(b)), axis=ax)
    s = np.where(s > 0, s, 1.0)
    return float(np.max(np.max(d, axis=ax) / s))


FIELD_CORE = {"filtered_means": 1, "predicted_means": 1, "smoothed_means": 1, "filtered_covariances": 2,
              "predicted_covariances": 2, "smoothed_covariances": 2, "smoothed_cross_covariances": 2}


def moment_err(post, ref, fld, prefix=""):
    """(gate_err, moment_norm_err) of one result field (`post`: result tuple, `ref`: dict of oracle / golden arrays)."""
    a = getattr(post, fld)
    a = a.cpu().numpy() if hasattr(a, "cpu") else a
    return gate_err(a, ref[prefix + fld]), moment_norm_err(a, ref[prefix + fld], core_ndim=FIELD_CORE[fld])


_RECORD = {}


def record(name, value):
    """Keep the measured parity errors of a GPU run (written to gpurun_out/parity_errors_*.json at session end)."""
    _RECORD[name] = float(value)


def scaled_err(a, b):
    """max |a-b| / max|b| -- error relative to the array's scale."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.size == 0:
        return 0.0
    both_nan = np.isnan(a) & np.isnan(b)
    d = np.where(both_nan, 0.0, np.abs(a - b))
    d = np.where(np.isnan(d), np.inf, d)
    s = np.nanmax(np.abs(b))
    return float(np.max(d) / (s if s > 0 else 1.0))
