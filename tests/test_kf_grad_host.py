"""CPU side of the linear CD-KF gradient (cdk_kf_grad_f64): the torch arbiter (oracle/cd_torch_kf.py) against the NumPy
oracle, its autograd gradient against central differences of the oracle, and the host-side checks of the entry point."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import cd_oracle as o
from oracle import cd_torch_kf as tk
from tests.test_gpu_time_grids import degenerate_grid, edge_grid

SOLVERS = list(o.TABLEAUX)
BLOCKS = ("F", "b", "Sigma", "H", "d", "R", "m0", "P0")
SYMMETRIC = ("Sigma", "R", "P0")


def random_model(n, m, seed, N=None):
    """Stable F, SPD Sigma / R / P0; with N, every parameter carries a leading N."""
    rng = np.random.default_rng(seed)
    lead = () if N is None else (N,)

    def spd(k, scale):
        A = rng.standard_normal(lead + (k, k))
        return scale * (A @ np.swapaxes(A, -1, -2) / k + np.eye(k))

    L = np.eye(n) + 0.2 * rng.standard_normal(lead + (n, n))
    Qc = spd(n, 0.3)
    return dict(F=-0.6 * np.eye(n) + 0.4 * rng.standard_normal(lead + (n, n)) / np.sqrt(n),
                b=0.1 * rng.standard_normal(lead + (n,)), L=L, Qc=Qc, Sigma=L @ Qc @ np.swapaxes(L, -1, -2),
                H=rng.standard_normal(lead + (m, n)) / np.sqrt(n), d=0.1 * rng.standard_normal(lead + (m,)),
                R=spd(m, 0.5), m0=rng.standard_normal(lead + (n,)), P0=spd(n, 1.0))


def random_grid(N, K, seed, mean_gap=0.05):
    rng = np.random.default_rng(seed)
    gaps = mean_gap * rng.uniform(0.2, 1.8, size=(N, K))
    gaps[:, 0] = 0.0
    return 0.3 * np.arange(N)[:, None] + np.cumsum(gaps, axis=1)


def oracle_filter(p, y, t, settings, dt_final=1e-10):
    lp = o.LinearParams(m0=p["m0"], P0=p["P0"], F=p["F"], L=p["L"], Qc=p["Qc"], H=p["H"], R=p["R"], b=p["b"], d=p["d"])
    return o.cdlgssm_filter(lp, y, t, dt_final=dt_final, settings=settings)


def arbiter(p, y, t, settings, dt_final=1e-10, requires_grad=False):
    ts = {k: torch.tensor(np.asarray(p[k], np.float64), requires_grad=requires_grad) for k in BLOCKS}
    return ts, tk.cdlgssm_filter(*(ts[k] for k in BLOCKS), y, t, dt_final, settings)


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _check_against_oracle(p, y, t, settings, dt_final=1e-10):
    ref = oracle_filter(p, y, t, settings, dt_final)
    _, out = arbiter(p, y, t, settings, dt_final)
    for fld in ("marginal_loglik", "filtered_means", "filtered_covariances", "predicted_means", "predicted_covariances"):
        assert rel(out[fld].numpy(), ref[fld]) < 1e-12, fld
    assert np.array_equal(out["status"], ref["status"])


@pytest.mark.parametrize("solver", SOLVERS)
def test_arbiter_matches_oracle_every_solver(solver):
    N, K, n, m = 3, 9, 4, 3
    p = random_model(n, m, seed=1)
    y = np.random.default_rng(2).standard_normal((N, K, m))
    _check_against_oracle(p, y, random_grid(N, K, 3), o.SolverSettings(solver, 0.02))


@pytest.mark.parametrize("n,m", [(1, 1), (2, 3), (4, 8), (16, 1), (16, 3), (16, 8)])
def test_arbiter_matches_oracle_every_size(n, m):
    N, K = 2, 7
    p = random_model(n, m, seed=n * 10 + m, N=N)  # per-trajectory parameters
    y = np.random.default_rng(4).standard_normal((N, K, m))
    _check_against_oracle(p, y, random_grid(N, K, 5), o.SolverSettings("rk4", 0.02))


@pytest.mark.parametrize("grid", ["edge", "degenerate"])
@pytest.mark.parametrize("solver,dt0", [("rk4", 0.0025), ("dopri5", 0.01)])
def test_arbiter_matches_oracle_on_edge_grids(grid, solver, dt0):
    N, K, n, m = 5, 10, 2, 2
    t = edge_grid(N, K, dt0) if grid == "edge" else degenerate_grid(N, K, dt0)
    p = random_model(n, m, seed=7)
    y = np.random.default_rng(8).standard_normal((N, K, m))
    _check_against_oracle(p, y, t, o.SolverSettings(solver, dt0))


@pytest.mark.parametrize("solver", ["heun", "rk4", "dopri5"])
def test_arbiter_gradient_matches_central_differences_of_the_oracle(solver):
    N, K, n, m = 2, 8, 3, 2
    settings = o.SolverSettings(solver, 0.02)
    p = random_model(n, m, seed=11)
    y = np.random.default_rng(12).standard_normal((N, K, m))
    t = random_grid(N, K, 13)
    ts, out = arbiter(p, y, t, settings, requires_grad=True)
    grads = torch.autograd.grad(out["marginal_loglik"].sum(), [ts[k] for k in BLOCKS])
    rng = np.random.default_rng(14)
    for name, g in zip(BLOCKS, grads):
        v = rng.standard_normal(p[name].shape)
        if name in SYMMETRIC:
            v = 0.5 * (v + v.T)
        h = 1e-5

        def ll_at(s):
            q = dict(p)
            q[name] = p[name] + s * v
            if name == "Sigma":  # the oracle takes L and Qc: move Qc so that L Qc L^T moves by s v
                q["Qc"] = p["Qc"] + s * np.linalg.solve(p["L"], np.linalg.solve(p["L"], v).T).T
            return oracle_filter(q, y, t, settings)["marginal_loglik"].sum()

        fd = (ll_at(h) - ll_at(-h)) / (2 * h)
        an = float(np.sum(g.numpy() * v))
        assert abs(an - fd) <= 1e-6 * max(abs(fd), 1.0), (name, an, fd)


# ---- host-side checks of cdk_kf_grad_f64 (no CUDA call is made before they return) ----------------------------------
@pytest.fixture(scope="module")
def lib():
    from cd_dynamax_b200 import _lib as L
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("libcdk.so not built")
    return L.lib()


def _call(lib, **fields):
    from cd_dynamax_b200 import _lib as L
    d = L.new_desc()
    d.N, d.K, d.n, d.m = 4, 5, 3, 2
    flags = fields.pop("flags", 0)
    null_out = fields.pop("null_out", ())
    for k, v in fields.items():
        setattr(d, k, v)
    d.reserved[2] = flags
    fake = ctypes.c_void_p(0x1000)  # never dereferenced: every check below returns before any device work
    ins = (ctypes.c_void_p * L.NUM_IN)(*([fake] * L.NUM_IN))
    outs = (ctypes.c_void_p * L.NUM_OUT)(*([fake] * L.NUM_OUT))
    for s in null_out:
        outs[s] = None
    return lib.cdk_kf_grad_f64(ctypes.byref(d), ins, outs, None), lib.cdk_last_error().decode()


def test_unsupported_requests_are_rejected_on_the_host(lib):
    from cd_dynamax_b200 import _lib as L
    E_NULL, E_UNSUPPORTED = -1, -4
    for fields, code in ((dict(n=17), E_UNSUPPORTED), (dict(m=9), E_UNSUPPORTED), (dict(d_u=2), E_UNSUPPORTED),
                         (dict(flags=L.FLAG_DIAG_R), E_UNSUPPORTED), (dict(flags=L.FLAG_PREDICT_ONLY), E_UNSUPPORTED),
                         (dict(null_out=(L.OUT_GRAD,)), E_NULL), (dict(null_out=(L.OUT_SCRATCH,)), E_NULL)):
        rc, msg = _call(lib, **fields)
        assert rc == code and "cdk_kf_grad_f64" in msg, (fields, rc, msg)


def test_reserved_3_must_be_zero(lib):
    from cd_dynamax_b200 import _lib as L
    d = L.new_desc()
    d.N, d.K, d.n, d.m = 4, 5, 3, 2
    d.reserved[3] = 1
    fake = ctypes.c_void_p(0x1000)
    ins = (ctypes.c_void_p * L.NUM_IN)(*([fake] * L.NUM_IN))
    outs = (ctypes.c_void_p * L.NUM_OUT)(*([fake] * L.NUM_OUT))
    assert lib.cdk_kf_grad_f64(ctypes.byref(d), ins, outs, None) == -4


def test_scratch_bytes_kf_grad_and_ekf_grad_are_distinct(lib):
    from cd_dynamax_b200 import _lib as L
    d = L.new_desc()
    d.K, d.n, d.m = 50, 16, 4
    sizes = []
    for N in (1, 2, 7):
        d.N = N
        sizes.append(lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_kf_grad"))
    assert sizes[0] > 0 and sizes[1] == 2 * sizes[0] and sizes[2] == 7 * sizes[0]  # linear in N
    d.N = 1
    d.reserved[3] = L.GRAD_REVERSE
    ekf = lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad")
    assert ekf == 1 * 50 * 24 * 8  # the EKF's own size, not the linear model's
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_kf_grad") == sizes[0]
    # the kf branch holds the forward moments (K (2 n + 2 n^2) doubles) besides the checkpoints
    assert sizes[0] > 50 * (2 * 16 + 2 * 256) * 8
