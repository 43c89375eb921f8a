"""CPU side of the gradient of the CD-UKF with literal sigma points (cdk_ukf_grad_sigma_f64): the torch sigma-point
restatement with a drift written in torch (`sigma_filter`, the reference of tests/test_gpu_ukf_sigma_grad.py) against the
registry restatement of oracle/cd_torch_ukf.py and against central differences, the Cholesky VJP the kernel uses against
torch autograd, and the host-side checks of the entry point and of ukf_sigma_points_marginal_log_prob_and_grad."""
import ctypes
import os
import shutil

import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200 import build as b
from oracle import cd_oracle as o
from oracle import cd_torch_ukf as tu
from oracle.cd_torch_ekf import drift_fns
from oracle.cd_torch_kf import _mvn_logpdf, _sym
from tests.helpers import record
from tests.test_ekf_grad_host import BLOCKS, SYMMETRIC, _stages, api_params, no_device, random_data, random_model, rel  # noqa: F401
from tests.test_kf_grad_host import random_grid
from tests.test_user_drift_grad_host import VDP, _Sentinel, _params

E_NULL, E_SIZE, E_UNSUPPORTED = -1, -2, -4


# ---- the sigma-point restatement with the drift as torch functions ---------------------------------------------------
def sigma_filter(fns, theta, Sigma, H, d, R, m0, P0, y, t, settings, dt_final=1e-10, alpha=float(np.sqrt(3.0)), beta=2.0,
                 kappa=1.0):
    """The log-likelihood [N] of cd_torch_ukf.unscented_kalman_filter(closed="sigma") with the drift given as torch
    functions fns = (f, jac, graddiv) of (theta [N, n_theta], x [N, n]) instead of a registry kind: the literal sigma
    points of every predict stage and update, step for step the same arithmetic."""
    f = fns[0]
    y = torch.as_tensor(np.asarray(y, np.float64))
    t = np.asarray(t, np.float64)
    N, K, mdim = y.shape
    c = lambda x, core: x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))
    theta, Sigma, H, R, P0, d, m0 = c(theta, 1), c(Sigma, 2), c(H, 2), c(R, 2), c(P0, 2), c(d, 1), c(m0, 1)
    n = Sigma.shape[-1]
    lamb, w_m, w_c, W = tu.ukf_weights(n, alpha, beta, kappa)

    def rhs(mm, PP):  # inference_ukf.py:130-152
        X = tu._sigmas(mm, PP, n, lamb)
        p = X.shape[1]
        fX = f(theta[:, None, :].expand(N, p, theta.shape[-1]).reshape(N * p, -1), X.reshape(N * p, n)).reshape(N, p, n)
        dm = torch.einsum("npi,p->ni", fX, w_m)
        foo = fX.transpose(-1, -2) @ W @ X
        return dm, foo + foo.transpose(-1, -2) + Sigma

    t0s, t1s = o._gap_times(t, dt_final)
    m, P = m0, P0
    ll = torch.zeros(N, dtype=torch.float64)
    eye = torch.eye(mdim, dtype=torch.float64)
    for k in range(K):  # inference_ukf.py:162-203
        X = tu._sigmas(m, P, n, lamb)
        Yp = torch.einsum("nij,npj->npi", H, X) + d[:, None, :]
        yhat = torch.einsum("p,npi->ni", w_m, Yp)
        dY = Yp - yhat[:, None, :]
        S = torch.einsum("p,npi,npj->nij", w_c, dY, dY) + R
        Ct = torch.einsum("p,npi,npj->nji", w_c, X - m[:, None, :], dY)
        ll = ll + _mvn_logpdf(y[:, k], yhat, S)
        Kt = torch.cholesky_solve(Ct, torch.linalg.cholesky(_sym(S) + 1e-9 * eye))
        Kg = Kt.transpose(-1, -2)
        mf = m + (Kg @ (y[:, k] - yhat)[..., None])[..., 0]
        Pf = P - Kg @ S @ Kt
        m, P, hit = tu._rk(rhs, mf, Pf, t0s[:, k], t1s[:, k], settings)
        assert not hit.any()
    return ll


def _leaves(p, N):
    out = {}
    for k in BLOCKS:
        x = torch.tensor(np.asarray(p[k], np.float64))
        core = 1 if k in ("theta", "d", "m0") else 2
        out[k] = (x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))).clone().requires_grad_(True)
    return out


def vdp_torch():
    from tests.test_gpu_user_drift_grad import vdp_fns
    return vdp_fns()


@pytest.mark.parametrize("kind,n", [("quadratic", 2), ("lorenz63", 3)])
def test_fns_restatement_equals_the_registry_restatement(kind, n):
    N, K, m = 2, 8, 2
    settings = o.SolverSettings("rk4", 0.01)
    p = random_model(kind, n, m, seed=11 + n)
    y = random_data(p, N, K, 12)
    t = random_grid(N, K, 13, mean_gap=0.03)
    a, bl = _leaves(p, N), _leaves(p, N)
    ll_f = sigma_filter(drift_fns(kind, n), *(a[k] for k in BLOCKS), y, t, settings)
    ll_r = tu.marginal_log_prob(kind, *(bl[k] for k in BLOCKS), y, t, settings=settings, closed="sigma")
    assert torch.equal(ll_f, ll_r)
    ga = torch.autograd.grad(ll_f.sum(), list(a.values()))
    gb = torch.autograd.grad(ll_r.sum(), list(bl.values()))
    for k, u, v in zip(BLOCKS, ga, gb):
        assert torch.equal(u, v), k


def test_vdp_restatement_gradient_matches_central_differences():
    N, K, m = 2, 8, 1
    settings = o.SolverSettings("rk4", 0.01)
    from tests.test_gpu_user_drift_grad import user_model
    p = user_model("vdp", m, 21)
    y = 0.7 * np.random.default_rng(22).standard_normal((N, K, m))
    t = random_grid(N, K, 23, mean_gap=0.05)
    fns = vdp_torch()
    lv = _leaves(p, N)
    grads = dict(zip(BLOCKS, torch.autograd.grad(sigma_filter(fns, *(lv[k] for k in BLOCKS), y, t, settings).sum(),
                                                 list(lv.values()))))
    rng = np.random.default_rng(24)
    worst = 0.0
    for name in BLOCKS:
        v = rng.standard_normal(np.shape(p[name]))
        if name in SYMMETRIC:
            v = 0.5 * (v + v.T)
        h = 1e-6

        def ll_at(s):
            q = {k: torch.tensor(np.asarray(p[k] + (s * v if k == name else 0.0), np.float64)) for k in BLOCKS}
            return float(sigma_filter(fns, *(q[k] for k in BLOCKS), y, t, settings).sum())

        fd = (ll_at(h) - ll_at(-h)) / (2 * h)
        an = float(np.sum(grads[name].sum(0).numpy() * v))
        err = abs(an - fd) / max(abs(fd), 1.0)
        worst = max(worst, err)
        assert err <= 1e-6, (name, an, fd)
    record("ukf_sigma_torch_vdp_vs_central_differences", worst)


def cholesky_vjp(Lc, Lb):
    """P_bar = sym(Lc^-T Phi(Lc^T tril(Lb)) Lc^-1), Phi = the lower triangle with the diagonal halved: what
    eg_sigma_rhs_vjp computes (a product, two solves with Lc^T and the symmetric part)."""
    Phi = torch.tril(Lc.T @ torch.tril(Lb))
    Phi = Phi - 0.5 * torch.diag(torch.diagonal(Phi))
    Y = torch.linalg.solve_triangular(Lc.T, Phi, upper=True)
    Z = torch.linalg.solve_triangular(Lc.T, Y.T, upper=True).T
    return 0.5 * (Z + Z.T)


@pytest.mark.parametrize("n", [1, 3, 8, 40])
def test_cholesky_vjp_formula_matches_autograd(n):
    rng = np.random.default_rng(n)
    G = rng.standard_normal((n, n))
    A = torch.tensor(G @ G.T + n * np.eye(n), requires_grad=True)
    Lb = torch.tensor(rng.standard_normal((n, n)))
    ref, = torch.autograd.grad(torch.linalg.cholesky(A), A, Lb)
    got = cholesky_vjp(torch.linalg.cholesky(A.detach()), Lb)
    err = float((got - ref).abs().max() / ref.abs().max())
    record(f"ukf_sigma_cholesky_vjp_vs_autograd:n{n}", err)
    assert err < 1e-12, err


# ---- host-side checks of cdk_ukf_grad_sigma_f64 (no CUDA call is made before they return) -----------------------------
@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("libcdk.so not built")
    return L.lib()


def _lib_or_skip(grad):
    if shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"):
        pytest.skip("nvcc is not available")
    return L.lib(b.build_user_drift(VDP, grad=grad))


def _call(lib, **fields):
    d = L.new_desc()
    d.N, d.K, d.n, d.m = 4, 5, 5, 2
    d.drift_id, d.n_theta = L.DRIFT_LORENZ96, 1
    flags = fields.pop("flags", 0)
    null_out = fields.pop("null_out", ())
    for k, v in fields.items():
        if k == "reserved3":
            d.reserved[3] = v
        else:
            setattr(d, k, v)
    d.reserved[2] = flags
    fake = ctypes.c_void_p(0x1000)  # never dereferenced: every check below returns before any device work
    ins = (ctypes.c_void_p * L.NUM_IN)(*([fake] * L.NUM_IN))
    outs = (ctypes.c_void_p * L.NUM_OUT)(*([fake] * L.NUM_OUT))
    for s in null_out:
        outs[s] = None
    return lib.cdk_ukf_grad_sigma_f64(ctypes.byref(d), ins, outs, None), lib.cdk_last_error().decode()


def test_unsupported_requests_are_rejected_on_the_host(lib):
    cases = ((dict(flags=L.FLAG_PREDICT_ONLY), E_UNSUPPORTED), (dict(flags=L.FLAG_DIAG_R), E_UNSUPPORTED),
             (dict(d_u=2), E_UNSUPPORTED), (dict(reserved3=1), E_UNSUPPORTED),
             (dict(reserved3=L.GRAD_REVERSE), E_UNSUPPORTED),
             (dict(null_out=(L.OUT_GRAD,)), E_NULL), (dict(null_out=(L.OUT_SCRATCH,)), E_NULL),
             (dict(n=64, m=64), E_SIZE))
    for fields, code in cases:
        rc, msg = _call(lib, **fields)
        assert rc == code and "cdk_ukf_grad_sigma_f64" in msg, (fields, rc, msg)
    assert "227 KB" in _call(lib, n=64, m=64)[1]
    # the caller's sigma flag is accepted (the entry point sets it on its own copy anyway)
    assert _call(lib, N=0, flags=L.FLAG_UKF_SIGMA_POINTS)[0] == 0


def test_user_drift_by_variant(lib):
    user = dict(drift_id=L.DRIFT_USER, n=2, m=1, n_theta=2, N=0)
    for stock_or_filter in (lib, _lib_or_skip(False)):
        rc, msg = _call(stock_or_filter, **user)
        assert rc == E_UNSUPPORTED and "cdk_ukf_grad_sigma_f64" in msg and "differentiable=True" in msg, msg
    var = _lib_or_skip(True)
    rc, msg = _call(var, **user)
    assert rc == 0, msg
    rc, msg = _call(var, **dict(user, n_theta=8000))
    assert rc == E_SIZE and "cdk_ukf_grad_sigma_f64" in msg and "n_theta = 8000" in msg, msg
    assert _call(var, **dict(user, null_out=(L.OUT_GRAD,), N=3))[0] == E_NULL
    # the closed-form UKF gradient keeps rejecting user drifts, and names the new entry point
    d = L.new_desc()
    d.N, d.K, d.n, d.m, d.drift_id, d.n_theta = 0, 5, 2, 1, L.DRIFT_USER, 2
    fake = ctypes.c_void_p(0x1000)
    ins = (ctypes.c_void_p * L.NUM_IN)(*([fake] * L.NUM_IN))
    outs = (ctypes.c_void_p * L.NUM_OUT)(*([fake] * L.NUM_OUT))
    assert var.cdk_ukf_grad_dense_f64(ctypes.byref(d), ins, outs, None) == E_UNSUPPORTED
    assert "cdk_ukf_grad_sigma_f64" in var.cdk_last_error().decode()
    d.N, d.K, d.solver = 3, 7, L.SOLVERS["rk4"]
    assert var.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ukf_grad_sigma") == lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ukf_grad_sigma")


def test_the_c4_shape_fits_with_every_solver(lib):
    for solver in L.SOLVERS.values():
        rc, msg = _call(lib, n=40, m=20, solver=solver, N=0)
        assert rc == 0, (solver, msg)


def test_scratch_bytes_of_the_new_name_and_the_unchanged_ones(lib):
    d = L.new_desc()
    for (n, m, K, solver) in ((40, 20, 50, "rk4"), (3, 2, 7, "dopri5"), (5, 5, 11, "euler")):
        d.K, d.n, d.m, d.solver = K, n, m, L.SOLVERS[solver]
        st = 2 * ((n + 1) // 2) + n * (n | 1)
        per = 8 * (K * (2 * n + 2 * n * n) + (64 + 2 * _stages(solver)) * st + 1)  # the formula of cdk.h
        for N in (1, 2, 7):
            d.N = N
            assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ukf_grad_sigma") == N * per
    # "cdk_ukf_grad_sigma" contains "kf_grad": it must not be sized as the linear gradient, and the names that existed
    # before keep their sizes
    d.N, d.K, d.n, d.m, d.solver = 3, 20, 4, 2, L.SOLVERS["rk4"]
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_kf_grad") == 805656
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ukf_grad_sigma") == 60696
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ukf_grad_dense") == 60696
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad_dense") == 60696
    d.N, d.K, d.n, d.m = 1, 50, 3, 1
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad") == 0
    d.reserved[3] = L.GRAD_REVERSE
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad") == 50 * 24 * 8


def test_the_entry_point_is_exported_and_in_the_xla_table(lib):
    assert "cdk_ukf_grad_sigma_f64" in L.ENTRY_POINTS
    assert hasattr(lib, "cdk_ukf_grad_sigma_f64")
    src = open(os.path.join(os.path.dirname(L.__file__), "csrc", "cdk_api.cu")).read()
    assert '{"cdk_ukf_grad_sigma_f64", cdk_ukf_grad_sigma_f64}' in src


# ---- ukf_sigma_points_marginal_log_prob_and_grad on the host --------------------------------------------------------
def test_mis_shaped_inputs_raise_before_the_library_is_loaded(no_device):  # noqa: F811
    N, K, n, m = 4, 5, 5, 2
    p = random_model("lorenz96", n, m, seed=1)
    y = np.zeros((N, K, m))
    t = np.tile(np.arange(K) * 0.01, (N, 1))[..., None]
    for key, bad in (("H", np.zeros((m, n + 1))), ("R", np.eye(m + 1)), ("P0", np.eye(n - 1)), ("m0", np.zeros((3, n))),
                     ("L", np.zeros((N + 1, n, n)))):
        q = dict(p)
        q[key] = bad
        with pytest.raises(ValueError):
            cd.ukf_sigma_points_marginal_log_prob_and_grad(api_params("lorenz96", n, m, q), y, t, wrt="all")


def test_host_rejections_of_the_python_entry(no_device, monkeypatch):  # noqa: F811
    N, K, n, m = 2, 4, 5, 2
    p = random_model("lorenz96", n, m, seed=2)
    params = api_params("lorenz96", n, m, p)
    y, t = np.zeros((N, K, m)), np.tile(np.arange(K) * 0.01, (N, 1))[..., None]
    with pytest.raises(NotImplementedError):
        cd.ukf_sigma_points_marginal_log_prob_and_grad(params, y.astype(np.float32), t)
    with pytest.raises(NotImplementedError):
        cd.ukf_sigma_points_marginal_log_prob_and_grad(params, y, t, inputs=np.ones((N, K, 1)))
    with pytest.raises(ValueError):
        cd.ukf_sigma_points_marginal_log_prob_and_grad(params, y, t, wrt=("nonsense",))
    for flag in ("0", "1"):  # the sigma-point filter is differentiated whatever the environment says
        monkeypatch.setenv("CDK_UKF_SIGMA_POINTS", flag)
        with pytest.raises(Exception) as e:
            cd.ukf_sigma_points_marginal_log_prob_and_grad(params, y, t, inputs=np.zeros((N, K, 1)))
        assert type(e.value).__name__ == "_Sentinel"


def test_non_differentiable_user_drift_is_rejected_before_any_build(monkeypatch):
    def boom(*a, **k):
        raise _Sentinel()
    monkeypatch.setattr(b, "build_user_drift", boom)
    monkeypatch.setattr(L, "lib", boom)
    y, t = np.zeros((3, 5, 1)), np.cumsum(np.full((3, 5), 0.1), 1)[..., None]
    p = _params(cd.LearnableUserDrift(device_code=VDP, theta=np.array([1.3, 0.4])))
    from cd_dynamax_b200.autograd import ukf_sigma_points_marginal_log_prob
    for fn in (cd.ukf_sigma_points_marginal_log_prob_and_grad, ukf_sigma_points_marginal_log_prob):
        with pytest.raises(NotImplementedError, match="differentiable=True"):
            fn(p, y, t)
    seen = []
    monkeypatch.setattr(b, "build_user_drift", lambda code, grad=False: seen.append(grad) or boom())
    with pytest.raises(_Sentinel):
        cd.ukf_sigma_points_marginal_log_prob_and_grad(
            _params(cd.LearnableUserDrift(VDP, np.array([1.3, 0.4]), differentiable=True)), y, t)
    assert seen == [True]
    # the closed-form entry keeps rejecting user drifts, and points to the new function
    with pytest.raises(NotImplementedError, match="ukf_sigma_points_marginal_log_prob_and_grad"):
        cd.ukf_marginal_log_prob_and_grad(_params(cd.LearnableUserDrift(VDP, np.array([1.3, 0.4]), differentiable=True)),
                                          y, t)


def test_exports():
    from cd_dynamax_b200 import autograd
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm import ukf_sigma_points_marginal_log_prob_and_grad
    assert cd.ukf_sigma_points_marginal_log_prob_and_grad is ukf_sigma_points_marginal_log_prob_and_grad
    assert callable(autograd.ukf_sigma_points_marginal_log_prob)
