"""CPU side of the CD-UKF gradient for every registry drift (cdk_ukf_grad_dense_f64): the two torch restatements
(oracle/cd_torch_ukf.py, closed form and literal sigma points) against the NumPy oracle, their autograd gradients against
central differences of the oracle and against each other, and the host-side checks of the entry point and of
ukf_marginal_log_prob_and_grad."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import cd_oracle as o
from oracle import cd_torch_ukf as tu
from tests.helpers import make_drift, record
from tests.test_ekf_grad_host import (BLOCKS, SYMMETRIC, _stages, api_params, no_device, random_data,  # noqa: F401
                                     random_model, rel)
from tests.test_kf_grad_host import random_grid

DRIFTS = ("linear", "lorenz63", "lorenz96", "quadratic")


def oracle_filter(p, y, t, settings, dt_final=1e-10):
    n = p["m0"].shape[-1]
    op = o.NonlinearParams(m0=p["m0"], P0=p["P0"], drift=make_drift(p["kind"], p["theta"], n), L=p["L"], Qc=p["Qc"],
                           H=p["H"], R=p["R"], d=p["d"])
    return o.unscented_kalman_filter(op, y, t, dt_final=dt_final, settings=settings)


def restated(p, y, t, settings, closed, requires_grad=False):
    ts = {k: torch.tensor(np.asarray(p[k], np.float64), requires_grad=requires_grad) for k in BLOCKS}
    return ts, tu.unscented_kalman_filter(p["kind"], *(ts[k] for k in BLOCKS), y, t, settings=settings, closed=closed)


FIELDS = ("marginal_loglik", "filtered_means", "filtered_covariances", "predicted_means", "predicted_covariances")


@pytest.mark.parametrize("solver", ["euler", "rk4", "dopri5"])
@pytest.mark.parametrize("kind", DRIFTS)
def test_restatements_match_the_oracle(kind, solver):
    N, K, m = 3, 8, 2
    n = 5 if kind == "lorenz96" else 3
    p = random_model(kind, n, m, seed=DRIFTS.index(kind) + 40, N=N if kind == "quadratic" else None)
    y = random_data(p, N, K, 2)
    t = random_grid(N, K, 3, mean_gap=0.03)
    settings = o.SolverSettings(solver, 0.01)
    ref = oracle_filter(p, y, t, settings)
    _, lit = restated(p, y, t, settings, "sigma")
    _, cf = restated(p, y, t, settings, "closed")
    gap = 0.0
    for fld in FIELDS:
        assert rel(lit[fld].numpy(), ref[fld]) < 1e-12, fld
        gap = max(gap, rel(cf[fld].numpy(), ref[fld]))
    record(f"ukf_torch_closed_vs_oracle:{kind}:{solver}", gap)
    # the closed form differs from the sigma-point sums by the rounding of their f(X+) - f(X-) cancellation
    assert gap < 1e-11, gap
    assert np.array_equal(lit["status"], ref["status"]) and np.array_equal(cf["status"], ref["status"])


@pytest.mark.parametrize("closed", ["closed", "sigma"])
@pytest.mark.parametrize("kind,solver", [("linear", "heun"), ("lorenz63", "rk4"), ("lorenz96", "dopri5"),
                                         ("quadratic", "rk4")])
def test_restated_gradient_matches_central_differences_of_the_oracle(kind, solver, closed):
    N, K, m = 2, 6, 2
    n = 3 if kind != "lorenz96" else 5
    settings = o.SolverSettings(solver, 0.01)
    p = random_model(kind, n, m, seed=61)
    y = random_data(p, N, K, 62)
    t = random_grid(N, K, 63, mean_gap=0.03)
    ts, out = restated(p, y, t, settings, closed, requires_grad=True)
    grads = torch.autograd.grad(out["marginal_loglik"].sum(), [ts[k] for k in BLOCKS])
    rng = np.random.default_rng(64)
    for name, g in zip(BLOCKS, grads):
        v = rng.standard_normal(np.shape(p[name]))
        if name in SYMMETRIC:
            v = 0.5 * (v + v.T)
        h = 1e-6 if name == "theta" else 1e-5

        def ll_at(s):
            q = dict(p)
            q[name] = p[name] + s * v
            if name == "Sigma":  # the oracle takes L and Qc: move Qc so that L Qc L^T moves by s v
                q["Qc"] = p["Qc"] + s * np.linalg.solve(p["L"], np.linalg.solve(p["L"], v).T).T
            return oracle_filter(q, y, t, settings)["marginal_loglik"].sum()

        fd = (ll_at(h) - ll_at(-h)) / (2 * h)
        an = float(np.sum(g.numpy() * v))
        assert abs(an - fd) <= 1e-6 * max(abs(fd), 1.0), (name, an, fd)


@pytest.mark.parametrize("kind", DRIFTS)
def test_closed_form_and_sigma_point_gradients_agree(kind):
    N, K, m = 2, 10, 2
    n = 5 if kind == "lorenz96" else 3
    settings = o.SolverSettings("rk4", 0.01)
    p = random_model(kind, n, m, seed=70 + DRIFTS.index(kind))
    y = random_data(p, N, K, 71)
    t = random_grid(N, K, 72, mean_gap=0.03)
    g = {}
    for closed in ("closed", "sigma"):
        ts, out = restated(p, y, t, settings, closed, requires_grad=True)
        g[closed] = torch.autograd.grad(out["marginal_loglik"].sum(), [ts[k] for k in BLOCKS])
    worst = 0.0
    for name, a, b in zip(BLOCKS, g["closed"], g["sigma"]):
        a, b = a.numpy(), b.numpy()
        if name in SYMMETRIC:  # only the symmetric parts are parameter gradients
            a, b = 0.5 * (a + a.T), 0.5 * (b + b.T)
        worst = max(worst, rel(a, b))
    record(f"ukf_torch_closed_vs_sigma_grad:{kind}", worst)
    assert worst < 1e-9, worst


# ---- host-side checks of cdk_ukf_grad_dense_f64 (no CUDA call is made before they return) ----------------------------
@pytest.fixture(scope="module")
def lib():
    from cd_dynamax_b200 import _lib as L
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("libcdk.so not built")
    return L.lib()


def _call(lib, **fields):
    from cd_dynamax_b200 import _lib as L
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
    return lib.cdk_ukf_grad_dense_f64(ctypes.byref(d), ins, outs, None), lib.cdk_last_error().decode()


def test_unsupported_requests_are_rejected_on_the_host(lib):
    from cd_dynamax_b200 import _lib as L
    E_NULL, E_SIZE, E_UNSUPPORTED = -1, -2, -4
    cases = ((dict(drift_id=L.DRIFT_USER), E_UNSUPPORTED), (dict(flags=L.FLAG_UKF_SIGMA_POINTS), E_UNSUPPORTED),
             (dict(flags=L.FLAG_PREDICT_ONLY), E_UNSUPPORTED), (dict(flags=L.FLAG_DIAG_R), E_UNSUPPORTED),
             (dict(d_u=2), E_UNSUPPORTED), (dict(reserved3=1), E_UNSUPPORTED),
             (dict(reserved3=L.GRAD_REVERSE), E_UNSUPPORTED),
             (dict(null_out=(L.OUT_GRAD,)), E_NULL), (dict(null_out=(L.OUT_SCRATCH,)), E_NULL),
             (dict(n=64, m=64), E_SIZE))
    for fields, code in cases:
        rc, msg = _call(lib, **fields)
        assert rc == code and "cdk_ukf_grad_dense_f64" in msg, (fields, rc, msg)
    rc, msg = _call(lib, n=64, m=64)
    assert "227 KB" in msg


def test_state_order_and_num_iter_are_ignored(lib):
    for fields in (dict(state_order=0), dict(state_order=1), dict(num_iter=3)):
        rc, msg = _call(lib, N=0, **fields)
        assert rc == 0, (fields, msg)


def test_the_c4_shape_fits_with_every_solver(lib):
    from cd_dynamax_b200 import _lib as L
    for solver in L.SOLVERS.values():
        rc, msg = _call(lib, n=40, m=20, solver=solver, N=0)
        assert rc == 0, (solver, msg)


def test_scratch_bytes_of_the_new_name_and_the_unchanged_ones(lib):
    from cd_dynamax_b200 import _lib as L
    d = L.new_desc()
    for (n, m, K, solver) in ((40, 20, 50, "rk4"), (3, 2, 7, "dopri5"), (5, 5, 11, "euler")):
        d.K, d.n, d.m, d.solver = K, n, m, L.SOLVERS[solver]
        st = 2 * ((n + 1) // 2) + n * (n | 1)
        per = 8 * (K * (2 * n + 2 * n * n) + (64 + 2 * _stages(solver)) * st + 1)
        for N in (1, 2, 7):
            d.N = N
            assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ukf_grad_dense") == N * per
            assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad_dense") == N * per
    # the names that existed before keep their sizes: the linear gradient's (the value before this entry point existed;
    # "cdk_ukf_grad_dense" contains "kf_grad" too, and must not be sized as the linear gradient) ...
    d.N, d.K, d.n, d.m, d.solver = 3, 20, 4, 2, L.SOLVERS["rk4"]
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_kf_grad") == 805656
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ukf_grad_dense") == 60696
    # ... and the Lorenz-63 kernels' (reverse mode only)
    d.N, d.K, d.n, d.m = 1, 50, 3, 1
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad") == 0
    d.reserved[3] = L.GRAD_REVERSE
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad") == 50 * 24 * 8


# ---- ukf_marginal_log_prob_and_grad on the host ---------------------------------------------------------------------
def test_mis_shaped_inputs_raise_before_the_library_is_loaded(no_device):  # noqa: F811
    import cd_dynamax_b200 as cd
    N, K, n, m = 4, 5, 5, 2
    p = random_model("lorenz96", n, m, seed=1)
    y = np.zeros((N, K, m))
    t = np.tile(np.arange(K) * 0.01, (N, 1))[..., None]
    for key, bad in (("H", np.zeros((m, n + 1))), ("R", np.eye(m + 1)), ("P0", np.eye(n - 1)), ("m0", np.zeros((3, n))),
                     ("L", np.zeros((N + 1, n, n)))):
        q = dict(p)
        q[key] = bad
        with pytest.raises(ValueError):
            cd.ukf_marginal_log_prob_and_grad(api_params("lorenz96", n, m, q), y, t, cd.UKFHyperParams(), wrt="all")
    q = dict(p, theta=np.full((N + 2, 1), 8.0))  # a batched forcing whose leading axis is not N
    with pytest.raises(ValueError):
        cd.ukf_marginal_log_prob_and_grad(api_params("lorenz96", n, m, q), y, t, cd.UKFHyperParams(), wrt="all")


def test_host_rejections_of_the_python_entry(no_device, monkeypatch):  # noqa: F811
    import cd_dynamax_b200 as cd
    N, K, n, m = 2, 4, 5, 2
    p = random_model("lorenz96", n, m, seed=2)
    params = api_params("lorenz96", n, m, p)
    y, t = np.zeros((N, K, m)), np.tile(np.arange(K) * 0.01, (N, 1))[..., None]
    with pytest.raises(NotImplementedError):
        cd.ukf_marginal_log_prob_and_grad(params, y.astype(np.float32), t)
    with pytest.raises(NotImplementedError):
        cd.ukf_marginal_log_prob_and_grad(params, y, t, inputs=np.ones((N, K, 1)))
    user = params._replace(
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableUserDrift(device_code="", theta=np.zeros(1)),
                                           diffusion_coefficient=p["L"], diffusion_cov=p["Qc"]))
    with pytest.raises(NotImplementedError):
        cd.ukf_marginal_log_prob_and_grad(user, y, t)
    with pytest.raises(ValueError):
        cd.ukf_marginal_log_prob_and_grad(params, y, t, wrt=("nonsense",))
    monkeypatch.setenv("CDK_UKF_SIGMA_POINTS", "1")
    with pytest.raises(NotImplementedError):
        cd.ukf_marginal_log_prob_and_grad(params, y, t)
    monkeypatch.setenv("CDK_UKF_SIGMA_POINTS", "0")
    with pytest.raises(Exception) as e:  # zero inputs are accepted: the call goes on to the (absent) device
        cd.ukf_marginal_log_prob_and_grad(params, y, t, inputs=np.zeros((N, K, 1)))
    assert type(e.value).__name__ == "_Sentinel"


def test_exports():
    import cd_dynamax_b200 as cd
    from cd_dynamax_b200 import autograd
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm import ukf_marginal_log_prob_and_grad
    assert cd.ukf_marginal_log_prob_and_grad is ukf_marginal_log_prob_and_grad
    assert callable(autograd.ukf_marginal_log_prob)
