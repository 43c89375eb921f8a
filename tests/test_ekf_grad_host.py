"""CPU side of the CD-EKF gradient for every registry drift (cdk_ekf_grad_dense_f64): the torch arbiter
(oracle/cd_torch_ekf.py) against the NumPy oracle, its autograd gradient against central differences of the oracle, and
the host-side checks of the entry point and of ekf_marginal_log_prob_and_grad."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import cd_oracle as o
from oracle import cd_torch_ekf as te
from tests.helpers import make_drift
from tests.test_kf_grad_host import random_grid

DRIFTS = ("linear", "lorenz63", "lorenz96", "quadratic")
BLOCKS = ("theta", "Sigma", "H", "d", "R", "m0", "P0")
SYMMETRIC = ("Sigma", "R", "P0")


def n_theta(kind, n):
    return {"linear": n * n + n, "lorenz63": 3, "lorenz96": 1, "quadratic": n + n * n + n ** 3}[kind]


def random_theta(kind, n, rng, lead=()):
    if kind == "lorenz63":
        return np.array([10.0, 28.0, 8.0 / 3.0]) * (1.0 + 0.05 * rng.standard_normal(lead + (3,)))
    if kind == "lorenz96":
        return 8.0 + 0.5 * rng.standard_normal(lead + (1,))
    if kind == "linear":
        W = -0.6 * np.eye(n) + 0.4 * rng.standard_normal(lead + (n, n)) / np.sqrt(n)
        return np.concatenate([W.reshape(lead + (n * n,)), 0.1 * rng.standard_normal(lead + (n,))], -1)
    a = 0.1 * rng.standard_normal(lead + (n,))
    B = (-0.8 * np.eye(n) + 0.3 * rng.standard_normal(lead + (n, n)) / np.sqrt(n)).reshape(lead + (n * n,))
    C = 0.1 * rng.standard_normal(lead + (n ** 3,)) / n
    return np.concatenate([a, B, C], -1)


def random_model(kind, n, m, seed, N=None):
    """theta of the drift, SPD Sigma / R / P0, with every parameter carrying a leading N when N is given."""
    rng = np.random.default_rng(seed)
    lead = () if N is None else (N,)

    def spd(k, scale):
        A = rng.standard_normal(lead + (k, k))
        return scale * (A @ np.swapaxes(A, -1, -2) / k + np.eye(k))

    L = np.eye(n) + 0.2 * rng.standard_normal(lead + (n, n))
    Qc = spd(n, 0.3)
    chaotic = kind in ("lorenz63", "lorenz96")
    return dict(kind=kind, theta=random_theta(kind, n, rng, lead), L=L, Qc=Qc, Sigma=L @ Qc @ np.swapaxes(L, -1, -2),
                H=rng.standard_normal(lead + (m, n)) / np.sqrt(n), d=0.1 * rng.standard_normal(lead + (m,)),
                R=spd(m, 0.5), m0=(1.0 if chaotic else 0.3) * rng.standard_normal(lead + (n,)) + (2.0 if chaotic else 0.0),
                P0=spd(n, 0.5))


def random_data(p, N, K, seed):
    m = p["H"].shape[-2]
    rng = np.random.default_rng(seed)
    scale = 3.0 if p["kind"] in ("lorenz63", "lorenz96") else 0.5
    return scale * rng.standard_normal((N, K, m))


def oracle_filter(p, y, t, settings, order, dt_final=1e-10):
    n = p["m0"].shape[-1]
    op = o.NonlinearParams(m0=p["m0"], P0=p["P0"], drift=make_drift(p["kind"], p["theta"], n), L=p["L"], Qc=p["Qc"],
                           H=p["H"], R=p["R"], d=p["d"])
    return o.extended_kalman_filter(op, y, t, dt_final=dt_final, state_order=order, settings=settings)


def arbiter(p, y, t, settings, order, dt_final=1e-10, requires_grad=False):
    ts = {k: torch.tensor(np.asarray(p[k], np.float64), requires_grad=requires_grad) for k in BLOCKS}
    return ts, te.extended_kalman_filter(p["kind"], *(ts[k] for k in BLOCKS), y, t, dt_final, order, settings)


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.mark.parametrize("solver", ["euler", "rk4", "dopri5"])
@pytest.mark.parametrize("order", ["first", "second"])
@pytest.mark.parametrize("kind", DRIFTS)
def test_arbiter_matches_oracle(kind, order, solver):
    N, K, m = 3, 8, 2
    n = 3 if kind == "lorenz63" else (5 if kind == "lorenz96" else 3)
    p = random_model(kind, n, m, seed=DRIFTS.index(kind) * 2 + (order == "second"), N=N if kind == "quadratic" else None)
    y = random_data(p, N, K, 2)
    t = random_grid(N, K, 3, mean_gap=0.03)
    settings = o.SolverSettings(solver, 0.01)
    ref = oracle_filter(p, y, t, settings, order)
    _, out = arbiter(p, y, t, settings, order)
    for fld in ("marginal_loglik", "filtered_means", "filtered_covariances", "predicted_means", "predicted_covariances"):
        assert rel(out[fld].numpy(), ref[fld]) < 1e-12, fld
    assert np.array_equal(out["status"], ref["status"])


@pytest.mark.parametrize("kind,order,solver", [("linear", "first", "heun"), ("lorenz63", "second", "rk4"),
                                               ("lorenz96", "first", "dopri5"), ("quadratic", "second", "rk4"),
                                               ("quadratic", "first", "bosh3")])
def test_arbiter_gradient_matches_central_differences_of_the_oracle(kind, order, solver):
    N, K, m = 2, 6, 2
    n = 3 if kind != "lorenz96" else 5
    settings = o.SolverSettings(solver, 0.01)
    p = random_model(kind, n, m, seed=21)
    y = random_data(p, N, K, 22)
    t = random_grid(N, K, 23, mean_gap=0.03)
    ts, out = arbiter(p, y, t, settings, order, requires_grad=True)
    grads = torch.autograd.grad(out["marginal_loglik"].sum(), [ts[k] for k in BLOCKS])
    rng = np.random.default_rng(24)
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
            return oracle_filter(q, y, t, settings, order)["marginal_loglik"].sum()

        fd = (ll_at(h) - ll_at(-h)) / (2 * h)
        an = float(np.sum(g.numpy() * v))
        assert abs(an - fd) <= 1e-6 * max(abs(fd), 1.0), (name, an, fd)


# ---- host-side checks of cdk_ekf_grad_dense_f64 (no CUDA call is made before they return) ----------------------------
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
    d.drift_id, d.n_theta, d.state_order = L.DRIFT_LORENZ96, 1, 1
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
    return lib.cdk_ekf_grad_dense_f64(ctypes.byref(d), ins, outs, None), lib.cdk_last_error().decode()


def test_unsupported_requests_are_rejected_on_the_host(lib):
    from cd_dynamax_b200 import _lib as L
    E_NULL, E_SIZE, E_UNSUPPORTED = -1, -2, -4
    cases = ((dict(state_order=0), E_UNSUPPORTED), (dict(num_iter=2), E_UNSUPPORTED),
             (dict(drift_id=L.DRIFT_USER), E_UNSUPPORTED), (dict(flags=L.FLAG_DIAG_R), E_UNSUPPORTED),
             (dict(flags=L.FLAG_PREDICT_ONLY), E_UNSUPPORTED), (dict(d_u=2), E_UNSUPPORTED),
             (dict(reserved3=1), E_UNSUPPORTED), (dict(reserved3=L.GRAD_REVERSE), E_UNSUPPORTED),
             (dict(null_out=(L.OUT_GRAD,)), E_NULL), (dict(null_out=(L.OUT_SCRATCH,)), E_NULL),
             (dict(n=64, m=64), E_SIZE))
    for fields, code in cases:
        rc, msg = _call(lib, **fields)
        assert rc == code and "cdk_ekf_grad_dense_f64" in msg, (fields, rc, msg)
    rc, msg = _call(lib, n=64, m=64)
    assert "227 KB" in msg


def test_the_c4_shape_fits_with_every_solver(lib):
    from cd_dynamax_b200 import _lib as L
    for solver in L.SOLVERS.values():
        rc, msg = _call(lib, n=40, m=20, solver=solver, N=0)
        assert rc == 0, (solver, msg)


def test_column_count():
    from cd_dynamax_b200 import _lib as L
    for kind, n, m in (("linear", 4, 2), ("lorenz63", 3, 3), ("lorenz96", 40, 20), ("quadratic", 2, 1)):
        nt = n_theta(kind, n)
        assert L.grad_cols_ekf(n, m, nt) == nt + n * n + m * n + m + m * m + n + n * n
    # a LearnableLinear drift: theta = W | bias is the F | b of the linear model's layout
    assert L.grad_cols_ekf(5, 3, 30) == L.grad_cols_kf(5, 3)


def _stages(solver):
    return len(o.TABLEAUX[solver]["b"])


def test_scratch_bytes_formula_and_names(lib):
    from cd_dynamax_b200 import _lib as L
    d = L.new_desc()
    for (n, m, K, solver) in ((40, 20, 50, "rk4"), (3, 2, 7, "dopri5"), (5, 5, 11, "euler")):
        d.K, d.n, d.m, d.solver = K, n, m, L.SOLVERS[solver]
        st = 2 * ((n + 1) // 2) + n * (n | 1)
        sizes = []
        for N in (1, 2, 7):
            d.N = N
            sizes.append(lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad_dense"))
        per = 8 * (K * (2 * n + 2 * n * n) + (64 + 2 * _stages(solver)) * st + 1)
        assert sizes == [per, 2 * per, 7 * per], (n, m, K, solver)
    # the existing names keep their sizes
    d.N, d.K, d.n, d.m = 1, 50, 3, 1
    d.reserved[3] = L.GRAD_REVERSE
    assert lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad") == 50 * 24 * 8


# ---- ekf_marginal_log_prob_and_grad on the host ---------------------------------------------------------------------
class _Sentinel(Exception):
    pass


@pytest.fixture
def no_device(monkeypatch):
    from cd_dynamax_b200 import _engine, _lib

    def boom(*a, **k):
        raise _Sentinel()

    monkeypatch.setattr(_lib, "lib", boom)
    monkeypatch.setattr(_engine, "device", boom)


def api_params(kind, n, m, p, batched_drift=False):
    import cd_dynamax_b200 as cd
    th = np.asarray(p["theta"])
    if kind == "linear":
        drift = cd.LearnableLinear(weights=th[..., :n * n].reshape(th.shape[:-1] + (n, n)), bias=th[..., n * n:])
    elif kind == "lorenz63":
        drift = cd.LearnableLorenz63(sigma=th[..., 0], rho=th[..., 1], beta=th[..., 2])
    elif kind == "lorenz96":
        drift = cd.LearnableLorenz96(forcing=th[..., 0])
    else:
        lead = th.shape[:-1]
        drift = cd.LearnableQuadratic(a=th[..., :n], B=th[..., n:n + n * n].reshape(lead + (n, n)),
                                      C=th[..., n + n * n:].reshape(lead + (n, n, n)))
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(p["m0"]), cov=cd.LearnableMatrix(p["P0"])),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=drift, diffusion_coefficient=cd.LearnableMatrix(p["L"]),
                                           diffusion_cov=cd.LearnableMatrix(p["Qc"])),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=p["H"], bias=p["d"]),
                                             emission_cov=cd.LearnableMatrix(p["R"])))


def test_mis_shaped_inputs_raise_before_the_library_is_loaded(no_device):
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
            cd.ekf_marginal_log_prob_and_grad(api_params("lorenz96", n, m, q), y, t, cd.EKFHyperParams(), wrt="all")
    q = dict(p, theta=np.full((N + 2, 1), 8.0))  # a batched forcing whose leading axis is not N
    with pytest.raises(ValueError):
        cd.ekf_marginal_log_prob_and_grad(api_params("lorenz96", n, m, q), y, t, cd.EKFHyperParams(), wrt="all")


def test_host_rejections_of_the_python_entry(no_device):
    import cd_dynamax_b200 as cd
    N, K, n, m = 2, 4, 5, 2
    p = random_model("lorenz96", n, m, seed=2)
    y, t = np.zeros((N, K, m)), np.tile(np.arange(K) * 0.01, (N, 1))[..., None]
    with pytest.raises(NotImplementedError):
        cd.ekf_marginal_log_prob_and_grad(api_params("lorenz96", n, m, p), y, t, cd.EKFHyperParams(state_order="zeroth"))
    with pytest.raises(NotImplementedError):
        cd.ekf_marginal_log_prob_and_grad(api_params("lorenz96", n, m, p), y.astype(np.float32), t)
    user = api_params("lorenz96", n, m, p)._replace(
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableUserDrift(device_code="", theta=np.zeros(1)),
                                           diffusion_coefficient=p["L"], diffusion_cov=p["Qc"]))
    with pytest.raises(NotImplementedError):
        cd.ekf_marginal_log_prob_and_grad(user, y, t)


@pytest.mark.parametrize("kind", DRIFTS)
def test_unflatten_theta_per_drift(kind):
    import cd_dynamax_b200 as cd
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm import inference_ekf as ie
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm.cdnlgssm_utils import drift_to_theta
    N, n = 3, 3
    p = random_model(kind, n, 1, seed=5, N=N)
    drift = api_params(kind, n, 1, p).dynamics.drift
    _, theta, nt = drift_to_theta(drift, n)
    assert theta.shape == (N, nt) == (N, n_theta(kind, n))
    parts = ie.unflatten_theta(theta, drift, n)
    assert list(parts) == [name for name, _ in ie.drift_leaves(drift, n)]
    for name, v in parts.items():  # the batched leaves come back with their own shapes, bit for bit
        np.testing.assert_array_equal(v.numpy(), np.asarray(getattr(drift, name), np.float64).reshape(v.shape))


def test_lorenz63_entry_keeps_its_scalar_emission_contract(no_device):
    """ekf_marginal_log_prob_and_grad serves Lorenz-63 with a scalar emission only (its own kernels); the dense entry
    point takes the model with two components and reaches the shape checks (here: a mis-shaped R)."""
    import cd_dynamax_b200 as cd
    N, K, m = 2, 4, 2
    p = random_model("lorenz63", 3, m, seed=3)
    y, t = np.zeros((N, K, m)), np.tile(np.arange(K) * 0.01, (N, 1))[..., None]
    with pytest.raises(NotImplementedError, match="ekf_dense_marginal_log_prob_and_grad"):
        cd.ekf_marginal_log_prob_and_grad(api_params("lorenz63", 3, m, p), y, t)
    with pytest.raises(ValueError):
        cd.ekf_dense_marginal_log_prob_and_grad(api_params("lorenz63", 3, m, dict(p, R=np.eye(3))), y, t)
