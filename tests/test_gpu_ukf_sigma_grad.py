"""cdk_ukf_grad_sigma_f64 / ukf_sigma_points_marginal_log_prob_and_grad / autograd.ukf_sigma_points_marginal_log_prob on
the GPU: the gradient of the CD-UKF with literal sigma points, for every registry drift and for user-defined drifts
(LearnableUserDrift(..., differentiable=True)).

The reference is torch autograd of the sigma-point restatement (oracle/cd_torch_ukf.py, closed="sigma", and for user
drifts tests/test_ukf_sigma_grad_host.sigma_filter with the same drift in torch), gated at 1e-9 of each block's max
|value|; Sigma, R and P0 are compared on their symmetric parts.  Cross-checks: the closed-form gradient
(cdk_ukf_grad_dense_f64) of the same registry models, user restatements of registry drifts against the registry's
sigma-point gradient, and central differences of the sigma-point filter itself."""
import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _engine as E
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200 import build as b
from cd_dynamax_b200.autograd import ukf_sigma_points_marginal_log_prob
from oracle import cd_oracle as o
from tests.helpers import record, scaled_err
from tests.test_ekf_grad_host import BLOCKS, n_theta, random_model
from tests.test_gpu_ekf_grad import _ins, blocks, sym
from tests.test_gpu_time_grids import degenerate_grid, edge_grid, long_grid, regular_grid
from tests.test_gpu_ukf_grad import _fields, case, dense, reference
from tests.test_gpu_user_drift_grad import CODE, FNS, L63, MLP, QUAD, VDP, user_model
from tests.test_kf_grad_host import random_grid
from tests.test_ukf_sigma_grad_host import sigma_filter

pytestmark = pytest.mark.gpu
GATE = 1e-9         # against torch autograd of the sigma-point restatement
GATE_CLOSED = 1e-8  # against the closed-form gradient of the same registry model


def sigma(p, y, t, solver, dt0, max_steps=100000, fields=None):
    """(ll, status, G [N, cols]) of cdk_ukf_grad_sigma_f64, device tensors."""
    N, K, m = y.shape
    n = np.shape(p["m0"])[-1]
    nt = np.shape(p["theta"])[-1]
    out = E.run("cdk_ukf_grad_sigma", "f64", N, K, n, m, _ins(p, y, t), (L.OUT_LL, L.OUT_GRAD),
                fields or _fields(p, solver, dt0, max_steps), out_shapes={L.OUT_GRAD: (N, L.grad_cols_ekf(n, m, nt))})
    return out[L.OUT_LL], out[L.OUT_STATUS], out[L.OUT_GRAD]


def sigma_filter_ll(p, y, t, fields):
    N, K, m = y.shape
    n = np.shape(p["m0"])[-1]
    return E.run("cdk_ukf_filter", "f64", N, K, n, m, _ins(p, y, t), (L.OUT_LL,),
                 dict(fields, flags=L.FLAG_UKF_SIGMA_POINTS))[L.OUT_LL]


def check(name, got, ref, gate):
    worst = 0.0
    for k, r in ref.items():
        r = sym(r) if k in ("Sigma", "R", "P0") else r
        err = scaled_err(got[k], r)
        record(f"ukf_grad_sigma:{name}:{k}", err)
        worst = max(worst, err)
        assert err < gate, (name, k, err)
    return worst


def compare(name, p, y, t, solver, dt0):
    """Every block against torch autograd of closed="sigma" and against the closed-form gradient."""
    ll, status, G = sigma(p, y, t, solver, dt0)
    assert int(status.abs().sum()) == 0, name
    assert torch.equal(ll, sigma_filter_ll(p, y, t, _fields(p, solver, dt0))), name
    n, m = np.shape(p["m0"])[-1], y.shape[-1]
    got = blocks(G, n, m, n_theta(p["kind"], n))
    ref_ll, ref = reference(p, y, t, solver, dt0, "sigma")
    err_ll = scaled_err(ll.cpu().numpy(), ref_ll)
    record(f"ukf_grad_sigma:{name}:ll", err_ll)
    assert err_ll < 1e-11, (name, err_ll)
    worst = check(name, got, ref, GATE)
    _, _, Gc = dense(p, y, t, solver, dt0)
    closed = blocks(Gc, n, m, n_theta(p["kind"], n))
    check(f"{name}:vs_closed_form", got, {k: v for k, v in closed.items()}, GATE_CLOSED)
    return worst


@pytest.mark.parametrize("m", [1, 2, 3])
def test_lorenz63_every_emission_size(m):
    p, y, t = case("lorenz63", 3, m, seed=m)
    compare(f"l63_m{m}", p, y, t, "rk4", 0.01)


@pytest.mark.parametrize("n,solver", [(5, "dopri5"), (40, "rk4"), (40, "dopri5")])
def test_lorenz96(n, solver):
    p, y, t = case("lorenz96", n, n // 2, N=2, K=8, seed=n)
    compare(f"l96_n{n}_{solver}", p, y, t, solver, 0.01)


@pytest.mark.parametrize("n", [1, 4])
def test_linear_drift(n):
    p, y, t = case("linear", n, 2, seed=10 + n, batched=(n == 4))
    compare(f"linear_n{n}", p, y, t, "rk4", 0.01)


def test_quadratic_drift():
    p, y, t = case("quadratic", 2, 2, seed=22, batched=True)
    compare("quadratic_n2", p, y, t, "rk4", 0.01)


@pytest.mark.parametrize("solver", list(L.SOLVERS))
def test_every_solver(solver):
    p, y, t = case("lorenz96", 5, 3, seed=30)
    compare(f"solver_{solver}", p, y, t, solver, 0.01)


@pytest.mark.parametrize("grid", ["t0_1e4", "edge", "degenerate", "long"])
def test_time_grids(grid):
    N, K, dt0 = 3, 8, 0.01
    p = random_model("linear", 4, 2, seed=40)
    t = {"t0_1e4": lambda: regular_grid(N, K, t0=1e4, h=0.013), "edge": lambda: edge_grid(N, K, dt0),
         "degenerate": lambda: degenerate_grid(N, K, dt0), "long": lambda: long_grid(N, 6, dt0)}[grid]()
    from tests.test_ekf_grad_host import random_data
    y = random_data(p, N, t.shape[1], 41)
    compare(f"grid_{grid}", p, y, t, "rk4", dt0)


@pytest.mark.parametrize("slot", ("theta", "L", "Qc", "H", "d", "R", "m0", "P0"))
def test_each_leaf_batched_alone(slot):
    N = 4
    p, y, t = case("quadratic", 2, 2, N=N, K=8, seed=90)
    _, _, G0 = sigma(p, y, t, "rk4", 0.01)
    q = dict(p)
    q[slot] = np.broadcast_to(np.asarray(p[slot]), (N,) + np.shape(p[slot])).copy()
    _, _, G = sigma(q, y, t, "rk4", 0.01)
    assert torch.equal(G, G0), slot
    rng = np.random.default_rng(91)
    q[slot] = q[slot] * (1.0 + 0.05 * rng.standard_normal(q[slot].shape))
    if slot in ("Qc", "R", "P0"):
        q[slot] = 0.5 * (q[slot] + np.swapaxes(q[slot], -1, -2))
    q["Sigma"] = q["L"] @ q["Qc"] @ np.swapaxes(q["L"], -1, -2)
    compare(f"batched_{slot}", q, y, t, "rk4", 0.01)


# ---- user drifts ---------------------------------------------------------------------------------------------------
def user_fields(code, nt, solver, dt0, max_steps=100000):
    return dict(solver=L.SOLVERS[solver], dt0=dt0, max_steps=max_steps, dt_final=1e-10, alpha=float(np.sqrt(3.0)),
                beta=2.0, kappa=1.0, drift_id=L.DRIFT_USER, n_theta=nt, emission_id=0,
                lib_path=b.build_user_drift(code, grad=True))


def compare_user(name, which, p, y, t, solver, dt0):
    N, K, m = y.shape
    n, nt = np.shape(p["m0"])[-1], np.shape(p["theta"])[-1]
    fields = user_fields(CODE[which], nt, solver, dt0)
    ll, status, G = sigma(p, y, t, solver, dt0, fields=fields)
    assert int(status.abs().sum()) == 0, name
    assert torch.equal(ll, sigma_filter_ll(p, y, t, fields)), name
    leaves = {}
    for k in BLOCKS:
        x = torch.tensor(np.asarray(p[k], np.float64))
        core = 1 if k in ("theta", "d", "m0") else 2
        leaves[k] = (x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))).clone().requires_grad_(True)
    ref_ll = sigma_filter(FNS[which](), *(leaves[k] for k in BLOCKS), y, t, o.SolverSettings(solver, dt0))
    ref = {k: g.numpy() for k, g in zip(leaves, torch.autograd.grad(ref_ll.sum(), list(leaves.values())))}
    err_ll = scaled_err(ll.cpu().numpy(), ref_ll.detach().numpy())
    record(f"ukf_grad_sigma_user:{name}:ll", err_ll)
    assert err_ll < 1e-11, (name, err_ll)
    return check(f"user:{name}", blocks(G, n, m, nt), ref, GATE)


def user_case(which, m=1, N=3, K=10, seed=0, batched=False, theta_batched=False, gap=0.05):
    p = user_model(which, m, seed, N=N if batched else None, theta_batched=theta_batched)
    rng = np.random.default_rng(seed + 1)
    return p, 0.7 * rng.standard_normal((N, K, m)), random_grid(N, K, seed + 2, mean_gap=gap)


@pytest.mark.parametrize("solver", list(L.SOLVERS))
def test_vdp_every_solver(solver):
    p, y, t = user_case("vdp", seed=1)
    compare_user(f"vdp_{solver}", "vdp", p, y, t, solver, 0.01)


@pytest.mark.parametrize("solver", ["rk4", "dopri5"])
def test_mlp(solver):
    p, y, t = user_case("mlp", seed=2)
    compare_user(f"mlp_{solver}", "mlp", p, y, t, solver, 0.01)


@pytest.mark.parametrize("which", ["vdp", "mlp"])
def test_theta_batched_and_m3(which):
    p, y, t = user_case(which, m=3, N=4, seed=3, batched=True, theta_batched=True)
    compare_user(f"{which}_batched_m3", which, p, y, t, "rk4", 0.01)


@pytest.mark.parametrize("kind,code,n,m", [("quadratic", QUAD, 2, 2), ("lorenz63", L63, 3, 3)])
def test_user_restatement_matches_the_registry(kind, code, n, m):
    p = random_model(kind, n, m, seed=7, N=3 if kind == "quadratic" else None)
    y = (3.0 if kind == "lorenz63" else 0.5) * np.random.default_rng(8).standard_normal((3, 12, m))
    t = random_grid(3, 12, 9, mean_gap=0.03)
    _, st_r, G_r = sigma(p, y, t, "rk4", 0.01)
    nt = np.shape(p["theta"])[-1]
    _, st_u, G_u = sigma(p, y, t, "rk4", 0.01, fields=user_fields(code, nt, "rk4", 0.01))
    assert int(st_r.abs().sum()) == 0 and int(st_u.abs().sum()) == 0
    r, u = blocks(G_r, n, m, nt), blocks(G_u, n, m, nt)
    for k in r:
        err = scaled_err(u[k], r[k])
        record(f"ukf_grad_sigma:{kind}_user_vs_registry:{k}", err)
        assert err < 1e-10, (k, err)


# ---- bits, status rows, central differences, the public entry ------------------------------------------------------
def test_log_likelihood_and_gradient_are_the_same_bits_run_to_run():
    for kind, n, m, solver in (("lorenz63", 3, 2, "rk4"), ("lorenz96", 40, 20, "dopri5"), ("quadratic", 3, 1, "rk4")):
        p, y, t = case(kind, n, m, N=4, K=12, seed=60)
        ll1, _, G1 = sigma(p, y, t, solver, 0.01)
        ll2, _, G2 = sigma(p, y, t, solver, 0.01)
        assert torch.equal(ll1, sigma_filter_ll(p, y, t, _fields(p, solver, 0.01))), kind
        assert torch.equal(ll1, ll2) and torch.equal(G1, G2), kind
    p, y, t = user_case("mlp", m=2, N=4, K=8, seed=61)
    fields = user_fields(MLP, 82, "rk4", 0.01)
    ll1, _, G1 = sigma(p, y, t, "rk4", 0.01, fields=fields)
    ll2, _, G2 = sigma(p, y, t, "rk4", 0.01, fields=fields)
    assert torch.equal(ll1, sigma_filter_ll(p, y, t, fields)) and torch.equal(ll1, ll2) and torch.equal(G1, G2)


def test_a_failed_trajectory_gets_a_nan_row_and_leaves_the_others_alone():
    N = 4
    p, y, t = case("lorenz96", 5, 2, N=N, K=6, seed=80, batched=True)
    _, st0, G0 = sigma(p, y, t, "rk4", 0.01)
    assert int(st0.abs().sum()) == 0
    q = dict(p)
    q["P0"] = np.broadcast_to(p["P0"], (N, 5, 5)).copy()
    q["P0"][2] = -np.eye(5)  # indefinite: the first predict's Cholesky factor is NaN
    _, st, G = sigma(q, y, t, "rk4", 0.01)
    st = st.cpu().numpy()
    assert st[2] != 0 and (np.delete(st, 2) == 0).all()
    assert torch.isnan(G[2]).all()
    keep = [0, 1, 3]
    assert torch.equal(G[keep], G0[keep])


def test_directional_derivatives_match_central_differences_of_the_filter():
    n, m, N, K = 5, 3, 4, 100
    p, y, t = case("lorenz96", n, m, N=N, K=K, seed=130, gap=0.02)
    _, st, G = sigma(p, y, t, "rk4", 0.01)
    assert int(st.abs().sum()) == 0
    got = blocks(G, n, m, 1)
    rng = np.random.default_rng(131)
    for name in BLOCKS:
        v = rng.standard_normal(np.shape(p[name]))
        if name in ("Sigma", "R", "P0"):
            v = 0.5 * (v + v.T)
        h = 1e-6 * max(1.0, float(np.max(np.abs(p[name]))))

        def ll_at(s):
            q = dict(p)
            q[name] = p[name] + s * v
            if name == "Sigma":  # the kernels take L and Qc: move Qc so that L Qc L^T moves by s v
                q["Qc"] = p["Qc"] + s * np.linalg.solve(p["L"], np.linalg.solve(p["L"], v).T).T
            return float(sigma_filter_ll(q, y, t, _fields(p, "rk4", 0.01)).sum())

        fd = (ll_at(h) - ll_at(-h)) / (2 * h)
        an = float(np.sum(got[name].sum(0) * v))
        err = abs(an - fd) / max(abs(fd), 1.0)
        record(f"ukf_grad_sigma:directional_vs_filter_fd:{name}", err)
        assert err <= 1e-6, (name, an, fd)


def test_adam_fit_of_vdp_through_the_autograd_wrapper():
    N, K = 16, 60
    truth = np.array([1.3, 0.4])
    tt = (0.1 * np.arange(K))[:, None]

    def params_for(theta):
        return cd.ParamsCDNLGSSM(
            initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(np.array([1.0, 0.0])), cov=cd.LearnableMatrix(0.5 * np.eye(2))),
            dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableUserDrift(VDP, theta, differentiable=True),
                                               diffusion_coefficient=cd.LearnableMatrix(np.eye(2)),
                                               diffusion_cov=cd.LearnableMatrix(0.05 * np.eye(2))),
            emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=np.eye(2), bias=np.zeros(2)),
                                                 emission_cov=cd.LearnableMatrix(0.01 * np.eye(2))))
    _, ys = cd.cdnlgssm_path_sample(params_for(truth), 5, K, tt, diffeqsolve_settings={"solver": "heun", "dt0": 0.005},
                                    num_sequences=N)
    ys = np.asarray(ys)
    T = np.broadcast_to(tt, (N, K, 1))
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    ll, g = cd.ukf_sigma_points_marginal_log_prob_and_grad(params_for(truth), ys, T, hp, wrt="all")
    assert set(g) == {"theta", "diffusion_coefficient", "diffusion_cov", "emission_cov", "emission_bias",
                      "emission_weights", "initial_mean", "initial_cov"} and g["theta"].shape == (N, 2)
    f = cd.cdnlgssm_filter(params_for(truth), ys, T, hp, output_fields=[])  # a user drift runs sigma points
    assert np.array_equal(ll, f.marginal_loglik)
    theta = torch.tensor([0.8, 0.1], dtype=torch.float64, requires_grad=True)
    opt = torch.optim.Adam([theta], lr=0.05)
    losses = []
    for _ in range(50):
        opt.zero_grad()
        loss = -ukf_sigma_points_marginal_log_prob(params_for(theta), ys, T, hp).sum() / (N * K)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    record("ukf_grad_sigma:adam_vdp_mu_final", float(theta.detach()[0]))
    record("ukf_grad_sigma:adam_vdp_eps_final", float(theta.detach()[1]))
    assert losses[-1] < losses[0]
    assert abs(float(theta[0]) - truth[0]) <= 0.5 * abs(0.8 - truth[0]), theta
