"""cdk_ekf_grad_dense_f64 / ekf_marginal_log_prob_and_grad / autograd.ekf_marginal_log_prob on the GPU, for every
registry drift and emission size.

The reference is the torch float64 restatement of the oracle's EKF (oracle/cd_torch_ekf.py) differentiated by torch
autograd: the gradient of the same discrete function.  Every gate is on one block's max error over that block's max
|value|; the symmetric blocks (Sigma, R, P0) are compared on their symmetric parts."""
import ctypes

import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _engine as E
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200.autograd import ekf_marginal_log_prob
from cd_dynamax_b200.continuous_discrete_linear_gaussian_ssm import inference as kfi
from oracle import cd_oracle as o
from oracle import cd_torch_ekf as te
from tests.helpers import make_drift, record, scaled_err
from tests.test_ekf_grad_host import BLOCKS, api_params, n_theta, random_data, random_model
from tests.test_gpu_time_grids import degenerate_grid, edge_grid, long_grid, regular_grid
from tests.test_gpu_parity import c3_problem, nonlinear_params_api
from tests.test_kf_grad_host import random_grid

pytestmark = pytest.mark.gpu
GATE = 1e-9
dev = torch.device("cuda", 0) if torch.cuda.is_available() else None
DRIFT_ID = {"linear": L.DRIFT_LINEAR, "lorenz63": L.DRIFT_LORENZ63, "lorenz96": L.DRIFT_LORENZ96,
            "quadratic": L.DRIFT_QUADRATIC}


def _ins(p, y, t):
    return {L.IN_Y: y, L.IN_T: t, L.IN_M0: p["m0"], L.IN_P0: p["P0"], L.IN_F: p["theta"], L.IN_L: p["L"],
            L.IN_QC: p["Qc"], L.IN_H: p["H"], L.IN_D: p["d"], L.IN_R: p["R"]}


def _fields(p, solver, dt0, order, max_steps=100000):
    n = np.shape(p["m0"])[-1]
    return dict(solver=L.SOLVERS[solver], dt0=dt0, max_steps=max_steps, dt_final=1e-10, state_order=L.ORDERS[order],
                num_iter=1, drift_id=DRIFT_ID[p["kind"]], n_theta=n_theta(p["kind"], n), emission_id=0)


def dense(p, y, t, solver, dt0, order="second", max_steps=100000):
    """(ll, status, G [N, cols]) of cdk_ekf_grad_dense_f64, device tensors."""
    N, K, m = y.shape
    n = np.shape(p["m0"])[-1]
    cols = L.grad_cols_ekf(n, m, n_theta(p["kind"], n))
    out = E.run("cdk_ekf_grad_dense", "f64", N, K, n, m, _ins(p, y, t), (L.OUT_LL, L.OUT_GRAD),
                _fields(p, solver, dt0, order, max_steps), out_shapes={L.OUT_GRAD: (N, cols)})
    return out[L.OUT_LL], out[L.OUT_STATUS], out[L.OUT_GRAD]


def blocks(G, n, m, nt):
    G = G.cpu().numpy() if isinstance(G, torch.Tensor) else G
    out, o_ = {}, 0
    for name, shp in (("theta", (nt,)), ("Sigma", (n, n)), ("H", (m, n)), ("d", (m,)), ("R", (m, m)), ("m0", (n,)),
                      ("P0", (n, n))):
        size = int(np.prod(shp))
        out[name] = G[:, o_:o_ + size].reshape((G.shape[0],) + shp)
        o_ += size
    return out


def reference(p, y, t, solver, dt0, order):
    N = y.shape[0]
    leaves = {}
    for k in BLOCKS:
        x = torch.tensor(np.asarray(p[k], np.float64))
        core = 1 if k in ("theta", "d", "m0") else 2
        x = x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))
        leaves[k] = x.clone().requires_grad_(True)
    ll = te.marginal_log_prob(p["kind"], *(leaves[k] for k in BLOCKS), y, t, 1e-10, order, o.SolverSettings(solver, dt0))
    g = torch.autograd.grad(ll.sum(), list(leaves.values()))
    return ll.detach().numpy(), {k: v.numpy() for k, v in zip(leaves, g)}


def sym(x):
    return 0.5 * (x + np.swapaxes(x, -1, -2))


def compare(name, p, y, t, solver, dt0, order="second", gate=GATE):
    ll, status, G = dense(p, y, t, solver, dt0, order)
    assert int(status.abs().sum()) == 0, name
    n, m = np.shape(p["m0"])[-1], y.shape[-1]
    got = blocks(G, n, m, n_theta(p["kind"], n))
    ref_ll, ref = reference(p, y, t, solver, dt0, order)
    err_ll = scaled_err(ll.cpu().numpy(), ref_ll)
    record(f"ekf_grad_dense:{name}:ll", err_ll)
    assert err_ll < 1e-11, (name, err_ll)
    worst = 0.0
    for k, r in ref.items():
        r = sym(r) if k in ("Sigma", "R", "P0") else r
        err = scaled_err(got[k], r)
        record(f"ekf_grad_dense:{name}:{k}", err)
        worst = max(worst, err)
        assert err < gate, (name, k, err)
    return worst


def case(kind, n, m, N=3, K=10, seed=0, batched=False, gap=0.03):
    p = random_model(kind, n, m, seed=seed, N=N if batched else None)
    return p, random_data(p, N, K, seed + 1), random_grid(N, K, seed + 2, mean_gap=gap)


@pytest.mark.parametrize("m", [1, 2, 3])
def test_lorenz63_every_emission_size(m):
    p, y, t = case("lorenz63", 3, m, seed=m)
    compare(f"l63_m{m}", p, y, t, "rk4", 0.01)


@pytest.mark.parametrize("n,solver", [(5, "dopri5"), (40, "rk4"), (40, "dopri5")])
def test_lorenz96(n, solver):
    p, y, t = case("lorenz96", n, n // 2, N=2, K=8, seed=n)
    compare(f"l96_n{n}_{solver}", p, y, t, solver, 0.01, order="first")


@pytest.mark.parametrize("n", [1, 4, 16])
def test_linear_drift(n):
    p, y, t = case("linear", n, 2, seed=10 + n, batched=(n == 4))
    compare(f"linear_n{n}", p, y, t, "rk4", 0.01)


@pytest.mark.parametrize("n", [2, 4])
@pytest.mark.parametrize("order", ["first", "second"])
def test_quadratic_drift(n, order):
    p, y, t = case("quadratic", n, 2, seed=20 + n, batched=True)
    compare(f"quadratic_n{n}_{order}", p, y, t, "rk4", 0.01, order=order)


@pytest.mark.parametrize("solver", list(L.SOLVERS))
def test_every_solver(solver):
    p, y, t = case("lorenz96", 5, 3, seed=30)
    compare(f"solver_{solver}", p, y, t, solver, 0.01, order="first")


@pytest.mark.parametrize("grid", ["t0_1e4", "edge", "degenerate", "long"])
def test_time_grids(grid):
    N, K, dt0 = 3, 8, 0.01
    p = random_model("linear", 4, 2, seed=40)
    t = {"t0_1e4": lambda: regular_grid(N, K, t0=1e4, h=0.013), "edge": lambda: edge_grid(N, K, dt0),
         "degenerate": lambda: degenerate_grid(N, K, dt0), "long": lambda: long_grid(N, 6, dt0)}[grid]()
    y = random_data(p, N, t.shape[1], 41)
    compare(f"grid_{grid}", p, y, t, "rk4", dt0)


def _fits(n, m, solver):
    d = L.new_desc()
    d.N, d.K, d.n, d.m, d.solver = 0, 4, n, m, L.SOLVERS[solver]
    d.drift_id, d.n_theta, d.state_order = L.DRIFT_LINEAR, n * n + n, 1
    fake = ctypes.c_void_p(0x1000)
    ins = (ctypes.c_void_p * L.NUM_IN)(*([fake] * L.NUM_IN))
    outs = (ctypes.c_void_p * L.NUM_OUT)(*([fake] * L.NUM_OUT))
    return L.lib().cdk_ekf_grad_dense_f64(ctypes.byref(d), ins, outs, None) == 0


def test_largest_n_the_layout_admits_at_m_eq_n():
    n = max(k for k in range(1, 65) if _fits(k, k, "rk4"))
    record("ekf_grad_dense:largest_n_m_eq_n_rk4", n)
    assert not _fits(n + 1, n + 1, "rk4")
    p, y, t = case("linear", n, n, N=1, K=4, seed=50, gap=0.02)
    compare(f"largest_n{n}", p, y, t, "rk4", 0.01)


def test_log_likelihood_is_bit_identical_to_the_filter():
    for kind, n, m in (("lorenz63", 3, 2), ("lorenz96", 40, 20), ("quadratic", 3, 1)):
        p, y, t = case(kind, n, m, N=4, K=12, seed=60)
        ll, _, _ = dense(p, y, t, "rk4", 0.01)
        f = E.run("cdk_ekf_filter", "f64", 4, 12, n, m, _ins(p, y, t), (L.OUT_LL,), _fields(p, "rk4", 0.01, "second"))
        assert torch.equal(ll, f[L.OUT_LL]), kind


@pytest.mark.parametrize("order", ["first", "second"])
def test_lorenz63_scalar_emission_agrees_with_the_existing_reverse_kernel(order):
    p, y, t = case("lorenz63", 3, 1, N=5, K=20, seed=70)
    _, _, G = dense(p, y, t, "rk4", 0.01, order)
    b = blocks(G, 3, 1, 3)
    f = dict(_fields(p, "rk4", 0.01, order), grad_groups=127 | L.GRAD_REVERSE)
    ref = E.run("cdk_ekf_grad", "f64", 5, 20, 3, 1, _ins(p, y, t), (L.OUT_LL, L.OUT_GRAD), f)[L.OUT_GRAD].cpu().numpy()
    iu = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]

    def pack(M):
        return np.stack([M[:, i, j] if i == j else 2.0 * M[:, i, j] for i, j in iu], -1)

    mine = np.concatenate([b["theta"], pack(b["Sigma"]), b["R"].reshape(5, 1), b["d"], b["H"].reshape(5, 3), b["m0"],
                           pack(b["P0"])], -1)
    for lo, hi, name in ((0, 3, "theta"), (3, 9, "Sigma"), (9, 10, "R"), (10, 11, "d"), (11, 14, "H"), (14, 17, "m0"),
                         (17, 23, "P0")):
        err = scaled_err(mine[:, lo:hi], ref[:, lo:hi])
        record(f"ekf_grad_dense:l63_m1_vs_reverse_{order}:{name}", err)
        assert err < 1e-10, (name, err)


def test_status_rows():
    p, y, t = case("lorenz96", 5, 2, N=4, K=6, seed=80)
    _, st, G = dense(p, y, t, "rk4", 0.001, "first", max_steps=5)  # every gap needs ~30 substeps
    assert (st.cpu().numpy() == 2).all() and torch.isnan(G).all()
    y2 = y.copy()
    y2[1, 3, 0] = np.nan
    _, st, G = dense(p, y2, t, "rk4", 0.01, "first")
    st = st.cpu().numpy()
    assert st[1] == 1 and (st[[0, 2, 3]] == 0).all()
    assert torch.isnan(G[1]).all() and torch.isfinite(G[[0, 2, 3]]).all()


SLOTS = ("theta", "L", "Qc", "H", "d", "R", "m0", "P0")


def test_each_slot_batched_alone_is_bit_identical_to_the_shared_value():
    N = 5
    p, y, t = case("quadratic", 3, 2, N=N, K=8, seed=90)
    _, _, G0 = dense(p, y, t, "rk4", 0.01)
    for slot in SLOTS:
        q = dict(p)
        q[slot] = np.broadcast_to(np.asarray(p[slot]), (N,) + np.shape(p[slot])).copy()
        _, _, G = dense(q, y, t, "rk4", 0.01)
        assert torch.equal(G, G0), slot


def test_shards_permutations_and_chunks_are_bit_identical(monkeypatch):
    N = 6
    p, y, t = case("lorenz96", 5, 2, N=N, K=8, seed=100, batched=True)
    ll0, _, G0 = dense(p, y, t, "dopri5", 0.01)
    sub = lambda q, idx: {k: (v[idx] if k != "kind" else v) for k, v in q.items()}
    for idx in (np.arange(0, 2), np.arange(2, N), np.array([5, 0, 3, 1, 4, 2])):
        ll, _, G = dense(sub(p, idx), y[idx], t[idx], "dopri5", 0.01)
        assert torch.equal(G, G0[torch.as_tensor(idx, device=dev)]) and torch.equal(ll, ll0[torch.as_tensor(idx, device=dev)])
    hp = cd.EKFHyperParams(state_order="second", diffeqsolve_settings={"solver": "dopri5", "dt0": 0.01})
    params = api_params("lorenz96", 5, 2, p)
    ll1, g1 = cd.ekf_marginal_log_prob_and_grad(params, y, t[..., None], hp, wrt="all")
    monkeypatch.setattr(kfi, "_grad_chunk", lambda N_, row: 2)
    ll2, g2 = cd.ekf_marginal_log_prob_and_grad(params, y, t[..., None], hp, wrt="all")
    assert np.array_equal(ll1, ll2) and set(g1) == set(g2)
    for k in g1:
        assert np.array_equal(np.asarray(g1[k]), np.asarray(g2[k])), k
    assert np.array_equal(np.asarray(g1["forcing"]), blocks(G0, 5, 2, 1)["theta"][:, 0])


def test_api_keys_and_chain_rule():
    p, y, t = case("linear", 3, 2, N=3, K=8, seed=110)
    hp = cd.EKFHyperParams(state_order="second", diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    ll, g = cd.ekf_marginal_log_prob_and_grad(api_params("linear", 3, 2, p), y, t[..., None], hp, wrt="all")
    assert set(g) == {"weights", "bias", "diffusion_coefficient", "diffusion_cov", "emission_cov", "emission_bias",
                      "emission_weights", "initial_mean", "initial_cov"}
    assert g["weights"].shape == (3, 3, 3) and g["emission_cov"].shape == (3, 2, 2)
    ref_ll, ref = reference(p, y, t, "rk4", 0.01, "second")
    assert scaled_err(ll, ref_ll) < 1e-11
    Sb = ref["Sigma"]
    Lm, Qc = p["L"], p["Qc"]
    assert scaled_err(g["diffusion_cov"], np.swapaxes(Lm, -1, -2) @ sym(Sb) @ Lm) < GATE
    assert scaled_err(g["diffusion_coefficient"], sym(Sb) @ Lm @ (Qc + Qc.T)) < GATE
    _, gd = cd.ekf_marginal_log_prob_and_grad(api_params("linear", 3, 2, p), y, t[..., None], hp, wrt="drift")
    assert set(gd) == {"weights", "bias"}


def test_autograd_wrapper_on_lorenz96():
    n, m, N = 6, 3, 4
    p, y, t = case("lorenz96", n, m, N=N, K=10, seed=120)
    F = torch.tensor(float(p["theta"][0]), dtype=torch.float64, requires_grad=True)
    H = torch.tensor(p["H"], requires_grad=True)
    params = api_params("lorenz96", n, m, p)
    params = params._replace(
        dynamics=params.dynamics._replace(drift=cd.LearnableLorenz96(forcing=F)),
        emissions=params.emissions._replace(emission_function=cd.LearnableLinear(weights=H, bias=p["d"])))
    hp = cd.EKFHyperParams(state_order="first", diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    ll = ekf_marginal_log_prob(params, y, t[..., None], hp)
    ll.sum().backward()
    _, ref = reference(p, y, t, "rk4", 0.01, "first")
    assert scaled_err(F.grad.numpy(), ref["theta"].sum(0)[0]) < GATE
    assert scaled_err(H.grad.numpy(), ref["H"].sum(0)) < GATE


def test_adam_fits_the_lorenz96_forcing():
    n, m, N, K = 8, 4, 32, 40
    truth = 8.0
    H = np.eye(n)[::2]
    def params_for(F):
        return cd.ParamsCDNLGSSM(
            initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(np.full(n, truth + 1.0)),
                                          cov=cd.LearnableMatrix(np.eye(n))),
            dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableLorenz96(forcing=F),
                                               diffusion_coefficient=cd.LearnableMatrix(np.eye(n)),
                                               diffusion_cov=cd.LearnableMatrix(0.1 * np.eye(n))),
            emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=H, bias=np.zeros(m)),
                                                 emission_cov=cd.LearnableMatrix(0.25 * np.eye(m))))
    tt = (0.05 * np.arange(K))[:, None]
    xs, ys = cd.cdnlgssm_path_sample(params_for(truth), 7, K, tt, diffeqsolve_settings={"solver": "heun", "dt0": 0.005},
                                     num_sequences=N)
    ys = np.asarray(ys)
    F = torch.tensor(6.5, dtype=torch.float64, requires_grad=True)
    opt = torch.optim.Adam([F], lr=0.05)
    hp = cd.EKFHyperParams(state_order="first", diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    losses = []
    for _ in range(50):
        opt.zero_grad()
        loss = -ekf_marginal_log_prob(params_for(F), ys, np.broadcast_to(tt, (N, K, 1)), hp).sum() / (N * K)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    record("ekf_grad_dense:adam_l96_forcing_final", float(F))
    assert losses[-1] < losses[0]
    assert abs(float(F) - truth) <= 0.5 * abs(6.5 - truth), float(F)


@pytest.mark.parametrize("solver,dt0", [("rk4", 0.0025), ("dopri5", 0.01), ("heun", 0.002)])
def test_lorenz63_two_component_emission_through_the_public_entry(solver, dt0):
    """ekf_dense_marginal_log_prob_and_grad on Lorenz-63 observed in two components (which ekf_marginal_log_prob_and_grad
    leaves to it): the filter's log-likelihood, d ll / d (sigma, rho, beta) against central differences of the oracle,
    and the autograd wrapper, which takes this path for such a model."""
    N, K = 6, 40
    t, y = c3_problem(N, K, seed=21)
    theta = np.array([10.0, 28.0, 8.0 / 3.0])
    g = dict(m0=np.array([1.0, 1.0, 20.0]), P0=2 * np.eye(3), drift="lorenz63", theta=theta,
             L=np.eye(3) + 0.1 * np.arange(9).reshape(3, 3) / 9, Qc=np.eye(3) + 0.05,
             H=np.array([[1.0, 0.3, -0.2], [0.0, 1.0, 0.5]]), R=np.array([[0.7, 0.1], [0.1, 0.9]]), d=np.array([0.1, -0.2]))
    y = np.concatenate([y, 0.5 * y + 1.0], -1)
    hp = cd.EKFHyperParams(dt_final=0.004, diffeqsolve_settings={"solver": solver, "dt0": dt0})
    ll, grad = cd.ekf_dense_marginal_log_prob_and_grad(nonlinear_params_api(g), y, t[..., None], hp)
    assert set(grad) == {"sigma", "rho", "beta"}
    f = cd.cdnlgssm_filter(nonlinear_params_api(g), y, t[..., None], hp, output_fields=[])
    assert np.array_equal(ll, f.marginal_loglik)

    def oracle_ll(th):
        po = o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift("lorenz63", th, 3), L=g["L"], Qc=g["Qc"],
                               H=g["H"], R=g["R"], d=g["d"])
        return o.extended_kalman_filter(po, y, t, dt_final=0.004, settings=o.SolverSettings(solver, dt0))["marginal_loglik"]

    for p, name in enumerate(("sigma", "rho", "beta")):
        h = 1e-5 * theta[p]
        tp, tm = theta.copy(), theta.copy()
        tp[p] += h
        tm[p] -= h
        np.testing.assert_allclose(grad[name], (oracle_ll(tp) - oracle_ll(tm)) / (2 * h), rtol=2e-6, atol=2e-7,
                                   err_msg=name)
    rho = torch.tensor(28.0, dtype=torch.float64, requires_grad=True)
    params = nonlinear_params_api(g)
    params = params._replace(dynamics=params.dynamics._replace(drift=cd.LearnableLorenz63(sigma=10.0, rho=rho, beta=8.0 / 3.0)))
    ekf_marginal_log_prob(params, y, t[..., None], hp).sum().backward()
    assert abs(float(rho.grad) - float(np.sum(grad["rho"]))) <= 1e-12 * abs(float(np.sum(grad["rho"])))
