"""cdk_ukf_grad_dense_f64 / ukf_marginal_log_prob_and_grad / autograd.ukf_marginal_log_prob on the GPU, for every
registry drift and emission size.

The reference is torch autograd of the closed-form restatement of the oracle's UKF (oracle/cd_torch_ukf.py,
closed="closed"), gated at 1e-9 of each block's max |value|, and of the literal sigma-point restatement (closed="sigma"),
gated at 1e-8.  The symmetric blocks (Sigma, R, P0) are compared on their symmetric parts."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _engine as E
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200.autograd import ukf_marginal_log_prob
from cd_dynamax_b200.continuous_discrete_linear_gaussian_ssm import inference as kfi
from oracle import cd_oracle as o
from oracle import cd_torch_ukf as tu
from tests.helpers import record, scaled_err
from tests.test_ekf_grad_host import BLOCKS, api_params, n_theta, random_data, random_model
from tests.test_gpu_ekf_grad import DRIFT_ID, _ins, blocks, sym
from tests.test_gpu_time_grids import degenerate_grid, edge_grid, long_grid, regular_grid
from tests.test_kf_grad_host import random_grid

pytestmark = pytest.mark.gpu
GATE = 1e-9        # against the closed form the kernels compute
GATE_SIGMA = 1e-8  # against the literal sigma points of the reference
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fields(p, solver, dt0, max_steps=100000):
    n = np.shape(p["m0"])[-1]
    return dict(solver=L.SOLVERS[solver], dt0=dt0, max_steps=max_steps, dt_final=1e-10, alpha=float(np.sqrt(3.0)),
                beta=2.0, kappa=1.0, drift_id=DRIFT_ID[p["kind"]], n_theta=n_theta(p["kind"], n), emission_id=0)


def dense(p, y, t, solver, dt0, max_steps=100000):
    """(ll, status, G [N, cols]) of cdk_ukf_grad_dense_f64, device tensors."""
    N, K, m = y.shape
    n = np.shape(p["m0"])[-1]
    cols = L.grad_cols_ekf(n, m, n_theta(p["kind"], n))
    out = E.run("cdk_ukf_grad_dense", "f64", N, K, n, m, _ins(p, y, t), (L.OUT_LL, L.OUT_GRAD),
                _fields(p, solver, dt0, max_steps), out_shapes={L.OUT_GRAD: (N, cols)})
    return out[L.OUT_LL], out[L.OUT_STATUS], out[L.OUT_GRAD]


def filter_ll(p, y, t, solver, dt0):
    N, K, m = y.shape
    n = np.shape(p["m0"])[-1]
    return E.run("cdk_ukf_filter", "f64", N, K, n, m, _ins(p, y, t), (L.OUT_LL,), _fields(p, solver, dt0))[L.OUT_LL]


def reference(p, y, t, solver, dt0, closed="closed"):
    N = y.shape[0]
    leaves = {}
    for k in BLOCKS:
        x = torch.tensor(np.asarray(p[k], np.float64))
        core = 1 if k in ("theta", "d", "m0") else 2
        x = x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))
        leaves[k] = x.clone().requires_grad_(True)
    ll = tu.marginal_log_prob(p["kind"], *(leaves[k] for k in BLOCKS), y, t, 1e-10,
                              settings=o.SolverSettings(solver, dt0), closed=closed)
    g = torch.autograd.grad(ll.sum(), list(leaves.values()))
    return ll.detach().numpy(), {k: v.numpy() for k, v in zip(leaves, g)}


def compare(name, p, y, t, solver, dt0):
    """Every block against both restatements; -> the worst block error against the closed form."""
    ll, status, G = dense(p, y, t, solver, dt0)
    assert int(status.abs().sum()) == 0, name
    n, m = np.shape(p["m0"])[-1], y.shape[-1]
    got = blocks(G, n, m, n_theta(p["kind"], n))
    worst = 0.0
    for closed, gate in (("closed", GATE), ("sigma", GATE_SIGMA)):
        ref_ll, ref = reference(p, y, t, solver, dt0, closed)
        err_ll = scaled_err(ll.cpu().numpy(), ref_ll)
        record(f"ukf_grad_dense:{name}:{closed}:ll", err_ll)
        assert err_ll < 1e-11, (name, closed, err_ll)
        for k, r in ref.items():
            r = sym(r) if k in ("Sigma", "R", "P0") else r
            err = scaled_err(got[k], r)
            record(f"ukf_grad_dense:{name}:{closed}:{k}", err)
            if closed == "closed":
                worst = max(worst, err)
            assert err < gate, (name, closed, k, err)
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
    compare(f"l96_n{n}_{solver}", p, y, t, solver, 0.01)


def shared_memory_ode_child():
    """Run in a child process with CDK_GENERIC_REG_ODE=0 (read once per process): Lorenz-96 n = 40 on the shared-memory
    moment ODE -- every block against the reference, and the log-likelihood bit for bit against the filter."""
    assert os.environ.get("CDK_GENERIC_REG_ODE") == "0"
    for solver in ("rk4", "dopri5"):
        p, y, t = case("lorenz96", 40, 20, N=2, K=8, seed=40)
        print("WORST", solver, compare(f"l96_n40_{solver}_shared_memory_ode", p, y, t, solver, 0.01))
        ll, _, _ = dense(p, y, t, solver, 0.01)
        assert torch.equal(ll, filter_ll(p, y, t, solver, 0.01)), solver


def test_lorenz96_n40_on_the_shared_memory_ode():
    env = dict(os.environ, CDK_GENERIC_REG_ODE="0")
    r = subprocess.run([sys.executable, "-c", "import tests.test_gpu_ukf_grad as t; t.shared_memory_ode_child()"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-4000:]
    for line in r.stdout.splitlines():
        if line.startswith("WORST"):
            _, solver, err = line.split()
            record(f"ukf_grad_dense:l96_n40_{solver}_shared_memory_ode:worst_closed", float(err))


@pytest.mark.parametrize("n", [1, 4, 16])
def test_linear_drift(n):
    p, y, t = case("linear", n, 2, seed=10 + n, batched=(n == 4))
    compare(f"linear_n{n}", p, y, t, "rk4", 0.01)


@pytest.mark.parametrize("n", [2, 4])
def test_quadratic_drift(n):
    p, y, t = case("quadratic", n, 2, seed=20 + n, batched=True)
    compare(f"quadratic_n{n}", p, y, t, "rk4", 0.01)


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
    y = random_data(p, N, t.shape[1], 41)
    compare(f"grid_{grid}", p, y, t, "rk4", dt0)


SLOTS = ("theta", "L", "Qc", "H", "d", "R", "m0", "P0")


@pytest.mark.parametrize("slot", SLOTS)
def test_each_leaf_batched_alone(slot):
    """One parameter batched (a different value per trajectory), the rest shared: against the reference, and the same
    value expanded to N rows is bit-identical to the shared call."""
    N = 4
    p, y, t = case("quadratic", 3, 2, N=N, K=8, seed=90)
    _, _, G0 = dense(p, y, t, "rk4", 0.01)
    q = dict(p)
    q[slot] = np.broadcast_to(np.asarray(p[slot]), (N,) + np.shape(p[slot])).copy()
    _, _, G = dense(q, y, t, "rk4", 0.01)
    assert torch.equal(G, G0), slot
    rng = np.random.default_rng(91)
    q[slot] = q[slot] * (1.0 + 0.05 * rng.standard_normal(q[slot].shape))
    if slot in ("Qc", "R", "P0"):
        q[slot] = 0.5 * (q[slot] + np.swapaxes(q[slot], -1, -2))
    q["Sigma"] = q["L"] @ q["Qc"] @ np.swapaxes(q["L"], -1, -2)
    compare(f"batched_{slot}", q, y, t, "rk4", 0.01)


def test_log_likelihood_is_bit_identical_to_the_filter():
    for kind, n, m, solver in (("lorenz63", 3, 2, "rk4"), ("lorenz96", 40, 20, "rk4"), ("lorenz96", 40, 20, "dopri5"),
                               ("quadratic", 3, 1, "rk4"), ("linear", 4, 2, "dopri5")):
        p, y, t = case(kind, n, m, N=4, K=12, seed=60)
        ll, _, _ = dense(p, y, t, solver, 0.01)
        assert torch.equal(ll, filter_ll(p, y, t, solver, 0.01)), (kind, solver)


def test_directional_derivative_against_central_differences_of_the_filter_at_c4():
    """<G, v> for a random direction v in every block against central differences of cdk_ukf_filter_f64 itself."""
    n, m, N, K = 40, 20, 2, 100
    p, y, t = case("lorenz96", n, m, N=N, K=K, seed=130, gap=0.02)
    _, st, G = dense(p, y, t, "rk4", 0.01)
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
            return float(filter_ll(q, y, t, "rk4", 0.01).sum())

        fd = (ll_at(h) - ll_at(-h)) / (2 * h)
        an = float(np.sum(got[name].sum(0) * v))
        err = abs(an - fd) / max(abs(fd), 1.0)
        record(f"ukf_grad_dense:c4_directional_vs_filter_fd:{name}", err)
        assert err <= 1e-6, (name, an, fd)


def test_status_rows():
    p, y, t = case("lorenz96", 5, 2, N=4, K=6, seed=80)
    _, st, G = dense(p, y, t, "rk4", 0.001, max_steps=5)  # every gap needs ~30 substeps
    assert (st.cpu().numpy() == 2).all() and torch.isnan(G).all()


def test_forced_small_chunks_are_bit_identical(monkeypatch):
    N = 6
    p, y, t = case("lorenz96", 5, 2, N=N, K=8, seed=100, batched=True)
    _, _, G0 = dense(p, y, t, "dopri5", 0.01)
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": "dopri5", "dt0": 0.01})
    params = api_params("lorenz96", 5, 2, p)
    ll1, g1 = cd.ukf_marginal_log_prob_and_grad(params, y, t[..., None], hp, wrt="all")
    monkeypatch.setattr(kfi, "_grad_chunk", lambda N_, row: 2)
    ll2, g2 = cd.ukf_marginal_log_prob_and_grad(params, y, t[..., None], hp, wrt="all")
    assert np.array_equal(ll1, ll2) and set(g1) == set(g2)
    for k in g1:
        assert np.array_equal(np.asarray(g1[k]), np.asarray(g2[k])), k
    assert np.array_equal(np.asarray(g1["forcing"]), blocks(G0, 5, 2, 1)["theta"][:, 0])


def test_api_keys_chain_rule_and_filter_log_likelihood():
    p, y, t = case("linear", 3, 2, N=3, K=8, seed=110)
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    params = api_params("linear", 3, 2, p)
    ll, g = cd.ukf_marginal_log_prob_and_grad(params, y, t[..., None], hp, wrt="all")
    assert set(g) == {"weights", "bias", "diffusion_coefficient", "diffusion_cov", "emission_cov", "emission_bias",
                      "emission_weights", "initial_mean", "initial_cov"}
    assert g["weights"].shape == (3, 3, 3) and g["emission_cov"].shape == (3, 2, 2)
    f = cd.cdnlgssm_filter(params, y, t[..., None], hp, output_fields=[])
    assert np.array_equal(ll, f.marginal_loglik)
    ref_ll, ref = reference(p, y, t, "rk4", 0.01)
    assert scaled_err(ll, ref_ll) < 1e-11
    Sb, Lm, Qc = ref["Sigma"], p["L"], p["Qc"]
    assert scaled_err(g["diffusion_cov"], np.swapaxes(Lm, -1, -2) @ sym(Sb) @ Lm) < GATE
    assert scaled_err(g["diffusion_coefficient"], sym(Sb) @ Lm @ (Qc + Qc.T)) < GATE
    _, gd = cd.ukf_marginal_log_prob_and_grad(params, y, t[..., None], hp, wrt="drift")
    assert set(gd) == {"weights", "bias"}


@pytest.mark.parametrize("batched", [False, True])
def test_autograd_wrapper_equals_the_function(batched):
    n, m, N = 6, 3, 4
    p, y, t = case("lorenz96", n, m, N=N, K=10, seed=120)
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    F0 = np.full(N, float(p["theta"][0])) + (0.1 * np.arange(N) if batched else 0.0)
    H0 = np.broadcast_to(p["H"], (N, m, n)).copy() if batched else p["H"]
    F = torch.tensor(F0 if batched else float(F0[0]), dtype=torch.float64, requires_grad=True)
    H = torch.tensor(H0, requires_grad=True)
    params = api_params("lorenz96", n, m, p)
    params = params._replace(
        dynamics=params.dynamics._replace(drift=cd.LearnableLorenz96(forcing=F)),
        emissions=params.emissions._replace(emission_function=cd.LearnableLinear(weights=H, bias=p["d"])))
    ll = ukf_marginal_log_prob(params, y, t[..., None], hp)
    ll.sum().backward()
    plain = params._replace(
        dynamics=params.dynamics._replace(drift=cd.LearnableLorenz96(forcing=F0 if batched else float(F0[0]))),
        emissions=params.emissions._replace(emission_function=cd.LearnableLinear(weights=H0, bias=p["d"])))
    ll_ref, g = cd.ukf_marginal_log_prob_and_grad(plain, y, t[..., None], hp, wrt="all")
    assert np.array_equal(ll.detach().numpy(), ll_ref)
    gF, gH = np.asarray(g["forcing"]), np.asarray(g["emission_weights"])
    if not batched:
        gF, gH = gF.sum(0), gH.sum(0)
    assert np.allclose(F.grad.numpy(), gF, rtol=1e-14, atol=0) and np.allclose(H.grad.numpy(), gH, rtol=1e-14, atol=0)


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
    hp = cd.UKFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    losses = []
    for _ in range(50):
        opt.zero_grad()
        loss = -ukf_marginal_log_prob(params_for(F), ys, np.broadcast_to(tt, (N, K, 1)), hp).sum() / (N * K)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    record("ukf_grad_dense:adam_l96_forcing_final", F.item())
    assert losses[-1] < losses[0]
    assert abs(F.item() - truth) <= 0.5 * abs(6.5 - truth), F.item()
