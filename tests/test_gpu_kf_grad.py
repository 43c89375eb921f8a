"""cdk_kf_grad_f64 / cdlgssm_marginal_log_prob_and_grad / autograd.cdlgssm_marginal_log_prob on the GPU.

The reference is the torch float64 restatement of the oracle's filter (oracle/cd_torch_kf.py) differentiated by torch
autograd: the gradient of the same discrete function.  Every gate is on one block's max error over that block's max
|value|; symmetric parameters (R, P0 and, through Sigma = L Qc L^T, Qc) are compared on their symmetric parts."""
import numpy as np
import pytest
import torch
from scipy.linalg import expm

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _engine
from cd_dynamax_b200.autograd import cdlgssm_marginal_log_prob
from cd_dynamax_b200.continuous_discrete_linear_gaussian_ssm import inference as kfi
from oracle import cd_oracle as o
from oracle import cd_torch_kf as tk
from tests.helpers import record, scaled_err
from tests.test_gpu_time_grids import degenerate_grid, edge_grid, long_grid, probe_grid, regular_grid
from tests.test_kf_grad_host import random_grid, random_model

pytestmark = pytest.mark.gpu
GATE = 1e-9
dev = torch.device("cuda", 0) if torch.cuda.is_available() else None


def api_params(p, as_torch=False):
    T = (lambda x: torch.as_tensor(np.asarray(x, np.float64), device=dev)) if as_torch else (lambda x: x)
    return cd.make_cdlgssm_params(initial_mean=T(p["m0"]), initial_cov=T(p["P0"]), dynamics_weights=T(p["F"]),
                                  dynamics_diffusion_coeff=T(p["L"]), dynamics_diffusion_cov=T(p["Qc"]),
                                  emissions_weights=T(p["H"]), emissions_cov=T(p["R"]), dynamics_bias=T(p["b"]),
                                  emissions_bias=T(p["d"]))


def hyper(solver, dt0, max_steps=100000, dt_final=1e-10):
    return cd.KFHyperParams(dt_final=dt_final, diffeqsolve_settings={"solver": solver, "dt0": dt0, "max_steps": max_steps})


def reference(p, y, t, solver, dt0, dt_final=1e-10):
    """(ll [N], per-trajectory gradients keyed like the API's leaves) from torch autograd of the arbiter."""
    N = y.shape[0]
    leaves = {}
    for k in ("F", "b", "L", "Qc", "H", "d", "R", "m0", "P0"):
        x = torch.tensor(np.asarray(p[k], np.float64))
        core = 1 if k in ("b", "d", "m0") else 2
        x = x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))
        leaves[k] = x.clone().requires_grad_(True)  # per-trajectory copies: autograd gives one gradient row each
    Sigma = leaves["L"] @ leaves["Qc"] @ leaves["L"].transpose(-1, -2)
    ll = tk.marginal_log_prob(leaves["F"], leaves["b"], Sigma, leaves["H"], leaves["d"], leaves["R"], leaves["m0"],
                              leaves["P0"], y, t, dt_final, o.SolverSettings(solver, dt0))
    g = torch.autograd.grad(ll.sum(), list(leaves.values()))
    return ll.detach().numpy(), {k: v.numpy() for k, v in zip(leaves, g)}


def sym(x):
    return 0.5 * (x + np.swapaxes(x, -1, -2))


def kernel_blocks(grads):
    c = lambda x: x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    return dict(F=c(grads.dynamics.weights), b=c(grads.dynamics.bias), L=c(grads.dynamics.diffusion_coefficient),
                Qc=c(grads.dynamics.diffusion_cov), H=c(grads.emissions.weights), d=c(grads.emissions.bias),
                R=c(grads.emissions.cov), m0=c(grads.initial.mean), P0=c(grads.initial.cov))


def compare(name, p, y, t, solver, dt0, gate=GATE, dt_final=1e-10):
    y_dev = torch.as_tensor(y, device=dev)
    ll, grads = cd.cdlgssm_marginal_log_prob_and_grad(api_params(p), y_dev, torch.as_tensor(t, device=dev)[..., None],
                                                      hyper(solver, dt0, dt_final=dt_final))
    ref_ll, ref = reference(p, y, t, solver, dt0, dt_final)
    assert scaled_err(ll.cpu().numpy(), ref_ll) < 1e-12
    got = kernel_blocks(grads)
    worst = 0.0
    for k, r in ref.items():
        r = sym(r) if k in ("R", "P0", "Qc") else r
        err = scaled_err(got[k], r)
        record(f"kf_grad:{name}:{k}", err)
        worst = max(worst, err)
        assert err < gate, (name, k, err)
    return worst


CASES = [("euler", 1, 1, False), ("heun", 2, 2, True), ("midpoint", 4, 4, False), ("ralston", 5, 8, True),
         ("bosh3", 16, 1, False), ("rk4", 16, 4, True), ("rk4", 5, 2, False), ("dopri5", 1, 8, True),
         ("dopri5", 4, 2, False), ("dopri5", 16, 8, True), ("dopri5", 16, 4, False), ("heun", 16, 8, False)]


@pytest.mark.parametrize("solver,n,m,batched", CASES)
def test_gradient_matches_arbiter(solver, n, m, batched):
    N, K = 7, 40  # ragged: not a multiple of the warps per CTA
    p = random_model(n, m, seed=100 + n * 9 + m, N=N if batched else None)
    y = np.random.default_rng(n + m).standard_normal((N, K, m))
    compare(f"{solver}:n{n}:m{m}:{'batched' if batched else 'shared'}", p, y, random_grid(N, K, 5), solver, 0.02)


GRIDS = {
    "arange@1e4:rk4": (lambda: regular_grid(6, 20, "arange", 1e4), "rk4", 0.0025),
    "arange@1e4:dopri5": (lambda: regular_grid(6, 20, "arange", 1e4), "dopri5", 0.01),
    "edge:rk4": (lambda: edge_grid(6, 20, 0.0025), "rk4", 0.0025),
    "edge:dopri5": (lambda: edge_grid(6, 20, 0.01), "dopri5", 0.01),
    "degenerate:rk4": (lambda: degenerate_grid(6, 20, 0.0025), "rk4", 0.0025),
    "degenerate:dopri5": (lambda: degenerate_grid(6, 20, 0.01), "dopri5", 0.01),
    "long:rk4": (lambda: long_grid(5, 6, 0.0025), "rk4", 0.0025),
    "long:dopri5": (lambda: long_grid(5, 6, 0.01), "dopri5", 0.01),
}


@pytest.mark.parametrize("grid", list(GRIDS))
def test_gradient_on_time_grids(grid):
    make, solver, dt0 = GRIDS[grid]
    t = make()
    N, K = t.shape
    p = random_model(3, 2, seed=21)
    y = np.random.default_rng(22).standard_normal((N, K, 2))
    compare(grid, p, y, t, solver, dt0)


@pytest.mark.parametrize("solver", ["rk4", "dopri5"])
def test_loglik_is_bit_identical_to_the_filter(solver):
    N, K, n, m = 37, 30, 6, 3
    p = random_model(n, m, seed=31)
    y = torch.as_tensor(np.random.default_rng(32).standard_normal((N, K, m)), device=dev)
    t = torch.as_tensor(random_grid(N, K, 33), device=dev)[..., None]
    hp = hyper(solver, 0.01)
    ll, _ = cd.cdlgssm_marginal_log_prob_and_grad(api_params(p, True), y, t, hp)
    post = cd.cdlgssm_filter(api_params(p, True), y, t, hp)
    assert torch.equal(ll, post.marginal_loglik)


def test_max_steps_rows_are_nan_and_raise_for_host_callers():
    N, K, dt0, max_steps = 20, 12, 0.01, 4
    t = probe_grid(N, K, dt0)
    count = o.substep_counts(t[:, :-1], t[:, 1:], dt0).max(axis=1)
    over = count > max_steps
    assert over.any() and not over.all()
    p = random_model(2, 1, seed=41)
    y = np.random.default_rng(42).standard_normal((N, K, 1))
    hp = hyper("rk4", dt0, max_steps)
    ll, grads = cd.cdlgssm_marginal_log_prob_and_grad(api_params(p), torch.as_tensor(y, device=dev),
                                                      torch.as_tensor(t, device=dev)[..., None], hp)
    status = _engine.last_status().cpu().numpy()
    assert np.array_equal(status == 2, over) and np.all(status[~over] == 0)
    F = grads.dynamics.weights.cpu().numpy()
    assert np.all(np.isnan(F[over])) and np.all(np.isfinite(F[~over]))
    with pytest.raises(_engine.MaxStepsReached):
        cd.cdlgssm_marginal_log_prob_and_grad(api_params(p), y, t[..., None], hp)


def test_batch_equals_its_shards_permutations_and_chunks(monkeypatch):
    N, K, n, m = 23, 25, 5, 3
    p = random_model(n, m, seed=51, N=N)
    y = np.random.default_rng(52).standard_normal((N, K, m))
    t = random_grid(N, K, 53)
    hp = hyper("dopri5", 0.01)
    run = lambda idx: cd.cdlgssm_marginal_log_prob_and_grad(
        api_params({k: v[idx] for k, v in p.items()}, True), torch.as_tensor(y[idx], device=dev),
        torch.as_tensor(t[idx], device=dev)[..., None], hp)
    flat = lambda r: [r[0].cpu().numpy()] + list(kernel_blocks(r[1]).values())
    full = flat(run(np.arange(N)))
    for lo, hi in ((0, 9), (9, 10), (10, N)):
        part = flat(run(np.arange(lo, hi)))
        for i, (a, b) in enumerate(zip(full, part)):
            assert np.array_equal(a[lo:hi], b), (lo, hi, i, np.nanmax(np.abs(a[lo:hi] - b)))
    perm = np.random.default_rng(54).permutation(N)
    for i, (a, b) in enumerate(zip(full, flat(run(perm)))):
        assert np.array_equal(a[perm], b), ("permuted", i)
    monkeypatch.setattr(kfi, "_grad_chunk", lambda N, row: 4)  # several launches when the scratch does not fit
    for i, (a, b) in enumerate(zip(full, flat(run(np.arange(N))))):
        assert np.array_equal(a, b), ("chunked", i)


@pytest.mark.parametrize("solver", ["rk4", "dopri5"])
def test_c2_shape_long_run(solver):
    N, K, n, m = 64, 500, 16, 4
    rng = np.random.default_rng(1235)
    p = random_model(n, m, seed=61)
    p["F"] = -0.5 * np.eye(n) + 0.3 * rng.standard_normal((n, n)) / np.sqrt(n)
    y = rng.standard_normal((N, K, m))
    t = random_grid(N, K, 62, mean_gap=0.04)
    compare(f"c2:{solver}", p, y, t, solver, 0.01, gate=1e-8)


def test_autograd_wrapper_sums_shared_leaves():
    N, K, n, m = 9, 30, 4, 2
    p = random_model(n, m, seed=71)
    y = torch.as_tensor(np.random.default_rng(72).standard_normal((N, K, m)), device=dev)
    t = torch.as_tensor(random_grid(N, K, 73), device=dev)[..., None]
    hp = hyper("dopri5", 0.01)
    params = api_params(p, True)
    leaves = [params.dynamics.weights, params.dynamics.bias, params.dynamics.diffusion_coefficient,
              params.dynamics.diffusion_cov, params.emissions.weights, params.emissions.bias, params.emissions.cov,
              params.initial.mean, params.initial.cov]
    for x in leaves:
        x.requires_grad_(True)
    ll = cdlgssm_marginal_log_prob(params, y, t, hp)
    (-ll.sum()).backward()
    with torch.no_grad():
        ll_f, g = cd.cdlgssm_marginal_log_prob_and_grad(params, y, t, hp)
    assert torch.equal(ll.detach(), ll_f)
    ref = [g.dynamics.weights, g.dynamics.bias, g.dynamics.diffusion_coefficient, g.dynamics.diffusion_cov,
           g.emissions.weights, g.emissions.bias, g.emissions.cov, g.initial.mean, g.initial.cov]
    for x, r in zip(leaves, ref):
        assert scaled_err(x.grad.cpu().numpy(), -r.sum(0).cpu().numpy()) < 1e-12


def test_adam_on_a_damped_oscillator_raises_the_loglik():
    N, K, n, m = 32, 60, 2, 1
    F_true = np.array([[0.0, 1.0], [-4.0, -0.5]])
    p = dict(F=F_true, b=np.zeros(n), L=np.eye(n), Qc=0.05 * np.eye(n), H=np.array([[1.0, 0.0]]), d=np.zeros(m),
             R=0.1 * np.eye(m), m0=np.array([1.0, 0.0]), P0=0.1 * np.eye(n))
    t = random_grid(N, K, 81, mean_gap=0.1)
    x = np.stack([[expm(F_true * (tk_ - t[i, 0])) @ p["m0"] for tk_ in t[i]] for i in range(N)])  # the noiseless path
    y = x[..., :1] + 0.3 * np.random.default_rng(82).standard_normal((N, K, m))
    params = api_params(p, True)
    F = (params.dynamics.weights + torch.tensor([[0.3, -0.4], [1.0, 0.5]], device=dev)).requires_grad_(True)
    params = params._replace(dynamics=params.dynamics._replace(weights=F))
    yt, tt = torch.as_tensor(y, device=dev), torch.as_tensor(t, device=dev)[..., None]
    hp = hyper("dopri5", 0.01)
    opt = torch.optim.Adam([F], lr=0.02)
    first = None
    for _ in range(50):
        opt.zero_grad()
        ll = cdlgssm_marginal_log_prob(params, yt, tt, hp).sum()
        first = float(ll.detach()) if first is None else first
        (-ll).backward()
        opt.step()
    last = float(cdlgssm_marginal_log_prob(params, yt, tt, hp).sum().detach())
    record("kf_grad:adam:ll_gain", last - first)
    assert last > first + 1.0, (first, last)
