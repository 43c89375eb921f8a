"""cdk_ekf_grad_dense_f64 for USER-DEFINED drifts (LearnableUserDrift(..., differentiable=True)) on the GPU: the variant
library built with build_user_drift(code, grad=True) takes the drift's derivatives from dual-number evaluations of the
user's own device code (csrc/cdk_dual.cuh).

The reference is a torch float64 restatement of the EKF with the same drift written in torch, differentiated by
autograd, under the gate of tests/test_gpu_ekf_grad.py (every block's max error <= 1e-9 of its max |value|, Sigma, R and
P0 on symmetric parts).  Cross-checks without torch: user drifts that restate the registry's quadratic and Lorenz-63
drifts against the registry's own gradient, and central differences of the filter."""
import os

import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _engine as E
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200 import build as b
from cd_dynamax_b200.autograd import ekf_marginal_log_prob
from oracle import cd_oracle as o
from oracle.cd_torch_kf import _mvn_logpdf, _sym, substeps
from tests.helpers import record, scaled_err
from tests.test_ekf_grad_host import BLOCKS, random_model
from tests.test_gpu_ekf_grad import GATE, _ins, blocks, dense, sym
from tests.test_gpu_time_grids import degenerate_grid, edge_grid, long_grid, regular_grid
from tests.test_kf_grad_host import random_grid

pytestmark = pytest.mark.gpu
EXAMPLES = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cd_dynamax_b200", "examples")
VDP = open(os.path.join(EXAMPLES, "vdp_drift.cuh")).read()
MLP = open(os.path.join(EXAMPLES, "mlp_drift.cuh")).read()

# the registry's quadratic drift (n = 2) and Lorenz-63, restated as user code
QUAD = r'''
namespace cdk_user {
template <typename T, class XF> __device__ T f(const T* th, int n, int i, XF x) {
  T s = th[i];
  for (int j = 0; j < 2; ++j) {
    T c = th[2 + i * 2 + j];
    for (int k = 0; k < 2; ++k) c += th[6 + (i * 2 + j) * 2 + k] * x(k);
    s += c * x(j);
  }
  return s;
}
template <typename T> __device__ T jac(const T* th, int n, int i, int j, const T* x) {
  T s = th[2 + i * 2 + j];
  for (int k = 0; k < 2; ++k) s += (th[6 + (i * 2 + j) * 2 + k] + th[6 + (i * 2 + k) * 2 + j]) * x[k];
  return s;
}
template <typename T> __device__ T graddiv(const T* th, int n, int k, const T* x) {
  T s = T(0);
  for (int i = 0; i < 2; ++i) s += th[6 + (i * 2 + i) * 2 + k] + th[6 + (i * 2 + k) * 2 + i];
  return s;
}
}
'''
L63 = r'''
namespace cdk_user {
template <typename T, class XF> __device__ T f(const T* th, int n, int i, XF x) {
  if (i == 0) return th[0] * (x(1) - x(0));
  if (i == 1) return x(0) * (th[1] - x(2)) - x(1);
  return x(0) * x(1) - th[2] * x(2);
}
template <typename T> __device__ T jac(const T* th, int n, int i, int j, const T* x) {
  if (i == 0) return j == 0 ? -th[0] : (j == 1 ? th[0] : T(0));
  if (i == 1) return j == 0 ? th[1] - x[2] : (j == 1 ? T(-1) : -x[0]);
  return j == 0 ? x[1] : (j == 1 ? x[0] : -th[2]);
}
template <typename T> __device__ T graddiv(const T* th, int n, int k, const T* x) { return T(0); }
}
'''


# ---- the same drifts in torch: f(theta, x) [N, n], jac [N, n, n], graddiv(theta, x) [N, n] -----------------------------
def vdp_fns():
    def f(th, x):
        mu, eps, x0, x1 = th[:, 0], th[:, 1], x[:, 0], x[:, 1]
        return torch.stack([x1, mu * (1 - x0 * x0) * x1 - x0 - eps * x0 ** 3], -1)

    def jac(th, x):
        mu, eps, x0, x1 = th[:, 0], th[:, 1], x[:, 0], x[:, 1]
        z, one = torch.zeros_like(x0), torch.ones_like(x0)
        return torch.stack([torch.stack([z, one], -1),
                            torch.stack([-2 * mu * x0 * x1 - 1 - 3 * eps * x0 * x0, mu * (1 - x0 * x0)], -1)], -2)

    return f, jac, lambda th, x: torch.stack([-2 * th[:, 0] * x[:, 0], torch.zeros_like(x[:, 0])], -1)


def mlp_fns(Hd=16):
    def split(th):
        return (th[:, :2 * Hd].reshape(-1, Hd, 2), th[:, 2 * Hd:3 * Hd], th[:, 3 * Hd:5 * Hd].reshape(-1, 2, Hd),
                th[:, 5 * Hd:])

    def hidden(th, x):
        W1, b1, _, _ = split(th)
        return torch.tanh((W1 @ x[..., None])[..., 0] + b1)

    def f(th, x):
        _, _, W2, b2 = split(th)
        return (W2 @ hidden(th, x)[..., None])[..., 0] + b2

    def jac(th, x):
        W1, _, W2, _ = split(th)
        t = hidden(th, x)
        return W2 @ ((1 - t * t)[..., None] * W1)

    def graddiv(th, x):
        W1, _, W2, _ = split(th)
        t = hidden(th, x)
        c = torch.einsum("nih,nhi->nh", W2, W1)
        return torch.einsum("nh,nhk->nk", c * (-2 * t * (1 - t * t)), W1)

    return f, jac, graddiv


def torch_ll(fns, theta, Sigma, H, d, R, m0, P0, y, t, state_order, settings):
    """cd_torch_ekf.extended_kalman_filter's log-likelihood with an x-dependent graddiv(theta, x) (the filter's
    'second'-order term for a user drift), batched over N."""
    f, jac, graddiv = fns
    y = torch.as_tensor(np.asarray(y, np.float64))
    N, K, mdim = y.shape
    c = lambda x, core: x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))
    theta, Sigma, H, R, P0, d, m0 = c(theta, 1), c(Sigma, 2), c(H, 2), c(R, 2), c(P0, 2), c(d, 1), c(m0, 1)
    tab = o.TABLEAUX[settings.solver]
    a, bw = tab["a"], tab["b"]

    def rhs(mm, PP):
        J = jac(theta, mm)
        dm = f(theta, mm)
        if state_order == "second":
            dm = dm + 0.5 * torch.einsum("nk,nkl->nl", graddiv(theta, mm), PP)
        return dm, J @ PP + PP @ J.transpose(-1, -2) + Sigma

    t0s, t1s = o._gap_times(np.asarray(t, np.float64), 1e-10)
    m, P = m0, P0
    ll = torch.zeros(N, dtype=torch.float64)
    eye = torch.eye(mdim, dtype=torch.float64)
    for k in range(K):
        Hm = (H @ m[..., None])[..., 0]
        S = R + H @ P @ H.transpose(-1, -2)
        ll = ll + _mvn_logpdf(y[:, k], Hm + d, S)
        Kt = torch.cholesky_solve(H @ P, torch.linalg.cholesky(_sym(S) + 1e-9 * eye))
        Kg = Kt.transpose(-1, -2)
        m = m + (Kg @ (y[:, k] - (Hm + d))[..., None])[..., 0]
        P = _sym(P - Kg @ S @ Kt)
        dts, acts, hit = substeps(t0s[:, k], t1s[:, k], settings)
        assert not hit.any()
        for dt_np, act_np in zip(dts, acts):
            dtm = torch.as_tensor(dt_np)[:, None]
            ks = []
            for i in range(len(bw)):
                ym = m + sum(a[i][j] * ks[j][0] for j in range(i) if a[i][j] != 0.0) if i else m
                yP = P + sum(a[i][j] * ks[j][1] for j in range(i) if a[i][j] != 0.0) if i else P
                km, kP = rhs(ym, yP)
                ks.append((dtm * km, dtm[..., None] * kP))
            act = torch.as_tensor(act_np)
            m = torch.where(act[:, None], m + sum(bw[j] * ks[j][0] for j in range(len(bw)) if bw[j] != 0.0), m)
            P = torch.where(act[:, None, None], P + sum(bw[j] * ks[j][1] for j in range(len(bw)) if bw[j] != 0.0), P)
    return ll


def user_model(which, m, seed, N=None, theta_batched=False):
    """A random model (tests.test_ekf_grad_host.random_model) with the drift's theta."""
    rng = np.random.default_rng(seed)
    p = random_model("linear", 2, m, seed, N=N)
    lead = (N,) if theta_batched else ()
    if which == "vdp":
        p["theta"] = np.array([1.3, 0.4]) * (1.0 + 0.1 * rng.standard_normal(lead + (2,)))
    else:
        W1 = 0.8 * rng.standard_normal(lead + (16, 2))
        W2 = 0.4 * rng.standard_normal(lead + (2, 16)) / 4.0
        p["theta"] = np.concatenate([W1.reshape(lead + (32,)), 0.3 * rng.standard_normal(lead + (16,)),
                                     W2.reshape(lead + (32,)), 0.1 * rng.standard_normal(lead + (2,))], -1)
    p["m0"] = p["m0"] + np.array([1.0, 0.5])
    p["kind"] = which
    return p


CODE = {"vdp": VDP, "mlp": MLP}
FNS = {"vdp": vdp_fns, "mlp": mlp_fns}


def user_fields(code, nt, solver, dt0, order, max_steps=100000):
    return dict(solver=L.SOLVERS[solver], dt0=dt0, max_steps=max_steps, dt_final=1e-10, state_order=L.ORDERS[order],
                num_iter=1, drift_id=L.DRIFT_USER, n_theta=nt, emission_id=0,
                lib_path=b.build_user_drift(code, grad=True))


def dense_user(code, p, y, t, solver, dt0, order):
    N, K, m = y.shape
    nt = np.shape(p["theta"])[-1]
    n = np.shape(p["m0"])[-1]
    out = E.run("cdk_ekf_grad_dense", "f64", N, K, n, m, _ins(p, y, t), (L.OUT_LL, L.OUT_GRAD),
                user_fields(code, nt, solver, dt0, order), out_shapes={L.OUT_GRAD: (N, L.grad_cols_ekf(n, m, nt))})
    return out[L.OUT_LL], out[L.OUT_STATUS], out[L.OUT_GRAD]


def compare_user(name, which, p, y, t, solver, dt0, order):
    ll, status, G = dense_user(CODE[which], p, y, t, solver, dt0, order)
    assert int(status.abs().sum()) == 0, name
    N, K, m = y.shape
    n = np.shape(p["m0"])[-1]
    nt = np.shape(p["theta"])[-1]
    f = E.run("cdk_ekf_filter", "f64", N, K, n, m, _ins(p, y, t), (L.OUT_LL,), user_fields(CODE[which], nt, solver, dt0, order))
    assert torch.equal(ll, f[L.OUT_LL]), name  # the forward pass is the filter's launch
    leaves = {}
    for k in BLOCKS:
        x = torch.tensor(np.asarray(p[k], np.float64))
        core = 1 if k in ("theta", "d", "m0") else 2
        leaves[k] = (x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))).clone().requires_grad_(True)
    ref_ll = torch_ll(FNS[which](), *(leaves[k] for k in BLOCKS), y, t, order, o.SolverSettings(solver, dt0))
    ref = dict(zip(leaves, torch.autograd.grad(ref_ll.sum(), list(leaves.values()))))
    err_ll = scaled_err(ll.cpu().numpy(), ref_ll.detach().numpy())
    record(f"user_drift_grad:{name}:ll", err_ll)
    assert err_ll < 1e-11, (name, err_ll)
    got = blocks(G, n, m, nt)
    worst = 0.0
    for k, r in ref.items():
        r = r.numpy()
        r = sym(r) if k in ("Sigma", "R", "P0") else r
        err = scaled_err(got[k], r)
        record(f"user_drift_grad:{name}:{k}", err)
        worst = max(worst, err)
        assert err < GATE, (name, k, err)
    return worst


def case(which, m=1, N=3, K=10, seed=0, batched=False, theta_batched=False, gap=0.05):
    p = user_model(which, m, seed, N=N if batched else None, theta_batched=theta_batched)
    rng = np.random.default_rng(seed + 1)
    return p, 0.7 * rng.standard_normal((N, K, m)), random_grid(N, K, seed + 2, mean_gap=gap)


@pytest.mark.parametrize("solver", list(L.SOLVERS))
@pytest.mark.parametrize("order", ["first", "second"])
def test_vdp_every_solver(order, solver):
    p, y, t = case("vdp", seed=1)
    compare_user(f"vdp_{order}_{solver}", "vdp", p, y, t, solver, 0.01, order)


@pytest.mark.parametrize("solver", ["rk4", "dopri5"])
@pytest.mark.parametrize("order", ["first", "second"])
def test_mlp(order, solver):
    p, y, t = case("mlp", seed=2)
    compare_user(f"mlp_{order}_{solver}", "mlp", p, y, t, solver, 0.01, order)


@pytest.mark.parametrize("which", ["vdp", "mlp"])
def test_theta_batched_and_m3(which):
    p, y, t = case(which, m=3, N=4, seed=3, batched=True, theta_batched=True)
    compare_user(f"{which}_batched_m3", which, p, y, t, "rk4", 0.01, "second")


@pytest.mark.parametrize("grid", ["t0_1e4", "edge", "degenerate", "long"])
def test_time_grids(grid):
    N, K, dt0 = 3, 8, 0.01
    p = user_model("vdp", 1, 40)
    t = {"t0_1e4": lambda: regular_grid(N, K, t0=1e4, h=0.013), "edge": lambda: edge_grid(N, K, dt0),
         "degenerate": lambda: degenerate_grid(N, K, dt0), "long": lambda: long_grid(N, 6, dt0)}[grid]()
    y = 0.7 * np.random.default_rng(41).standard_normal((N, t.shape[1], 1))
    compare_user(f"grid_{grid}", "vdp", p, y, t, "rk4", dt0, "second")


def test_each_slot_batched_alone_is_bit_identical_to_the_shared_value():
    N = 5
    p, y, t = case("mlp", m=2, N=N, K=8, seed=90)
    _, _, G0 = dense_user(MLP, p, y, t, "rk4", 0.01, "second")
    _, _, G1 = dense_user(MLP, p, y, t, "rk4", 0.01, "second")
    assert torch.equal(G0, G1)  # run to run
    for slot in ("theta", "L", "Qc", "H", "d", "R", "m0", "P0"):
        q = dict(p)
        q[slot] = np.broadcast_to(np.asarray(p[slot]), (N,) + np.shape(p[slot])).copy()
        _, _, G = dense_user(MLP, q, y, t, "rk4", 0.01, "second")
        assert torch.equal(G, G0), slot


def _registry_pair(kind, code, n, m, order, K, solver="rk4"):
    p = random_model(kind, n, m, seed=7, N=3 if kind == "quadratic" else None)
    y = (3.0 if kind == "lorenz63" else 0.5) * np.random.default_rng(8).standard_normal((3, K, m))
    t = random_grid(3, K, 9, mean_gap=0.03)
    _, st_r, G_r = dense(p, y, t, solver, 0.01, order)
    _, st_u, G_u = dense_user(code, p, y, t, solver, 0.01, order)
    assert int(st_r.abs().sum()) == 0 and int(st_u.abs().sum()) == 0
    return blocks(G_r, n, m, np.shape(p["theta"])[-1]), blocks(G_u, n, m, np.shape(p["theta"])[-1])


def test_restated_quadratic_matches_the_registry():
    """'second' order: the theta-derivative of graddiv (VdP's graddiv checks its x-derivative against torch)."""
    r, u = _registry_pair("quadratic", QUAD, 2, 2, "second", 12)
    for k in r:
        err = scaled_err(u[k], r[k])
        record(f"user_drift_grad:quadratic_vs_registry:{k}", err)
        assert err < 1e-11, (k, err)


def test_restated_lorenz63_matches_the_registry():
    r, u = _registry_pair("lorenz63", L63, 3, 3, "first", 12)
    for k in r:
        err = scaled_err(u[k], r[k])
        record(f"user_drift_grad:lorenz63_vs_registry:{k}", err)
        assert err < 1e-10, (k, err)


def test_directional_derivatives_match_central_differences_of_the_filter():
    N, K = 4, 100
    p, y, t = case("mlp", m=2, N=N, K=K, seed=60, gap=0.03)
    _, _, G = dense_user(MLP, p, y, t, "rk4", 0.01, "second")
    got = blocks(G, 2, 2, 82)
    rng = np.random.default_rng(61)
    nt = 82

    def ll_at(q):
        f = E.run("cdk_ekf_filter", "f64", N, K, 2, 2, _ins(q, y, t), (L.OUT_LL,), user_fields(MLP, nt, "rk4", 0.01, "second"))
        return float(f[L.OUT_LL].sum())

    for name in ("theta", "Sigma", "H", "d", "R", "m0", "P0"):
        key = "Qc" if name == "Sigma" else name
        v = rng.standard_normal(np.shape(p[key]))
        if name in ("Sigma", "R", "P0"):
            v = 0.5 * (v + v.T)
        h = 1e-5

        def moved(s):
            q = dict(p)
            if name == "Sigma":  # the filter takes L and Qc: move Qc so that L Qc L^T moves by s v
                q["Qc"] = p["Qc"] + s * np.linalg.solve(p["L"], np.linalg.solve(p["L"], v).T).T
            else:
                q[name] = p[name] + s * v
            return q

        fd = (ll_at(moved(h)) - ll_at(moved(-h))) / (2 * h)
        an = float(np.sum(got[name].sum(0) * v))
        record(f"user_drift_grad:central_difference:{name}", abs(an - fd) / max(abs(fd), 1e-300))
        assert abs(an - fd) <= 1e-6 * max(abs(fd), 1.0), (name, an, fd)


def test_public_entry_and_adam_fit_of_vdp():
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
    hp = cd.EKFHyperParams(state_order="second", diffeqsolve_settings={"solver": "rk4", "dt0": 0.01})
    ll, g = cd.ekf_marginal_log_prob_and_grad(params_for(truth), ys, T, hp, wrt="all")
    assert set(g) == {"theta", "diffusion_coefficient", "diffusion_cov", "emission_cov", "emission_bias",
                      "emission_weights", "initial_mean", "initial_cov"} and g["theta"].shape == (N, 2)
    f = cd.cdnlgssm_filter(params_for(truth), ys, T, hp, output_fields=[])
    assert np.array_equal(ll, f.marginal_loglik)
    theta = torch.tensor([0.8, 0.1], dtype=torch.float64, requires_grad=True)
    opt = torch.optim.Adam([theta], lr=0.05)
    losses = []
    for _ in range(50):
        opt.zero_grad()
        loss = -ekf_marginal_log_prob(params_for(theta), ys, T, hp).sum() / (N * K)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    record("user_drift_grad:adam_vdp_mu_final", float(theta.detach()[0]))
    assert losses[-1] < losses[0]
    assert abs(float(theta[0]) - truth[0]) <= 0.5 * abs(0.8 - truth[0]), theta


def test_filter_only_variant_and_ukf_reject():
    import ctypes
    var = L.lib(b.build_user_drift(VDP))
    d = L.new_desc()
    d.N, d.K, d.n, d.m, d.drift_id, d.n_theta = 2, 3, 2, 1, L.DRIFT_USER, 2
    fake = ctypes.c_void_p(0x1000)
    ins = (ctypes.c_void_p * L.NUM_IN)(*([fake] * L.NUM_IN))
    outs = (ctypes.c_void_p * L.NUM_OUT)(*([fake] * L.NUM_OUT))
    assert var.cdk_ekf_grad_dense_f64(ctypes.byref(d), ins, outs, None) == -4
    assert "differentiable=True" in var.cdk_last_error().decode()
    p, y, t = case("vdp", seed=5)
    params = cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=p["m0"], cov=p["P0"]),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableUserDrift(VDP, p["theta"], differentiable=True),
                                           diffusion_coefficient=p["L"], diffusion_cov=p["Qc"]),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=p["H"], bias=p["d"]),
                                             emission_cov=p["R"]))
    with pytest.raises(NotImplementedError):
        cd.ukf_marginal_log_prob_and_grad(params, y, t[..., None])
