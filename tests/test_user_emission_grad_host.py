"""Host side of the CD-EKF gradient for user-defined emissions (no GPU).

A torch float64 EKF with the drift AND the emission given as torch callables (drift: the registry's torch functions or
VdP's; emission: range, wide tanh network, square, linear) is the reference of tests/test_gpu_user_emission_grad.py.
Here it is pinned to the NumPy oracle of tests/user_emission_oracle.py (log-likelihood to 1e-12) and its phi gradient to
central differences of that oracle (1e-6).  Also: the Python gates and `wrt` errors, the variant's build flags, units
and hashes (with a faked compiler), and the C-ABI answers of the stock, filter-only and gradient libraries."""
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200 import build as b
from oracle import cd_oracle as o
from oracle.cd_torch_ekf import drift_fns
from oracle.cd_torch_kf import _mvn_logpdf, _sym, substeps
from tests.test_ekf_grad_host import random_model
from tests.test_gpu_user_drift_grad import vdp_fns
from tests.test_gpu_user_emission_matrix import SQUARE_CODE, WIDE_CODE, WIDTH, SquareEmission, WideEmission
from tests.test_gpu_user_emission import RangeEmission

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EX = os.path.join(ROOT, "cd_dynamax_b200", "examples")
RANGE_CODE = open(os.path.join(EX, "range_emission.cuh")).read()
LIN_CODE = open(os.path.join(EX, "linear_emission.cuh")).read()
VDP_CODE = open(os.path.join(EX, "vdp_drift.cuh")).read()
# the largest n_phi the backward layout admits at n = 40, m = 20 (EgLay: 21,624 doubles + 2 n_phi for phi and its
# cotangent; the dual scratch 256 * 4 + (40 + n_phi) * 5 aliases the 6,720 doubles of YC..ACC; 227 KiB = 29,056 doubles)
C4_MAX_NPHI = 1099


def fixed_params_code(k):
    """A linear-in-x emission with exactly k parameters (k >= 1), for the n_phi limit: h_a = sum_j phi[(a n + j) % k] x_j."""
    return ("namespace cdk_user_emission {\n"
            f"__host__ __device__ inline int num_params(int n, int m) {{ return {k}; }}\n"
            "template <typename T, class XF> __device__ __forceinline__ T h(const T* phi, int n, int m, int a, XF x) {\n"
            f"  T s = T(0);\n  for (int j = 0; j < n; ++j) s += phi[(a * n + j) % {k}] * x(j);\n  return s;\n}}\n"
            "template <typename T> __device__ __forceinline__ T jac(const T* phi, int n, int m, int a, int j, const T* x) {\n"
            f"  return phi[(a * n + j) % {k}];\n}}\n}}\n")


CODE = {"range": RANGE_CODE, "wide": WIDE_CODE, "square": SQUARE_CODE, "linear": LIN_CODE}


# ---- the emissions in torch: h(phi, x) [N, m] and jac(phi, x) [N, m, n] for phi [N, n_phi], x [N, n] --------------------
def emission_fns(kind, n, m):
    if kind == "range":
        def h(phi, x):
            r = x[:, None, :] - phi[:, :m * n].reshape(-1, m, n)
            return torch.sqrt(phi[:, m * n:m * n + 1] + (r * r).sum(-1))
        return h, lambda phi, x: (x[:, None, :] - phi[:, :m * n].reshape(-1, m, n)) / h(phi, x)[..., None]
    if kind == "linear":
        H = lambda phi: phi[:, :m * n].reshape(-1, m, n)
        return lambda phi, x: (H(phi) @ x[..., None])[..., 0] + phi[:, m * n:], lambda phi, x: H(phi)
    if kind == "wide":
        def split(phi):
            o_ = WIDTH * n
            return (phi[:, :o_].reshape(-1, WIDTH, n), phi[:, o_:o_ + WIDTH],
                    phi[:, o_ + WIDTH:o_ + WIDTH + m * WIDTH].reshape(-1, m, WIDTH), phi[:, o_ + WIDTH + m * WIDTH:])

        def hidden(phi, x):
            W1, b1, _, _ = split(phi)
            return torch.tanh((W1 @ x[..., None])[..., 0] + b1)

        def h(phi, x):
            _, _, W2, b2 = split(phi)
            return (W2 @ hidden(phi, x)[..., None])[..., 0] + b2

        def jac(phi, x):
            W1, _, W2, _ = split(phi)
            t = hidden(phi, x)
            return W2 @ ((1 - t * t)[..., None] * W1)
        return h, jac
    if kind == "square":
        idx = torch.arange(m) % n
        onehot = torch.nn.functional.one_hot(idx, n).to(torch.float64)
        return lambda phi, x: x[:, idx] ** 2, lambda phi, x: 2.0 * x[:, idx][..., None] * onehot
    raise ValueError(kind)


def emission_model(drift, em, n, m, seed, N=None, nphi=None):
    """A random model (tests.test_ekf_grad_host.random_model) with a user emission `em` and its phi; drift 'vdp' is the
    user drift of examples/vdp_drift.cuh (n = 2), the others registry drifts."""
    rng = np.random.default_rng(seed + 100)
    p = random_model("linear" if drift == "vdp" else drift, n, m, seed, N=N)
    lead = () if N is None else (N,)
    if drift == "vdp":
        p["theta"] = np.array([1.3, 0.4]) * (1.0 + 0.1 * rng.standard_normal(lead + (2,)))
        p["m0"] = p["m0"] + np.array([1.0, 0.5])
    if em == "range":
        phi = np.concatenate([3.0 * rng.standard_normal(lead + (m * n,)), 0.1 + 0.05 * rng.uniform(size=lead + (1,))], -1)
    elif em == "linear":
        phi = np.concatenate([p["H"].reshape(lead + (m * n,)), p["d"]], -1)
    elif em == "wide":
        phi = np.stack([WideEmission(n, m, rng).phi() for _ in range(N)]) if N else WideEmission(n, m, rng).phi()
    elif em == "square":
        phi = np.zeros(lead + (0,))
    else:  # "fixed": fixed_params_code(nphi)
        phi = 0.1 * rng.standard_normal(lead + (nphi,))
    p.update(phi=phi, em=em, drift=drift, drift_id={"linear": L.DRIFT_LINEAR, "lorenz63": L.DRIFT_LORENZ63,
                                                    "lorenz96": L.DRIFT_LORENZ96, "vdp": L.DRIFT_USER}.get(drift))
    return p


def _drift_fns(p):
    n = np.shape(p["m0"])[-1]
    if p["drift"] == "vdp":
        return vdp_fns()
    f, jac, gd = drift_fns(p["drift"], n)
    return f, jac, lambda th, x: gd(th)


def _predict(fns, theta, Sigma, m, P, t0, t1, order, settings):
    """The moment ODE over one gap, with an x-dependent graddiv(theta, x) (the filter's 'second'-order term)."""
    f, jac, graddiv = fns
    tab = o.TABLEAUX[settings.solver]
    a, bw = tab["a"], tab["b"]

    def rhs(mm, PP):
        J = jac(theta, mm)
        dm = f(theta, mm)
        if order == "second":
            dm = dm + 0.5 * torch.einsum("nk,nkl->nl", graddiv(theta, mm), PP)
        return dm, J @ PP + PP @ J.transpose(-1, -2) + Sigma

    dts, acts, hit = substeps(t0, t1, settings)
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
    return m, P


def torch_ll(p, y, t, solver, dt0, order, grad=False, leaves=None):
    """The EKF's log-likelihood [N] with drift and emission as torch callables (num_iter = 1, the filter's update:
    H = J(m), r = y - h(m), Kt from chol(sym(S) + 1e-9 I)).  grad=True: also {block: d ll.sum() / d block} as NumPy,
    every block per trajectory (theta, Sigma, phi, R, m0, P0)."""
    y = torch.as_tensor(np.asarray(y, np.float64))
    N, K, m = y.shape
    n = np.shape(p["m0"])[-1]
    if leaves is None:
        leaves = {}
        for k, core in (("theta", 1), ("Sigma", 2), ("phi", 1), ("R", 2), ("m0", 1), ("P0", 2)):
            x = torch.tensor(np.asarray(p[k], np.float64))
            leaves[k] = (x if x.dim() == core + 1 else x.expand((N,) + tuple(x.shape))).clone().requires_grad_(grad)
    theta, Sigma, phi, R, m_, P = (leaves[k] for k in ("theta", "Sigma", "phi", "R", "m0", "P0"))
    fns = _drift_fns(p)
    h, jac = emission_fns(p["em"], n, m)
    settings = o.SolverSettings(solver, dt0)
    t0s, t1s = o._gap_times(np.asarray(t, np.float64).reshape(N, -1), 1e-10)
    ll = torch.zeros(N, dtype=torch.float64)
    eye = torch.eye(m, dtype=torch.float64)
    for k in range(K):
        J = jac(phi, m_)
        hm = h(phi, m_)
        S = R + J @ P @ J.transpose(-1, -2)
        ll = ll + _mvn_logpdf(y[:, k], hm, S)
        Kt = torch.cholesky_solve(J @ P, torch.linalg.cholesky(_sym(S) + 1e-9 * eye))
        Kg = Kt.transpose(-1, -2)
        m_ = m_ + (Kg @ (y[:, k] - hm)[..., None])[..., 0]
        P = _sym(P - Kg @ S @ Kt)
        if k < K - 1:
            m_, P = _predict(fns, theta, Sigma, m_, P, t0s[:, k], t1s[:, k], order, settings)
    if not grad:
        return ll.detach().numpy()
    gs = torch.autograd.grad(ll.sum(), list(leaves.values()), allow_unused=True)
    return ll.detach().numpy(), {k: (np.zeros(tuple(v.shape)) if g is None else g.numpy())
                                 for (k, v), g in zip(leaves.items(), gs)}


def ue_blocks(G, n, m, nt, nph):
    """The row theta | Sigma | phi | R | m0 | P0 (CDK_GRAD_COLS_EKF_UE) as {block: [N, ...]}."""
    G = G.cpu().numpy() if isinstance(G, torch.Tensor) else G
    out, o_ = {}, 0
    for name, shp in (("theta", (nt,)), ("Sigma", (n, n)), ("phi", (nph,)), ("R", (m, m)), ("m0", (n,)), ("P0", (n, n))):
        size = int(np.prod(shp))
        out[name] = G[:, o_:o_ + size].reshape((G.shape[0],) + shp)
        o_ += size
    return out


def _oracle_em(p, n, m):
    phi = np.asarray(p["phi"], np.float64)
    if p["em"] == "range":
        return RangeEmission(phi[:m * n].reshape(m, n), phi[m * n])
    if p["em"] == "square":
        return SquareEmission(n, m)
    em = WideEmission.__new__(WideEmission)
    o_ = WIDTH * n
    em.W1, em.b1 = phi[:o_].reshape(WIDTH, n), phi[o_:o_ + WIDTH]
    em.W2, em.b2 = phi[o_ + WIDTH:o_ + WIDTH + m * WIDTH].reshape(m, WIDTH), phi[o_ + WIDTH + m * WIDTH:]
    return em


def _oracle_ll(p, y, t, solver, dt0, order):
    from tests.user_emission_oracle import extended_kalman_filter
    n, m = np.shape(p["m0"])[-1], np.shape(p["R"])[-1]
    drift = (o.LinearDrift(p["theta"][:n * n].reshape(n, n), p["theta"][n * n:]) if p["drift"] == "linear"
             else __import__("tests.test_gpu_user_emission_matrix", fromlist=["VdpDrift"]).VdpDrift(*p["theta"]))
    po = o.NonlinearParams(m0=p["m0"], P0=p["P0"], drift=drift, L=p["L"], Qc=p["Qc"], H=None, R=p["R"])
    return extended_kalman_filter(po, _oracle_em(p, n, m), y, np.asarray(t).reshape(np.shape(y)[0], -1),
                                  state_order=order, settings=o.SolverSettings(solver, dt0))["marginal_loglik"]


def _data(p, N=2, K=6, seed=0):
    from tests.test_kf_grad_host import random_grid
    rng = np.random.default_rng(seed)
    return 2.0 + 0.7 * rng.standard_normal((N, K, np.shape(p["R"])[-1])), random_grid(N, K, seed + 1, mean_gap=0.05)


@pytest.mark.parametrize("solver", ["euler", "rk4", "dopri5"])
@pytest.mark.parametrize("order", ["first", "second"])
@pytest.mark.parametrize("drift", ["vdp", "linear"])
@pytest.mark.parametrize("em", ["range", "wide", "square"])
def test_torch_reference_matches_the_oracle(em, drift, order, solver):
    p = emission_model(drift, em, 2, 3, seed=1)
    y, t = _data(p)
    ref = _oracle_ll(p, y, t, solver, 0.01, order)
    got = torch_ll(p, y, t, solver, 0.01, order)
    assert np.max(np.abs(got - ref)) <= 1e-12 * max(1.0, np.max(np.abs(ref))), (got, ref)


@pytest.mark.parametrize("em", ["range", "wide"])
def test_torch_phi_gradient_matches_central_differences_of_the_oracle(em):
    p = emission_model("vdp", em, 2, 3, seed=2)
    y, t = _data(p, N=1)
    _, g = torch_ll(p, y, t, "rk4", 0.01, "second", grad=True)
    rng = np.random.default_rng(3)
    v = rng.standard_normal(np.shape(p["phi"]))
    eps = 1e-6
    fd = (_oracle_ll(dict(p, phi=p["phi"] + eps * v), y, t, "rk4", 0.01, "second")
          - _oracle_ll(dict(p, phi=p["phi"] - eps * v), y, t, "rk4", 0.01, "second")) / (2 * eps)
    an = g["phi"][0] @ v
    assert abs(an - fd[0]) <= 1e-6 * max(1.0, abs(fd[0])), (an, fd)


# ---- Python gates -------------------------------------------------------------------------------------------------
def api_params(p, phi=None, differentiable=True, drift=None):
    n, m = np.shape(p["m0"])[-1], np.shape(p["R"])[-1]
    if drift is None:
        th = p["theta"]
        drift = cd.LearnableLinear(weights=th[:n * n].reshape(n, n), bias=th[n * n:])
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(p["m0"]), cov=cd.LearnableMatrix(p["P0"])),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=drift, diffusion_coefficient=cd.LearnableMatrix(p["L"]),
                                           diffusion_cov=cd.LearnableMatrix(p["Qc"])),
        emissions=cd.ParamsCDNLGSSMEmissions(
            emission_function=cd.LearnableUserEmission(CODE[p["em"]], p["phi"] if phi is None else phi,
                                                       differentiable=differentiable),
            emission_cov=cd.LearnableMatrix(p["R"])))


class _Sentinel(Exception):
    pass


def test_the_field_is_last_and_defaults_to_false():
    e = cd.LearnableUserEmission(device_code="", phi=np.zeros(3))
    assert e.differentiable is False and cd.LearnableUserEmission._fields[-1] == "differentiable"


def test_non_differentiable_emission_is_rejected_before_any_build(monkeypatch):
    def boom(*a, **k):
        raise _Sentinel()
    monkeypatch.setattr(b, "build_variant", boom)
    monkeypatch.setattr(L, "lib", boom)
    p = emission_model("linear", "range", 2, 3, seed=4)
    y, t = _data(p)
    from cd_dynamax_b200 import autograd
    for fn in (cd.ekf_marginal_log_prob_and_grad, cd.ekf_dense_marginal_log_prob_and_grad, autograd.ekf_marginal_log_prob):
        with pytest.raises(NotImplementedError, match=r"LearnableUserEmission.*differentiable=True"):
            fn(api_params(p, differentiable=False), y, t)
    # the UKF gradients keep refusing a user emission, differentiable or not
    for fn in (cd.ukf_marginal_log_prob_and_grad, cd.ukf_sigma_points_marginal_log_prob_and_grad,
               autograd.ukf_marginal_log_prob, autograd.ukf_sigma_points_marginal_log_prob):
        with pytest.raises(NotImplementedError, match="LearnableUserEmission"):
            fn(api_params(p), y, t)
    # the flags reach the build: a differentiable emission asks for the emission's gradient unit, Lorenz-63 included
    seen = []
    monkeypatch.setattr(b, "build_variant", lambda d, e, grad=False, verbose=False, emission_grad=False:
                        seen.append((d is None, grad, emission_grad)) or boom())
    with pytest.raises(_Sentinel):
        cd.ekf_marginal_log_prob_and_grad(api_params(p), y, t)
    l63 = emission_model("lorenz63", "range", 3, 1, seed=5)
    y3, t3 = _data(l63)
    with pytest.raises(_Sentinel):
        cd.ekf_marginal_log_prob_and_grad(api_params(l63, drift=cd.LearnableLorenz63(10.0, 28.0, 8.0 / 3.0)), y3, t3)
    # a user drift that is not differentiable still gets a variant for the filter; the gradient raises on the drift
    ud = cd.LearnableUserDrift(VDP_CODE, np.array([1.3, 0.4]))
    with pytest.raises(NotImplementedError, match="LearnableUserDrift"):
        cd.ekf_dense_marginal_log_prob_and_grad(api_params(p, drift=ud), y, t)
    with pytest.raises(_Sentinel):
        cd.cdnlgssm_filter(api_params(p, drift=ud), y, t, cd.EKFHyperParams())
    assert seen == [(True, False, True), (True, False, True), (False, False, True)]


def test_wrt_names(monkeypatch):
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm.inference_ekf import _parse_wrt
    assert "phi" in _parse_wrt("all", True) and "emission_weights" not in _parse_wrt("all", True)
    assert "phi" not in _parse_wrt("all") and "emission_bias" in _parse_wrt("all")
    for bad in ("emission_weights", "emission_bias"):
        with pytest.raises(ValueError):
            _parse_wrt((bad,), True)
    with pytest.raises(ValueError):
        _parse_wrt(("phi",))
    p = emission_model("linear", "range", 2, 3, seed=6)
    y, t = _data(p)
    with pytest.raises(ValueError):
        cd.ekf_dense_marginal_log_prob_and_grad(api_params(p), y, t, wrt=("emission_weights",))


def test_autograd_leaves_name_phi():
    from cd_dynamax_b200.autograd import _leaves
    p = emission_model("linear", "range", 2, 3, seed=7)
    phi = torch.zeros(7, dtype=torch.float64, requires_grad=True)
    leaves = _leaves(api_params(p, phi=phi))
    assert leaves["phi"] is phi and "emission_weights" not in leaves and "emission_bias" not in leaves


# ---- build flags, units and hashes (faked compiler) ------------------------------------------------------------------
def test_build_flags_units_and_hashes(monkeypatch, tmp_path):
    calls = []

    def fake_run(cmd, capture_output=True, text=True):
        calls.append(cmd)
        out = cmd[cmd.index("-o") + 1]
        os.makedirs(os.path.dirname(out), exist_ok=True)
        open(out, "w").close()
        return subprocess.CompletedProcess(cmd, 0, "", "")

    monkeypatch.setattr(b, "build", lambda *a, **k: None)
    monkeypatch.setattr(b, "LIBDIR", str(tmp_path / "lib"))
    monkeypatch.setattr(b, "OBJ", str(tmp_path / "obj"))
    monkeypatch.setattr(b.subprocess, "run", fake_run)

    def units():
        out = {os.path.basename(c[c.index("-c") + 1]): (any("CDK_USER_DRIFT_HEADER" in a for a in c),
                                                         any("CDK_USER_EMISSION_HEADER" in a for a in c))
               for c in calls if "-c" in c}
        calls.clear()
        return out

    libs = {}
    for args, kw in (((None, RANGE_CODE), {}), ((None, RANGE_CODE), dict(emission_grad=True)),
                     ((VDP_CODE, RANGE_CODE, True), dict(emission_grad=True)),
                     ((VDP_CODE, RANGE_CODE, False), dict(emission_grad=True)),
                     ((VDP_CODE, RANGE_CODE, True), {})):
        libs[(args[0] is None, args[2] if len(args) > 2 else False, kw.get("emission_grad", False))] = \
            (b.build_variant(*args, **kw), units())
    assert len({lib for lib, _ in libs.values()}) == len(libs)  # five content hashes
    _, u = libs[(True, False, False)]
    assert sorted(u) == sorted(b.USER_SOURCES)
    _, u = libs[(True, False, True)]
    assert sorted(u) == sorted(b.USER_GRAD_SOURCES) and u["cdk_ekfgrad.cu"] == (False, True)
    assert all(v == (False, True) for v in u.values())
    _, u = libs[(False, True, True)]
    assert u["cdk_ekfgrad.cu"] == (True, True) and u["cdk_api.cu"] == (True, True)
    _, u = libs[(False, False, True)]  # a non-differentiable drift stays out of the gradient unit
    assert u["cdk_ekfgrad.cu"] == (False, True) and u["cdk_generic.cu"] == (True, True)
    _, u = libs[(False, True, False)]  # ... and so does a non-differentiable emission
    assert u["cdk_ekfgrad.cu"] == (True, False) and u["cdk_generic.cu"] == (True, True)
    assert b.variant_key(None, RANGE_CODE) == b.variant_key(None, RANGE_CODE, False, emission_grad=False)
    assert b.variant_key(None, RANGE_CODE) != b.variant_key(None, RANGE_CODE, emission_grad=True)
    with pytest.raises(ValueError):
        b.build_variant(VDP_CODE, None, emission_grad=True)


# ---- C-ABI answers of the stock, filter-only and gradient libraries ----------------------------------------------------
def _nvcc_or_skip():
    if shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"):
        pytest.skip("nvcc is not available")


def test_abi_answers_by_library():
    _nvcc_or_skip()
    from tests.test_gpu_user_emission_grad import _grad_call
    stock = L.lib()
    filt = L.lib(b.build_variant(None, RANGE_CODE))
    grad = L.lib(b.build_variant(None, RANGE_CODE, emission_grad=True))
    for lib in (stock, filt):
        rc, msg = _grad_call(lib, 4, 1, "rk4")
        assert rc == -4 and "differentiable=True" in msg, msg
    assert grad.cdk_has_user_emission() == 1
    assert _grad_call(grad, 4, 1, "rk4")[0] == 0  # N = 0: every check passes, nothing is launched
    for solver in ("rk4", "dopri5"):
        assert _grad_call(grad, 40, 20, solver)[0] == 0  # n_phi = 801 fits at the C4 shape
    import ctypes
    for name in ("cdk_ekf_grad_f64", "cdk_ukf_grad_dense_f64", "cdk_ukf_grad_sigma_f64"):
        d = L.new_desc()
        d.N, d.K, d.n, d.m, d.emission_id = 0, 5, 2, 1, L.EMISSION_USER
        assert getattr(grad, name)(ctypes.byref(d), None, None, None) == -4, name
