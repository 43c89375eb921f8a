"""cdk_ekf_grad_dense_f64 for USER-DEFINED emissions (LearnableUserEmission(..., differentiable=True)) on the GPU: the
variant library built with build_variant(..., emission_grad=True) re-linearises h at every predicted mean and takes the
emission's second derivatives from dual-number evaluations of the user's own h / jac (csrc/cdk_dual.cuh).

The reference is the torch float64 EKF of tests/test_user_emission_grad_host.py (drift and emission as torch callables),
differentiated by autograd, under the gate of tests/test_gpu_ekf_grad.py: every block's max error <= 1e-9 of its max
|value|, Sigma, R and P0 on symmetric parts.  Cross-checks without torch: the linear emission written as user code
against the stock LearnableLinear gradient, and central differences of the filter."""
import ctypes

import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _engine as E
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200 import build as b
from oracle import cd_oracle as o
from tests.helpers import record, scaled_err
from tests.test_gpu_ekf_grad import GATE, dense, sym
from tests.test_gpu_time_grids import degenerate_grid, edge_grid, long_grid, regular_grid
from tests.test_user_emission_grad_host import (CODE, LIN_CODE, RANGE_CODE, emission_model, torch_ll, ue_blocks)

pytestmark = pytest.mark.gpu


def ue_fields(p, solver, dt0, order, drift_code=None):
    n, m = np.shape(p["m0"])[-1], np.shape(p["R"])[-1]
    user_drift = drift_code is not None
    lib = b.build_variant(drift_code, p.get("code", CODE.get(p["em"])), user_drift, emission_grad=True)
    return dict(solver=L.SOLVERS[solver], dt0=dt0, max_steps=100000, dt_final=1e-10, state_order=L.ORDERS[order],
                num_iter=1, drift_id=L.DRIFT_USER if user_drift else p["drift_id"], n_theta=np.shape(p["theta"])[-1],
                emission_id=L.EMISSION_USER, n_phi=np.shape(p["phi"])[-1], lib_path=lib)


def ue_ins(p, y, t):
    return {L.IN_Y: y, L.IN_T: t, L.IN_M0: p["m0"], L.IN_P0: p["P0"], L.IN_F: p["theta"], L.IN_L: p["L"],
            L.IN_QC: p["Qc"], L.IN_H: p["phi"], L.IN_D: None, L.IN_R: p["R"]}


def ue_dense(p, y, t, solver, dt0, order, drift_code=None):
    N, K, m = y.shape
    n, nt, nph = np.shape(p["m0"])[-1], np.shape(p["theta"])[-1], np.shape(p["phi"])[-1]
    out = E.run("cdk_ekf_grad_dense", "f64", N, K, n, m, ue_ins(p, y, t), (L.OUT_LL, L.OUT_GRAD),
                ue_fields(p, solver, dt0, order, drift_code),
                out_shapes={L.OUT_GRAD: (N, L.grad_cols_ekf_ue(n, m, nt, nph))})
    return out[L.OUT_LL], out[L.OUT_STATUS], out[L.OUT_GRAD]


def ue_filter(p, y, t, solver, dt0, order, drift_code=None):
    N, K, m = y.shape
    out = E.run("cdk_ekf_filter", "f64", N, K, np.shape(p["m0"])[-1], m, ue_ins(p, y, t), (L.OUT_LL,),
                ue_fields(p, solver, dt0, order, drift_code))
    return out[L.OUT_LL], out[L.OUT_STATUS]


def compare(name, p, y, t, solver, dt0, order, drift_code=None):
    ll, status, G = ue_dense(p, y, t, solver, dt0, order, drift_code)
    assert int(status.abs().sum()) == 0, name
    fl, _ = ue_filter(p, y, t, solver, dt0, order, drift_code)
    assert torch.equal(ll, fl), name  # the forward pass is the filter's launch
    N, K, m = y.shape
    n, nt = np.shape(p["m0"])[-1], np.shape(p["theta"])[-1]
    ref_ll, ref = torch_ll(p, y, t, solver, dt0, order, grad=True)
    err_ll = scaled_err(ll.cpu().numpy(), ref_ll)
    record(f"user_emission_grad:{name}:ll", err_ll)
    assert err_ll < 1e-11, (name, err_ll)
    got = ue_blocks(G, n, m, nt, np.shape(p["phi"])[-1])
    for k, r in ref.items():
        r = sym(r) if k in ("Sigma", "R", "P0") else r
        err = scaled_err(got[k], r)
        record(f"user_emission_grad:{name}:{k}", err)
        assert err < GATE, (name, k, err)
    return G


def data(p, N, K, seed, gap=0.05):
    from tests.test_kf_grad_host import random_grid
    rng = np.random.default_rng(seed)
    m = np.shape(p["R"])[-1]
    return 2.0 + 0.7 * rng.standard_normal((N, K, m)), random_grid(N, K, seed + 1, mean_gap=gap)


@pytest.mark.parametrize("em", ["range", "wide", "square"])
@pytest.mark.parametrize("drift", ["linear", "lorenz96", "lorenz63"])
def test_emissions_with_registry_drifts(em, drift):
    n = {"linear": 2, "lorenz96": 5, "lorenz63": 3}[drift]
    p = emission_model(drift, em, n, 3, seed=1)
    y, t = data(p, 3, 8, 2, gap=0.03)
    compare(f"{drift}_{em}", p, y, t, "rk4", 0.01, "second")


@pytest.mark.parametrize("solver", list(L.SOLVERS))
@pytest.mark.parametrize("order", ["first", "second"])
def test_vdp_range_every_solver_and_order(order, solver):
    from tests.test_user_emission_grad_host import VDP_CODE
    p = emission_model("vdp", "range", 2, 3, seed=3)
    y, t = data(p, 3, 8, 4)
    compare(f"vdp_range_{order}_{solver}", p, y, t, solver, 0.01, order, drift_code=VDP_CODE)


@pytest.mark.parametrize("shape", ["m1", "m_gt_n", "m_gt_32"])
def test_emission_sizes_and_batched_phi(shape):
    n, m = {"m1": (2, 1), "m_gt_n": (3, 7), "m_gt_32": (4, 35)}[shape]
    p = emission_model("linear", "range", n, m, seed=5, N=3)  # every parameter, phi included, per trajectory
    y, t = data(p, 3, 6, 6)
    compare(f"batched_{shape}", p, y, t, "rk4", 0.01, "second")


@pytest.mark.parametrize("grid", ["t0_1e4", "edge", "degenerate", "long"])
def test_time_grids(grid):
    N, K, dt0 = 3, 6, 0.01
    p = emission_model("linear", "range", 2, 2, seed=7)
    t = {"t0_1e4": lambda: regular_grid(N, K, t0=1e4, h=0.013), "edge": lambda: edge_grid(N, K, dt0),
         "degenerate": lambda: degenerate_grid(N, K, dt0), "long": lambda: long_grid(N, 5, dt0)}[grid]()
    y = 2.0 + 0.7 * np.random.default_rng(8).standard_normal((N, t.shape[1], 2))
    compare(f"grid_{grid}", p, y, t, "dopri5", dt0, "second")


def test_linear_emission_as_user_code_matches_the_stock_gradient():
    """phi = [H | d]: the row has the stock row's layout and every block agrees within 1e-13 of its scale."""
    n, m = 3, 2
    p = emission_model("linear", "linear", n, m, seed=9)
    y, t = data(p, 4, 10, 10)
    ll, st, G = ue_dense(p, y, t, "rk4", 0.01, "second")
    q = dict(p, kind="linear", H=p["phi"][:m * n].reshape(m, n), d=p["phi"][m * n:])
    ll0, st0, G0 = dense(q, y, t, "rk4", 0.01, "second")
    assert int(st.abs().sum()) == 0 and int(st0.abs().sum()) == 0
    assert G.shape == G0.shape
    nt = np.shape(p["theta"])[-1]
    got, ref = ue_blocks(G, n, m, nt, m * n + m), ue_blocks(G0, n, m, nt, m * n + m)
    for k in ref:
        err = scaled_err(got[k], ref[k])
        record(f"user_emission_grad:linear_as_user:{k}", err)
        assert err < 1e-13, (k, err)
    assert scaled_err(ll.cpu().numpy(), ll0.cpu().numpy()) < 1e-13


def test_bit_identity_run_to_run_per_slot_and_status_rows():
    p = emission_model("linear", "range", 2, 3, seed=11)
    y, t = data(p, 4, 8, 12)
    ll, st, G = ue_dense(p, y, t, "rk4", 0.01, "second")
    ll2, _, G2 = ue_dense(p, y, t, "rk4", 0.01, "second")
    assert torch.equal(G, G2) and torch.equal(ll, ll2)
    for k in ("phi", "theta", "R", "m0"):  # each slot batched alone gives the same bits
        q = dict(p)
        q[k] = np.broadcast_to(p[k], (4,) + np.shape(p[k])).copy()
        _, _, Gk = ue_dense(q, y, t, "rk4", 0.01, "second")
        assert torch.equal(G, Gk), k
    y_bad = y.copy()
    y_bad[1, 3, 0] = np.nan  # a NaN observation: status != 0 for that row only
    _, stb, Gb = ue_dense(p, y_bad, t, "rk4", 0.01, "second")
    if int(stb[1]) != 0:
        assert torch.isnan(Gb[1]).all()
        keep = [i for i in range(4) if int(stb[i]) == 0]
        assert torch.equal(Gb[keep], G[keep])


def test_directional_derivatives_match_central_differences_of_the_filter():
    from tests.test_user_emission_grad_host import VDP_CODE
    p = emission_model("vdp", "range", 2, 3, seed=13)
    y, t = data(p, 2, 8, 14)
    ll, st, G = ue_dense(p, y, t, "rk4", 0.01, "second", VDP_CODE)
    n, m = 2, 3
    nt, nph = np.shape(p["theta"])[-1], np.shape(p["phi"])[-1]
    got = ue_blocks(G, n, m, nt, nph)
    rng = np.random.default_rng(15)
    for k in ("theta", "phi", "R", "m0", "P0", "Qc"):
        v = rng.standard_normal(np.shape(p[k]))
        if k in ("R", "P0", "Qc"):
            v = 0.5 * (v + v.T)
        eps = 1e-6 * max(1.0, float(np.max(np.abs(p[k]))))
        lp, _ = ue_filter(dict(p, **{k: p[k] + eps * v}), y, t, "rk4", 0.01, "second", VDP_CODE)
        lm, _ = ue_filter(dict(p, **{k: p[k] - eps * v}), y, t, "rk4", 0.01, "second", VDP_CODE)
        fd = (lp - lm).cpu().numpy() / (2 * eps)
        if k == "Qc":  # through Sigma = L Qc L^T
            Lm = p["L"]
            an = np.einsum("nij,ij->n", got["Sigma"], Lm @ v @ Lm.T)
        else:
            an = (got[k].reshape(len(fd), -1) * v.reshape(-1)).sum(-1)
        err = np.max(np.abs(an - fd)) / max(np.max(np.abs(fd)), 1e-12)
        record(f"user_emission_grad:fd:{k}", err)
        assert err < 1e-6, (k, err)


def _grad_call(lib, n, m, solver):
    d = L.new_desc()
    d.N, d.K, d.n, d.m, d.solver = 0, 5, n, m, L.SOLVERS[solver]
    d.drift_id, d.n_theta, d.state_order, d.num_iter = L.DRIFT_LORENZ96, 1, 1, 1
    d.emission_id = L.EMISSION_USER
    fake = ctypes.c_void_p(0x1000)
    ins = (ctypes.c_void_p * L.NUM_IN)(*([fake] * L.NUM_IN))
    outs = (ctypes.c_void_p * L.NUM_OUT)(*([fake] * L.NUM_OUT))
    return lib.cdk_ekf_grad_dense_f64(ctypes.byref(d), ins, outs, None), lib.cdk_last_error().decode()


def test_the_largest_n_phi_at_the_c4_shape_runs_and_one_more_is_refused():
    from tests.test_user_emission_grad_host import C4_MAX_NPHI, fixed_params_code
    n, m = 40, 20
    for solver in ("rk4", "dopri5"):
        for code in (RANGE_CODE, LIN_CODE):
            assert _grad_call(L.lib(b.build_variant(None, code, emission_grad=True)), n, m, solver)[0] == 0
    big = L.lib(b.build_variant(None, fixed_params_code(C4_MAX_NPHI + 1), emission_grad=True))
    rc, msg = _grad_call(big, n, m, "rk4")
    assert rc == -2 and f"n_phi = {C4_MAX_NPHI + 1}" in msg, msg
    p = emission_model("lorenz96", "fixed", n, m, seed=17, nphi=C4_MAX_NPHI)
    p["code"] = fixed_params_code(C4_MAX_NPHI)
    y, t = data(p, 2, 3, 18)
    ll, st, G = ue_dense(p, y, t, "rk4", 0.005, "second")
    assert int(st.abs().sum()) == 0 and torch.isfinite(G).all()


def test_adam_moves_the_beacons_towards_the_true_ones():
    """50 Adam steps through autograd.ekf_marginal_log_prob on perturbed beacon positions."""
    from cd_dynamax_b200.autograd import ekf_marginal_log_prob
    from tests.test_user_emission_grad_host import api_params
    n, m, N, K = 2, 3, 16, 30
    p = emission_model("linear", "range", n, m, seed=19)
    true_phi = p["phi"].copy()
    rng = np.random.default_rng(20)
    t = np.tile(np.arange(K) * 0.1, (N, 1))[..., None]
    _, y = cd.cdnlgssm_path_sample(api_params(p), 21, K, t_emissions=t, num_sequences=N)
    y = np.asarray(y)
    phi = torch.tensor(true_phi.copy(), dtype=torch.float64)
    phi[:m * n] += 0.3 * torch.tensor(rng.standard_normal(m * n))
    phi.requires_grad_(True)
    d0 = float(torch.linalg.norm(phi.detach()[:m * n] - torch.tensor(true_phi[:m * n])))
    opt = torch.optim.Adam([phi], lr=0.02)
    for _ in range(50):
        opt.zero_grad()
        loss = -ekf_marginal_log_prob(api_params(p, phi=phi), y, t).sum()
        loss.backward()
        opt.step()
    d1 = float(torch.linalg.norm(phi.detach()[:m * n] - torch.tensor(true_phi[:m * n])))
    record("user_emission_grad:adam_beacon_distance_ratio", d1 / d0)
    assert d1 < 0.7 * d0, (d0, d1)
