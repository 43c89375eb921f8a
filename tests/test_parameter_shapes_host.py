"""CPU: model parameters whose per-trajectory shape is not what the kernels read are rejected on the host, and per-sample
(batched) parameters are laid out as the kernels index them.

Every kernel reads `slot_elems` entries of a parameter slot (cdk_api.cu: n*n for P0 / L / Qc, m*n for H, n_theta for the
drift, ...) at `in[slot] + traj * in_stride[slot]`.  A shared L of shape [4, 4] for n = 3, an H one column wide, or a
batched leaf whose leading axis is not N would therefore be read past its end, or as the wrong numbers, on the device.
`_engine.run` must raise ValueError for all of them, whichever public entry point the parameters come through.

`_lib.lib` and `_engine.device` are replaced by functions that raise `_Reached`: a call that passes validation stops
there, so none of these tests loads the library, allocates device memory or launches anything, with or without a GPU.

The second half checks the batched parameter layout itself: `drift_to_theta` for every registry drift with each leaf
batched alone, and the oracle's batched parameters (what the GPU sweep of tests/test_gpu_batched_parameters.py compares
with) against N single-sample oracle runs."""
import numpy as np
import pytest
import torch

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _engine as E
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm.cdnlgssm_utils import drift_to_theta
from oracle import cd_oracle as o
from tests.helpers import make_drift


class _Reached(Exception):
    pass


@pytest.fixture
def no_device(monkeypatch):
    def boom(*a, **k):
        raise _Reached()

    monkeypatch.setattr(L, "lib", boom)
    monkeypatch.setattr(E, "device", boom)
    # the shims size optional device caches from the free memory before they call run(); a query, not device work
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a, **k: (1 << 40, 1 << 40))


N, K = 5, 6


def _grid(batched=True):
    t = np.cumsum(np.full((N, K), 0.05), axis=1)
    return t[..., None] if batched else t[0][:, None]


# ---- the models the entry points are called with -------------------------------------------------------------------
def _nl_model(drift="quadratic", n=3, m=2):
    """Nonlinear model leaves by slot name (drift leaves under 'drift')."""
    rng = np.random.default_rng(0)
    if drift == "quadratic":
        leaves = dict(a=0.1 * np.ones(n), B=-np.eye(n), C=0.01 * rng.standard_normal((n, n, n)))
    elif drift == "lorenz63":
        leaves = dict(sigma=10.0, rho=28.0, beta=8.0 / 3.0)
    else:
        raise ValueError(drift)
    return dict(drift_kind=drift, drift=leaves, m0=np.zeros(n), P0=np.eye(n), L=np.eye(n), Qc=np.eye(n),
                H=np.eye(m, n), d=np.zeros(m), R=np.eye(m))


def _nl_api(g):
    kind = g["drift_kind"]
    drift = cd.LearnableQuadratic(**g["drift"]) if kind == "quadratic" else cd.LearnableLorenz63(**g["drift"])
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(g["m0"]), cov=cd.LearnableMatrix(g["P0"])),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=drift, diffusion_coefficient=cd.LearnableMatrix(g["L"]),
                                           diffusion_cov=cd.LearnableMatrix(g["Qc"])),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=g["H"], bias=g["d"]),
                                             emission_cov=cd.LearnableMatrix(g["R"])))


def _lin_model(n=3, m=2, d_u=0):
    g = dict(m0=np.zeros(n), P0=np.eye(n), F=-np.eye(n), b=np.zeros(n), L=np.eye(n), Qc=np.eye(n), H=np.eye(m, n),
             d=np.zeros(m), R=np.eye(m))
    if d_u:
        g.update(BU=np.zeros((n, d_u)), DU=np.zeros((m, d_u)))
    return g


def _lin_api(g):
    return cd.make_cdlgssm_params(g["m0"], g["P0"], g["F"], g["L"], g["Qc"], g["H"], g["R"], dynamics_bias=g["b"],
                                  dynamics_input_weights=g.get("BU"), emissions_bias=g["d"],
                                  emissions_input_weights=g.get("DU"))


# ---- entry points: name -> (model factory, call) -------------------------------------------------------------------
def _y(m):
    return np.zeros((N, K, m))


ENTRIES = {
    "cdlgssm_filter": (lambda: _lin_model(),
                       lambda g: cd.cdlgssm_filter(_lin_api(g), _y(2), _grid())),
    "cdlgssm_filter_inputs": (lambda: _lin_model(d_u=2),
                              lambda g: cd.cdlgssm_filter(_lin_api(g), _y(2), _grid(), inputs=np.ones((N, K, 2)))),
    "cdlgssm_filter_diag_r": (lambda: dict(_lin_model(), R=np.ones(2)),
                              lambda g: cd.cdlgssm_filter(_lin_api(g), _y(2), _grid())),
    "cdlgssm_smoother_1": (lambda: _lin_model(),
                           lambda g: cd.cdlgssm_smoother(_lin_api(g), _y(2), _grid(), smoother_type="cd_smoother_1")),
    "cdlgssm_smoother_2": (lambda: _lin_model(),
                           lambda g: cd.cdlgssm_smoother(_lin_api(g), _y(2), _grid(), smoother_type="cd_smoother_2")),
    "cdlgssm_grad": (lambda: _lin_model(),
                     lambda g: cd.cdlgssm_marginal_log_prob_and_grad(_lin_api(g), _y(2), _grid())),
    "ekf_filter": (lambda: _nl_model(),
                   lambda g: cd.cdnlgssm_filter(_nl_api(g), _y(2), _grid(), cd.EKFHyperParams())),
    "ukf_filter": (lambda: _nl_model(),
                   lambda g: cd.cdnlgssm_filter(_nl_api(g), _y(2), _grid(), cd.UKFHyperParams())),
    "enkf_filter": (lambda: _nl_model(),
                    lambda g: cd.cdnlgssm_filter(_nl_api(g), _y(2), _grid(), cd.EnKFHyperParams(N_particles=16))),
    "ekf_smoother": (lambda: _nl_model(),
                     lambda g: cd.cdnlgssm_smoother(_nl_api(g), _y(2), _grid(), cd.EKFHyperParams())),
    "ekf_l63_filter": (lambda: _nl_model("lorenz63", m=1),
                       lambda g: cd.cdnlgssm_filter(_nl_api(g), _y(1), _grid(), cd.EKFHyperParams())),
    "ekf_l63_grad": (lambda: _nl_model("lorenz63", m=1),
                     lambda g: cd.ekf_marginal_log_prob_and_grad(_nl_api(g), _y(1), _grid(), wrt="all")),
    "ekf_forecast": (lambda: _nl_model(),
                     lambda g: cd.cdnlgssm_forecast(_nl_api(g), (g["m0"], g["P0"]), 0.0, _grid())),
    "path_sample": (lambda: _nl_model(),
                    lambda g: cd.cdnlgssm_path_sample(_nl_api(g), 0, K, _grid(False), num_sequences=N)),
}

# slot name of every leaf, for the message check
SLOT = dict(m0="IN_M0", P0="IN_P0", F="IN_F", drift="IN_F", b="IN_B", BU="IN_BU", L="IN_L", Qc="IN_QC", H="IN_H",
            d="IN_D", DU="IN_DU", R="IN_R")


def _wider(shape, axis):
    s = list(shape)
    s[axis] += 1
    return tuple(s)


def _bad(value, case, axis=-2):
    """A mis-shaped version of a well-shaped shared leaf: 'shared' one row (or entry) too many, 'lead' batched with a
    leading axis of N + 2 (not N, not the broadcast 1), 'core' batched over N but one row too many.  Rows, not columns,
    by default: the shims take n from the last axis of H (linear model) or of Qc (nonlinear model)."""
    shape = np.shape(value)
    axis = axis if len(shape) >= 2 else -1
    if case == "shared":
        return np.zeros(_wider(shape, axis)) if shape else np.zeros(2)
    if case == "lead":
        return np.ones((N + 2,) + shape)
    return np.ones((N,) + _wider(shape, axis)) if shape else np.ones((N, 2))


def _cases():
    for entry, (model, _) in ENTRIES.items():
        g = model()
        for slot in g:
            if slot == "drift_kind":
                continue
            for case in ("shared", "lead", "core"):
                yield pytest.param(entry, slot, case, id=f"{entry}-{slot}-{case}")


def _break(g, slot, case, entry):
    g = dict(g)
    if slot != "drift":
        # the forecast and the sampler take m from the rows of H: widen its columns there
        g[slot] = _bad(g[slot], case, -1 if slot == "H" and entry in ("ekf_forecast", "path_sample") else -2)
        return g
    leaves = dict(g["drift"])
    if g["drift_kind"] == "quadratic":
        # every leaf of a quadratic drift is an array: break B (shared / lead) or a (per-sample rows one entry long)
        if case == "core":
            leaves["a"] = _bad(leaves["a"], case)
        else:
            leaves["B"] = _bad(leaves["B"], case)
    else:
        # Lorenz-63 leaves are scalars or [N]: a shared one cannot be mis-shaped, a batched one can be N + 2 long
        leaves["rho"] = np.full(N + 2, 28.0)
    g["drift"] = leaves
    return g


@pytest.mark.parametrize("entry,slot,case", list(_cases()))
def test_mis_shaped_parameter_is_rejected_on_the_host(entry, slot, case, no_device):
    model, call = ENTRIES[entry]
    g = model()
    with pytest.raises(_Reached):  # the well-shaped model gets as far as the library
        call(g)
    bad = _break(g, slot, case, entry)
    if entry == "cdlgssm_grad" and slot == "R" and case == "shared":
        # a 2-D emissions.cov that is not square is a batch of diagonals, which the gradient does not take
        with pytest.raises(NotImplementedError, match="diagonal"):
            call(bad)
        return
    with pytest.raises(ValueError, match="input slot IN_"):
        call(bad)
    if entry == "ekf_forecast" and slot == "m0" and case == "lead":
        return  # the forecast takes N from the initial mean, so the mismatch is reported on the covariance
    with pytest.raises(ValueError, match=SLOT[slot]):
        call(bad)


@pytest.mark.parametrize("slot,shape", [("L", (4, 4)), ("Qc", (2, 2)), ("P0", (3, 4)), ("H", (1, 5)), ("R", (2, 2)),
                                        ("d", (3,)), ("m0", (4,)), ("H", (5, 1, 5))])
def test_issue_shapes_stop_on_the_host(slot, shape, no_device):
    """n = 3 taken from Qc (run_filter), m = 1 from the emissions: each of these reached the launch before the per-slot
    shape check."""
    g = _nl_model("lorenz63", m=1)
    g[slot] = np.ones(shape)
    with pytest.raises(ValueError, match="input slot IN_"):
        cd.cdnlgssm_filter(_nl_api(g), _y(1), _grid(), cd.EKFHyperParams())


def test_theta_of_the_wrong_length_is_rejected(no_device):
    g = _nl_model()
    g["drift"] = dict(g["drift"], C=np.zeros((3, 3, 2)))
    with pytest.raises(ValueError, match=r"IN_F.*\(39,\)"):
        cd.cdnlgssm_filter(_nl_api(g), _y(2), _grid(), cd.EKFHyperParams())


@pytest.mark.parametrize("slot,value", [("H", np.ones((2, 4))), ("H", np.ones((N + 2, 2, 3))), ("d", np.ones(3)),
                                        ("d", np.ones((N, 3))), ("R", np.ones((2, 3))), ("R", np.ones((N + 2, 2, 2)))])
def test_emission_moments_reject_mis_shaped_parameters(slot, value, no_device):
    g = _nl_model()
    p = _nl_api(g)
    em = dict(H=g["H"], d=g["d"], R=g["R"])
    em[slot] = value
    p = p._replace(emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=em["H"], bias=em["d"]),
                                                        emission_cov=cd.LearnableMatrix(em["R"])))
    sm = np.zeros((N, K, 3))
    with pytest.raises(_Reached):
        cd.cdnlgssm_emissions(_nl_api(g), _grid(), sm, np.zeros((N, K, 3, 3)), hyperparams=cd.EKFHyperParams())
    with pytest.raises(ValueError, match=SLOT[slot]):
        cd.cdnlgssm_emissions(p, _grid(), sm, np.zeros((N, K, 3, 3)), hyperparams=cd.EKFHyperParams())
    with pytest.raises(ValueError, match="IN_FP"):
        cd.cdnlgssm_emissions(_nl_api(g), _grid(), sm, np.zeros((N, K, 3, 4)), hyperparams=cd.EKFHyperParams())


def test_well_shaped_batched_leaves_pass(no_device):
    """Every leaf batched over N (and the broadcast leading axis of 1) passes validation on every entry point."""
    for entry, (model, call) in ENTRIES.items():
        g = model()
        for slot in g:
            if slot == "drift_kind":
                continue
            for lead in (N, 1):
                h = dict(g)
                if slot == "drift":
                    h["drift"] = {k: np.broadcast_to(np.asarray(v), (lead,) + np.shape(v)).copy() for k, v in g["drift"].items()}
                else:
                    h[slot] = np.broadcast_to(g[slot], (lead,) + np.shape(g[slot])).copy()
                with pytest.raises(_Reached):
                    call(h)


# ---- drift_to_theta: each leaf of every registry drift batched alone -------------------------------------------------
def _factor(i):
    return 1.0 + 0.04 * ((7 * i) % 11)


DRIFTS = {
    "LearnableLinear": (3, lambda: dict(weights=-np.eye(3) + 0.1, bias=np.arange(3.0))),
    "LearnableLorenz63": (3, lambda: dict(sigma=10.0, rho=28.0, beta=8.0 / 3.0)),
    "LearnableLorenz96": (6, lambda: dict(forcing=8.0)),
    "LearnableQuadratic": (3, lambda: dict(a=np.arange(3.0), B=np.arange(9.0).reshape(3, 3),
                                           C=np.arange(27.0).reshape(3, 3, 3))),
    "LearnableUserDrift": (2, lambda: dict(device_code="", theta=np.array([1.0, 2.0, 3.0]))),
}


@pytest.mark.parametrize("name,leaf", [(nm, lf) for nm, (_, mk) in DRIFTS.items() for lf in mk() if lf != "device_code"])
@pytest.mark.parametrize("torch_leaf", [False, True])
def test_drift_to_theta_batches_each_leaf_alone(name, leaf, torch_leaf):
    n, make = DRIFTS[name]
    cls = getattr(cd, name)
    shared = make()
    samples = [dict(shared, **{leaf: _factor(i) * np.asarray(shared[leaf], np.float64)}) for i in range(N)]
    stacked = np.stack([s[leaf] for s in samples])
    batched = dict(shared, **{leaf: torch.as_tensor(stacked) if torch_leaf else stacked})
    did, theta, n_theta = drift_to_theta(cls(**batched), n)
    assert tuple(theta.shape) == (N, n_theta), (name, leaf, tuple(theta.shape))
    for i, s in enumerate(samples):
        did_i, th_i, nt_i = drift_to_theta(cls(**s), n)
        assert did_i == did and nt_i == n_theta and tuple(th_i.shape) == (n_theta,)
        assert torch.equal(theta[i], th_i), (name, leaf, i)
    # a leading axis of 1 stays a single row the engine broadcasts; leaves that disagree on N are an error
    one = dict(shared, **{leaf: stacked[:1]})
    assert tuple(drift_to_theta(cls(**one), n)[1].shape) in ((1, n_theta), (n_theta,))


def test_quadratic_leaves_disagreeing_on_n_are_rejected():
    q = cd.LearnableQuadratic(a=np.zeros((4, 3)), B=np.zeros((5, 3, 3)), C=np.zeros((3, 3, 3)))
    with pytest.raises(ValueError, match="leading axis"):
        drift_to_theta(q, 3)


# ---- the oracle takes batched leaves: a batched run is the stack of N single runs --------------------------------------
def _per_sample(v, i, core):
    v = np.asarray(v)
    return v[i] if v.ndim == core + 1 else v


def _nl_oracle_case(kind, n, m, Nb=3, Kb=4, seed=2):
    rng = np.random.default_rng(seed)
    f = np.array([_factor(i) for i in range(Nb)])
    if kind == "lorenz63":
        theta = np.array([10.0, 28.0, 8.0 / 3.0])[None] * f[:, None]
    elif kind == "lorenz96":
        theta = 8.0 * f[:, None]
    elif kind == "linear":
        th = np.concatenate([(-0.5 * np.eye(n) + 0.1 * rng.standard_normal((n, n))).ravel(), 0.1 * rng.standard_normal(n)])
        theta = th[None] * f[:, None]
    else:
        th = np.concatenate([0.1 * rng.standard_normal(n), (-np.eye(n)).ravel(), 0.02 * rng.standard_normal(n ** 3)])
        theta = th[None] * f[:, None]
    g = dict(m0=0.5 + 0.1 * rng.standard_normal((Nb, n)), P0=f[:, None, None] * np.eye(n),
             L=f[:, None, None] * (np.eye(n) + 0.05), Qc=0.3 * f[:, None, None] * np.eye(n),
             H=f[:, None, None] * np.eye(m, n), d=0.1 * f[:, None] * np.ones(m), R=0.5 * f[:, None, None] * np.eye(m))
    t = np.cumsum(np.full((Nb, Kb), 0.02), axis=1)
    y = rng.standard_normal((Nb, Kb, m))
    return g, theta, t, y


def _nl_params(g, theta, kind, n, i=None):
    pick = (lambda v, core: v) if i is None else (lambda v, core: _per_sample(v, i, core))
    return o.NonlinearParams(m0=pick(g["m0"], 1), P0=pick(g["P0"], 2), drift=make_drift(kind, pick(theta, 1), n),
                             L=pick(g["L"], 2), Qc=pick(g["Qc"], 2), H=pick(g["H"], 2), R=pick(g["R"], 2),
                             d=pick(g["d"], 1))


ORACLE_RUNS = {
    "ekf": lambda p, y, t: o.extended_kalman_filter(p, y, t, settings=o.SolverSettings("rk4", 0.01)),
    "ekf_zeroth": lambda p, y, t: o.extended_kalman_filter(p, y, t, state_order="zeroth", cov_rescaling=0.7,
                                                          settings=o.SolverSettings("bosh3", 0.01)),
    "eks": lambda p, y, t: o.extended_kalman_smoother(p, y, t, settings=o.SolverSettings("rk4", 0.01)),
    "ukf": lambda p, y, t: o.unscented_kalman_filter(p, y, t, settings=o.SolverSettings("rk4", 0.01)),
    "enkf": lambda p, y, t: o.ensemble_kalman_filter(p, y, t, E=8, seed=3, settings=o.SolverSettings("euler", 0.01)),
    "sample": lambda p, y, t: dict(zip(("x", "y"), o.sample_paths(p, t, seed=4, settings=o.SolverSettings("heun", 0.01)))),
}


@pytest.mark.parametrize("algo", list(ORACLE_RUNS))
@pytest.mark.parametrize("kind,n,m", [("lorenz63", 3, 1), ("lorenz96", 5, 2), ("linear", 3, 2), ("quadratic", 3, 2)])
def test_batched_oracle_equals_stack_of_single_runs(kind, n, m, algo):
    g, theta, t, y = _nl_oracle_case(kind, n, m)
    run = ORACLE_RUNS[algo]
    batched = run(_nl_params(g, theta, kind, n), y, t)
    for i in range(t.shape[0]):
        single = run(_nl_params(g, theta, kind, n, i), y[i:i + 1], t[i:i + 1])
        for key, v in single.items():
            if algo in ("enkf", "sample"):
                continue  # the random stream is indexed by the trajectory number: row i of a batch is not trajectory 0
            np.testing.assert_allclose(batched[key][i], v[0], rtol=1e-15, atol=1e-15, err_msg=f"{kind} {algo} {key} {i}")
    if algo in ("enkf", "sample"):
        # compare against the batch of N identical copies of sample i instead: same trajectory numbers, same deviates
        for i in range(t.shape[0]):
            gi = {k: np.broadcast_to(_per_sample(v, i, {"m0": 1, "d": 1}.get(k, 2)), np.shape(v)) for k, v in g.items()}
            thi = np.broadcast_to(theta[i], theta.shape)
            rep = run(_nl_params(gi, thi, kind, n), y, t)
            for key, v in rep.items():
                np.testing.assert_allclose(batched[key][i], v[i], rtol=1e-15, atol=1e-15, err_msg=f"{kind} {algo} {key} {i}")
    # and the shared model is what a stack of identical rows computes
    shared = run(_nl_params({k: v[0] for k, v in g.items()}, theta[0], kind, n), y, t)
    rows = run(_nl_params({k: np.broadcast_to(v[0], v.shape) for k, v in g.items()}, np.broadcast_to(theta[0], theta.shape),
                          kind, n), y, t)
    for key in shared:
        np.testing.assert_allclose(rows[key], shared[key], rtol=1e-15, atol=1e-15, err_msg=key)


@pytest.mark.parametrize("smoother_type", [1, 2])
def test_batched_linear_oracle_equals_stack_of_single_runs(smoother_type):
    rng = np.random.default_rng(9)
    Nb, Kb, n, m, d_u = 3, 4, 3, 2, 2
    f = np.array([_factor(i) for i in range(Nb)])
    p = o.LinearParams(m0=0.1 * rng.standard_normal((Nb, n)), P0=f[:, None, None] * np.eye(n),
                       F=f[:, None, None] * (-0.5 * np.eye(n) + 0.1 * rng.standard_normal((n, n))),
                       L=f[:, None, None] * np.eye(n), Qc=0.3 * f[:, None, None] * np.eye(n),
                       H=f[:, None, None] * np.eye(m, n), R=0.5 * f[:, None, None] * np.eye(m),
                       b=0.1 * f[:, None] * np.ones(n), d=0.1 * f[:, None] * np.ones(m),
                       B=f[:, None, None] * np.ones((n, d_u)), D=f[:, None, None] * np.ones((m, d_u)))
    t = np.cumsum(np.full((Nb, Kb), 0.03), axis=1)
    y, u = rng.standard_normal((Nb, Kb, m)), rng.standard_normal((Nb, Kb, d_u))
    s = o.SolverSettings("rk4", 0.01)
    batched = o.cdlgssm_smoother(p, y, t, settings=s, inputs=u, smoother_type=smoother_type)
    for i in range(Nb):
        pi = o.LinearParams(**{k: (v[i] if v is not None else None) for k, v in vars(p).items()})
        single = o.cdlgssm_smoother(pi, y[i:i + 1], t[i:i + 1], settings=s, inputs=u[i:i + 1], smoother_type=smoother_type)
        for key, v in single.items():
            np.testing.assert_allclose(batched[key][i], v[0], rtol=1e-15, atol=1e-15, err_msg=f"{key} {i}")
