"""Every kernel's substep loop under the diffrax ConstantStepSize rule, on time grids that reach its last-bit branches.

The kernels call one rule, StepClock (csrc/cdk_common.cuh; its host build is tested against the oracle in
test_step_rule_host), from many loops; each loop still owns its bounds, its max_steps check and what it does per substep,
so each call site below is probed on its own.

The rule: the first substep of a gap is tnext = min(t0 + dt0, t1); every later one is cand = tprev + dt0, tnext = t1 if
cand > t1 - tol else cand (tol = 1e-10 for fp64 times, 1e-6 for fp32).  A grid of random gaps almost never lands within
tol of a multiple of dt0, so these grids are built to: regular grids (where t0 + dt0 rounds just below or above t1),
gaps of q dt0 +- a few tol, repeated time stamps, tiny gaps, and gaps of up to ~300 substeps mixed inside one warp.

Three checks per kernel:
  * grid self-checks (CPU, unmarked): each grid provably hits the edge it exists for, on the oracle's rule;
  * substep-count probe (GPU): with max_steps = M, status 2 must appear exactly on the trajectories whose oracle substep
    count exceeds M -- an exact test of the kernel's count, independent of how small the extra substep is;
  * values (GPU): every output against the oracle on the same grid at the suite's gates.

Entry point -> kernel -> what runs here (a reviewer can hold this against the dispatch in cdk_api.cu, kf_warp_eligible and
the ekf_small_lw launch conditions):

  entry point                     kernel (call site of the rule)             grids            probe  values
  cdk_ekf_filter  L63 m=1 f64     ekf_small_lw (cdk_small.cu)                all              yes    yes
  cdk_ekf_filter  L63 sliced      ekf_small_lw, time-sliced launch           probe, K = 200   yes    (= unsliced, test_gpu_parity)
  cdk_ekf_filter  L63 m=1 f32     ekf_small_lw<float>                        probe, fp32      yes    yes (fp32 step oracle)
  cdk_ekf_smooth  L63             eks_small_lw (filter + backward in s)      all              yes    yes
  cdk_ekf_filter  linear n=4      generic_filter_kernel, ode_solve           all              yes    yes
  cdk_ekf_filter  L96 n=8 rk4     generic_filter_kernel<1>, ode_solve_stencil        all      yes    yes
  cdk_ekf_filter  L96 n=8 dopri5  generic_filter_kernel<2>, ode_solve_stencil_dopri5 all      yes    yes
  cdk_ukf_filter  L96 n=8         generic_filter_kernel<1|2> (closed form)   all              yes    yes
  cdk_ukf_filter  L63 sigma pts   generic_filter_kernel<0>, ode_solve        all              yes    yes
  cdk_kf_filter   n=5, no inputs  kf_warp_filter, pushforward (cdk_kfwarp.cu)        all      yes    yes
  cdk_kf_smooth   type 1, cache   kf_warp_smooth reading the filter's (A, Q) all              yes    yes
  cdk_kf_smooth   type 1, no cache kf_warp_smooth, pushforward               all              yes    yes
  cdk_kf_filter   n=4, inputs     generic_filter_kernel, ode_solve           all              yes    yes
  cdk_kf_smooth   type 1 / 2      generic_smooth_kernel (type 2: Dopri5, 0.01, 1e5 backward) all yes (filter) yes
  cdk_enkf_filter linear n=4      enkf kernel (cdk_enkf.cu)                  all              yes    yes
  cdk_sample_path linear n=4      sample_path_kernel (cdk_aux.cu)            all              yes    yes
  cdk_ekf_filter  PREDICT_ONLY    ekf_small_lw (forecast)                    all              yes    yes
  cdk_ukf_filter  PREDICT_ONLY    generic_filter_kernel (forecast)           all              yes    yes
  cdk_ekf_grad    forward mode    ekf_l63_grad_kernel                        all              NaN*   vs reverse, vs FD
  cdk_ekf_grad    reverse mode    ekf_small_lw + ekf_l63_grad_rev_kernel     all              yes    vs forward
  (* the forward-mode gradient kernels write no status: a trajectory past max_steps has a NaN log-likelihood instead)
"""
import numpy as np
import pytest

from oracle import cd_oracle as o
from tests.helpers import FIELD_CORE, gate_err, make_drift, max_rel_err, moment_norm_err, record, scaled_err
from tests.test_gpu_parity import FIELDS, linear_params_api, nonlinear_params_api

gpu = pytest.mark.gpu
TOL = 1e-9
EDGE_DELTAS = (-3e-10, -3e-11, 3e-11, 3e-10)
# substeps of a gap q dt0 + delta (fp64 rule, tol = 1e-10): q = 1, delta > 0 is the first-step special case (a full step,
# then a sub-tol tail); q = 4, delta = +3e-11 is the later-step clip (the 4th step absorbs the excess)
EDGE_COUNTS = {(1, -3e-10): 1, (1, -3e-11): 1, (1, 3e-11): 2, (1, 3e-10): 2,
               (4, -3e-10): 4, (4, -3e-11): 4, (4, 3e-11): 4, (4, 3e-10): 5}


# ---- the stepping rule, replayed with the decisions it takes ------------------------------------------------------------
def replay(t0, t1, dt0, dtype=np.float64):
    """-> (count, first_rounded, tail, clip) per gap: the oracle's substep count; the first step was cut to t1 although
    the gap is dt0 to within rounding; a later step shorter than tol was taken; a later step was clipped to t1 from a
    candidate that was not t1 itself."""
    t0, t1 = np.asarray(t0, dtype), np.asarray(t1, dtype)
    dt0, tol = dtype(dt0), dtype(o._tol_for(dtype))
    first_rounded = (t0 + dt0 >= t1) & (t1 - t0 != dt0) & (np.abs((t1 - t0) - dt0) < dtype(100) * tol)
    tail, clip = np.zeros(t0.shape, bool), np.zeros(t0.shape, bool)
    tprev, tnext = t0.copy(), np.minimum(t0 + dt0, t1)
    q = np.zeros(t0.shape, np.int64)
    while True:
        act = tprev < t1
        if not act.any():
            break
        q += act
        tail |= act & (q > 1) & (tnext - tprev < tol)
        tprev = np.where(act, tnext, tprev)
        cand = tprev + dt0
        clip |= act & (tprev < t1) & (cand > t1 - tol) & (cand != t1)
        tnext = np.where(cand > t1 - tol, t1, cand)
    assert np.array_equal(q, o.substep_counts(t0, t1, dt0, dtype))
    return q, first_rounded, tail, clip


# ---- grids (built in fp64 as t[k+1] = t[k] + gap unless stated) ----------------------------------------------------------
def regular_grid(N, K, kind="arange", t0=0.0, h=0.01):
    """Consecutive pieces of one long regular grid: row i holds stamps i K .. i K + K - 1 of `arange * h` or `linspace`."""
    j = np.arange(N * K)
    t = j * h if kind == "arange" else np.linspace(0.0, h * (N * K - 1), N * K)
    return (t0 + t).reshape(N, K)


def edge_grid(N, K, dt0, t0=0.0):
    """Every gap is q dt0 + delta, (q, delta) cycling through EDGE_COUNTS along and across trajectories."""
    combos = list(EDGE_COUNTS)
    t = np.empty((N, K))
    t[:, 0] = t0 + 0.37 * np.arange(N)
    for k in range(K - 1):
        for i in range(N):
            q, dl = combos[(i + 3 * k) % len(combos)]
            t[i, k + 1] = t[i, k] + (q * dt0 + dl)
    return t


def degenerate_grid(N, K, dt0):
    """Repeated stamps at k = 0 -> 1 (odd rows) and in mid-run (every row), a gap of 1e-11, the rest 1.3 dt0 or 0.6 dt0."""
    gaps = np.where(np.arange(K)[None, :] % 2 == 0, 1.3 * dt0, 0.6 * dt0) * np.ones((N, 1))
    gaps[1::2, 0] = 0.0
    gaps[:, K // 2] = 0.0
    gaps[:, K // 3] = 1e-11
    t = np.zeros((N, K))
    t[:, 0] = 0.5 * np.arange(N)
    for k in range(K - 1):
        t[:, k + 1] = t[:, k] + gaps[:, k]
    return t


def long_grid(N, K, dt0, dtype=np.float64):
    """Gaps of 0 .. ~300 dt0, different in every lane of a warp; N ragged (not a multiple of 32)."""
    i, k = np.arange(N)[:, None], np.arange(K - 1)[None, :]
    mult = (i * 37 + k * 101) % 301 + np.where((i + k) % 3 == 0, 0.0, 0.37)
    mult = np.where((i + k) % 11 == 5, 0.0, mult)
    t = np.zeros((N, K), dtype)
    t[:, 0] = dtype(0.25) * np.arange(N)
    for kk in range(K - 1):
        t[:, kk + 1] = t[:, kk] + dtype(dt0) * mult[:, kk].astype(dtype)
    return t


def probe_grid(N, K, dt0, dtype=np.float64, seed=0):
    """Every gap 0.6 dt0 (one substep) except ONE designed gap per trajectory, q dt0 + delta with q in {1, 2, 4, 7}: the
    trajectory's largest substep count is that gap's."""
    tol = o._tol_for(dtype)
    deltas = (-3 * tol, -0.3 * tol, 0.0, 0.3 * tol, 3 * tol)
    designs = [(q, dl) for q in (1, 2, 4, 7) for dl in deltas]
    t = np.zeros((N, K), dtype)
    t[:, 0] = dtype(0.5) * np.arange(N, dtype=dtype)
    where = (np.arange(N) * 5 + seed) % (K - 1)
    for kk in range(K - 1):
        for i in range(N):
            q, dl = designs[(i + seed) % len(designs)]
            gap = q * dt0 + dl if kk == where[i] else 0.6 * dt0
            t[i, kk + 1] = t[i, kk] + dtype(gap)
    return t


REGULAR = [("arange", 0.0, "rk4", 0.0025), ("arange", 0.0, "dopri5", 0.01), ("arange", 0.0, "rk4", 0.01 / 3),
           ("linspace", 0.0, "dopri5", 0.01), ("arange", 1e4, "rk4", 0.0025), ("arange", 1e4, "dopri5", 0.01),
           ("linspace", 1e4, "rk4", 0.01 / 3), ("arange", -3.7, "rk4", 0.0025), ("arange", -3.7, "dopri5", 0.01),
           ("linspace", -3.7, "rk4", 0.01 / 3)]
N_VAL, K_VAL = 36, 14


def value_grids():
    """name -> (t [N_VAL, K_VAL], solver, dt0, dt_final) of the value checks."""
    g = {}
    for kind, t0, solver, dt0 in REGULAR:
        g[f"{kind}@{t0:g}:{solver}:{dt0:.4g}"] = (regular_grid(N_VAL, K_VAL, kind, t0), solver, dt0, 1e-10)
    for solver, dt0 in (("rk4", 0.0025), ("dopri5", 0.01)):
        g[f"edge:{solver}"] = (edge_grid(N_VAL, K_VAL, dt0), solver, dt0, 1e-10)
    g["degenerate:dt_final=1e-10"] = (degenerate_grid(N_VAL, K_VAL, 0.0025), "rk4", 0.0025, 1e-10)
    g["degenerate:dt_final=0"] = (degenerate_grid(N_VAL, K_VAL, 0.0025), "rk4", 0.0025, 0.0)
    g["long"] = (long_grid(45, 5, 0.001), "rk4", 0.001, 1e-10)
    return g


GRIDS = value_grids()


# ---- grid self-checks (CPU) ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,t0,solver,dt0", REGULAR)
def test_regular_grid_hits_a_rounding_edge(kind, t0, solver, dt0):
    t = regular_grid(N_VAL, K_VAL, kind, t0)
    q, first, tail, clip = replay(t[:, :-1], t[:, 1:], dt0)
    assert (first | tail | clip).any(), (kind, t0, solver, dt0)
    if (kind, solver, t0) in (("arange", "dopri5", 0.0), ("arange", "dopri5", -3.7)):
        # t0 + dt0 rounds just below t1: a second substep of ~1e-17 on some gaps, one substep on the others
        assert set(np.unique(q)) == {1, 2} and tail.any()
    if solver == "rk4" and t0 == 0.0:
        assert clip.any()  # the 4th (3rd) substep is clipped to t1 from a candidate an ulp away


@pytest.mark.parametrize("dt0", [0.0025, 0.01])
def test_edge_grid_takes_the_sub_tol_tail_and_the_clip(dt0):
    t = edge_grid(N_VAL, K_VAL, dt0)
    q, first, tail, clip = replay(t[:, :-1], t[:, 1:], dt0)
    combos = list(EDGE_COUNTS)
    for i in range(N_VAL):
        for k in range(K_VAL - 1):
            assert q[i, k] == EDGE_COUNTS[combos[(i + 3 * k) % len(combos)]], (i, k)
    assert tail.any() and clip.any()


def test_degenerate_grid():
    t = degenerate_grid(N_VAL, K_VAL, 0.0025)
    q = o.substep_counts(t[:, :-1], t[:, 1:], 0.0025)
    assert (q[1::2, 0] == 0).all() and (q[:, K_VAL // 2] == 0).all() and (q[:, K_VAL // 3] == 1).all()
    assert (q[0::2, 0] == 2).all()  # 1.3 dt0
    t0s, t1s = o._gap_times(t, 0.0)
    assert (o.substep_counts(t0s, t1s, 0.0025)[:, -1] == 0).all()  # dt_final = 0: a last gap of length 0
    t0s, t1s = o._gap_times(t, 1e-10)
    assert (o.substep_counts(t0s, t1s, 0.0025)[:, -1] == 1).all()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_long_grid_mixes_lengths_inside_each_warp(dtype):
    t = long_grid(45, 5, 0.0025, dtype)
    q = o.substep_counts(t[:, :-1], t[:, 1:], dtype(0.0025), dtype)
    assert q.max() >= 250 and (q == 0).any()
    for w in range(0, 45, 32):
        assert len(np.unique(q[w:w + 32].max(axis=1))) > 5  # lanes of one warp need very different trip counts
    stride = np.maximum(-(-q // 8), 1)
    assert ((q > 8) & (q % stride != 0)).any()  # reverse-mode checkpoints: stride > 1 that does not divide q


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_probe_grid_designed_gap_sets_the_maximum(dtype):
    for dt0 in (0.0025, 0.01):
        t = probe_grid(40, 8, dt0, dtype)
        q = o.substep_counts(t[:, :-1], t[:, 1:], dtype(dt0), dtype)
        assert (np.sort(q, axis=1)[:, :-1] == 1).all()  # every other gap: one substep
        assert set(np.unique(q.max(axis=1))) >= {1, 2, 4, 5, 7, 8}


def test_fp32_rule_differs_from_the_fp64_rule_on_fp32_times():
    """Why the fp32 checks need an oracle that steps in fp32: on the same fp32 stamps the two rules disagree."""
    t = np.arange(1000, dtype=np.float32) * np.float32(0.01)
    q32 = o.substep_counts(t[:-1], t[1:], np.float32(0.0025), np.float32)
    q64 = o.substep_counts(t[:-1].astype(np.float64), t[1:].astype(np.float64), float(np.float32(0.0025)))
    assert (q32 != q64).sum() > 100
    # the oracle's fp32 time dtype takes the fp32 rule's substeps with an fp64 state
    s = o.SolverSettings("rk4", 0.0025, time_dtype=np.float32)
    _, n, _ = o.rk_solve(lambda tt, y: (-y[0],), t[:-1], t[1:], (np.ones((999, 1)),), s)
    assert np.array_equal(n, q32)


# ---- models -------------------------------------------------------------------------------------------------------------
L63 = dict(m0=np.array([1.0, 1.0, 20.0]), P0=2 * np.eye(3), drift="lorenz63", theta=np.array([10.0, 28.0, 8.0 / 3.0]),
           L=np.eye(3) + 0.1 * np.arange(9).reshape(3, 3) / 9, Qc=np.eye(3) + 0.05, H=np.array([[1.0, 0.3, -0.2]]),
           R=0.7 * np.eye(1), d=np.array([0.1]))


def _lin_nl(seed=3):
    rng = np.random.default_rng(seed)
    n, m = 4, 2
    F = -0.5 * np.eye(n) + 0.15 * rng.standard_normal((n, n))
    A = rng.standard_normal((m, m))
    return dict(m0=rng.standard_normal(n), P0=np.eye(n), drift="linear",
                theta=np.concatenate([F.ravel(), 0.1 * rng.standard_normal(n)]), L=np.eye(n) + 0.2 * rng.standard_normal((n, n)),
                Qc=0.3 * np.eye(n) + 0.05, H=rng.standard_normal((m, n)), R=A @ A.T + np.eye(m), d=np.array([0.3, -0.2]))


LIN = _lin_nl()
L96 = dict(m0=8.0 + np.random.default_rng(5).standard_normal(8), P0=np.eye(8), drift="lorenz96", theta=np.array([8.0]),
           L=np.eye(8), Qc=0.1 * np.eye(8), H=np.eye(8)[::2], R=np.eye(4), d=np.zeros(4))


def _kf(n, m, d_u, seed):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((m, m))
    return dict(m0=rng.standard_normal(n), P0=0.7 * np.eye(n), F=-0.5 * np.eye(n) + 0.3 * rng.standard_normal((n, n)) / np.sqrt(n),
                b=0.1 * rng.standard_normal(n), B=0.2 * rng.standard_normal((n, d_u)) if d_u else None,
                L=np.eye(n) + 0.1 * rng.standard_normal((n, n)), Qc=0.1 * np.eye(n) + 0.01, H=rng.standard_normal((m, n)),
                d=0.2 * rng.standard_normal(m), D=0.2 * rng.standard_normal((m, d_u)) if d_u else None,
                R=0.1 * (A @ A.T + np.eye(m)))


KF_WARP, KF_GEN = _kf(5, 2, 0, 11), _kf(4, 2, 2, 12)


def _po_nl(g):
    n = g["m0"].shape[0]
    return o.NonlinearParams(m0=g["m0"], P0=g["P0"], drift=make_drift(g["drift"], g["theta"], n), L=g["L"], Qc=g["Qc"],
                             H=g["H"], R=g["R"], d=g["d"])


def _po_lin(g):
    return o.LinearParams(m0=g["m0"], P0=g["P0"], F=g["F"], L=g["L"], Qc=g["Qc"], H=g["H"], R=g["R"], b=g["b"], d=g["d"],
                          B=g["B"], D=g["D"])


def _data(t, m, seed=1, d_u=0):
    rng = np.random.default_rng(seed)
    N, K = t.shape
    y = 2.0 * rng.standard_normal((N, K, m))
    u = rng.standard_normal((N, K, d_u)) if d_u else None
    return y, u


# ---- entry points: (GPU call, oracle call, which gaps it integrates) -----------------------------------------------------
# run(t, y, u, solver, dt0, dt_final, max_steps, dtype) -> dict of numpy outputs; the status is read separately
def _settings(solver, dt0, max_steps):
    s = {"solver": solver, "dt0": dt0}
    if max_steps is not None:
        s["max_steps"] = max_steps
    return s


def _np(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _nl_filter(model, hp_kind, sigma=False):
    def run(t, y, u, solver, dt0, dtf, ms, env):
        import cd_dynamax_b200 as cd
        hpc = {"ekf": cd.EKFHyperParams, "ukf": cd.UKFHyperParams}[hp_kind]
        env["CDK_UKF_SIGMA_POINTS"] = "1" if sigma else "0"
        f = cd.cdnlgssm_filter(nonlinear_params_api(model), y, t[..., None],
                               hpc(dt_final=dtf, diffeqsolve_settings=_settings(solver, dt0, ms)))
        return {k: _np(getattr(f, k)) for k in ["marginal_loglik"] + FIELDS}

    def ref(t, y, u, settings, dtf):
        fn = o.extended_kalman_filter if hp_kind == "ekf" else o.unscented_kalman_filter
        return fn(_po_nl(model), y, t, dt_final=dtf, settings=settings)
    return run, ref, "filter"


def _eks():
    def run(t, y, u, solver, dt0, dtf, ms, env):
        import cd_dynamax_b200 as cd
        s = cd.cdnlgssm_smoother(nonlinear_params_api(L63), y, t[..., None],
                                 cd.EKFHyperParams(dt_final=dtf, diffeqsolve_settings=_settings(solver, dt0, ms)))
        return {k: _np(getattr(s, k)) for k in ("marginal_loglik", "filtered_means", "filtered_covariances",
                                                  "smoothed_means", "smoothed_covariances")}

    def ref(t, y, u, settings, dtf):
        return o.extended_kalman_smoother(_po_nl(L63), y, t, dt_final=dtf, settings=settings)
    return run, ref, "eks"


def _kf_run(model, mode):
    """mode: filter | s1 | s1_nocache | s2."""
    def run(t, y, u, solver, dt0, dtf, ms, env):
        import cd_dynamax_b200 as cd
        from cd_dynamax_b200 import _engine as E
        from cd_dynamax_b200 import _lib as L
        from cd_dynamax_b200.continuous_discrete_linear_gaussian_ssm import inference as I
        p = linear_params_api(model)
        hp = cd.KFHyperParams(dt_final=dtf, diffeqsolve_settings=_settings(solver, dt0, ms))
        if mode == "filter":
            f = cd.cdlgssm_filter(p, y, t[..., None], hp, u)
            return {k: _np(getattr(f, k)) for k in ["marginal_loglik"] + FIELDS}
        if mode == "s1_nocache":
            # what cdlgssm_smoother does when the (A, Q) cache is not affordable: the smoother re-integrates every gap
            out, ins, fields, (N, K, n, m, dt, _) = I._filter_device(p, y, t[..., None], hp, u, (L.OUT_LL, L.OUT_FM, L.OUT_FP))
            ins = {**ins, L.IN_FM: out[L.OUT_FM], L.IN_FP: out[L.OUT_FP]}
            sm = E.run("cdk_kf_smooth", dt, N, K, n, m, ins, (L.OUT_SM, L.OUT_SP, L.OUT_SCROSS), dict(fields, smoother_type=1),
                       theta_core_ndim=2, status=out[L.OUT_STATUS])
            assert L.OUT_SCRATCH not in sm
            return {"marginal_loglik": _np(out[L.OUT_LL]), "smoothed_means": _np(sm[L.OUT_SM]),
                    "smoothed_covariances": _np(sm[L.OUT_SP]), "smoothed_cross_covariances": _np(sm[L.OUT_SCROSS])}
        s = cd.cdlgssm_smoother(p, y, t[..., None], hp, u, smoother_type="cd_smoother_1" if mode == "s1" else "cd_smoother_2")
        keys = ["marginal_loglik", "smoothed_means", "smoothed_covariances"] + (["smoothed_cross_covariances"] if mode == "s1" else [])
        return {k: _np(getattr(s, k)) for k in keys}

    def ref(t, y, u, settings, dtf):
        r = o.cdlgssm_smoother(_po_lin(model), y, t, dt_final=dtf, settings=settings, inputs=u,
                               smoother_type=2 if mode == "s2" else 1)
        return r
    return run, ref, "filter"


E_ENKF, KEY = 64, 4242


def _enkf():
    def run(t, y, u, solver, dt0, dtf, ms, env):
        import cd_dynamax_b200 as cd
        f = cd.cdnlgssm_filter(nonlinear_params_api(LIN), y, t[..., None],
                               cd.EnKFHyperParams(N_particles=E_ENKF, key=KEY, dt_final=dtf,
                                                  diffeqsolve_settings=_settings("euler", dt0, ms)))
        return {k: _np(getattr(f, k)) for k in ["marginal_loglik"] + FIELDS}

    def ref(t, y, u, settings, dtf):
        s = o.SolverSettings("euler", settings.dt0, settings.max_steps, settings.time_dtype)
        return o.ensemble_kalman_filter(_po_nl(LIN), y, t, dt_final=dtf, E=E_ENKF, seed=KEY, settings=s)
    return run, ref, "filter"


def _sampler():
    def run(t, y, u, solver, dt0, dtf, ms, env):
        import cd_dynamax_b200 as cd
        xs, ys = cd.cdnlgssm_path_sample(nonlinear_params_api(LIN), KEY, t.shape[1], t_emissions=t[..., None],
                                         diffeqsolve_settings=_settings("heun", dt0, ms), num_sequences=t.shape[0])
        return {"states": _np(xs), "emissions": _np(ys)}

    def ref(t, y, u, settings, dtf):
        s = o.SolverSettings("heun", settings.dt0, settings.max_steps, settings.time_dtype)
        xs, ys = o.sample_paths(_po_nl(LIN), t, seed=KEY, settings=s)
        return {"states": xs, "emissions": ys}
    return run, ref, "between"


def _forecast(model, hp_kind):
    def run(t, y, u, solver, dt0, dtf, ms, env):
        import cd_dynamax_b200 as cd
        hpc = {"ekf": cd.EKFHyperParams, "ukf": cd.UKFHyperParams}[hp_kind]
        env["CDK_UKF_SIGMA_POINTS"] = "0"
        fc = cd.cdnlgssm_forecast(nonlinear_params_api(model), (model["m0"], model["P0"]), t[:, 0], t[:, 1:, None],
                                  hpc(diffeqsolve_settings=_settings(solver, dt0, ms)))
        return {"predicted_means": _np(fc.forecasted_state_means), "predicted_covariances": _np(fc.forecasted_state_covariances)}

    def ref(t, y, u, settings, dtf):
        fn = o.extended_kalman_filter if hp_kind == "ekf" else o.unscented_kalman_filter
        yy = np.zeros((t.shape[0], t.shape[1] - 1, model["H"].shape[0]))
        return fn(_po_nl(model), yy, t, settings=settings, forecast=True)
    return run, ref, "between"


ENTRIES = {
    "ekf_small_lw": _nl_filter(L63, "ekf"),
    "eks_small_lw": _eks(),
    "ekf_generic_ode_solve": _nl_filter(LIN, "ekf"),
    "ekf_l96_register_stencil": _nl_filter(L96, "ekf"),
    "ukf_l96_register_stencil": _nl_filter(L96, "ukf"),
    "ukf_sigma_points": _nl_filter(L63, "ukf", sigma=True),
    "kf_warp_filter": _kf_run(KF_WARP, "filter"),
    "kf_warp_smooth_cache": _kf_run(KF_WARP, "s1"),
    "kf_warp_smooth_nocache": _kf_run(KF_WARP, "s1_nocache"),
    "kf_generic_filter": _kf_run(KF_GEN, "filter"),
    "kf_generic_smooth1": _kf_run(KF_GEN, "s1"),
    "kf_generic_smooth2": _kf_run(KF_GEN, "s2"),
    "kf_warp_smooth2_generic": _kf_run(KF_WARP, "s2"),
    "enkf": _enkf(),
    "path_sampler": _sampler(),
    "forecast_ekf_small_lw": _forecast(L63, "ekf"),
    "forecast_ukf_generic": _forecast(L63, "ukf"),
}
_M_OF = {"ekf_small_lw": 1, "eks_small_lw": 1, "ekf_generic_ode_solve": 2, "ekf_l96_register_stencil": 4,
         "ukf_l96_register_stencil": 4, "ukf_sigma_points": 1, "kf_warp_filter": 2, "kf_warp_smooth_cache": 2,
         "kf_warp_smooth_nocache": 2, "kf_generic_filter": 2, "kf_generic_smooth1": 2, "kf_generic_smooth2": 2,
         "kf_warp_smooth2_generic": 2, "enkf": 2, "path_sampler": 2, "forecast_ekf_small_lw": 1, "forecast_ukf_generic": 1}
_DU_OF = {k: (2 if k.startswith("kf_generic") else 0) for k in ENTRIES}
_MODEL_OF = {"kf_warp_filter": KF_WARP, "kf_warp_smooth_cache": KF_WARP, "kf_warp_smooth_nocache": KF_WARP,
             "kf_warp_smooth2_generic": KF_WARP}


def expected_counts(kind, t, dt_final, dt0, dtype=np.float64):
    """Largest substep count per trajectory over the gaps the entry point integrates with the caller's settings."""
    if kind in ("filter", "eks"):
        t0s, t1s = o._gap_times(t, dt_final)
    else:  # forecast / sampler: between consecutive stamps
        t0s, t1s = t[:, :-1], t[:, 1:]
    q = o.substep_counts(t0s, t1s, dtype(dt0), dtype).max(axis=1)
    if kind == "eks" and t.shape[1] > 1:  # backward pass: s from 0 to t_{k+1} - t_k
        span = t[:, 1:] - t[:, :-1]
        q = np.maximum(q, o.substep_counts(np.zeros_like(span), span, dtype(dt0), dtype).max(axis=1))
    return q


def _status():
    from cd_dynamax_b200 import _engine as E
    return _np(E.last_status()).astype(int)


@pytest.fixture
def env(monkeypatch):
    """Environment switches read per call (CDK_UKF_SIGMA_POINTS, CDK_LW_SLICE*, CDK_GRAD_MODE); restored afterwards."""
    from cd_dynamax_b200 import _engine as E
    monkeypatch.setattr(E, "RAISE_ON_MAX_STEPS", False)

    class Env(dict):
        def __setitem__(self, k, v):
            monkeypatch.setenv(k, v)

    return Env()


def _probe(name, run, kind, t, y, u, solver, dt0, env, dtype=np.float64, dt_final=1e-10):
    q = expected_counts(kind, t, dt_final, dt0, dtype)
    tried = set()
    for c in sorted(set(q.tolist())):
        for M in (c - 1, c):
            if M < 1 or M in tried:
                continue
            tried.add(M)
            run(t, y, u, solver, dt0, dt_final, M, env)
            st = _status()
            want = np.where(q > M, 2, 0)
            bad = np.nonzero(st != want)[0]
            assert bad.size == 0, (name, M, [(int(i), int(q[i]), int(st[i])) for i in bad[:8]])
    record(f"time_grids:probe:{name}:max_count", q.max())
    return tried


# ---- substep-count probes -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", sorted(ENTRIES))
@pytest.mark.parametrize("solver,dt0", [("rk4", 0.0025), ("dopri5", 0.01)])
def test_substep_count_probe(name, solver, dt0, env):
    run, _, kind = ENTRIES[name]
    t = probe_grid(40, 8, dt0, seed=len(name))
    y, u = _data(t, _M_OF[name], d_u=_DU_OF[name])
    if kind == "between":
        y = None
    tried = _probe(name, run, kind, t, y, u, solver, dt0, env)
    assert len(tried) >= 6


@gpu
@pytest.mark.parametrize("sliced", [False, True])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_substep_count_probe_ekf_small_lw_launches(sliced, dtype, env):
    """ekf_small_lw in fp64 and fp32 (the fp32 rule: fp32 times, tol 1e-6), unsliced and time-sliced (K = 200, a pretended
    one-SM GPU so that N = 96 is more than one wave)."""
    run, _, kind = ENTRIES["ekf_small_lw"]
    env["CDK_LW_SLICE"] = "2" if sliced else "0"
    env["CDK_LW_SLICE_SMS"] = "1"
    t = probe_grid(96, 200, 0.0025, dtype, seed=3)
    y = _data(t, 1)[0].astype(dtype)
    _probe(f"ekf_small_lw:{'sliced' if sliced else 'unsliced'}:{np.dtype(dtype).name}", run, kind, t, y, None, "rk4", 0.0025,
           env, dtype)


@gpu
@pytest.mark.parametrize("mode", ["forward", "reverse"])
def test_substep_count_probe_gradient(mode, env):
    """The reverse mode reports status through its forward filter pass (ekf_small_lw), over every gap including the last
    (dt_final); the forward-mode kernels write no status.  In both, the log-likelihood is NaN exactly where a gap BETWEEN
    observations needs more than max_steps (the gap after the last observation does not reach it, as in the oracle)."""
    import cd_dynamax_b200 as cd
    env["CDK_GRAD_MODE"] = mode
    t = probe_grid(40, 8, 0.0025, seed=7)
    y = _data(t, 1)[0]
    q_all = expected_counts("filter", t, 0.004, 0.0025)  # the last gap, 0.004, takes 2 substeps
    q_obs = o.substep_counts(t[:, :-1], t[:, 1:], 0.0025).max(axis=1)
    for M in sorted(set(q_obs.tolist()) | set((q_obs - 1).tolist()) | {1}):
        if M < 1:
            continue
        ll, g = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(L63), y, t[..., None],
                                                  cd.EKFHyperParams(dt_final=0.004, diffeqsolve_settings=_settings("rk4", 0.0025, M)),
                                                  wrt="all")
        ll = _np(ll)
        assert np.array_equal(~np.isfinite(ll), q_obs > M), (mode, M)
        if mode == "reverse":
            assert np.array_equal(_status(), np.where(q_all > M, 2, 0)), M


# ---- values against the oracle on the same grids ------------------------------------------------------------------------
def _compare(name, grid, got, ref):
    tag = f"time_grids:{name}:{grid}"
    if "marginal_loglik" in got:
        e = max_rel_err(got["marginal_loglik"], ref["marginal_loglik"])
        record(f"{tag}:marginal_loglik", e)
        assert e < TOL, (tag, e)
    for fld in FIELDS:
        if fld in got:
            e, en = gate_err(got[fld], ref[fld]), moment_norm_err(got[fld], ref[fld], core_ndim=FIELD_CORE[fld])
            record(f"{tag}:{fld}:gate", e)
            record(f"{tag}:{fld}:own_norm", en)
            assert e < TOL and en < 0.1 * TOL, (tag, fld, e, en)
    for fld in ("smoothed_means", "smoothed_covariances", "smoothed_cross_covariances"):
        if fld in got:
            e = scaled_err(got[fld], ref[fld])
            record(f"{tag}:{fld}:scaled", e)
            assert e < 1e-8, (tag, fld, e)
    for fld in ("states", "emissions"):
        if fld in got:
            e = scaled_err(got[fld], ref[fld])
            record(f"{tag}:{fld}:scaled", e)
            assert e < 1e-8, (tag, fld, e)


@gpu
@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("name", sorted(ENTRIES))
def test_values_vs_oracle_on_edge_grids(name, grid, env):
    run, ref, kind = ENTRIES[name]
    t, solver, dt0, dtf = GRIDS[grid]
    if kind == "between" and dtf == 0.0:
        pytest.skip("dt_final applies to the filters only")
    y, u = _data(t, _M_OF[name], seed=2, d_u=_DU_OF[name])
    got = run(t, y, u, solver, dt0, dtf, None, env)
    assert (_status() == 0).all(), name
    r = ref(t, y, u, o.SolverSettings(solver, dt0), dtf)
    _compare(name, grid, got, r)


@gpu
def test_repeated_time_stamps_are_two_updates_without_a_predict(env):
    """A zero gap takes no substep: the prediction is the filtered moment itself (A = I, Q = 0; the model has no drift
    bias, which the reference adds once per gap whatever its length), so the next filtered moment is a second Kalman
    update of the same state -- the oracle's closed-form update, in fp64 NumPy."""
    import cd_dynamax_b200 as cd
    t = degenerate_grid(N_VAL, K_VAL, 0.0025)
    y, _ = _data(t, 2, seed=4)
    g = dict(KF_WARP, b=np.zeros(5))
    f = cd.cdlgssm_filter(linear_params_api(g), y, t[..., None],
                          cd.KFHyperParams(diffeqsolve_settings={"solver": "rk4", "dt0": 0.0025}))
    k = K_VAL // 2
    assert (t[:, k + 1] == t[:, k]).all()
    assert scaled_err(f.predicted_means[:, k], f.filtered_means[:, k]) <= 1e-15
    assert scaled_err(f.predicted_covariances[:, k], f.filtered_covariances[:, k]) <= 1e-15
    N = t.shape[0]
    bN = lambda a: np.broadcast_to(a, (N,) + a.shape)
    m2, P2 = o._kf_condition_on(f.filtered_means[:, k], f.filtered_covariances[:, k], bN(g["H"]), bN(g["d"]),
                                np.zeros((N, 2)), bN(g["R"]), y[:, k + 1])
    e = max(scaled_err(f.filtered_means[:, k + 1], m2), scaled_err(f.filtered_covariances[:, k + 1], P2))
    record("time_grids:repeated_stamps_two_updates", e)
    assert e < 1e-9, e


@gpu
@pytest.mark.parametrize("grid", ["long", "degenerate:dt_final=1e-10", "edge:rk4"])
def test_gradient_reverse_vs_forward_on_edge_grids(grid, env):
    import cd_dynamax_b200 as cd
    t, solver, dt0, dtf = GRIDS[grid]
    y, _ = _data(t, 1, seed=6)
    hp = cd.EKFHyperParams(dt_final=dtf, diffeqsolve_settings={"solver": solver, "dt0": dt0})
    res = {}
    for mode in ("forward", "reverse"):
        env["CDK_GRAD_MODE"] = mode
        res[mode] = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(L63), y, t[..., None], hp, wrt="all")
    (ll_f, gf), (ll_r, gr) = res["forward"], res["reverse"]
    assert max_rel_err(ll_r, ll_f) < 1e-12
    for nm in sorted(gf):
        err = np.max(np.abs(gr[nm] - gf[nm])) / np.max(np.abs(gf[nm]))
        record(f"time_grids:grad_reverse_vs_forward:{grid}:{nm}", err)
        assert np.isfinite(gr[nm]).all() and err < 1e-9, (grid, nm, err)


@gpu
def test_gradient_forward_mode_vs_oracle_differences_on_the_edge_grid(env):
    import cd_dynamax_b200 as cd
    t, solver, dt0, dtf = GRIDS["edge:rk4"]
    t, y = t[:6], _data(t[:6], 1, seed=8)[0]
    env["CDK_GRAD_MODE"] = "forward"
    ll, grad = cd.ekf_marginal_log_prob_and_grad(nonlinear_params_api(L63), y, t[..., None],
                                                 cd.EKFHyperParams(dt_final=dtf, diffeqsolve_settings={"solver": solver, "dt0": dt0}))
    theta = L63["theta"]
    for p, nm in enumerate(("sigma", "rho", "beta")):
        h = 1e-5 * theta[p]
        lls = []
        for sgn in (1, -1):
            th = theta.copy()
            th[p] += sgn * h
            lls.append(o.extended_kalman_filter(_po_nl(dict(L63, theta=th)), y, t, dt_final=dtf,
                                                settings=o.SolverSettings(solver, dt0))["marginal_loglik"])
        fd = (lls[0] - lls[1]) / (2 * h)
        err = np.max(np.abs(grad[nm] - fd) / np.maximum(np.abs(fd), 1e-3 * np.abs(fd).max()))
        record(f"time_grids:grad_forward_vs_fd:{nm}", err)
        assert err < 5e-6, (nm, err)


# ---- fp32: against an fp64 oracle that takes the fp32 step grid ---------------------------------------------------------
@gpu
@pytest.mark.parametrize("name,grid", [("ekf_small_lw", "regular"), ("ekf_small_lw", "long"), ("ekf_l96_register_stencil", "regular"),
                                       ("kf_generic_filter", "regular"), ("kf_generic_filter", "long")])
def test_fp32_values_on_the_fp32_step_grid(name, grid, env):
    run, ref, kind = ENTRIES[name]
    dt0 = float(np.float32(0.0025))
    t = (np.arange(24 * 20, dtype=np.float32) * np.float32(0.01)).reshape(24, 20) if grid == "regular" \
        else long_grid(45, 4, 0.0025, np.float32)
    q32 = o.substep_counts(t[:, :-1], t[:, 1:], np.float32(dt0), np.float32)
    q64 = o.substep_counts(t[:, :-1].astype(np.float64), t[:, 1:].astype(np.float64), dt0)
    y, u = _data(t, _M_OF[name], seed=9, d_u=_DU_OF[name])
    y32 = y.astype(np.float32)
    u32 = None if u is None else u.astype(np.float32)
    got = run(t, y32, u32, "rk4", dt0, 1e-10, None, env)
    assert got["filtered_means"].dtype == np.float32
    assert (_status() == 0).all()
    r = ref(t.astype(np.float64), y32.astype(np.float64), None if u32 is None else u32.astype(np.float64),
            o.SolverSettings("rk4", dt0, time_dtype=np.float32), 1e-10)
    tag = f"time_grids:fp32:{name}:{grid}"
    record(f"{tag}:gaps_where_fp32_and_fp64_rules_differ", (q32 != q64).sum())
    e = max_rel_err(got["marginal_loglik"], r["marginal_loglik"])
    record(f"{tag}:marginal_loglik", e)
    errs = {fld: scaled_err(got[fld], r[fld]) for fld in FIELDS}
    for fld, v in errs.items():
        record(f"{tag}:{fld}:scaled", v)
    # fp32 rounding alone: ~1e-6 on these short regular grids (measured <= 2.5e-7 on the log-likelihood, 2.2e-5 on the
    # moments); the long Lorenz-63 gaps (up to 0.75 time units without an update) let the tangent flow amplify it to
    # 4.4e-3 / 2.5e-3 (B200)
    ll_bound, mom_bound = (1e-2, 1e-2) if (name, grid) == ("ekf_small_lw", "long") else (1e-5, 1e-4)
    assert e < ll_bound, (tag, e)
    assert max(errs.values()) < mom_bound, (tag, errs)
