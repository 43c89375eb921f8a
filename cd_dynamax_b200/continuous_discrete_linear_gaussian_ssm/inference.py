"""Drop-in for src/continuous_discrete_linear_gaussian_ssm/inference.py (filter :555-632, smoother :694-823):
same names, argument order and result tuples; the arithmetic runs in libcdk.so on the GPU.

Batched form (what `jax.vmap` produces in the reference, src/ssm_temissions.py:555-567): emissions [N,K,m],
t_emissions [N,K,1]; any parameter may carry a leading N as well.
"""
import ctypes
from typing import Any, NamedTuple, Optional

import numpy as np
import torch

from .. import _engine as E
from .. import _lib as L
from ..types import ParamsLGSSMEmissions, ParamsLGSSMInitial, PosteriorGSSMFiltered, PosteriorGSSMSmoothed


class KFHyperParams(NamedTuple):
    """cd_linear/inference.py:34-38"""
    dt_final: float = 1e-10
    diffeqsolve_settings: dict = {}


class ParamsCDLGSSMDynamics(NamedTuple):
    """cd_linear/inference.py:57-89"""
    weights: Any
    bias: Any
    input_weights: Any
    diffusion_coefficient: Any
    diffusion_cov: Any


class ParamsCDLGSSM(NamedTuple):
    """cd_linear/inference.py:92-102"""
    initial: ParamsLGSSMInitial
    dynamics: ParamsCDLGSSMDynamics
    emissions: ParamsLGSSMEmissions


def make_cdlgssm_params(initial_mean, initial_cov, dynamics_weights, dynamics_diffusion_coeff, dynamics_diffusion_cov,
                        emissions_weights, emissions_cov, dynamics_bias=None, dynamics_input_weights=None,
                        emissions_bias=None, emissions_input_weights=None):
    """cd_linear/inference.py:146-182"""
    return ParamsCDLGSSM(
        initial=ParamsLGSSMInitial(mean=initial_mean, cov=initial_cov),
        dynamics=ParamsCDLGSSMDynamics(weights=dynamics_weights, bias=dynamics_bias,
                                       input_weights=dynamics_input_weights,
                                       diffusion_coefficient=dynamics_diffusion_coeff,
                                       diffusion_cov=dynamics_diffusion_cov),
        emissions=ParamsLGSSMEmissions(weights=emissions_weights, bias=emissions_bias,
                                       input_weights=emissions_input_weights, cov=emissions_cov))


def _shape(x):
    return tuple(x.shape) if hasattr(x, "shape") else np.shape(x)


def _check_constant(x, name, core):
    if callable(x):
        raise NotImplementedError(f"{name}: callable (time-varying) parameters are not supported "
                                  "(cd_linear/inference.py:42-51 _get_params); pass constant arrays")
    return x


def prepare_data(emissions, t_emissions, inputs):
    """-> (Y [N,K,m], T [N,K], U [N,K,d_u] or None, batched?)"""
    ys = _shape(emissions)
    batched = len(ys) == 3
    if len(ys) not in (2, 3):
        raise ValueError(f"emissions must be [K,m] or [N,K,m], got {ys}")
    K = ys[-2]
    Y = emissions if batched else emissions[None]
    if t_emissions is None:
        # unit spacing (cd_linear/inference.py:590-593)
        T = np.arange(K, dtype=np.float64)[None]
    else:
        ts = _shape(t_emissions)
        if ts[-1] == 1 and len(ts) >= 2 and ts[-2] == K:
            T = t_emissions[..., 0]  # the reference's [K,1] column
        elif ts[-1] == K:
            T = t_emissions
        else:
            raise ValueError(f"t_emissions must be [K,1] (or [N,K,1]); got {ts} for K={K}")
        if len(_shape(T)) == 1:
            T = T[None]
    U = None
    if inputs is not None and _shape(inputs)[-1] > 0:
        U = inputs if len(_shape(inputs)) == 3 else inputs[None]
    return Y, T, U, batched


def _diag_r(params) -> bool:
    """A 1-D `emissions.cov` [m] is the diagonal of R: the reference's Woodbury update (cd_linear/inference.py:240-254).
    Batched over parameter samples it is [N, m], i.e. any 2-D covariance that is not square.  A square 2-D one is a full,
    shared R [m, m] whatever the weights look like (so diagonals batched over N = m samples must be passed as full
    matrices)."""
    rs = _shape(params.emissions.cov)
    return len(rs) == 1 or (len(rs) == 2 and rs[-1] != rs[-2])


def _linear_inputs(params: ParamsCDLGSSM, Y, T, U, n, m, d_u):
    dyn, em = params.dynamics, params.emissions
    for nm, v in (("dynamics.weights", dyn.weights), ("dynamics.diffusion_coefficient", dyn.diffusion_coefficient),
                  ("dynamics.diffusion_cov", dyn.diffusion_cov), ("emissions.weights", em.weights),
                  ("emissions.cov", em.cov)):
        assert v is not None, f"params.{nm} is required (cd_linear/inference.py:266-272)"
        _check_constant(v, nm, 2)
    zeros = lambda *s: np.zeros(s)
    ins = {
        L.IN_Y: Y, L.IN_T: T, L.IN_M0: params.initial.mean, L.IN_P0: params.initial.cov, L.IN_F: dyn.weights,
        L.IN_B: dyn.bias if dyn.bias is not None else zeros(n), L.IN_L: dyn.diffusion_coefficient,
        L.IN_QC: dyn.diffusion_cov, L.IN_H: em.weights, L.IN_D: em.bias if em.bias is not None else zeros(m),
        L.IN_R: em.cov,
    }
    if d_u > 0:
        ins[L.IN_U] = U
        ins[L.IN_BU] = dyn.input_weights if dyn.input_weights is not None else zeros(n, d_u)
        ins[L.IN_DU] = em.input_weights if em.input_weights is not None else zeros(m, d_u)
    return ins


def _filter_device(params, emissions, t_emissions, filter_hyperparams, inputs, want, host_out=False, flags=0):
    hp = filter_hyperparams if filter_hyperparams is not None else KFHyperParams()  # None crashes upstream (:585)
    Y, T, U, batched = prepare_data(emissions, t_emissions, inputs)
    N, K, m = _shape(Y)
    n = _shape(params.emissions.weights)[-1]
    d_u = _shape(U)[-1] if U is not None else 0
    dt = E.pick_dtype(emissions)
    ins = _linear_inputs(params, Y, T, U, n, m, d_u)
    fields = dict(E.parse_settings(hp.diffeqsolve_settings), dt_final=float(hp.dt_final), d_u=d_u)
    diag = _diag_r(params)
    if diag:
        fields["flags"] = L.FLAG_DIAG_R
    elif flags and dt == "f64" and K > 1:
        # keep (A_k, Q_k) of every gap for the type-1 smoother when the cache is affordable (a quarter of the free HBM)
        free, _ = torch.cuda.mem_get_info()
        if N * (K - 1) * 2 * n * n * 8 <= free // 4:
            fields["flags"] = flags
    dev_ins = {}
    out = E.run("cdk_kf_filter", dt, N, K, n, m, ins, want, fields, theta_core_ndim=2, host_out=host_out,
                dev_inputs=dev_ins, core_ndim_override={L.IN_R: 1} if diag else None)
    return out, {**ins, **dev_ins}, fields, (N, K, n, m, dt, batched)


def _sq(t, batched):
    return t if (batched or t is None) else t[0]


def cdlgssm_filter(params: ParamsCDLGSSM, emissions, t_emissions=None,
                   filter_hyperparams: Optional[KFHyperParams] = KFHyperParams(), inputs=None) -> PosteriorGSSMFiltered:
    """Continuous-discrete Kalman filter (cd_linear/inference.py:555-632)."""
    kind = E.kind_of(emissions)
    want = (L.OUT_LL, L.OUT_FM, L.OUT_FP, L.OUT_PM, L.OUT_PP)
    out, _, _, (N, K, n, m, dt, batched) = _filter_device(params, emissions, t_emissions, filter_hyperparams, inputs,
                                                          want, host_out=(kind != "cuda"))
    g = lambda s: E.from_dev(_sq(out[s], batched), kind)
    return PosteriorGSSMFiltered(marginal_loglik=g(L.OUT_LL), filtered_means=g(L.OUT_FM),
                                 filtered_covariances=g(L.OUT_FP), predicted_means=g(L.OUT_PM),
                                 predicted_covariances=g(L.OUT_PP))


def cdlgssm_smoother(params: ParamsCDLGSSM, emissions, t_emissions=None,
                     filter_hyperparams: Optional[KFHyperParams] = None, inputs=None,
                     smoother_type: Optional[str] = "cd_smoother_1") -> PosteriorGSSMSmoothed:
    """Forward filter + backward smoother (cd_linear/inference.py:694-823): 'cd_smoother_1' = Sarkka Alg. 3.17,
    'cd_smoother_2' = Alg. 3.18 (backward ODE; cross-covariances are NaN as upstream, :792)."""
    if smoother_type not in ("cd_smoother_1", "cd_smoother_2"):
        raise ValueError("CD Kalman Smoother type = {} not implemented yet".format(smoother_type))  # :798-799
    kind = E.kind_of(emissions)
    want = (L.OUT_LL, L.OUT_FM, L.OUT_FP)
    out, ins, fields, (N, K, n, m, dt, batched) = _filter_device(
        params, emissions, t_emissions, filter_hyperparams, inputs, want,
        flags=L.FLAG_KEEP_PUSHFORWARD if smoother_type == "cd_smoother_1" else 0)
    ins = dict(ins)
    ins[L.IN_FM], ins[L.IN_FP] = out[L.OUT_FM], out[L.OUT_FP]
    fields = dict(fields, smoother_type=1 if smoother_type == "cd_smoother_1" else 2)
    if L.OUT_SCRATCH not in out and "flags" in fields:
        # the filter kept nothing (not the warp kernel): the smoother re-integrates the pushforward
        fields["flags"] = int(fields["flags"]) & ~L.FLAG_KEEP_PUSHFORWARD
    sm = E.run("cdk_kf_smooth", dt, N, K, n, m, ins, (L.OUT_SM, L.OUT_SP, L.OUT_SCROSS), fields, theta_core_ndim=2,
               status=out[L.OUT_STATUS], scratch=out.get(L.OUT_SCRATCH),
               core_ndim_override={L.IN_R: 1} if _diag_r(params) else None)
    g = lambda t: E.from_dev(_sq(t, batched), kind)
    return PosteriorGSSMSmoothed(marginal_loglik=g(out[L.OUT_LL]), filtered_means=g(out[L.OUT_FM]),
                                 filtered_covariances=g(out[L.OUT_FP]), smoothed_means=g(sm[L.OUT_SM]),
                                 smoothed_covariances=g(sm[L.OUT_SP]),
                                 smoothed_cross_covariances=g(sm[L.OUT_SCROSS]))


def _grad_chunk(N: int, row_bytes: int) -> int:
    """Trajectories per launch of cdk_kf_grad whose device scratch fits half of the free device memory."""
    free, _ = torch.cuda.mem_get_info()
    return max(1, min(N, (free // 2) // max(row_bytes, 1)))


def _rows(ins, lo, hi, N, theta_core_ndim=2):
    """The [lo, hi) trajectories of every input that carries a leading N (see _engine.run's classification)."""
    out = {}
    for slot, x in ins.items():
        core = E._CORE_NDIM[slot] if E._CORE_NDIM[slot] is not None else theta_core_ndim
        shp = _shape(x)
        out[slot] = x[lo:hi] if (len(shp) == core + 1 and shp[0] == N and N > 1) else x
    return out


def _mm(A, B):
    """A @ B for the small [.., n, n] blocks of the gradient, one elementwise pass per inner index: every row of a batch
    gets the same bits whatever the batch size (a batched GEMM may pick a different kernel per batch size)."""
    acc = A[..., :, :1] * B[..., :1, :]
    for k in range(1, A.shape[-1]):
        acc = acc + A[..., :, k:k + 1] * B[..., k:k + 1, :]
    return acc


def cdlgssm_marginal_log_prob_and_grad(params: ParamsCDLGSSM, emissions, t_emissions=None,
                                       filter_hyperparams: Optional[KFHyperParams] = None, inputs=None):
    """Marginal log-likelihood of `cdlgssm_filter` and its gradient with respect to the model parameters.

    -> (marginal_loglik, grads): `grads` is a ParamsCDLGSSM shaped like `params` -- what
    `jax.value_and_grad(lambda p: cdlgssm_filter(p, ...).marginal_loglik)` gives the reference's fit_sgd
    (src/utils/optimize_utils.py:102, src/ssm_temissions.py:550-568) -- with a leading N for batched emissions (one
    gradient per trajectory).  Leaves absent from `params` (a None bias, the input weights) are None.  It is the
    derivative of exactly the discrete filter cdlgssm_filter runs, from cdk_kf_grad_f64 (one forward filter pass and one
    reverse-mode launch).  The symmetric parameters (emissions.cov, initial.cov) get the symmetric part (G + G^T)/2 of
    the entry-wise gradient G, which is what a PSD parameterisation consumes; diffusion_coefficient L and diffusion_cov
    Qc get the chain rule through Sigma = L Qc L^T: L_bar = Sigma_bar L (Qc + Qc^T), Qc_bar = L^T Sigma_bar L.

    Coverage: fp64, n <= 16, m <= 8, full R, no inputs, every solver; anything else raises NotImplementedError.  A
    batch whose scratch does not fit half of the free device memory runs in several launches (same result, bit for bit).
    """
    hp = filter_hyperparams if filter_hyperparams is not None else KFHyperParams()
    if inputs is not None and _shape(inputs)[-1] > 0:
        raise NotImplementedError("cdlgssm_marginal_log_prob_and_grad: inputs (B, D) are not supported")
    if _diag_r(params):
        raise NotImplementedError("cdlgssm_marginal_log_prob_and_grad: a diagonal (1-D) emissions.cov is not supported")
    if E.pick_dtype(emissions) != "f64":
        raise NotImplementedError("cdlgssm_marginal_log_prob_and_grad: gradients are fp64 only")
    kind = E.kind_of(emissions)
    Y, T, _, batched = prepare_data(emissions, t_emissions, None)
    N, K, m = _shape(Y)
    n = _shape(params.emissions.weights)[-1]
    if n > 16 or m > 8:
        raise NotImplementedError(f"cdlgssm_marginal_log_prob_and_grad: needs n <= 16 and m <= 8 (n = {n}, m = {m})")
    ins = _linear_inputs(params, Y, T, None, n, m, 0)
    fields = dict(E.parse_settings(hp.diffeqsolve_settings), dt_final=float(hp.dt_final), d_u=0)
    cols = L.grad_cols_kf(n, m)
    E.classify(N, K, n, m, ins, fields, theta_core_ndim=2)  # reject mis-shaped parameters before the library is loaded
    d = L.new_desc()
    d.N, d.K, d.n, d.m = 1, K, n, m
    chunk = _grad_chunk(N, int(L.lib().cdk_scratch_bytes(ctypes.byref(d), b"cdk_kf_grad")))
    parts = []
    for lo in range(0, N, chunk):
        hi = min(N, lo + chunk)
        dev_ins = {}
        try:
            out = E.run("cdk_kf_grad", "f64", hi - lo, K, n, m, _rows(ins, lo, hi, N), (L.OUT_LL, L.OUT_GRAD), fields,
                        theta_core_ndim=2, host_out=(kind != "cuda"), dev_inputs=dev_ins,
                        out_shapes={L.OUT_GRAD: (hi - lo, cols)})
        except L.CdkError as e:
            raise NotImplementedError(str(e)) from e
        G = out[L.OUT_GRAD]
        Sb = G[:, n * n + n:2 * n * n + n].reshape(hi - lo, n, n)
        Lm, Qc = dev_ins[L.IN_L].detach().to(G.device), dev_ins[L.IN_QC].detach().to(G.device)
        parts.append((out[L.OUT_LL], G, _mm(_mm(Sb, Lm), Qc + Qc.transpose(-1, -2)), _mm(_mm(Lm.transpose(-1, -2), Sb), Lm)))
    ll, G, gL, gQc = (torch.cat(p) for p in zip(*parts))
    o = 0
    blocks = {}
    for name, shp in (("F", (n, n)), ("b", (n,)), ("Sigma", (n, n)), ("H", (m, n)), ("d", (m,)), ("R", (m, m)),
                      ("m0", (n,)), ("P0", (n, n))):
        size = int(np.prod(shp))
        blocks[name] = G[:, o:o + size].reshape((N,) + shp)
        o += size
    g = lambda t: E.from_dev(_sq(t, batched), kind)
    dyn, em = params.dynamics, params.emissions
    grads = ParamsCDLGSSM(
        initial=ParamsLGSSMInitial(mean=g(blocks["m0"]), cov=g(blocks["P0"])),
        dynamics=ParamsCDLGSSMDynamics(weights=g(blocks["F"]), bias=g(blocks["b"]) if dyn.bias is not None else None,
                                       input_weights=None, diffusion_coefficient=g(gL), diffusion_cov=g(gQc)),
        emissions=ParamsLGSSMEmissions(weights=g(blocks["H"]), bias=g(blocks["d"]) if em.bias is not None else None,
                                       input_weights=None, cov=g(blocks["R"])))
    return g(ll), grads
