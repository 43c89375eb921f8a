"""Drop-in for src/continuous_discrete_nonlinear_gaussian_ssm/inference_ekf.py: EKFHyperParams :34-44,
extended_kalman_filter :202-326, iterated_extended_kalman_filter :328-361, extended_kalman_smoother :450-539,
iterated_extended_kalman_smoother :541-593."""
from typing import List, NamedTuple, Optional

import numpy as np

from .. import _engine as E
from .. import _lib as L
from ..continuous_discrete_linear_gaussian_ssm.inference import _sq
from ..types import PosteriorGSSMFiltered, PosteriorGSSMSmoothed
from ._common import DEFAULT_FIELDS, reject_user_emission, run_filter


class EKFHyperParams(NamedTuple):
    dt_final: float = 1e-10
    state_order: str = "second"
    emission_order: str = "first"
    smooth_order: str = "first"
    cov_rescaling: float = 1.0
    diffeqsolve_settings: dict = {}


def _ekf_fields(hp: EKFHyperParams, num_iter: int):
    if hp.state_order not in L.ORDERS:
        raise ValueError("EKF hyperparams.state_order = {} not implemented yet".format(hp.state_order))  # :118
    return dict(dt_final=float(hp.dt_final), state_order=L.ORDERS[hp.state_order], num_iter=int(num_iter),
                cov_rescaling=float(hp.cov_rescaling))


def extended_kalman_filter(params, emissions, t_emissions=None, hyperparams: EKFHyperParams = EKFHyperParams(),
                           inputs=None, num_iter: int = 1,
                           output_fields: Optional[List[str]] = DEFAULT_FIELDS) -> PosteriorGSSMFiltered:
    post, _, _ = run_filter("cdk_ekf_filter", params, emissions, t_emissions, inputs, output_fields,
                            _ekf_fields(hyperparams, num_iter), diffeqsolve_settings=hyperparams.diffeqsolve_settings)
    return post


def iterated_extended_kalman_filter(params, emissions, t_emissions=None, hyperparams: EKFHyperParams = EKFHyperParams(),
                                    inputs=None, num_iter: int = 2,
                                    output_fields: Optional[List[str]] = DEFAULT_FIELDS) -> PosteriorGSSMFiltered:
    return extended_kalman_filter(params, emissions, t_emissions, hyperparams, inputs, num_iter, output_fields)


def extended_kalman_smoother(params, emissions, hyperparams: EKFHyperParams = EKFHyperParams(), t_emissions=None,
                             filtered_posterior: Optional[PosteriorGSSMFiltered] = None,
                             inputs=None) -> PosteriorGSSMSmoothed:
    """Forward EKF (num_iter = 1, as upstream :503-509) then the backward ODE with the Jacobian frozen at the filtered
    mean (:363-448)."""
    if hyperparams.smooth_order != "first":
        raise ValueError("EKF hyperparams.smooth_order = {} not implemented yet".format(hyperparams.smooth_order))
    post, out, (ins, fields, N, K, n, m, dt, batched, kind) = run_filter(
        "cdk_ekf_filter", params, emissions, t_emissions, inputs, ["filtered_means", "filtered_covariances"],
        _ekf_fields(hyperparams, 1), diffeqsolve_settings=hyperparams.diffeqsolve_settings, keep_on_device=True)
    fm, fp = out[L.OUT_FM], out[L.OUT_FP]
    if filtered_posterior is not None:
        # upstream uses a caller-supplied filtered posterior verbatim (:497-512)
        dev = fm.device
        fm = E.to_dev(filtered_posterior.filtered_means, dt, dev).reshape(N, K, n)
        fp = E.to_dev(filtered_posterior.filtered_covariances, dt, dev).reshape(N, K, n, n)
    ins = dict(ins)
    ins[L.IN_FM], ins[L.IN_FP] = fm, fp
    sm = E.run("cdk_ekf_smooth", dt, N, K, n, m, ins, (L.OUT_SM, L.OUT_SP), fields, status=out[L.OUT_STATUS])
    g = lambda t: E.from_dev(_sq(t, batched), kind)
    ll = filtered_posterior.marginal_loglik if filtered_posterior is not None else g(out[L.OUT_LL])
    return PosteriorGSSMSmoothed(marginal_loglik=ll, filtered_means=g(fm), filtered_covariances=g(fp),
                                 smoothed_means=g(sm[L.OUT_SM]), smoothed_covariances=g(sm[L.OUT_SP]))


def iterated_extended_kalman_smoother(params, emissions, hyperparams: EKFHyperParams = EKFHyperParams(),
                                      t_emissions=None, num_iter: int = 2, inputs=None) -> PosteriorGSSMSmoothed:
    """Upstream silently runs a single smoothing pass (:577-586); so does this."""
    return extended_kalman_smoother(params, emissions, hyperparams, t_emissions, None, inputs)


_GRAD_GROUPS = {"drift": 1, "diffusion_coefficient": 2, "diffusion_cov": 2, "emission_cov": 4, "emission_bias": 8,
                "emission_weights": 16, "initial_mean": 32, "initial_cov": 64}


def ekf_marginal_log_prob_and_grad(params, emissions, t_emissions=None, hyperparams: EKFHyperParams = EKFHyperParams(),
                                   inputs=None, wrt=("drift",)):
    """Marginal log-likelihood of the CD-EKF and its gradient with respect to the model parameters.

    -> (marginal_loglik, grads): `grads` maps the drift's own field names (wrt "drift": "sigma", "rho", "beta" for
    LearnableLorenz63, "weights" [n,n] / "bias" [n] for LearnableLinear, "forcing" for LearnableLorenz96, "a" / "B" / "C"
    for LearnableQuadratic), "diffusion_coefficient" [n,n], "diffusion_cov" [n,n], "emission_cov" [m,m],
    "emission_bias" [m], "emission_weights" [m,n], "initial_mean" [n], "initial_cov" [n,n] to arrays, with a leading N
    for batched emissions.  `wrt` = any of the group names of _GRAD_GROUPS, or "all".

    LearnableLinear, LearnableLorenz96 and LearnableQuadratic drifts, with any emission size, run through
    `ekf_dense_marginal_log_prob_and_grad` (cdk_ekf_grad_dense_f64).  A LearnableLorenz63 drift keeps the contract of
    its own kernels (cdk_ekf_grad_f64, below): a scalar emission only, anything else raises NotImplementedError; call
    `ekf_dense_marginal_log_prob_and_grad` for Lorenz-63 with a multi-component emission.  A LearnableUserDrift with
    differentiable=True runs through the dense function too and gets its gradient under "theta" ([n_theta] or
    [N, n_theta]); with differentiable=False it raises NotImplementedError before any build or device work.

    This is what `jax.value_and_grad(lambda p: model.marginal_log_prob(p, ...))` yields upstream
    (src/utils/optimize_utils.py:102, src/ssm_temissions.py:550-568) -- here as the derivative of exactly the discrete
    filter `cdnlgssm_filter` runs.  For Lorenz-63 with a scalar emission (cdk_ekf_grad_f64): REVERSE mode for more than
    the drift group (a forward filter pass
    + one backward launch for all 23 columns, ~4 filter passes), forward mode otherwise (one launch per column), so that
    a `jax.custom_vjp` around the filter can be fed (INTEGRATION.md).  Symmetric matrices (diffusion_cov, initial_cov) are differentiated
    along symmetric directions: the result is the symmetric part (G + G^T)/2 of the entry-wise gradient G, which is what
    any PSD parameterisation consumes; diffusion_coefficient's gradient is exact.  Both paths: num_iter = 1, fp64.
    A LearnableUserEmission raises NotImplementedError: a user-defined emission has no gradient."""
    reject_user_emission(params, "ekf_marginal_log_prob_and_grad")
    import torch
    from ._common import nonlinear_inputs, _val
    from ..continuous_discrete_linear_gaussian_ssm.inference import _shape, prepare_data
    if type(params.dynamics.drift).__name__ != "LearnableLorenz63":
        return ekf_dense_marginal_log_prob_and_grad(params, emissions, t_emissions, hyperparams, inputs, wrt)
    wrt = _parse_wrt(wrt)
    groups = 0
    for w in wrt:
        groups |= _GRAD_GROUPS[w]
    kind = E.kind_of(emissions)
    Y, T, U, batched = prepare_data(emissions, t_emissions, None)
    N, K, m = _shape(Y)
    if m != 1:
        raise NotImplementedError("the Lorenz-63 gradient kernels take a scalar emission; "
                                  "ekf_dense_marginal_log_prob_and_grad serves any emission size")
    n = 3
    dt = E.pick_dtype(emissions)
    if dt != "f64":
        raise NotImplementedError("gradients are fp64 only")
    ins, drift_fields = nonlinear_inputs(params, Y, T, n, m)
    fields = dict(E.parse_settings(hyperparams.diffeqsolve_settings), **drift_fields, **_ekf_fields(hyperparams, 1))
    # more than the three drift columns: REVERSE mode (one backward launch for all 23 columns behind a forward filter pass
    # whose moments go to device scratch, N*K*192 bytes) when that scratch is affordable; else forward mode, one launch
    # per column.  CDK_GRAD_MODE=forward|reverse overrides.
    import os
    mode = os.environ.get("CDK_GRAD_MODE", "auto")
    free, _ = torch.cuda.mem_get_info()
    reverse = mode == "reverse" or (mode == "auto" and groups != 1 and N * K * 192 <= free // 2)
    fields["grad_groups"] = groups | (L.GRAD_REVERSE if reverse else 0)
    dev_ins = {}
    try:
        out = E.run("cdk_ekf_grad", dt, N, K, n, m, ins, (L.OUT_LL, L.OUT_GRAD), fields, dev_inputs=dev_ins)
    except L.CdkError as e:
        raise NotImplementedError(str(e)) from e
    G = out[L.OUT_GRAD]  # [N, 23] on the device: theta 3 | LQL 6 | R | d | H 3 | m0 3 | P0 6
    g = lambda t: E.from_dev(_sq(t, batched), kind)

    def sym(cols):  # packed symmetric-direction derivatives -> symmetric gradient matrix Gs (off-diagonals halved)
        M = torch.zeros((N, 3, 3), dtype=G.dtype, device=G.device)
        iu = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
        for c, (i, j) in enumerate(iu):
            v = cols[:, c] if i == j else 0.5 * cols[:, c]
            M[:, i, j] = v
            M[:, j, i] = v
        return M

    grads = {}
    if groups & 1:
        grads.update(sigma=g(G[:, 0]), rho=g(G[:, 1]), beta=g(G[:, 2]))
    if groups & 2:
        Gs = sym(G[:, 3:9])
        Lm, Qc = dev_ins[L.IN_L].to(G.dtype), dev_ins[L.IN_QC].to(G.dtype)
        Lm = Lm.expand(N, 3, 3) if Lm.dim() == 2 else Lm
        Qc = Qc.expand(N, 3, 3) if Qc.dim() == 2 else Qc
        if "diffusion_cov" in wrt:
            grads["diffusion_cov"] = g(Lm.transpose(1, 2) @ Gs @ Lm)  # d(L Qc L^T) = L dQc L^T
        if "diffusion_coefficient" in wrt:
            grads["diffusion_coefficient"] = g(2.0 * Gs @ Lm @ Qc)  # d(L Qc L^T) = dL Qc L^T + L Qc dL^T
    if groups & 4:
        grads["emission_cov"] = g(G[:, 9].reshape(N, 1, 1))
    if groups & 8:
        grads["emission_bias"] = g(G[:, 10].reshape(N, 1))
    if groups & 16:
        grads["emission_weights"] = g(G[:, 11:14].reshape(N, 1, 3))
    if groups & 32:
        grads["initial_mean"] = g(G[:, 14:17])
    if groups & 64:
        grads["initial_cov"] = g(sym(G[:, 17:23]))
    return g(out[L.OUT_LL]), grads


# drift leaves in the order of their theta layout (include/cdk.h drift registry), with their per-trajectory shapes
_DRIFT_LEAVES = {
    "LearnableLinear": lambda n: (("weights", (n, n)), ("bias", (n,))),
    "LearnableLorenz63": lambda n: (("sigma", ()), ("rho", ()), ("beta", ())),
    "LearnableLorenz96": lambda n: (("forcing", ()),),
    "LearnableQuadratic": lambda n: (("a", (n,)), ("B", (n, n)), ("C", (n, n, n))),
}


def drift_leaves(drift, n):
    """(name, per-trajectory shape) of the drift's parameters, in the order of its theta layout."""
    name = type(drift).__name__
    if name == "LearnableUserDrift":
        shp = np.shape(drift.theta)
        return (("theta", (int(shp[-1]) if len(shp) else 1,)),)
    if name not in _DRIFT_LEAVES:
        raise NotImplementedError(f"drift {name!r} has no gradient: it is not in the kernel registry")
    return _DRIFT_LEAVES[name](n)


def unflatten_theta(G_theta, drift, n):
    """theta_bar [N, n_theta] -> {drift field name: [N, *shape]}."""
    out, o = {}, 0
    for name, shp in drift_leaves(drift, n):
        size = int(np.prod(shp, dtype=np.int64))
        out[name] = G_theta[:, o:o + size].reshape((G_theta.shape[0],) + shp)
        o += size
    return out


def _parse_wrt(wrt):
    wrt = tuple(_GRAD_GROUPS) if wrt == "all" else ((wrt,) if isinstance(wrt, str) else tuple(wrt))
    unknown = [w for w in wrt if w not in _GRAD_GROUPS]
    if unknown:
        raise ValueError(f"unknown gradient groups {unknown}; choose from {sorted(_GRAD_GROUPS)}")
    return wrt


def ekf_dense_marginal_log_prob_and_grad(params, emissions, t_emissions=None,
                                         hyperparams: EKFHyperParams = EKFHyperParams(), inputs=None, wrt=("drift",)):
    """Marginal log-likelihood of the CD-EKF and its gradient for every registry drift (LearnableLinear,
    LearnableLorenz63, LearnableLorenz96, LearnableQuadratic) and any emission size: cdk_ekf_grad_dense_f64, one forward
    filter pass (the log-likelihood is the filter's, bit for bit) and one reverse-mode launch for all columns.

    -> (marginal_loglik, grads) keyed as in `ekf_marginal_log_prob_and_grad`: the drift's own field names (wrt "drift"),
    then "diffusion_coefficient", "diffusion_cov", "emission_cov", "emission_bias", "emission_weights", "initial_mean",
    "initial_cov", with a leading N for batched emissions.  A batch whose scratch does not fit half of the free device
    memory runs in several launches, with the same result bit for bit.  fp64, state_order first / second, num_iter = 1.
    A LearnableUserDrift with differentiable=True gets its gradient under "theta": the variant library built with
    build_user_drift(code, grad=True) takes the drift's derivatives from dual-number evaluations of its own device code.
    A LearnableUserDrift with differentiable=False, the zeroth order and fp32 raise NotImplementedError, mis-shaped
    parameters ValueError (before any device work).  A LearnableUserEmission raises NotImplementedError."""
    reject_user_emission(params, "ekf_dense_marginal_log_prob_and_grad")
    drift = params.dynamics.drift
    if type(drift).__name__ == "LearnableUserDrift" and not drift.differentiable:
        raise NotImplementedError("the gradient of a user-defined drift needs LearnableUserDrift(..., differentiable=True), "
                                  "which declares that its device code stays within the dual-number contract "
                                  "(cd_dynamax_b200.build.build_user_drift)")
    wrt = _parse_wrt(wrt)
    if E.pick_dtype(emissions) != "f64":
        raise NotImplementedError("gradients are fp64 only")
    if hyperparams.state_order == "zeroth":
        raise NotImplementedError("gradients need state_order 'first' or 'second'")
    return dense_marginal_log_prob_and_grad("cdk_ekf_grad_dense", params, emissions, t_emissions,
                                            hyperparams.diffeqsolve_settings, _ekf_fields(hyperparams, 1), wrt)


def dense_marginal_log_prob_and_grad(entry, params, emissions, t_emissions, diffeqsolve_settings, filter_fields, wrt):
    """The body shared by the dense EKF and UKF gradients, after their own checks: `entry` is "cdk_ekf_grad_dense",
    "cdk_ukf_grad_dense" or "cdk_ukf_grad_sigma", `filter_fields` the descriptor fields of the filter it differentiates, `wrt` parsed by
    _parse_wrt.  -> (marginal_loglik, grads) as documented in `ekf_dense_marginal_log_prob_and_grad`."""
    import ctypes
    from ._common import nonlinear_inputs, _val
    from ..continuous_discrete_linear_gaussian_ssm.inference import _grad_chunk, _mm, _rows, _shape, prepare_data
    kind = E.kind_of(emissions)
    Y, T, _, batched = prepare_data(emissions, t_emissions, None)
    N, K, m = _shape(Y)
    n = _shape(_val(params.dynamics.diffusion_cov))[-1]
    drift_leaves(params.dynamics.drift, n)
    ins, drift_fields = nonlinear_inputs(params, Y, T, n, m)
    fields = dict(E.parse_settings(diffeqsolve_settings), **drift_fields, **filter_fields)
    n_theta = int(fields["n_theta"])
    E.classify(N, K, n, m, ins, fields)  # reject mis-shaped parameters before the library is loaded
    cols = L.grad_cols_ekf(n, m, n_theta)
    d = L.new_desc()
    d.N, d.K, d.n, d.m, d.solver = 1, K, n, m, int(fields["solver"])
    chunk = _grad_chunk(N, int(L.lib().cdk_scratch_bytes(ctypes.byref(d), entry.encode())))
    parts = []
    for lo in range(0, N, chunk):
        hi = min(N, lo + chunk)
        dev_ins = {}
        try:
            out = E.run(entry, "f64", hi - lo, K, n, m, _rows(ins, lo, hi, N, theta_core_ndim=1),
                        (L.OUT_LL, L.OUT_GRAD), fields, host_out=(kind != "cuda"), dev_inputs=dev_ins,
                        out_shapes={L.OUT_GRAD: (hi - lo, cols)})
        except L.CdkError as e:
            raise NotImplementedError(str(e)) from e
        G = out[L.OUT_GRAD]
        Sb = G[:, n_theta:n_theta + n * n].reshape(hi - lo, n, n)
        Lm, Qc = dev_ins[L.IN_L].detach().to(G.device), dev_ins[L.IN_QC].detach().to(G.device)
        parts.append((out[L.OUT_LL], G, _mm(_mm(Sb, Lm), Qc + Qc.transpose(-1, -2)), _mm(_mm(Lm.transpose(-1, -2), Sb), Lm)))
    import torch
    ll, G, gL, gQc = (torch.cat(p) for p in zip(*parts))
    g = lambda t: E.from_dev(_sq(t, batched), kind)
    o = n_theta
    blocks = {}
    for name, shp in (("Sigma", (n, n)), ("H", (m, n)), ("d", (m,)), ("R", (m, m)), ("m0", (n,)), ("P0", (n, n))):
        size = int(np.prod(shp))
        blocks[name] = G[:, o:o + size].reshape((N,) + shp)
        o += size
    grads = {}
    if "drift" in wrt:
        grads.update({k: g(v) for k, v in unflatten_theta(G[:, :n_theta], params.dynamics.drift, n).items()})
    for key, val in (("diffusion_coefficient", gL), ("diffusion_cov", gQc), ("emission_cov", blocks["R"]),
                     ("emission_bias", blocks["d"]), ("emission_weights", blocks["H"]), ("initial_mean", blocks["m0"]),
                     ("initial_cov", blocks["P0"])):
        if key in wrt:
            grads[key] = g(val)
    return g(ll), grads
