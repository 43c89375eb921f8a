"""Drop-in for src/continuous_discrete_nonlinear_gaussian_ssm/inference_ukf.py: UKFHyperParams :25-34,
unscented_kalman_filter :206-308 (the smoother does not exist upstream: raise NotImplementedError :332).

The unscented predict runs in CLOSED FORM by default: every drift of the registry is a polynomial of degree <= 2 and the
emission is linear, and for those the 2n + 1 sigma-point sums of inference_ukf.py:130-152 are exactly
f(m) + tr(Hess f P) / 2 and J P (csrc/cdk_generic.cu, ODE_UKFC) -- same moments up to rounding, no Cholesky factor of P at
every RK stage.  `CDK_UKF_SIGMA_POINTS=1` in the environment (read per call) selects the literal sigma-point kernel.

`ukf_marginal_log_prob_and_grad` differentiates the closed-form filter (cdk_ukf_grad_dense_f64),
`ukf_sigma_points_marginal_log_prob_and_grad` the literal sigma-point filter (cdk_ukf_grad_sigma_f64), which is also
the one a LearnableUserDrift runs."""
import math
import os
from typing import List, NamedTuple, Optional

from ..types import PosteriorGSSMFiltered
from ._common import DEFAULT_FIELDS, reject_user_emission, run_filter


class UKFHyperParams(NamedTuple):
    dt_final: float = 1e-10
    alpha: float = math.sqrt(3)
    beta: int = 2
    kappa: int = 1
    diffeqsolve_settings: dict = {}


def _ukf_fields(hp: UKFHyperParams):
    return dict(dt_final=float(hp.dt_final), alpha=float(hp.alpha), beta=float(hp.beta), kappa=float(hp.kappa))


def unscented_kalman_filter(params, emissions, t_emissions=None, hyperparams: UKFHyperParams = UKFHyperParams(),
                            inputs=None, output_fields: Optional[List[str]] = DEFAULT_FIELDS) -> PosteriorGSSMFiltered:
    from .. import _lib as L
    fields = _ukf_fields(hyperparams)
    if os.environ.get("CDK_UKF_SIGMA_POINTS", "0") == "1":
        fields["flags"] = L.FLAG_UKF_SIGMA_POINTS
    post, _, _ = run_filter("cdk_ukf_filter", params, emissions, t_emissions, inputs, output_fields, fields,
                            diffeqsolve_settings=hyperparams.diffeqsolve_settings)
    return post


def ukf_marginal_log_prob_and_grad(params, emissions, t_emissions=None, hyperparams: UKFHyperParams = UKFHyperParams(),
                                   inputs=None, wrt=("drift",)):
    """Marginal log-likelihood of the CD-UKF and its gradient with respect to the model parameters, for every registry
    drift (LearnableLinear, LearnableLorenz63, LearnableLorenz96, LearnableQuadratic) and any emission size:
    cdk_ukf_grad_dense_f64, one forward pass of the closed-form filter `unscented_kalman_filter` runs (the
    log-likelihood is the filter's, bit for bit) and one reverse-mode launch for all columns.

    -> (marginal_loglik, grads) keyed as in `ekf_dense_marginal_log_prob_and_grad`: the drift's own field names (wrt
    "drift"), then "diffusion_coefficient", "diffusion_cov", "emission_cov", "emission_bias", "emission_weights",
    "initial_mean", "initial_cov", with a leading N for batched emissions; `wrt` = any of those groups, or "all".  A batch
    whose scratch does not fit half of the free device memory runs in several launches, with the same result bit for
    bit.  alpha, beta and kappa reach the filter as `unscented_kalman_filter` passes them; they do not enter the closed
    form and get no gradient.  fp64 only.  LearnableUserDrift, fp32, non-zero inputs and CDK_UKF_SIGMA_POINTS=1 (literal
    sigma points) raise NotImplementedError, mis-shaped parameters ValueError (before any device work).  So does a
    LearnableUserEmission: a user-defined emission has no gradient."""
    import torch
    from .. import _engine as E
    from .inference_ekf import _parse_wrt, dense_marginal_log_prob_and_grad
    reject_user_emission(params, "ukf_marginal_log_prob_and_grad")
    if type(params.dynamics.drift).__name__ == "LearnableUserDrift":
        raise NotImplementedError("a user-defined drift runs literal sigma points: use "
                                  "ukf_sigma_points_marginal_log_prob_and_grad")
    wrt = _parse_wrt(wrt)
    if E.pick_dtype(emissions) != "f64":
        raise NotImplementedError("gradients are fp64 only")
    if inputs is not None and bool(torch.as_tensor(inputs).ne(0).any()):
        raise NotImplementedError("gradients with inputs are not supported")
    if os.environ.get("CDK_UKF_SIGMA_POINTS", "0") == "1":
        raise NotImplementedError("CDK_UKF_SIGMA_POINTS=1: the literal sigma-point filter is differentiated by "
                                  "ukf_sigma_points_marginal_log_prob_and_grad")
    return dense_marginal_log_prob_and_grad("cdk_ukf_grad_dense", params, emissions, t_emissions,
                                            hyperparams.diffeqsolve_settings, _ukf_fields(hyperparams), wrt)


def ukf_sigma_points_marginal_log_prob_and_grad(params, emissions, t_emissions=None,
                                                hyperparams: UKFHyperParams = UKFHyperParams(), inputs=None,
                                                wrt=("drift",)):
    """Marginal log-likelihood of the CD-UKF with LITERAL sigma points (inference_ukf.py:130-152: a Cholesky factor of P
    and 2n + 1 drift evaluations at every RK stage) and its gradient with respect to the model parameters:
    cdk_ukf_grad_sigma_f64, one forward pass of the sigma-point filter (`unscented_kalman_filter` with
    CDK_UKF_SIGMA_POINTS=1; the log-likelihood is that filter's, bit for bit) and one reverse-mode launch for all
    columns.  It always differentiates the sigma-point filter, whatever CDK_UKF_SIGMA_POINTS says.

    Every registry drift, and a LearnableUserDrift(..., differentiable=True), whose gradient comes under "theta" (the
    variant library built with build_user_drift(code, grad=True) takes the theta-derivatives of its f from dual numbers
    and its x-derivatives from its jac).  -> (marginal_loglik, grads) keyed as in `ekf_dense_marginal_log_prob_and_grad`;
    `wrt` = any of its groups, or "all".  alpha, beta and kappa get no gradient.  fp64 only.  fp32, non-zero inputs and
    a LearnableUserDrift with differentiable=False raise NotImplementedError, mis-shaped parameters ValueError (before any
    device work); so does a LearnableUserEmission."""
    import torch
    from .. import _engine as E
    from .inference_ekf import _parse_wrt, dense_marginal_log_prob_and_grad
    reject_user_emission(params, "ukf_sigma_points_marginal_log_prob_and_grad")
    drift = params.dynamics.drift
    if type(drift).__name__ == "LearnableUserDrift" and not drift.differentiable:
        raise NotImplementedError("the gradient of a user-defined drift needs LearnableUserDrift(..., differentiable=True), "
                                  "which declares that its device code stays within the dual-number contract "
                                  "(cd_dynamax_b200.build.build_user_drift)")
    wrt = _parse_wrt(wrt)
    if E.pick_dtype(emissions) != "f64":
        raise NotImplementedError("gradients are fp64 only")
    if inputs is not None and bool(torch.as_tensor(inputs).ne(0).any()):
        raise NotImplementedError("gradients with inputs are not supported")
    return dense_marginal_log_prob_and_grad("cdk_ukf_grad_sigma", params, emissions, t_emissions,
                                            hyperparams.diffeqsolve_settings, _ukf_fields(hyperparams), wrt)


def unscented_kalman_smoother(*args, **kwargs):
    raise NotImplementedError("UKS not implemented yet")  # as upstream (inference_ukf.py:332)
