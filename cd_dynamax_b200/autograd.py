"""Differentiable total log-likelihood for torch callers: the shape `jax.custom_vjp` gives the filter in the reference
stack (INTEGRATION.md section 2) -- forward = the CUDA filter, backward = the hand-written reverse-mode kernel
(cdk_ekf_grad_f64 with CDK_GRAD_REVERSE), no autodiff through the solver.

    ll = ekf_marginal_log_prob(params, emissions, t_emissions, hyperparams)   # [N] (or scalar), differentiable w.r.t. the
    ll.sum().backward()                                                       # torch leaves of `params`

What `fit_sgd` minimises upstream is `-vmap(marginal_log_prob)(...).sum()` (src/ssm_temissions.py:550-568,
src/utils/optimize_utils.py:102).  Every registry drift, linear emission of any size, fp64 (cdk_ekf_grad_f64 for
Lorenz-63 with a scalar emission, cdk_ekf_grad_dense_f64 otherwise); differentiable user drifts and emissions
(cdk_ekf_grad_dense_f64).  ukf_marginal_log_prob is the same for the
closed-form CD-UKF (backward = cdk_ukf_grad_dense_f64), ukf_sigma_points_marginal_log_prob for the CD-UKF with literal
sigma points (backward = cdk_ukf_grad_sigma_f64; registry drifts and differentiable user drifts).

The linear CD Kalman filter has the same shape, cdlgssm_marginal_log_prob (backward = cdk_kf_grad_f64)."""
import numpy as np
import torch

from .continuous_discrete_linear_gaussian_ssm.inference import cdlgssm_marginal_log_prob_and_grad

from .continuous_discrete_nonlinear_gaussian_ssm._common import (check_user_emission_grad, is_user_emission,
                                                                 reject_user_emission)
from .continuous_discrete_nonlinear_gaussian_ssm.inference_ekf import (EKFHyperParams, drift_leaves,
                                                                       ekf_dense_marginal_log_prob_and_grad,
                                                                       ekf_marginal_log_prob_and_grad)
from .continuous_discrete_nonlinear_gaussian_ssm.inference_ukf import (UKFHyperParams, ukf_marginal_log_prob_and_grad,
                                                                       ukf_sigma_points_marginal_log_prob_and_grad)

def _val(x):
    return x.params if hasattr(x, "params") and hasattr(x, "f") else x


def _leaves(params):
    """Leaf name -> value: the drift's own fields (sigma / rho / beta, weights / bias, forcing, a / B / C), then the rest
    (a user emission's parameters are the one leaf "phi")."""
    d, e = params.dynamics, params.emissions
    out = {name: getattr(d.drift, name) for name, _ in drift_leaves(d.drift, 0)}
    out.update(diffusion_coefficient=_val(d.diffusion_coefficient), diffusion_cov=_val(d.diffusion_cov),
               emission_cov=_val(e.emission_cov))
    if is_user_emission(params):
        out.update(phi=e.emission_function.phi)
    else:
        out.update(emission_bias=e.emission_function.bias, emission_weights=e.emission_function.weights)
    out.update(initial_mean=_val(params.initial.mean), initial_cov=_val(params.initial.cov))
    return out


class _NonlinearLogLik(torch.autograd.Function):
    """`grad_fn(params, emissions, t_emissions, hyperparams, wrt="all")` -> (ll, grads keyed by leaf name)."""
    @staticmethod
    def forward(ctx, grad_fn, params, emissions, t_emissions, hyperparams, names, *leaf_tensors):
        ll, grads = grad_fn(params, emissions, t_emissions, hyperparams, wrt="all")
        ll = torch.as_tensor(ll)
        ctx.grads = [torch.as_tensor(grads[name]) for name in names]
        ctx.shapes = [tuple(t.shape) for t in leaf_tensors]
        ctx.batched = ll.dim() == 1
        return ll

    @staticmethod
    def backward(ctx, grad_ll):
        out = []
        for g, shape in zip(ctx.grads, ctx.shapes):
            g = g.to(grad_ll.device)
            if ctx.batched:
                w = grad_ll.reshape((-1,) + (1,) * (g.dim() - 1))
                g = g * w
                if len(shape) < g.dim():  # a parameter shared by the batch: sum over trajectories
                    g = g.sum(0)
            else:
                g = g * grad_ll
            out.append(g.reshape(shape))
        return (None, None, None, None, None, None) + tuple(out)


def _nonlinear_log_prob(grad_fn, params, emissions, t_emissions, hyperparams):
    leaves = _leaves(params)
    names = tuple(leaves)
    tensors = [leaves[n] if isinstance(leaves[n], torch.Tensor) else torch.as_tensor(leaves[n]) for n in names]
    return _NonlinearLogLik.apply(grad_fn, params, emissions, t_emissions, hyperparams, names, *tensors)


def ekf_marginal_log_prob(params, emissions, t_emissions=None, hyperparams: EKFHyperParams = EKFHyperParams()):
    """Per-trajectory marginal log-likelihood of the CD-EKF as a differentiable torch tensor.  Every leaf of `params`
    that is a torch tensor with requires_grad receives its gradient on `.backward()`: the drift's fields (named as in its
    registry class) and the diffusion, emission and initial parameters; for a LearnableUserEmission(...,
    differentiable=True) the emission's parameters are a torch `phi`."""
    check_user_emission_grad(params, "ekf_marginal_log_prob")
    scalar_l63 = (type(params.dynamics.drift).__name__ == "LearnableLorenz63" and not is_user_emission(params)
                  and tuple(np.shape(params.emissions.emission_function.weights))[-2] == 1)
    fn = ekf_marginal_log_prob_and_grad if scalar_l63 else ekf_dense_marginal_log_prob_and_grad
    return _nonlinear_log_prob(fn, params, emissions, t_emissions, hyperparams)


def ukf_marginal_log_prob(params, emissions, t_emissions=None, hyperparams: UKFHyperParams = UKFHyperParams()):
    """Per-trajectory marginal log-likelihood of the closed-form CD-UKF as a differentiable torch tensor
    (ukf_marginal_log_prob_and_grad).  Every leaf of `params` that is a torch tensor with requires_grad receives its
    gradient on `.backward()`, as in `ekf_marginal_log_prob`."""
    reject_user_emission(params, "ukf_marginal_log_prob")
    return _nonlinear_log_prob(ukf_marginal_log_prob_and_grad, params, emissions, t_emissions, hyperparams)


def ukf_sigma_points_marginal_log_prob(params, emissions, t_emissions=None,
                                       hyperparams: UKFHyperParams = UKFHyperParams()):
    """Per-trajectory marginal log-likelihood of the CD-UKF with literal sigma points as a differentiable torch tensor
    (ukf_sigma_points_marginal_log_prob_and_grad).  Every leaf of `params` that is a torch tensor with requires_grad
    receives its gradient on `.backward()`, as in `ekf_marginal_log_prob`; for a LearnableUserDrift(...,
    differentiable=True) that includes a torch `theta`."""
    reject_user_emission(params, "ukf_sigma_points_marginal_log_prob")
    return _nonlinear_log_prob(ukf_sigma_points_marginal_log_prob_and_grad, params, emissions, t_emissions, hyperparams)


_KF_LEAVES = (("dynamics", "weights"), ("dynamics", "bias"), ("dynamics", "diffusion_coefficient"),
              ("dynamics", "diffusion_cov"), ("emissions", "weights"), ("emissions", "bias"), ("emissions", "cov"),
              ("initial", "mean"), ("initial", "cov"))


class _KFLogLik(torch.autograd.Function):
    @staticmethod
    def forward(ctx, params, emissions, t_emissions, filter_hyperparams, names, *leaf_tensors):
        ll, grads = cdlgssm_marginal_log_prob_and_grad(params, emissions, t_emissions, filter_hyperparams)
        ll = torch.as_tensor(ll)
        ctx.grads = [torch.as_tensor(getattr(getattr(grads, grp), fld)) for grp, fld in names]
        ctx.leaves = [(tuple(t.shape), t.device, t.dtype) for t in leaf_tensors]
        ctx.batched = ll.dim() == 1
        return ll

    @staticmethod
    def backward(ctx, grad_ll):
        out = []
        for g, (shape, device, dtype) in zip(ctx.grads, ctx.leaves):
            g = g.to(grad_ll.device)
            if ctx.batched:
                g = g * grad_ll.reshape((-1,) + (1,) * (g.dim() - 1))
                if len(shape) < g.dim():  # a parameter shared by the batch: sum over trajectories
                    g = g.sum(0)
            else:
                g = g * grad_ll
            out.append(g.reshape(shape).to(device=device, dtype=dtype))
        return (None, None, None, None, None) + tuple(out)


def cdlgssm_marginal_log_prob(params, emissions, t_emissions=None, filter_hyperparams=None):
    """Per-trajectory marginal log-likelihood of the linear CD Kalman filter as a differentiable torch tensor (fp64,
    n <= 16, m <= 8, full R, no inputs: the coverage of cdk_kf_grad_f64).  Every torch leaf among F, b, L, Qc, H, d, R,
    m0, P0 of `params` with requires_grad receives its gradient on `.backward()`; a leaf shared by a batch of
    trajectories receives the sum over them."""
    names = tuple(nm for nm in _KF_LEAVES if getattr(getattr(params, nm[0]), nm[1]) is not None)
    tensors = [torch.as_tensor(getattr(getattr(params, grp), fld)) for grp, fld in names]
    return _KFLogLik.apply(params, emissions, t_emissions, filter_hyperparams, names, *tensors)
