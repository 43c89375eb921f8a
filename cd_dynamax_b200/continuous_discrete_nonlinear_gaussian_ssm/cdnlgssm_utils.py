"""Parameter containers of the nonlinear model with the reference's names and fields
(src/continuous_discrete_nonlinear_gaussian_ssm/cdnlgssm_utils.py:13-206).

A CUDA kernel cannot take an arbitrary Python callable, so the drift must be one of the registry classes below
(`LearnableLinear`, `LearnableLorenz63` as upstream; `LearnableLorenz96` and `LearnableQuadratic` are additions) and
the emission function must be `LearnableLinear`; `LearnableUserDrift` and `LearnableUserEmission` take CUDA device code
instead.  Each class still carries `.f(x, u, t)` with the upstream signature
(NumPy) so that host code written against the reference keeps working.
"""
from typing import Any, NamedTuple, Optional

import numpy as np

from .. import _lib as L
from ..types import ParamsLGSSMInitial


def _np(x):
    import torch
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


class LearnableVector(NamedTuple):
    params: Any

    def f(self, x=None, u=None, t=None):
        return self.params


class LearnableMatrix(NamedTuple):
    params: Any

    def f(self, x=None, u=None, t=None):
        return self.params


class LearnableLinear(NamedTuple):
    """f(x) = weights @ x + bias (cdnlgssm_utils.py:50-61)"""
    weights: Any
    bias: Any

    def f(self, x, u=None, t=None):
        return _np(self.weights) @ _np(x) + _np(self.bias)


class LearnableLorenz63(NamedTuple):
    """cdnlgssm_utils.py:63-83"""
    sigma: Any
    rho: Any
    beta: Any

    def f(self, x, u=None, t=None):
        x = _np(x)
        s, r, b = (_np(v) for v in (self.sigma, self.rho, self.beta))
        return np.array([s * (x[1] - x[0]), x[0] * (r - x[2]) - x[1], x[0] * x[1] - b * x[2]])


class LearnableLorenz96(NamedTuple):
    """dx_i = (x_{i+1} - x_{i-2}) x_{i-1} - x_i + forcing, cyclic (BASELINE configs 4-5; not in the reference)."""
    forcing: Any

    def f(self, x, u=None, t=None):
        x = _np(x)
        return (np.roll(x, -1) - np.roll(x, 2)) * np.roll(x, 1) - x + _np(self.forcing)


class LearnableQuadratic(NamedTuple):
    """f_i = a_i + B_ij x_j + C_ijk x_j x_k (any quadratic vector field; not in the reference)."""
    a: Any
    B: Any
    C: Any

    def f(self, x, u=None, t=None):
        x = _np(x)
        return _np(self.a) + _np(self.B) @ x + np.einsum("ijk,j,k->i", _np(self.C), x, x)


class LearnableUserDrift(NamedTuple):
    """A user-defined drift (SURVEY 8f rank 4; upstream: any `LearnableFunction.f`, cdnlgssm_utils.py:13-36).  A CUDA kernel
    needs device code, so the drift is given as CUDA C++ source (see cd_dynamax_b200.build.build_user_drift for the three
    functions it must define in `namespace cdk_user`) plus its parameter vector `theta` ([n_theta] or [N, n_theta]); the
    first use compiles a variant of libcdk.so with that code in the drift registry (cached by content hash).  `py_f` is an
    optional NumPy callable f(x, theta) for host-side use (e.g. the reference-style `.f`).

    `differentiable=True` declares that the device code stays within the dual-number contract of
    cd_dynamax_b200.build.build_user_drift (T arithmetic and the unqualified math functions only), and selects the variant
    that also holds the EKF gradient: ekf_marginal_log_prob_and_grad then returns d ll / d theta under "theta", and
    autograd.ekf_marginal_log_prob takes a torch `theta`.  The drift's filter calls use that same variant."""
    device_code: str
    theta: Any
    py_f: Any = None
    differentiable: bool = False

    def f(self, x, u=None, t=None):
        if self.py_f is None:
            raise NotImplementedError("no host-side callable was given for this user drift")
        return self.py_f(_np(x), _np(self.theta))


class LearnableUserEmission(NamedTuple):
    """A user-defined emission function (upstream: any `LearnableFunction.f` as emission, cdnlgssm_utils.py:13-36), given
    as CUDA C++ source (see cd_dynamax_b200.build.build_variant for the three functions it must define in
    `namespace cdk_user_emission`) plus its parameter vector `phi` ([n_phi] or [N, n_phi], torch or NumPy); the first use
    compiles a variant of libcdk.so with that code -- and the drift's, when the drift is a LearnableUserDrift -- in the
    registries (cached by content hash).  The EKF, EKS, UKF, EnKF and the path sampler run it; the emission moments of
    cdnlgssm_emissions and the UKF gradients do not.  `py_h` is an optional NumPy callable h(x, phi) for host-side use
    (`.f`).  `differentiable=True` declares that the code stays within the dual-number contract (build_variant) and
    compiles the EKF gradient for it: ekf_marginal_log_prob_and_grad, ekf_dense_marginal_log_prob_and_grad and
    autograd.ekf_marginal_log_prob then differentiate every parameter, phi included (grads["phi"])."""
    device_code: str
    phi: Any
    py_h: Any = None
    differentiable: bool = False

    def f(self, x, u=None, t=None):
        if self.py_h is None:
            raise NotImplementedError("no host-side callable was given for this user emission")
        return self.py_h(_np(x), _np(self.phi))


class ParamsCDNLGSSMDynamics(NamedTuple):
    """cdnlgssm_utils.py:88-130"""
    drift: Any
    diffusion_coefficient: Any
    diffusion_cov: Any
    approx_order: Any = 2.0


class ParamsCDNLGSSMEmissions(NamedTuple):
    """cdnlgssm_utils.py:163-179"""
    emission_function: Any
    emission_cov: Any


class ParamsCDNLGSSM(NamedTuple):
    """cdnlgssm_utils.py:191-206"""
    initial: ParamsLGSSMInitial
    dynamics: ParamsCDNLGSSMDynamics
    emissions: ParamsCDNLGSSMEmissions


class GSSMForecast(NamedTuple):
    """cdnlgssm_utils.py:227-249 (container only; forecasting is outside the hot path)"""
    forecasted_state_means: Optional[Any] = None
    forecasted_state_covariances: Optional[Any] = None
    forecasted_emission_means: Optional[Any] = None
    forecasted_emission_covariances: Optional[Any] = None
    forecasted_state_path: Optional[Any] = None
    forecasted_emission_path: Optional[Any] = None


def drift_to_theta(drift, n: int):
    """-> (drift_id, theta tensor [n_theta] or [N, n_theta], n_theta).  Layouts: include/cdk.h drift registry."""
    import torch

    def T(x):
        t = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x, dtype=np.float64))
        return t.to(torch.float64)

    def same_device(parts):
        cuda = [p for p in parts if p.is_cuda]
        return [p.to(cuda[0].device) for p in parts] if cuda else parts

    def flat_theta(leaves):
        """(leaf, core rank) pairs -> theta: [sum of sizes] when no leaf carries a leading N, else [N, sum of sizes] with
        the shared leaves repeated on every row (vmap over parameter samples batches any subset of the leaves)."""
        lead = {int(x.shape[0]) for x, core in leaves if x.dim() == core + 1}
        if len(lead) > 1:
            raise ValueError(f"{name}: batched leaves disagree on the leading axis: "
                             f"{[tuple(x.shape) for x, _ in leaves]}")
        if not lead:
            return torch.cat([x.reshape(-1) for x, _ in leaves])
        N = lead.pop()
        return torch.cat([x.reshape(N, -1) if x.dim() == core + 1 else x.reshape(1, -1).expand(N, -1)
                          for x, core in leaves], dim=-1)

    name = type(drift).__name__
    if name == "LearnableLinear":
        W, b = same_device([T(drift.weights), T(drift.bias)])
        return L.DRIFT_LINEAR, flat_theta([(W, 2), (b, 1)]), n * n + n
    if name == "LearnableLorenz63":
        parts = same_device([T(drift.sigma), T(drift.rho), T(drift.beta)])
        N = max(p.numel() for p in parts)
        if N > 1:
            theta = torch.stack([p.reshape(-1).expand(N) for p in parts], dim=-1)
        else:
            theta = torch.stack([p.reshape(()) for p in parts])
        return L.DRIFT_LORENZ63, theta, 3
    if name == "LearnableLorenz96":
        F = T(drift.forcing)
        theta = F.reshape(-1, 1) if F.numel() > 1 else F.reshape(1)
        return L.DRIFT_LORENZ96, theta, 1
    if name == "LearnableQuadratic":
        a, B, C = same_device([T(drift.a), T(drift.B), T(drift.C)])
        return L.DRIFT_QUADRATIC, flat_theta([(a, 1), (B, 2), (C, 3)]), n + n * n + n * n * n
    if name == "LearnableUserDrift":
        th = T(drift.theta)
        return L.DRIFT_USER, th, int(th.shape[-1]) if th.dim() else 1
    raise NotImplementedError(
        f"drift {name!r} is not in the kernel registry (LearnableLinear, LearnableLorenz63, LearnableLorenz96, "
        "LearnableQuadratic) and is not a LearnableUserDrift (CUDA device code): arbitrary Python drift callables cannot "
        "run inside a CUDA kernel")
