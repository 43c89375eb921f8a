"""Drop-in for the callers either side of the filters in src/continuous_discrete_nonlinear_gaussian_ssm/models.py:

  cdnlgssm_forecast      :767-936   forecast a Gaussian (EKF / UKF / EnKF _predict scanned with no updates:
                                    forecast_extended_kalman_filter inference_ekf.py:679-761 and its twins) or a point
                                    estimate (one SDE sample path + sampled emissions)
  cdnlgssm_emissions     :939-1047  emission moments of state estimates (emissions_extended_kalman_filter
                                    inference_ekf.py:762-855: H m + d, H P H^T + R; or the model's own (H m + d, R))
  cdnlgssm_path_sample   :525-656   forward sample paths; batched = SSM.sample_batch(..., transition_type="path")
                                    (src/ssm_temissions.py:187-225)

All arithmetic runs in libcdk.so (cdk_*_filter with CDK_FLAG_PREDICT_ONLY, cdk_sample_path, cdk_emission_moments).
Random streams: the reference's `key` is a jax.random key whose stream cannot be reproduced outside JAX; here `key` seeds
a Philox4x32-10 stream (an int, or a 2-word PRNGKey-like array), so samples agree with the reference in distribution only
(and with oracle/cd_oracle.py bit-for-bit up to rounding)."""
import os
from typing import Any, List, NamedTuple, Optional

import numpy as np

from .. import _engine as E
from .. import _lib as L
from ..continuous_discrete_linear_gaussian_ssm.inference import _shape, _sq
from ._common import _val, emission_dim, is_user_emission, nonlinear_inputs, reject_user_emission
from .inference_ekf import EKFHyperParams, _ekf_fields
from .inference_enkf import EnKFHyperParams, key_to_seed
from .inference_ukf import UKFHyperParams


from .cdnlgssm_utils import GSSMForecast  # noqa: E402  (the reference's container, cdnlgssm_utils.py)


class MultivariateNormalFullCovariance:
    """Minimal stand-in for tfd.MultivariateNormalFullCovariance as `init_forecast` (only .mean() / .covariance() are used
    upstream, inference_ekf.py:753)."""

    def __init__(self, loc, covariance_matrix):
        self.loc, self.covariance_matrix = loc, covariance_matrix

    def mean(self):
        return self.loc

    def covariance(self):
        return self.covariance_matrix


def _times_with_init(t_init, t_forecast, like):
    """[t_init | t_forecast] along the time axis -> [N, K+1] (or [1, K+1] when shared)."""
    if t_forecast is None:
        raise ValueError("t_forecast must be provided for forecasting")  # models.py:858
    tf = t_forecast[..., 0] if _shape(t_forecast)[-1] == 1 and len(_shape(t_forecast)) >= 2 else t_forecast
    import torch
    if isinstance(tf, torch.Tensor):
        ti = torch.as_tensor(t_init, dtype=tf.dtype, device=tf.device).reshape(-1)
        tf2 = tf if tf.ndim == 2 else tf[None]
        ti2 = ti.reshape(-1, 1).expand(tf2.shape[0], 1) if ti.numel() in (1, tf2.shape[0]) else ti.reshape(tf2.shape[0], 1)
        return torch.cat([ti2, tf2], dim=1)
    tf = np.asarray(tf, dtype=np.float64)
    tf2 = tf if tf.ndim == 2 else tf[None]
    ti = np.asarray(t_init, dtype=np.float64).reshape(-1)
    ti2 = np.broadcast_to(ti.reshape(-1, 1), (tf2.shape[0], 1))
    return np.concatenate([ti2, tf2], axis=1)


def cdnlgssm_forecast(params, init_forecast, t_init, t_forecast=None, hyperparams=EKFHyperParams(), inputs=None,
                      output_fields: Optional[List[str]] = ("forecasted_state_means", "forecasted_state_covariances"),
                      key=0, diffeqsolve_settings: dict = {}) -> GSSMForecast:
    """cd_nonlinear/models.py:767-936.  `init_forecast` with .mean() / .covariance() (or a (mean, cov) pair) forecasts the
    Gaussian with the filter the hyper-parameter type names; an array is a point estimate and forecasts one sample path of
    the SDE plus sampled emissions.  Batched: leading N on the initial condition and / or `t_forecast [N, K, 1]`."""
    if hasattr(init_forecast, "mean") and hasattr(init_forecast, "covariance"):
        m0, P0 = init_forecast.mean(), init_forecast.covariance()
    elif isinstance(init_forecast, (tuple, list)) and len(init_forecast) == 2:
        m0, P0 = init_forecast
    else:
        return _forecast_path(params, init_forecast, t_init, t_forecast, key, diffeqsolve_settings)
    kind = E.kind_of(m0)
    T = _times_with_init(t_init, t_forecast, m0)
    n = _shape(_val(params.dynamics.diffusion_cov))[-1]
    m = emission_dim(params)
    if is_user_emission(params) and output_fields is not None and \
            {"forecasted_emission_means", "forecasted_emission_covariances"} & set(output_fields):
        reject_user_emission(params, "the forecasted emission moments")
    batched = len(_shape(m0)) == 2 or _shape(T)[0] > 1
    N = max(_shape(m0)[0] if len(_shape(m0)) == 2 else 1, _shape(T)[0])
    K = _shape(T)[1] - 1
    dt = E.pick_dtype(m0)
    ins, drift_fields = nonlinear_inputs(params, None, T, n, m)
    ins = {k: v for k, v in ins.items() if v is not None}
    ins[L.IN_M0], ins[L.IN_P0] = m0, P0
    if isinstance(hyperparams, EKFHyperParams):
        entry, fields, sde = "cdk_ekf_filter", _ekf_fields(hyperparams, 1), False
    elif isinstance(hyperparams, UKFHyperParams):
        entry, sde = "cdk_ukf_filter", False
        fields = dict(dt_final=float(hyperparams.dt_final), alpha=float(hyperparams.alpha), beta=float(hyperparams.beta),
                      kappa=float(hyperparams.kappa))
    elif isinstance(hyperparams, EnKFHyperParams):
        entry, sde = "cdk_enkf_filter", True
        fields = dict(dt_final=float(hyperparams.dt_final), E=int(hyperparams.N_particles), perturb_measurements=0,
                      rng_seed=key_to_seed(hyperparams.key))
    else:
        raise TypeError(f"hyperparams must be EKFHyperParams, UKFHyperParams or EnKFHyperParams, got {type(hyperparams)}")
    flags = L.FLAG_PREDICT_ONLY
    if entry == "cdk_ukf_filter" and os.environ.get("CDK_UKF_SIGMA_POINTS", "0") == "1":
        flags |= L.FLAG_UKF_SIGMA_POINTS
    fields = dict(E.parse_settings(hyperparams.diffeqsolve_settings, sde=sde), **drift_fields, **fields, flags=flags)
    want = []
    if output_fields is None or "forecasted_state_means" in output_fields:
        want.append(L.OUT_PM)
    if output_fields is None or "forecasted_state_covariances" in output_fields:
        want.append(L.OUT_PP)
    out = E.run(entry, dt, N, K, n, m, ins, want, fields, host_out=(kind != "cuda"))
    g = lambda s: E.from_dev(_sq(out[s], batched), kind) if s in out else None
    return GSSMForecast(forecasted_state_means=g(L.OUT_PM), forecasted_state_covariances=g(L.OUT_PP))


def _sample(params, m0, P0, T, N, K, fixed, key, diffeqsolve_settings, kind, dt, batched, want_states=True,
            want_emissions=True, rng_offset=0):
    n = _shape(_val(params.dynamics.diffusion_cov))[-1]
    m = emission_dim(params)
    ins, drift_fields = nonlinear_inputs(params, None, T, n, m)
    ins = {k: v for k, v in ins.items() if v is not None}
    ins[L.IN_M0] = m0
    if P0 is not None:
        ins[L.IN_P0] = P0
    else:
        ins.pop(L.IN_P0, None)
    fields = dict(E.parse_settings(diffeqsolve_settings, sde=True), **drift_fields, rng_seed=key_to_seed(key),
                  rng_offset=int(rng_offset), flags=L.FLAG_FIXED_INIT if fixed else 0)
    want = ([L.OUT_FM] if want_states else []) + ([L.OUT_PM] if want_emissions else [])
    out = E.run("cdk_sample_path", dt, N, K, n, m, ins, want, fields, host_out=(kind != "cuda"),
                out_shapes={L.OUT_PM: (N, K, m)})
    g = lambda s: E.from_dev(_sq(out[s], batched), kind) if s in out else None
    return g(L.OUT_FM), g(L.OUT_PM)


def _forecast_path(params, init_state, t_init, t_forecast, key, diffeqsolve_settings):
    kind = E.kind_of(init_state)
    T = _times_with_init(t_init, t_forecast, init_state)
    batched = len(_shape(init_state)) == 2 or _shape(T)[0] > 1
    N = max(_shape(init_state)[0] if len(_shape(init_state)) == 2 else 1, _shape(T)[0])
    K = _shape(T)[1] - 1
    xs, ys = _sample(params, init_state, None, T, N, K, True, key, diffeqsolve_settings, kind, E.pick_dtype(init_state), batched)
    return GSSMForecast(forecasted_state_path=xs, forecasted_emission_path=ys)


def cdnlgssm_path_sample(params, key, num_timesteps: int, t_emissions=None, inputs=None, diffeqsolve_settings={},
                         num_sequences: Optional[int] = None, rng_offset: int = 0, device_resident: bool = False):
    """cd_nonlinear/models.py:525-656: (states [K, n], emissions [K, m]) of one forward sample path; `num_sequences=N`
    gives the batch `SSM.sample_batch(params, key, N, K, t_emissions, inputs, transition_type="path")` returns
    ([N, K, n], [N, K, m]; src/ssm_temissions.py:187-225), all paths in ONE launch.  `t_emissions` may be [K, 1] (shared) or
    [N, K, 1]; None means unit spacing.  `device_resident=True` returns CUDA tensors (e.g. to feed a filter directly)."""
    import torch
    K = int(num_timesteps)
    if t_emissions is None:
        T = np.arange(K, dtype=np.float64)[None]  # models.py:633-634
    else:
        T = t_emissions[..., 0] if _shape(t_emissions)[-1] == 1 and len(_shape(t_emissions)) >= 2 else t_emissions
        if len(_shape(T)) == 1:
            T = T[None]
    if _shape(T)[-1] != K:
        raise ValueError(f"t_emissions has {_shape(T)[-1]} stamps, num_timesteps = {K}")
    batched = num_sequences is not None or _shape(T)[0] > 1
    N = int(num_sequences) if num_sequences is not None else _shape(T)[0]
    kind = "cuda" if (device_resident or isinstance(T, torch.Tensor) and T.is_cuda) else E.kind_of(T)
    m0, P0 = _val(params.initial.mean), _val(params.initial.cov)
    return _sample(params, m0, P0, T, N, K, False, key, diffeqsolve_settings, kind, E.pick_dtype(T), batched,
                   rng_offset=rng_offset)


def cdnlgssm_emissions(params, t_states, state_means, state_covs=None, inputs=None, hyperparams=None, key=0):
    """cd_nonlinear/models.py:939-1047: (emission means, emission covariances) for state estimates at `t_states`.  With EKF
    / UKF hyper-parameters and covariances: (H m + d, H P H^T + R) (the unscented transform of a linear emission is exact);
    with hyperparams=None: the model's own (H m + d, R) for point estimates."""
    if isinstance(hyperparams, EnKFHyperParams):
        raise NotImplementedError("emissions_ensemble_kalman_filter re-samples an ensemble from (m, P) with a jax.random "
                                  "key; use EKFHyperParams / UKFHyperParams for the exact Gaussian emission moments")
    reject_user_emission(params, "cdnlgssm_emissions")
    if t_states is None:
        raise ValueError("t_states must be provided for forecasting")
    em = params.emissions.emission_function
    if type(em).__name__ != "LearnableLinear":
        raise NotImplementedError("emission_function must be LearnableLinear (h(x) = H x + d)")
    kind = E.kind_of(state_means)
    sm = state_means
    batched = len(_shape(sm)) == 3
    if not batched:
        sm = sm[None]
        state_covs = None if state_covs is None else state_covs[None]
    N, K, n = _shape(sm)
    m = _shape(em.weights)[-2]
    dt = E.pick_dtype(state_means)
    use_cov = state_covs is not None and hyperparams is not None
    ins = {L.IN_FM: sm, L.IN_H: em.weights, L.IN_D: em.bias, L.IN_R: _val(params.emissions.emission_cov)}
    if use_cov:
        ins[L.IN_FP] = state_covs
    out = E.run("cdk_emission_moments", dt, N, K, n, m, ins, [L.OUT_PM, L.OUT_PP], {}, host_out=(kind != "cuda"),
                out_shapes={L.OUT_PM: (N, K, m), L.OUT_PP: (N, K, m, m)})
    g = lambda s: E.from_dev(_sq(out[s], batched), kind)
    return g(L.OUT_PM), g(L.OUT_PP)
