"""Shared marshalling for the nonlinear filters (EKF / UKF / EnKF)."""
import numpy as np

from .. import _engine as E
from .. import _lib as L
from ..continuous_discrete_linear_gaussian_ssm.inference import _shape, _sq, prepare_data
from ..types import PosteriorGSSMFiltered
from .cdnlgssm_utils import drift_to_theta

DEFAULT_FIELDS = ["filtered_means", "filtered_covariances", "predicted_means", "predicted_covariances"]
_FIELD_SLOT = {"filtered_means": L.OUT_FM, "filtered_covariances": L.OUT_FP, "predicted_means": L.OUT_PM,
               "predicted_covariances": L.OUT_PP, "marginal_loglik": L.OUT_LLCUM}


def _to_host(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else x


def _val(x):
    """LearnableVector / LearnableMatrix -> array; plain arrays pass through."""
    return x.params if hasattr(x, "params") and hasattr(x, "f") else x


def nonlinear_inputs(params, Y, T, n, m):
    em = params.emissions.emission_function
    if type(em).__name__ != "LearnableLinear":
        raise NotImplementedError("emission_function must be LearnableLinear (h(x) = H x + d): arbitrary Python "
                                  "emission callables cannot run inside a CUDA kernel")
    drift_id, theta, n_theta = drift_to_theta(params.dynamics.drift, n)
    ins = {
        L.IN_Y: Y, L.IN_T: T, L.IN_M0: _val(params.initial.mean), L.IN_P0: _val(params.initial.cov), L.IN_F: theta,
        L.IN_L: _val(params.dynamics.diffusion_coefficient), L.IN_QC: _val(params.dynamics.diffusion_cov),
        L.IN_H: em.weights, L.IN_D: em.bias, L.IN_R: _val(params.emissions.emission_cov),
    }
    fields = dict(drift_id=drift_id, n_theta=n_theta, emission_id=0)
    if drift_id == L.DRIFT_USER:
        from .. import build as _build
        drift = params.dynamics.drift
        fields["lib_path"] = _build.build_user_drift(drift.device_code, grad=bool(drift.differentiable))
    return ins, fields


def run_filter(entry, params, emissions, t_emissions, inputs, output_fields, desc_fields, settings_sde=False,
               diffeqsolve_settings=None, keep_on_device=False):
    """Common driver: returns (PosteriorGSSMFiltered, device outputs dict, context)."""
    kind = E.kind_of(emissions)
    if inputs is not None and _shape(inputs)[-1] > 0 and bool(np.any(np.asarray(_to_host(inputs)) != 0)):
        # the registry drifts and the linear emission take no inputs (upstream's LearnableLorenz63 / LearnableLinear
        # ignore `u` as well); silently dropping a non-zero input array would change the model without a word
        raise NotImplementedError("non-zero `inputs` are not supported on the nonlinear path: the registry drifts and "
                                  "emissions do not depend on u (cdnlgssm_utils.py:50-83)")
    Y, T, U, batched = prepare_data(emissions, t_emissions, None)
    N, K, m = _shape(Y)
    n = _shape(_val(params.dynamics.diffusion_cov))[-1]
    dt = E.pick_dtype(emissions)
    ins, drift_fields = nonlinear_inputs(params, Y, T, n, m)
    fields = dict(E.parse_settings(diffeqsolve_settings, sde=settings_sde), **drift_fields, **desc_fields)
    output_fields = list(DEFAULT_FIELDS if output_fields is None else output_fields)
    unknown = [f for f in output_fields if f not in _FIELD_SLOT]
    if unknown:
        raise ValueError(f"unknown output_fields {unknown}")
    want = [L.OUT_LL] + [_FIELD_SLOT[f] for f in output_fields]
    # host callers get their results streamed back chunk by chunk into pinned memory, unless a smoother is going to
    # consume them on the device (keep_on_device); either way the staged device inputs are handed on for reuse
    dev_ins = {}
    out = E.run(entry, dt, N, K, n, m, ins, want, fields, host_out=(kind != "cuda" and not keep_on_device),
                dev_inputs=dev_ins)
    ins = {**ins, **dev_ins}
    g = lambda s: E.from_dev(_sq(out[s], batched), kind) if s in out else None
    # listing "marginal_loglik" in output_fields replaces the scalar by the cumulative per-step array
    # (inference_ekf.py:313-315,322; SURVEY 8b)
    ll = g(L.OUT_LLCUM) if "marginal_loglik" in output_fields else g(L.OUT_LL)
    post = PosteriorGSSMFiltered(marginal_loglik=ll, filtered_means=g(L.OUT_FM), filtered_covariances=g(L.OUT_FP),
                                 predicted_means=g(L.OUT_PM), predicted_covariances=g(L.OUT_PP))
    return post, out, (ins, fields, N, K, n, m, dt, batched, kind)
