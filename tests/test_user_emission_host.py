"""Host-only checks of the user-emission plumbing (no GPU): the variant cache key of build.build_variant, the host-side
check of phi against the emission's num_params, and the entry points that must refuse a user emission before any build or
device work."""
import os

import numpy as np
import pytest

from cd_dynamax_b200 import build as B

_EX = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cd_dynamax_b200", "examples")
VDP = open(os.path.join(_EX, "vdp_drift.cuh")).read()
RANGE = open(os.path.join(_EX, "range_emission.cuh")).read()


def test_variant_key_separates_drift_emission_both_and_grad():
    keys = [B.variant_key(VDP, None, False), B.variant_key(None, RANGE, False), B.variant_key(VDP, RANGE, False),
            B.variant_key(VDP, None, True), B.variant_key(VDP, RANGE, True)]
    assert len(set(keys)) == len(keys)
    # the same code as drift or as emission is a different variant
    assert B.variant_key(RANGE, None) != B.variant_key(None, RANGE)
    assert B.variant_key(VDP, RANGE) == B.variant_key(VDP, RANGE)


def test_build_user_drift_is_build_variant_with_a_drift_only(monkeypatch):
    calls = []
    monkeypatch.setattr(B, "build_variant", lambda *a: calls.append(a) or "lib")
    assert B.build_user_drift(VDP) == "lib" and B.build_user_drift(VDP, True) == "lib"
    assert calls == [(VDP, None, False, False), (VDP, None, True, False)]
    assert B.variant_key(VDP, None, False) != B.variant_key(VDP, None, True)


def test_build_variant_rejects_empty_and_drift_less_grad_requests():
    with pytest.raises(ValueError):
        B.build_variant()
    with pytest.raises(ValueError):
        B.build_variant(None, RANGE, grad=True)


def _params(phi, m=2):
    import cd_dynamax_b200 as cd
    n = 2
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(np.zeros(n)), cov=cd.LearnableMatrix(np.eye(n))),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=cd.LearnableLinear(weights=-np.eye(n), bias=np.zeros(n)),
                                           diffusion_coefficient=cd.LearnableMatrix(np.eye(n)),
                                           diffusion_cov=cd.LearnableMatrix(np.eye(n))),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableUserEmission(RANGE, phi),
                                             emission_cov=cd.LearnableMatrix(np.eye(m))))


def test_gradients_autograd_and_emission_moments_refuse_a_user_emission():
    import cd_dynamax_b200 as cd
    from cd_dynamax_b200 import autograd
    p = _params(np.zeros(5))
    y, t = np.zeros((3, 2)), np.arange(3.0)[:, None]
    for fn in (cd.ekf_marginal_log_prob_and_grad, cd.ekf_dense_marginal_log_prob_and_grad, cd.ukf_marginal_log_prob_and_grad,
               cd.ukf_sigma_points_marginal_log_prob_and_grad, autograd.ekf_marginal_log_prob, autograd.ukf_marginal_log_prob,
               autograd.ukf_sigma_points_marginal_log_prob):
        with pytest.raises(NotImplementedError, match="LearnableUserEmission"):
            fn(p, y, t)
    with pytest.raises(NotImplementedError, match="LearnableUserEmission"):
        cd.cdnlgssm_emissions(p, t, np.zeros((3, 2)), np.zeros((3, 2, 2)), hyperparams=cd.EKFHyperParams())


def test_phi_of_the_wrong_length_raises_on_the_host():
    """nonlinear_inputs builds (or finds) the variant, asks it for num_params(n, m) = m n + 1 = 5 and rejects any other
    length before a kernel is launched."""
    from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm._common import nonlinear_inputs
    ins, fields = nonlinear_inputs(_params(np.zeros(5)), np.zeros((1, 3, 2)), np.zeros((1, 3)), 2, 2)
    assert fields["n_phi"] == 5 and fields["emission_id"] == 1 and ins[10].shape == (5,)
    ins, fields = nonlinear_inputs(_params(np.zeros((4, 5))), np.zeros((4, 3, 2)), np.zeros((4, 3)), 2, 2)
    assert fields["n_phi"] == 5
    for bad in (np.zeros(4), np.zeros((4, 6)), np.zeros((2, 2, 5))):
        with pytest.raises(ValueError, match="num_params"):
            nonlinear_inputs(_params(bad), np.zeros((1, 3, 2)), np.zeros((1, 3)), 2, 2)
