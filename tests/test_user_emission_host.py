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


@pytest.mark.parametrize("kind", ["range", "wide", "square"])
def test_test_emissions_jacobian_is_the_derivative_of_h(kind):
    """The NumPy twins of the GPU matrix's test emissions: the analytic jac against central differences of h."""
    from tests.test_gpu_user_emission_matrix import _emission
    n, m = 3, 5
    rng = np.random.default_rng(1)
    em = _emission(kind, n, m, rng)
    x = rng.standard_normal((4, n)) + 0.5
    eps = 1e-6
    fd = np.stack([(em.h(x + eps * e) - em.h(x - eps * e)) / (2 * eps) for e in np.eye(n)], axis=-1)
    J = em.jac(x)
    assert J.shape == (4, m, n)
    assert np.max(np.abs(J - fd)) < 1e-8 * max(1.0, np.max(np.abs(fd)))


def test_per_trajectory_phi_with_the_wrong_batch_raises_before_any_launch():
    """phi [N', n_phi] with N' != N (and N' != 1) is refused by the engine's host-side shape check, naming the slot."""
    import cd_dynamax_b200 as cd
    y, t = np.zeros((4, 3, 2)), np.tile(np.arange(3.0), (4, 1))[..., None]
    for bad in (np.zeros((3, 5)), np.zeros((5, 5))):
        with pytest.raises(ValueError, match="IN_H"):
            cd.cdnlgssm_filter(_params(bad), y, t, cd.EKFHyperParams())
    with pytest.raises(ValueError, match="num_params"):
        cd.cdnlgssm_filter(_params(np.zeros((4, 6))), y, t, cd.EKFHyperParams())


def test_parameter_free_emission_phi_classifies():
    """n_phi = 0: phi [0] is the shared call and [N, 0] a batched one with rows of 0 elements (a NULL device pointer)."""
    from cd_dynamax_b200 import _engine
    from cd_dynamax_b200 import _lib as L
    N, K, n, m = 4, 3, 2, 3
    fields = dict(emission_id=L.EMISSION_USER, n_phi=0)
    metas, mask = _engine.classify(N, K, n, m, {L.IN_H: np.zeros(0)}, fields)
    assert not metas[L.IN_H][1] and metas[L.IN_H][2] == 0 and mask == 0
    metas, mask = _engine.classify(N, K, n, m, {L.IN_H: np.zeros((N, 0))}, fields)
    assert metas[L.IN_H][1] and metas[L.IN_H][2] == 0 and mask == 1 << L.IN_H
    with pytest.raises(ValueError, match="IN_H"):
        _engine.classify(N, K, n, m, {L.IN_H: np.zeros(1)}, fields)
