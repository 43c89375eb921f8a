"""CPU: the host rejects time grids, emissions and inputs whose per-trajectory shape does not match (K, m, d_u) before it
touches the library or the device.  The kernels index these arrays with strides computed from K, m and d_u alone, so a
grid one column short would otherwise be read out of bounds on the GPU.

`_lib.lib` is replaced by a function that raises `_Reached`: a call that passes validation stops there, so none of these
tests loads the library or launches anything, with or without a GPU."""
import numpy as np
import pytest

from cd_dynamax_b200 import _engine as E
from cd_dynamax_b200 import _lib as L


class _Reached(Exception):
    pass


@pytest.fixture
def no_device(monkeypatch):
    def boom(*a, **k):
        raise _Reached()

    monkeypatch.setattr(L, "lib", boom)


N, K, n, m = 5, 7, 3, 2


def _run(ins, flags=0, d_u=0):
    fields = dict(flags=flags, d_u=d_u) if flags else dict(d_u=d_u)
    return E.run("cdk_ekf_filter", "f64", N, K, n, m, ins, [L.OUT_LL], fields)


def _ok_inputs(t_cols=K, d_u=0):
    ins = {L.IN_Y: np.zeros((N, K, m)), L.IN_T: np.zeros((N, t_cols)), L.IN_M0: np.zeros(n)}
    if d_u:
        ins[L.IN_U] = np.zeros((N, K, d_u))
    return ins


def test_well_shaped_inputs_pass_validation(no_device):
    for ins, flags, d_u in ((_ok_inputs(), 0, 0), (_ok_inputs(d_u=2), 0, 2), (_ok_inputs(K + 1), L.FLAG_PREDICT_ONLY, 0),
                            (_ok_inputs(K + 1), L.FLAG_FIXED_INIT, 0)):
        with pytest.raises(_Reached):
            _run(ins, flags, d_u)
    # a shared grid: [K] or a leading axis of 1
    for t in (np.zeros(K), np.zeros((1, K))):
        with pytest.raises(_Reached):
            _run({**_ok_inputs(), L.IN_T: t})


@pytest.mark.parametrize("slot,shape,flags,d_u", [
    (L.IN_T, (N, K - 1), 0, 0),  # one time stamp short
    (L.IN_T, (N, K + 1), 0, 0),  # a filter reads K stamps
    (L.IN_T, (N, K), L.FLAG_PREDICT_ONLY, 0),  # a forecast reads K + 1 (t_init first)
    (L.IN_T, (N, K), L.FLAG_FIXED_INIT, 0),
    (L.IN_T, (N, K + 2), L.FLAG_PREDICT_ONLY, 0),
    (L.IN_T, (K - 1,), 0, 0),  # shared grid
    (L.IN_T, (1, K - 1), 0, 0),  # shared grid with a leading axis of 1
    (L.IN_Y, (N, K - 1, m), 0, 0),
    (L.IN_Y, (N, K, m + 1), 0, 0),
    (L.IN_Y, (K + 1, m), 0, 0),
    (L.IN_U, (N, K - 1, 2), 0, 2),
    (L.IN_U, (N, K, 3), 0, 2),
])
def test_mis_shaped_time_grid_emissions_and_inputs_raise_on_host(no_device, slot, shape, flags, d_u):
    ins = _ok_inputs(K + 1 if flags else K, d_u)
    ins[slot] = np.zeros(shape)
    with pytest.raises(ValueError) as e:
        _run(ins, flags, d_u)
    msg = str(e.value)
    name = {L.IN_T: "IN_T", L.IN_Y: "IN_Y", L.IN_U: "IN_U"}[slot]
    assert name in msg and str(shape) in msg, msg


def test_public_api_rejects_inputs_of_the_wrong_length(no_device):
    """cdlgssm_filter takes K from the emissions; `inputs` one row short would be read past its end."""
    import cd_dynamax_b200 as cd
    d_u = 2
    p = cd.ParamsCDLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=np.zeros(n), cov=np.eye(n)),
        dynamics=cd.ParamsCDLGSSMDynamics(weights=-np.eye(n), bias=np.zeros(n), input_weights=np.ones((n, d_u)),
                                          diffusion_coefficient=np.eye(n), diffusion_cov=np.eye(n)),
        emissions=cd.ParamsLGSSMEmissions(weights=np.ones((m, n)), bias=np.zeros(m), input_weights=np.ones((m, d_u)),
                                          cov=np.eye(m)))
    y = np.zeros((N, K, m))
    t = np.cumsum(np.full((N, K), 0.1), axis=1)[..., None]
    with pytest.raises(_Reached):
        cd.cdlgssm_filter(p, y, t, cd.KFHyperParams(), np.ones((N, K, d_u)))
    with pytest.raises(ValueError, match="IN_U"):
        cd.cdlgssm_filter(p, y, t, cd.KFHyperParams(), np.ones((N, K - 1, d_u)))
    with pytest.raises(ValueError, match="IN_U"):
        cd.cdlgssm_filter(p, y, t, cd.KFHyperParams(), np.ones((K - 1, d_u)))
