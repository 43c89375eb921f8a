"""Host side of the CD-EKF gradient for user-defined drifts (no GPU): the Python gate on `differentiable`, the "theta"
leaf, the two variants build_user_drift makes of one device code, the C-ABI checks of the stock, filter-only and
gradient variants, and the dual-number type of csrc/cdk_dual.cuh compiled as host code and checked against analytic
derivatives."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import cd_dynamax_b200 as cd
from cd_dynamax_b200 import _lib as L
from cd_dynamax_b200 import build as b
from cd_dynamax_b200.continuous_discrete_nonlinear_gaussian_ssm import inference_ekf as ie
from tests.test_ekf_grad_host import _call, lib  # noqa: F401  (lib: the stock library fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXAMPLES = os.path.join(ROOT, "cd_dynamax_b200", "examples")
VDP = open(os.path.join(EXAMPLES, "vdp_drift.cuh")).read()
MLP = open(os.path.join(EXAMPLES, "mlp_drift.cuh")).read()


class _Sentinel(Exception):
    pass


def _params(drift, n=2, m=1):
    return cd.ParamsCDNLGSSM(
        initial=cd.ParamsLGSSMInitial(mean=cd.LearnableVector(np.zeros(n)), cov=cd.LearnableMatrix(np.eye(n))),
        dynamics=cd.ParamsCDNLGSSMDynamics(drift=drift, diffusion_coefficient=cd.LearnableMatrix(np.eye(n)),
                                           diffusion_cov=cd.LearnableMatrix(np.eye(n))),
        emissions=cd.ParamsCDNLGSSMEmissions(emission_function=cd.LearnableLinear(weights=np.eye(m, n), bias=np.zeros(m)),
                                             emission_cov=cd.LearnableMatrix(np.eye(m))))


def test_non_differentiable_user_drift_is_rejected_before_any_build(monkeypatch):
    def boom(*a, **k):
        raise _Sentinel()
    monkeypatch.setattr(b, "build_user_drift", boom)
    monkeypatch.setattr(L, "lib", boom)
    p = _params(cd.LearnableUserDrift(device_code=VDP, theta=np.array([1.3, 0.4])))
    y, t = np.zeros((3, 5, 1)), np.cumsum(np.full((3, 5), 0.1), 1)[..., None]
    for fn in (cd.ekf_marginal_log_prob_and_grad, cd.ekf_dense_marginal_log_prob_and_grad):
        with pytest.raises(NotImplementedError, match="differentiable=True"):
            fn(p, y, t)
    from cd_dynamax_b200.autograd import ekf_marginal_log_prob
    with pytest.raises(NotImplementedError, match="differentiable=True"):
        ekf_marginal_log_prob(p, y, t)
    # the flag reaches the build: a differentiable drift asks for the gradient variant
    seen = []
    monkeypatch.setattr(b, "build_user_drift", lambda code, grad=False: seen.append(grad) or boom())
    with pytest.raises(_Sentinel):
        cd.ekf_marginal_log_prob_and_grad(_params(cd.LearnableUserDrift(VDP, np.array([1.3, 0.4]), differentiable=True)),
                                          y, t)
    assert seen == [True]


def test_the_field_is_last_and_defaults_to_false():
    d = cd.LearnableUserDrift(device_code="", theta=np.zeros(3))
    assert d.differentiable is False and cd.LearnableUserDrift._fields[-1] == "differentiable"


@pytest.mark.parametrize("shape", [(5,), (4, 5)])
def test_theta_leaf_and_unflatten(shape):
    drift = cd.LearnableUserDrift(device_code="", theta=np.arange(np.prod(shape), dtype=float).reshape(shape),
                                  differentiable=True)
    assert ie.drift_leaves(drift, 2) == (("theta", (5,)),)
    G = np.arange(4 * 5, dtype=float).reshape(4, 5)
    out = ie.unflatten_theta(G, drift, 2)
    assert set(out) == {"theta"} and np.array_equal(out["theta"], G)
    import torch
    from cd_dynamax_b200.autograd import _leaves
    th = torch.zeros(shape, dtype=torch.float64, requires_grad=True)
    leaves = _leaves(_params(drift._replace(theta=th)))
    assert leaves["theta"] is th


def test_filter_and_gradient_variants_differ_in_hash_and_units(monkeypatch, tmp_path):
    """build_user_drift(code) and build_user_drift(code, grad=True): two content hashes, and the gradient unit is compiled
    with the user header only in the second (the compiler is faked: no nvcc runs)."""
    calls = []

    def fake_run(cmd, capture_output=True, text=True):
        calls.append(cmd)
        out = cmd[cmd.index("-o") + 1]
        os.makedirs(os.path.dirname(out), exist_ok=True)
        open(out, "w").close()
        return subprocess.CompletedProcess(cmd, 0, "", "")

    monkeypatch.setattr(b, "build", lambda *a, **k: None)
    monkeypatch.setattr(b, "LIBDIR", str(tmp_path / "lib"))
    monkeypatch.setattr(b, "OBJ", str(tmp_path / "obj"))
    monkeypatch.setattr(b.subprocess, "run", fake_run)

    def units(lib):
        compiled = [os.path.basename(c[c.index("-c") + 1]) for c in calls if "-c" in c]
        link = next(c for c in calls if "-shared" in c)
        calls.clear()
        return sorted(compiled), link, lib

    filt, link_f, lib_f = units(b.build_user_drift(VDP))
    grad, link_g, lib_g = units(b.build_user_drift(VDP, grad=True))
    assert lib_f != lib_g
    assert filt == sorted(b.USER_SOURCES) and grad == sorted(b.USER_SOURCES + ["cdk_ekfgrad.cu"])
    assert any(o.endswith(os.path.join("obj", "cdk_ekfgrad.o")) for o in link_f)  # the stock gradient unit
    assert not any(o.endswith(os.path.join("obj", "cdk_ekfgrad.o")) for o in link_g)
    assert b.build_user_drift(VDP, grad=True) == lib_g and not calls  # cached


def _lib_or_skip(grad):
    if shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"):
        pytest.skip("nvcc is not available")
    return L.lib(b.build_user_drift(VDP, grad=grad))


def test_gradient_entry_point_by_variant(lib):
    E_SIZE, E_UNSUPPORTED = -2, -4
    user = dict(drift_id=L.DRIFT_USER, n=2, m=1, n_theta=2, N=0)
    for stock_or_filter in (lib, _lib_or_skip(False)):
        rc, msg = _call(stock_or_filter, **user)
        assert rc == E_UNSUPPORTED and "cdk_ekf_grad_dense_f64" in msg and "differentiable=True" in msg, msg
    var = _lib_or_skip(True)
    assert var.cdk_has_user_drift() == 1
    rc, msg = _call(var, **user)
    assert rc == 0, msg
    for order in (1, 2):
        assert _call(var, **dict(user, state_order=order))[0] == 0
    rc, msg = _call(var, **dict(user, n_theta=8000))
    assert rc == E_SIZE and "n_theta = 8000" in msg, msg
    # the UKF gradient keeps rejecting user drifts (literal sigma points)
    d = L.new_desc()
    d.N, d.K, d.n, d.m, d.drift_id, d.n_theta = 0, 5, 2, 1, L.DRIFT_USER, 2
    fake = ctypes.c_void_p(0x1000)
    ins = (ctypes.c_void_p * L.NUM_IN)(*([fake] * L.NUM_IN))
    outs = (ctypes.c_void_p * L.NUM_OUT)(*([fake] * L.NUM_OUT))
    assert var.cdk_ukf_grad_dense_f64(ctypes.byref(d), ins, outs, None) == E_UNSUPPORTED
    # the scratch of the user drift is the registry formula
    d.N, d.K, d.solver, d.n_theta = 3, 7, L.SOLVERS["rk4"], 2
    assert var.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad_dense") == lib.cdk_scratch_bytes(ctypes.byref(d), b"cdk_ekf_grad_dense")


DUAL_PROGRAM = r'''
#include <cmath>
#include <cstdio>
#include "cdk_dual.cuh"
using D = cdk_dual::Dual<3>;
namespace cdk_user {  // unqualified calls from a user namespace: found by argument-dependent lookup
template <typename T> T all_ops(const T& x, const T& y, int which) {
  switch (which) {
    case 0: return x + y;   case 1: return x - y;   case 2: return x * y;   case 3: return x / y;
    case 4: return -x;      case 5: return 2 * x + 1;  case 6: return 3.5 - x;  case 7: return x * 2.5;
    case 8: return 1.5 / x; case 9: return x / 4;   case 10: return x - 2;  case 11: return 2.0 + x;
    case 12: { T s = x; s += y; s -= 0.5 * x; s *= y; s /= x + 3; s += 1; s -= 2.0; s *= 3; s /= 2.0; return s; }
    case 13: return x < y ? x * x : y * y;
    case 14: return x > 0.5 ? T(2) * x : T(1);
    case 15: return sqrt(x);  case 16: return exp(x);  case 17: return log(x);  case 18: return sin(x);
    case 19: return cos(x);   case 20: return tan(x);  case 21: return tanh(x); case 22: return sinh(x);
    case 23: return cosh(x);  case 24: return atan(x); case 25: return fabs(-x); case 26: return pow(x, 2.5);
    case 27: return pow(y, 3);
    default: return x;
  }
}
}
int main() {
  const double xv = 0.7, yv = 1.9;
  D x(xv), y(yv);
  x.d[0] = 1.0; y.d[1] = 1.0; x.d[2] = 0.5; y.d[2] = -2.0;  // direction 2: (0.5, -2)
  for (int w = 0; w < 28; ++w) {
    D r = cdk_user::all_ops<D>(x, y, w);
    const double v = cdk_user::all_ops<double>(xv, yv, w);
    printf("%d %.17g %.17g %.17g %.17g\n", w, r.v - v, r.d[0], r.d[1], r.d[2]);
  }
  printf("cmp %d %d %d %d %d %d %d\n", x < y, x <= 0.7, 0.7 >= x, y > x, x == 0.7, x != y, 2 > x);
  return 0;
}
'''


def test_dual_numbers_match_analytic_derivatives(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc is not available")
    src = tmp_path / "dual.cu"
    src.write_text(DUAL_PROGRAM)
    exe = tmp_path / "dual"
    r = subprocess.run([nvcc, "-std=c++17", "-I", b.CSRC, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    x, y = 0.7, 1.9
    grads = {0: (1, 1), 1: (1, -1), 2: (y, x), 3: (1 / y, -x / y ** 2), 4: (-1, 0), 5: (2, 0), 6: (-1, 0), 7: (2.5, 0),
             8: (-1.5 / x ** 2, 0), 9: (0.25, 0), 10: (1, 0), 11: (1, 0),
             12: None, 13: (2 * x, 0), 14: (2, 0), 15: (0.5 / np.sqrt(x), 0), 16: (np.exp(x), 0), 17: (1 / x, 0),
             18: (np.cos(x), 0), 19: (-np.sin(x), 0), 20: (1 / np.cos(x) ** 2, 0), 21: (1 - np.tanh(x) ** 2, 0),
             22: (np.cosh(x), 0), 23: (np.sinh(x), 0), 24: (1 / (1 + x * x), 0), 25: (1, 0), 26: (2.5 * x ** 1.5, 0),
             27: (0, 3 * y ** 2)}
    # case 12 by hand: s = (((x + y - x/2) y / (x + 3)) + 1 - 2) * 3 / 2
    u, du_dx, du_dy = (x / 2 + y) * y, 0.5 * y, x / 2 + 2 * y
    grads[12] = (1.5 * (du_dx * (x + 3) - u) / (x + 3) ** 2, 1.5 * du_dy / (x + 3))
    for line, (w, (gx, gy)) in zip(out[:28], sorted(grads.items())):
        k, dv, d0, d1, d2 = line.split()
        assert int(k) == w
        assert float(dv) == 0.0, (w, dv)  # the value is the double evaluation, bit for bit
        for got, want in ((float(d0), gx), (float(d1), gy), (float(d2), 0.5 * gx - 2.0 * gy)):
            assert abs(got - want) <= 1e-14 * max(1.0, abs(want)), (w, got, want)
    assert out[28] == "cmp 1 1 1 1 1 1 1"
