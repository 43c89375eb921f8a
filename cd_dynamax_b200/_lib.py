"""ctypes binding of libcdk.so (include/cdk.h). No CPU fallback: importing fails loudly when the library is missing."""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libcdk.so")

NUM_IN, NUM_OUT = 16, 12
(IN_Y, IN_T, IN_U, IN_M0, IN_P0, IN_F, IN_B, IN_BU, IN_L, IN_QC, IN_H, IN_D, IN_DU, IN_R, IN_FM, IN_FP) = range(16)
(OUT_LL, OUT_FM, OUT_FP, OUT_PM, OUT_PP, OUT_LLCUM, OUT_SM, OUT_SP, OUT_SCROSS, OUT_STATUS, OUT_SCRATCH,
 OUT_GRAD) = range(12)
SOLVERS = {"euler": 0, "heun": 1, "midpoint": 2, "ralston": 3, "bosh3": 4, "rk4": 5, "dopri5": 6}
DRIFT_LINEAR, DRIFT_LORENZ63, DRIFT_LORENZ96, DRIFT_QUADRATIC, DRIFT_USER = 0, 1, 2, 3, 4
EMISSION_LINEAR, EMISSION_USER = 0, 1
ORDERS = {"zeroth": 0, "first": 1, "second": 2}
FLAG_KEEP_PUSHFORWARD = 1  # CDK_FLAG_KEEP_PUSHFORWARD (desc.reserved[2])
FLAG_UKF_SIGMA_POINTS = 2  # CDK_FLAG_UKF_SIGMA_POINTS
FLAG_DIAG_R = 4  # CDK_FLAG_DIAG_R: in[IN_R] is the [m] diagonal of the emission covariance
FLAG_PREDICT_ONLY = 8  # CDK_FLAG_PREDICT_ONLY: forecast (no updates), in[IN_T] is [N, K+1]
FLAG_FIXED_INIT = 16  # CDK_FLAG_FIXED_INIT: cdk_sample_path starts from in[IN_M0] at t_init
GRAD_COLS_L63 = 23  # CDK_GRAD_COLS_L63: columns of out[CDK_OUT_GRAD]
GRAD_REVERSE = 128  # CDK_GRAD_REVERSE (desc.reserved[3] bit 7)


def grad_cols_kf(n, m):
    """CDK_GRAD_COLS_KF(n, m): columns of out[CDK_OUT_GRAD] of cdk_kf_grad_f64."""
    return 3 * n * n + m * n + m * m + 2 * n + m


def grad_cols_ekf(n, m, n_theta):
    """CDK_GRAD_COLS_EKF(n, m, n_theta): columns of out[CDK_OUT_GRAD] of cdk_ekf_grad_dense_f64, cdk_ukf_grad_dense_f64 and
    cdk_ukf_grad_sigma_f64."""
    return n_theta + 2 * n * n + m * n + m * m + n + m


def grad_cols_ekf_ue(n, m, n_theta, n_phi):
    """CDK_GRAD_COLS_EKF_UE(n, m, n_theta, n_phi): columns of out[CDK_OUT_GRAD] of cdk_ekf_grad_dense_f64 with a user
    emission (phi in place of H | d)."""
    return n_theta + 2 * n * n + n_phi + m * m + n


ENTRY_POINTS = [f"cdk_{a}_{d}_{t}" for a, d in (("kf", "filter"), ("kf", "smooth"), ("ekf", "filter"), ("ekf", "smooth"),
                                                  ("ukf", "filter"), ("enkf", "filter")) for t in ("f64", "f32")]
ENTRY_POINTS.append("cdk_ekf_grad_f64")
ENTRY_POINTS.append("cdk_kf_grad_f64")
ENTRY_POINTS.append("cdk_ekf_grad_dense_f64")
ENTRY_POINTS.append("cdk_ukf_grad_dense_f64")
ENTRY_POINTS.append("cdk_ukf_grad_sigma_f64")
ENTRY_POINTS += ["cdk_sample_path_f64", "cdk_sample_path_f32", "cdk_emission_moments_f64", "cdk_emission_moments_f32"]
OTHER_SYMBOLS = ["cdk_desc_init", "cdk_scratch_bytes", "cdk_ll_sum_f64", "cdk_ll_sum_f32", "cdk_ll_allreduce",
                 "cdk_xla_custom_call", "cdk_xla_custom_call_status", "cdk_xla_last_rc", "cdk_fma_probe_f64", "cdk_fma_probe_f32", "cdk_fma3_probe_f64", "cdk_dmma_probe_f64", "cdk_rng_probe_f64", "cdk_launch_count", "cdk_debug_set_trace", "cdk_has_user_drift", "cdk_has_user_emission", "cdk_user_emission_params", "cdk_version",
                 "cdk_last_error"]


class CdkDesc(ctypes.Structure):
    """Mirror of `struct cdk_desc` (include/cdk.h)."""
    _fields_ = [
        ("struct_size", ctypes.c_int32), ("K", ctypes.c_int32), ("N", ctypes.c_int64), ("n", ctypes.c_int32),
        ("m", ctypes.c_int32), ("d_u", ctypes.c_int32), ("E", ctypes.c_int32), ("solver", ctypes.c_int32),
        ("max_steps", ctypes.c_int32), ("dt0", ctypes.c_double), ("dt_final", ctypes.c_double),
        ("state_order", ctypes.c_int32), ("num_iter", ctypes.c_int32), ("smoother_type", ctypes.c_int32),
        ("drift_id", ctypes.c_int32), ("emission_id", ctypes.c_int32), ("n_theta", ctypes.c_int32),
        ("batched_mask", ctypes.c_uint32), ("perturb_measurements", ctypes.c_int32),
        ("cov_rescaling", ctypes.c_double), ("alpha", ctypes.c_double), ("beta", ctypes.c_double),
        ("kappa", ctypes.c_double), ("rng_seed", ctypes.c_uint64), ("rng_offset", ctypes.c_uint64),
        ("reserved", ctypes.c_int32 * 4),
    ]


class CdkError(RuntimeError):
    pass


_lib = None
_variants = {}


def lib(path=None):
    """Load libcdk.so once (or, with `path`, a variant built by build.build_variant: same ABI, a user drift and / or
    emission compiled in). Raises (never falls back) if the CUDA extension has not been built."""
    global _lib
    if path is None and _lib is not None:
        return _lib
    if path is not None and path in _variants:
        return _variants[path]
    target = path or LIB_PATH
    if not os.path.exists(target):
        raise ImportError(
            f"{target} is missing: build the CUDA extension first (python -m cd_dynamax_b200.build). "
            "cd_dynamax_b200 has no CPU fallback.")
    L = ctypes.CDLL(target, mode=ctypes.RTLD_GLOBAL if path is None else ctypes.RTLD_LOCAL)
    pp = ctypes.POINTER(ctypes.c_void_p)
    for name in ENTRY_POINTS:
        fn = getattr(L, name)
        fn.argtypes = [ctypes.POINTER(CdkDesc), pp, pp, ctypes.c_void_p]
        fn.restype = ctypes.c_int
    L.cdk_desc_init.argtypes = [ctypes.POINTER(CdkDesc)]
    L.cdk_desc_init.restype = None
    L.cdk_scratch_bytes.argtypes = [ctypes.POINTER(CdkDesc), ctypes.c_char_p]
    L.cdk_scratch_bytes.restype = ctypes.c_size_t
    for name in ("cdk_ll_sum_f64", "cdk_ll_sum_f32"):
        fn = getattr(L, name)
        fn.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
        fn.restype = ctypes.c_int
    L.cdk_ll_allreduce.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    L.cdk_ll_allreduce.restype = ctypes.c_int
    for name in ("cdk_fma_probe_f64", "cdk_fma_probe_f32", "cdk_dmma_probe_f64"):
        fn = getattr(L, name)
        fn.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        fn.restype = ctypes.c_int
    L.cdk_rng_probe_f64.argtypes = [ctypes.c_int64, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint64,
                                    ctypes.c_void_p, ctypes.c_void_p]
    L.cdk_rng_probe_f64.restype = ctypes.c_int
    L.cdk_fma3_probe_f64.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    L.cdk_fma3_probe_f64.restype = ctypes.c_int
    L.cdk_xla_custom_call.argtypes = [ctypes.c_void_p, pp, ctypes.c_char_p, ctypes.c_size_t]
    L.cdk_xla_custom_call.restype = None
    L.cdk_xla_custom_call_status.argtypes = [ctypes.c_void_p, pp, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p]
    L.cdk_xla_custom_call_status.restype = None
    L.cdk_xla_last_rc.restype = ctypes.c_int
    L.cdk_debug_set_trace.argtypes = [ctypes.c_void_p]
    L.cdk_debug_set_trace.restype = ctypes.c_int
    L.cdk_launch_count.restype = ctypes.c_int64
    L.cdk_version.restype = ctypes.c_int
    L.cdk_last_error.restype = ctypes.c_char_p
    assert ctypes.sizeof(CdkDesc) == _c_sizeof_desc(L), "cdk_desc layout mismatch between Python and C"
    L.cdk_has_user_drift.restype = ctypes.c_int
    L.cdk_has_user_emission.restype = ctypes.c_int
    L.cdk_user_emission_params.argtypes = [ctypes.c_int, ctypes.c_int]
    L.cdk_user_emission_params.restype = ctypes.c_int
    if path is None:
        _lib = L
    else:
        _variants[path] = L
    return L


def _c_sizeof_desc(L):
    d = CdkDesc()
    L.cdk_desc_init(ctypes.byref(d))
    return d.struct_size


def new_desc():
    d = CdkDesc()
    lib().cdk_desc_init(ctypes.byref(d))
    return d


def check(rc, what):
    if rc != 0:
        raise CdkError(f"{what} failed with code {rc}: {lib().cdk_last_error().decode()}")
