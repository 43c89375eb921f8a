"""Build libcdk.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m cd_dynamax_b200.build [--force]

The built library lives at cd_dynamax_b200/lib/libcdk.so; it is git-ignored but travels to the GPU box.
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
OBJ = os.path.join(PKG, "build")
LIBDIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIBDIR, "libcdk.so")
SOURCES = ["cdk_api.cu", "cdk_small.cu", "cdk_generic.cu", "cdk_enkf.cu", "cdk_kfwarp.cu", "cdk_aux.cu", "cdk_ekfgrad.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", CSRC,
]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(ROOT, "include", "cdk.h"))
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    jobs = []
    for s in srcs:
        src, obj = os.path.join(CSRC, s), os.path.join(OBJ, s.replace(".cu", ".o"))
        if force or _stale(obj, [src] + headers):
            cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append((s, cmd))
    if jobs:
        with concurrent.futures.ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            futs = {ex.submit(subprocess.run, cmd, capture_output=True, text=True): name for name, cmd in jobs}
            for f in concurrent.futures.as_completed(futs):
                r = f.result()
                if verbose or r.returncode != 0:
                    sys.stderr.write(f"--- {futs[f]} ---\n{r.stdout}{r.stderr}\n")
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed on {futs[f]}")
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in srcs]
    if force or jobs or _stale(LIB, objs):
        # -Bsymbolic: the library binds its own symbols internally, so a user-drift VARIANT (same symbol names, loaded next to
        # the stock library) cannot be interposed by it
        cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-ldl",
                                                       "-Xlinker", "-Bsymbolic"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


USER_SOURCES = ["cdk_api.cu", "cdk_generic.cu", "cdk_enkf.cu", "cdk_aux.cu"]  # the units that see the drift registry
USER_GRAD_SOURCES = USER_SOURCES + ["cdk_ekfgrad.cu"]  # ... plus the dense EKF gradient (grad or emission_grad)
USER_KEEP = 24  # variants kept in lib/user, newest first


def variant_key(drift_code=None, emission_code=None, grad=False, emission_grad=False) -> str:
    """Content hash naming the variant of build_variant(drift_code, emission_code, grad, emission_grad=...): the device
    codes (each marked present or absent), the two gradient flags, the library sources and this file."""
    import hashlib
    key = hashlib.sha1()
    for part in (drift_code, emission_code):
        key.update(b"-" if part is None else b"%d:" % len(part.encode()) + part.encode())
    key.update(b"grad" if grad else b"filter")
    if emission_grad:
        key.update(b"emission_grad")
    for f in sorted(os.listdir(CSRC)) + ["../../include/cdk.h", "../build.py"]:
        key.update(open(os.path.join(CSRC, f), "rb").read())
    return key.hexdigest()[:16]


def build_user_drift(device_code: str, grad: bool = False, verbose=False) -> str:
    """Compile a VARIANT of libcdk.so whose drift registry contains CDK_DRIFT_USER = the given CUDA device code
    (SURVEY 8f rank 4: the reference accepts any Python drift callable, cdnlgssm_utils.py:13-36; a CUDA kernel needs device
    code).  `device_code` must define, inside `namespace cdk_user { ... }`:

        template <typename T, class XF> __device__ T f(const T* th, int n, int i, XF x);      // f_i(x; theta); x(j) = x_j
        template <typename T> __device__ T jac(const T* th, int n, int i, int j, const T* x);  // d f_i / d x_j
        template <typename T> __device__ T graddiv(const T* th, int n, int k, const T* x);     // sum_i d2 f_i/dx_i dx_k
                                                                                               // (EKF 'second'; else 0)
    grad=True also compiles the dense EKF gradient (cdk_ekf_grad_dense_f64) for this drift.  It instantiates the three
    templates with T = cdk_dual::Dual<W> (csrc/cdk_dual.cuh), a forward-mode dual number, and takes every derivative the
    reverse pass needs (df/dtheta, dJ/dx, dJ/dtheta, dg/dx, dg/dtheta) from them, so the code must then stay within the
    dual-number contract: arithmetic on T only (+ - * / and unary -, mixed with int / double constants, compound
    assignment, comparisons, T(c)) and the UNQUALIFIED functions sqrt exp log sin cos tan tanh sinh cosh atan fabs
    pow(T, double).  Qualified calls (::sin, std::exp) and intrinsics (__expf) do not compile with the dual type.  The
    cost is n_theta (n^2 + 2n) / W dual drift evaluations per stage VJP: fine for up to about a hundred parameters, the
    wrong mode for thousands.  grad=False builds exactly the filter units, and code that compiles for float / double only
    keeps working there.

    The same as build_variant(device_code, None, grad): see there for the cache and the returned path."""
    return build_variant(device_code, None, grad, verbose)


def build_variant(drift_code=None, emission_code=None, grad: bool = False, verbose=False, emission_grad: bool = False) -> str:
    """Compile a VARIANT of libcdk.so with a user-defined drift (CDK_DRIFT_USER, `drift_code`: see build_user_drift), a
    user-defined emission (CDK_EMISSION_USER, `emission_code`), or both.  `emission_code` must define, inside
    `namespace cdk_user_emission { ... }`, for T = float and double:

        __host__ __device__ int num_params(int n, int m);                                        // n_phi, length of phi
        template <typename T, class XF> __device__ T h(const T* phi, int n, int m, int a, XF x);   // h_a(x; phi); x(j) = x_j
        template <typename T> __device__ T jac(const T* phi, int n, int m, int a, int j, const T* x); // d h_a / d x_j

    num_params may return 0 (an emission without parameters; phi is then [0] or [N, 0]), as a user drift may take
    n_theta = 0 parameters (theta [0]).  grad=True (the drift's dense EKF gradient) needs a drift.

    emission_grad=True also compiles the dense EKF gradient (cdk_ekf_grad_dense_f64) for this emission, the gradient
    with respect to phi included.  It instantiates h and jac with T = cdk_dual::Dual<W> (csrc/cdk_dual.cuh) and takes
    d2h/dx dphi, dJ/dx and dJ/dphi from them, so the emission code must then stay within the dual-number contract that
    build_user_drift states for drifts: arithmetic on T only (+ - * / and unary -, mixed with int / double constants,
    compound assignment, comparisons, T(c)) and the UNQUALIFIED functions sqrt exp log sin cos tan tanh sinh cosh atan
    fabs pow(T, double); num_params stays plain int.  examples/range_emission.cuh and examples/linear_emission.cuh do.
    The cost is (n + n_phi) / W dual evaluations of all m n entries of jac per update VJP: forward mode over phi, so it
    grows with n_phi.  emission_grad needs an emission.

    The gradient unit (cdk_ekfgrad.cu) is compiled when grad or emission_grad is set, and it sees the drift's code only
    with grad and the emission's only with emission_grad: code that is not declared dual-safe never reaches it.  The
    filter units see both codes whatever the flags.

    Returns the path of cd_dynamax_b200/lib/user/libcdk_user_<hash>.so, cached by content hash (variant_key: both codes
    and both flags; ~1 minute of nvcc the first time; the USER_KEEP newest variants are kept).  The variant exports the
    same C ABI (include/cdk.h); the units that do not see the registries (cdk_small.cu, cdk_kfwarp.cu, and cdk_ekfgrad.cu
    unless grad or emission_grad) are linked from the stock build."""
    if drift_code is None and emission_code is None:
        raise ValueError("build_variant needs a drift code, an emission code or both")
    if grad and drift_code is None:
        raise ValueError("grad=True compiles the gradient of a user drift: it needs drift_code")
    if emission_grad and emission_code is None:
        raise ValueError("emission_grad=True compiles the gradient of a user emission: it needs emission_code")
    build()  # the stock objects
    tag = variant_key(drift_code, emission_code, grad, emission_grad)
    udir = os.path.join(LIBDIR, "user")
    os.makedirs(udir, exist_ok=True)
    lib = os.path.join(udir, f"libcdk_user_{tag}.so")
    if os.path.exists(lib):
        return lib
    work = os.path.join(OBJ, f"user_{tag}")
    os.makedirs(work, exist_ok=True)
    flags = {}  # header macro -> (its -D flag, whether the gradient unit sees it)
    for code, name, macro, in_grad in ((drift_code, "cdk_user_drift.cuh", "CDK_USER_DRIFT_HEADER", grad),
                                       (emission_code, "cdk_user_emission.cuh", "CDK_USER_EMISSION_HEADER", emission_grad)):
        if code is None:
            continue
        header = os.path.join(work, name)
        with open(header, "w") as fh:
            fh.write("// generated by cd_dynamax_b200.build.build_variant\n#pragma once\n" + code + "\n")
        flags[macro] = (f'-D{macro}="{header}"', in_grad)
    units = USER_GRAD_SOURCES if grad or emission_grad else USER_SOURCES
    jobs = []
    for s in units:
        src, obj = os.path.join(CSRC, s), os.path.join(work, s.replace(".cu", ".o"))
        unit_flags = [f for f, in_grad in flags.values() if in_grad or s != "cdk_ekfgrad.cu"]
        jobs.append((s, [_nvcc()] + NVCC_FLAGS + unit_flags + ["-c", src, "-o", obj]))
    with concurrent.futures.ThreadPoolExecutor(max_workers=len(jobs)) as ex:
        futs = {ex.submit(subprocess.run, cmd, capture_output=True, text=True): name for name, cmd in jobs}
        for f in concurrent.futures.as_completed(futs):
            r = f.result()
            if verbose or r.returncode != 0:
                sys.stderr.write(f"--- {futs[f]} ---\n{r.stdout}{r.stderr}\n")
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {futs[f]} (user device code):\n{r.stderr[-4000:]}")
    objs = [os.path.join(work, s.replace(".cu", ".o")) for s in units]
    objs += [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES if s not in units]
    tmp = lib + ".tmp"
    r = subprocess.run([_nvcc(), "-shared", "-o", tmp] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-ldl",
                                                                "-Xlinker", "-Bsymbolic"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed (user device code):\n" + r.stdout + r.stderr)
    os.replace(tmp, lib)
    # housekeeping: every change of the sources or of the device code is a new content hash; keep the newest variants
    old = sorted((f for f in os.listdir(udir) if f.startswith("libcdk_user_") and f.endswith(".so")),
                 key=lambda f: os.path.getmtime(os.path.join(udir, f)), reverse=True)[USER_KEEP:]
    for f in old:
        os.remove(os.path.join(udir, f))
        shutil.rmtree(os.path.join(OBJ, "user_" + f[len("libcdk_user_"):-3]), ignore_errors=True)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
