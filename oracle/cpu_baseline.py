"""ctypes loader + timing harness for the C restatement (oracle/cd_oracle_c.c).  Test / baseline infrastructure only."""
import ctypes
import os
import subprocess
import tempfile
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "cd_oracle_c.c")
SO = os.path.join(HERE, "_build", "libcdoracle.so")
SOLVER_IDS = {"euler": 0, "heun": 1, "midpoint": 2, "ralston": 3, "bosh3": 4, "rk4": 5, "dopri5": 6}
_lib = None
_so = None  # the library load() opened


def _fresh(so):
    """The library at `so` is newer than the source and was built on a CPU of this model (see build())."""
    try:
        return os.path.getmtime(so) >= os.path.getmtime(SRC) and open(so + ".host").read() == _host_tag()
    except OSError:
        return False


def build(force=False, out_dir=os.path.dirname(SO)):
    """gcc -O3 -march=native -fopenmp into out_dir/libcdoracle.so.  -march=native binds the .so to the build host's ISA,
    so a marker next to it records the CPU model it was built on, and load() rebuilds it if the CPU differs."""
    so = os.path.join(out_dir, "libcdoracle.so")
    if force or not _fresh(so):
        # an exported CC may name a compiler without libgomp: prefer the system gcc, fall back to a serial build
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        make = ["make", "-C", HERE, "-B", f"BUILD={out_dir}", so, f"CC={cc}"]
        r = subprocess.run(make, capture_output=True, text=True)
        if r.returncode != 0:
            r = subprocess.run(make + ["CFLAGS=-O3 -fPIC -std=gnu11"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("building oracle/cd_oracle_c.c failed:\n" + r.stdout + r.stderr)
        with open(so + ".host", "w") as f:
            f.write(_host_tag())
    return so


def load():
    """Open the library build() left in the tree; if it is missing or was built for another CPU, build a private copy in
    the temporary directory instead, so that a read-only checkout works too."""
    global _lib, _so
    if _lib is None:
        _so = SO if _fresh(SO) else build(out_dir=os.path.join(tempfile.gettempdir(), f"cd_oracle_{os.getuid()}"))
        L = ctypes.CDLL(_so)
        dp, i, ll, d = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_double
        L.cdo_filter.argtypes = [i, ll, i, i, i, i, i, d, d, i, i] + [dp] * 11 + [dp] * 5 + [i]
        L.cdo_filter.restype = ll
        L.cdo_max_threads.restype = i
        _lib = L
    return _lib


def _has_openmp():
    try:
        return b"GOMP" in open(_so, "rb").read()
    except OSError:
        return False


def _host_tag():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def filter_c(algo, Y, T, m0, P0, theta, Lm, Qc, H, d, R, drift_id=0, solver="rk4", dt0=0.01, dt_final=1e-10,
             max_steps=100000, num_iter=1, bias=None, outputs=True, threads=0):
    """algo 'ekf' | 'kf'.  Shared parameters, batched data.  Returns dict like the NumPy oracle + 'substeps'."""
    L = load()
    c = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    Y, T, m0, P0, theta, Lm, Qc, H, d, R = map(c, (Y, T, m0, P0, theta, Lm, Qc, H, d, R))
    bias = None if bias is None else c(bias)
    N, K, m = Y.shape
    n = m0.shape[0]
    LL = np.empty(N)
    FM = np.empty((N, K, n)) if outputs else None
    FP = np.empty((N, K, n, n)) if outputs else None
    PM = np.empty((N, K, n)) if outputs else None
    PP = np.empty((N, K, n, n)) if outputs else None
    sub = L.cdo_filter(0 if algo == "ekf" else 1, N, K, n, m, drift_id, SOLVER_IDS[solver], dt0, dt_final, max_steps,
                       num_iter, _p(Y), _p(T), _p(m0), _p(P0), _p(theta), _p(bias), _p(Lm), _p(Qc), _p(H), _p(d), _p(R),
                       _p(LL), _p(FM), _p(FP), _p(PM), _p(PP), threads)
    if sub < 0:
        raise ValueError("cdo_filter rejected its arguments")
    return dict(marginal_loglik=LL, filtered_means=FM, filtered_covariances=FP, predicted_means=PM,
                predicted_covariances=PP, substeps=sub)


def time_ekf_l63(n_traj, K, cfg, steps=2, warmup=1):
    """BASELINE config 3 workload on the host cores: returns obs-steps/s with the core count."""
    L = load()
    rng = np.random.Generator(np.random.PCG64(cfg["seed"]))
    gaps = cfg["mean_gap"] * rng.uniform(0.5, 1.5, size=(n_traj, K))
    gaps[:, 0] = 0.0
    T = np.cumsum(gaps, axis=1)
    Y = 8.0 * rng.standard_normal((n_traj, K, 1))
    args = dict(m0=np.zeros(3), P0=5 * np.eye(3), theta=np.array([10.0, 28.0, 8.0 / 3.0]), Lm=np.eye(3), Qc=np.eye(3),
                H=np.array([[1.0, 0.0, 0.0]]), d=np.zeros(1), R=np.eye(1), drift_id=1, solver=cfg["solver"],
                dt0=cfg["dt0"])
    # all the host threads this process may use, set explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers,
    # which would silently turn the multi-threaded baseline into a single-core one at N > 1 GPUs
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    for _ in range(warmup):
        filter_c("ekf", Y, T, threads=cores, **args)
    t0 = time.perf_counter()
    for _ in range(steps):
        r = filter_c("ekf", Y, T, threads=cores, **args)
    el = time.perf_counter() - t0
    t0 = time.perf_counter()
    filter_c("ekf", Y, T, threads=cores, outputs=False, **args)  # log-likelihood only (what fit_sgd consumes)
    el_ll = time.perf_counter() - t0
    if L.cdo_max_threads() == 1 and cores > 1 and not _has_openmp():
        cores = 1  # serial fallback build (no libgomp)
    return {"value": n_traj * K * steps / el, "value_ll_only": n_traj * K / el_ll, "ms_per_step": 1e3 * el / steps,
            "cores": cores, "kind": "port",
            "sample": f"N={n_traj} of the workload's trajectories x K={K}, {steps} passes, C + OpenMP "
                      f"({cores} threads), naive dense arithmetic as in the reference"}
