"""Host-side marshalling between the reference-shaped Python API and the C ABI (include/cdk.h).

PyTorch is used only for device memory, streams and host<->device copies.  All arithmetic happens in libcdk.so.
"""
import ctypes
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _lib as L

_TORCH_DT = {"f64": torch.float64, "f32": torch.float32}
_NP_DT = {"f64": np.float64, "f32": np.float32}

# core (per-trajectory) rank of every input slot
_CORE_NDIM = {L.IN_Y: 2, L.IN_T: 1, L.IN_U: 2, L.IN_M0: 1, L.IN_P0: 2, L.IN_F: None, L.IN_B: 1, L.IN_BU: 2,
              L.IN_L: 2, L.IN_QC: 2, L.IN_H: 2, L.IN_D: 1, L.IN_DU: 2, L.IN_R: 2, L.IN_FM: 2, L.IN_FP: 3}
_SLOT_NAMES = {L.IN_Y: "IN_Y", L.IN_T: "IN_T", L.IN_U: "IN_U", L.IN_M0: "IN_M0", L.IN_P0: "IN_P0", L.IN_F: "IN_F",
               L.IN_B: "IN_B", L.IN_BU: "IN_BU", L.IN_L: "IN_L", L.IN_QC: "IN_QC", L.IN_H: "IN_H", L.IN_D: "IN_D",
               L.IN_DU: "IN_DU", L.IN_R: "IN_R", L.IN_FM: "IN_FM", L.IN_FP: "IN_FP"}


def _core_shapes(K: int, n: int, m: int, desc_fields: dict, theta_core_ndim: int) -> dict:
    """Per-trajectory shape of every input slot: exactly the slot_elems (cdk_api.cu) entries a kernel reads from it."""
    flags = int(desc_fields.get("flags", 0))
    d_u = int(desc_fields.get("d_u", 0))
    # a user emission (CDK_EMISSION_USER) reads its parameter vector phi [n_phi] from the H slot
    h_shape = (int(desc_fields["n_phi"]),) if int(desc_fields.get("emission_id", 0)) == L.EMISSION_USER else (m, n)
    # a forecast and a sampler started from a fixed state read K + 1 time stamps (t_init first), every other entry point K
    t_cols = K + 1 if flags & (L.FLAG_PREDICT_ONLY | L.FLAG_FIXED_INIT) else K
    return {
        L.IN_Y: (K, m), L.IN_T: (t_cols,), L.IN_U: (K, d_u), L.IN_M0: (n,), L.IN_P0: (n, n),
        L.IN_F: (n, n) if theta_core_ndim == 2 else (int(desc_fields.get("n_theta", 0)),),
        L.IN_B: (n,), L.IN_BU: (n, d_u), L.IN_L: (n, n), L.IN_QC: (n, n), L.IN_H: h_shape, L.IN_D: (m,),
        L.IN_DU: (m, d_u), L.IN_R: (m,) if flags & L.FLAG_DIAG_R else (m, m), L.IN_FM: (K, n), L.IN_FP: (K, n, n),
    }


def device():
    if not torch.cuda.is_available():
        raise RuntimeError("cd_dynamax_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def kind_of(x):
    """How the caller holds its data: 'cuda' (torch tensor on the GPU), 'torch' (torch CPU tensor) or 'numpy'."""
    if isinstance(x, torch.Tensor):
        return "cuda" if x.is_cuda else "torch"
    return "numpy"


def pick_dtype(x) -> str:
    """float32 data runs the fp32 kernels, everything else the fp64 kernels (the reference computes in the dtype of
    its inputs: fp32 unless jax_enable_x64, SURVEY F6)."""
    dt = x.dtype if hasattr(x, "dtype") else np.asarray(x).dtype
    return "f32" if dt in (torch.float32, np.float32, np.dtype("float32")) else "f64"


def to_dev(x, dt: str, dev) -> torch.Tensor:
    tdt = _TORCH_DT[dt]
    if isinstance(x, torch.Tensor):
        return x.to(device=dev, dtype=tdt, non_blocking=True).contiguous()
    if hasattr(x, "__cuda_array_interface__"):
        return torch.as_tensor(x, device=dev).to(tdt).contiguous()
    arr = np.ascontiguousarray(np.asarray(x), dtype=_NP_DT[dt])
    return torch.from_numpy(arr).to(dev, non_blocking=True)


def from_dev(t: Optional[torch.Tensor], kind: str):
    """Hand a result back in the caller's array kind (`t` may already be a host tensor, see run(host_out=True))."""
    if t is None:
        return None
    if kind == "cuda":
        return t
    if kind == "torch":
        return t.cpu()
    return t.cpu().numpy()


# Host-resident batched inputs larger than this are staged in N-chunks: chunk i+1 crosses PCIe on a copy stream while the
# kernels of earlier chunks run (and their results return on a third stream).  Trajectories are independent, so a chunk
# is just the same entry point with offset pointers and a smaller N.  The chunk kernels go to a small pool of compute
# streams so that they overlap EACH OTHER as well: one trajectory is a serial chain of K steps, so a chunk of N/8
# trajectories takes almost as long as the whole batch (the GPU is a single wave either way) and back-to-back chunk
# kernels would serialise that latency.
# Per-trajectory status of the kernels (include/cdk.h): 0 ok, 1 non-finite result (the reference's silent NaN), 2 the
# solver hit max_steps -- where diffrax RAISES ("The maximum number of solver steps was reached", diffeqsolve's default
# throw=True).  Host callers already wait for their results, so the check is free there and status 2 raises as upstream
# does; device-resident callers stay asynchronous and can inspect `last_status()` (a device tensor) themselves.
RAISE_ON_MAX_STEPS = True
_last_status = None


def last_status():
    """int32 [N] status tensor of the most recent kernel call in this process (device or pinned host memory)."""
    return _last_status


class MaxStepsReached(RuntimeError):
    pass


STREAM_MIN_BYTES = 32 << 20
STREAM_CHUNKS = 8
COMPUTE_STREAMS = 4
_side_streams: Dict[int, tuple] = {}


def _streams(dev):
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _side_streams:
        _side_streams[key] = (torch.cuda.Stream(dev), torch.cuda.Stream(dev),
                              [torch.cuda.Stream(dev) for _ in range(COMPUTE_STREAMS)])
    return _side_streams[key]


def _is_host(x) -> bool:
    if isinstance(x, torch.Tensor):
        return not x.is_cuda
    return not hasattr(x, "__cuda_array_interface__")


def _host_tensor(x, dt: str) -> torch.Tensor:
    """Host array-like -> contiguous CPU tensor of the kernel dtype (no copy when it already is one, so a pinned
    buffer stays pinned)."""
    if isinstance(x, torch.Tensor):
        return x.to(dtype=_TORCH_DT[dt]).contiguous()
    return torch.from_numpy(np.ascontiguousarray(np.asarray(x), dtype=_NP_DT[dt]))


def classify(N: int, K: int, n: int, m: int, inputs: Dict[int, object], desc_fields: dict, theta_core_ndim: int = 1,
             core_ndim_override: Optional[dict] = None):
    """The host-side half of `run`, which touches no device: check every input slot against the per-trajectory shape
    its kernels read and tell shared from batched (leading N) inputs.  -> ({slot: (array, batched, row elements, host?)},
    batched_mask).  Raises ValueError, naming the slot, on any other shape."""
    core_shape = _core_shapes(K, n, m, desc_fields, theta_core_ndim)
    if int(desc_fields.get("emission_id", 0)) == L.EMISSION_USER:
        core_ndim_override = {**(core_ndim_override or {}), L.IN_H: 1}
    metas = {}
    mask = 0
    for slot in range(L.NUM_IN):
        x = inputs.get(slot)
        if x is None:
            continue
        shape = full_shape = tuple(x.shape) if hasattr(x, "shape") else tuple(np.shape(x))
        core = _CORE_NDIM[slot] if _CORE_NDIM[slot] is not None else theta_core_ndim
        if core_ndim_override and slot in core_ndim_override:
            core = core_ndim_override[slot]  # e.g. IN_R as the [m] diagonal (CDK_FLAG_DIAG_R)
        batched = len(shape) == core + 1
        if batched and shape[0] == 1 and N > 1:
            # a leading axis of length 1 is a shared (broadcast) input: `t_emissions=None` or one [K, 1] time grid for
            # a whole batch of emissions, shared `inputs` -- what vmap(..., in_axes=None) does in the reference
            x, shape, batched = x[0], shape[1:], False
        if batched:
            if shape[0] != N:
                raise ValueError(f"input slot {_SLOT_NAMES[slot]}: leading axis {shape[0]} != N={N} "
                                 f"(full shape {full_shape})")
            mask |= 1 << slot
        elif len(shape) != core:
            raise ValueError(f"input slot {_SLOT_NAMES[slot]}: expected rank {core} or {core + 1}, got shape {shape}")
        if tuple(shape[1:] if batched else shape) != core_shape[slot]:
            raise ValueError(f"input slot {_SLOT_NAMES[slot]}: per-trajectory shape {tuple(shape[1:] if batched else shape)} "
                             f"!= {core_shape[slot]} (full shape {full_shape}, N={N}, K={K})")
        row = int(np.prod(shape[1:], dtype=np.int64)) if batched else 0
        metas[slot] = (x, batched, row, _is_host(x))
    return metas, mask


def run(entry: str, dt: str, N: int, K: int, n: int, m: int, inputs: Dict[int, object], want: Sequence[int],
        desc_fields: dict, theta_core_ndim: int = 1, scross_rows: Optional[int] = None,
        status: Optional[torch.Tensor] = None, host_out: bool = False,
        dev_inputs: Optional[dict] = None, scratch: Optional[torch.Tensor] = None,
        core_ndim_override: Optional[dict] = None,
        out_shapes: Optional[dict] = None) -> Dict[int, torch.Tensor]:
    """Call one C-ABI entry point. `inputs` maps slot -> array-like (None = absent); a leading N marks it batched.
    Every slot must have the per-trajectory shape the kernels read (`_core_shapes`: [K] time stamps, [K + 1] for a
    forecast or a sampler from a fixed initial state, [K, m] emissions, [n, n] covariances, [n_theta] drift parameters,
    ...); anything else raises ValueError before any device work.
    Returns slot -> tensor for every slot in `want` (+ OUT_STATUS): device tensors, or -- with `host_out`, which the
    API shims set when the caller handed in host arrays -- pinned host tensors whose copies have completed.
    `dev_inputs`, when given, receives slot -> staged device tensor (a smoother reuses the filter's staged inputs).
    `desc_fields["flags"]` sets the CDK_FLAG_* bits (desc.reserved[2]); when the entry point then asks for device scratch
    (cdk_scratch_bytes, sized per trajectory) it is allocated here -- or taken from `scratch`, which is how the type-1
    smoother gets the pushforward cache its filter wrote -- and returned as out[OUT_SCRATCH]."""
    desc_fields = dict(desc_fields)
    tdt = _TORCH_DT[dt]
    esz = 8 if dt == "f64" else 4
    # ---- classify inputs (before any device work: a mis-shaped batch is rejected here, not read out of bounds) ----
    metas, mask = classify(N, K, n, m, inputs, desc_fields, theta_core_ndim, core_ndim_override)
    stream_bytes = sum(N * row * esz for _, batched, row, host in metas.values() if batched and host)
    lib = L.lib(desc_fields.pop("lib_path", None))  # a variant library for user device code, else the stock one
    desc_fields.pop("n_phi", None)  # the kernels take it from the library's own num_params
    dev = device()
    d = L.new_desc()
    d.N, d.K, d.n, d.m = N, K, n, m
    for k, v in desc_fields.items():
        if k == "flags":
            d.reserved[2] = int(v)
        elif k == "grad_groups":
            d.reserved[3] = int(v)
        else:
            setattr(d, k, v)
    cur = torch.cuda.current_stream(dev)
    d.batched_mask = mask
    nchunks = STREAM_CHUNKS if (stream_bytes >= STREAM_MIN_BYTES and N >= 2 * STREAM_CHUNKS) else 1
    if host_out and N >= 2 * STREAM_CHUNKS:
        out_bytes = sum(int(np.prod(out_shapes[s] if out_shapes and s in out_shapes else
                                    _out_shape(s, N, K, n, scross_rows, int(desc_fields.get("n_theta", 0))),
                                    dtype=np.int64)) * esz for s in want)
        if out_bytes >= STREAM_MIN_BYTES:
            nchunks = STREAM_CHUNKS
    h2d, d2h, comp = _streams(dev) if (nchunks > 1 or host_out) else (None, None, None)
    # ---- stage inputs ----
    keep = []
    dev_in = {}
    staged = {}  # slot -> (host tensor, device tensor) copied chunk by chunk
    for slot, (x, batched, row, host) in metas.items():
        if nchunks > 1 and batched and host:
            ht = _host_tensor(x, dt)
            dtens = torch.empty(ht.shape, dtype=tdt, device=dev)
            staged[slot] = (ht, dtens)
            dev_in[slot] = dtens
        else:
            dev_in[slot] = to_dev(x, dt, dev)
        keep.append(dev_in[slot])
    if dev_inputs is not None:
        dev_inputs.update(dev_in)
    # ---- outputs ----
    out = {}
    for slot in want:
        shp = out_shapes[slot] if out_shapes and slot in out_shapes else \
            _out_shape(slot, N, K, n, scross_rows, int(desc_fields.get("n_theta", 0)))
        out[slot] = torch.empty(shp, dtype=tdt, device=dev)
    if status is None:
        status = torch.zeros((N,), dtype=torch.int32, device=dev)
    out[L.OUT_STATUS] = status
    hout = {}
    if host_out:
        for slot, t in out.items():
            hout[slot] = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    fn = getattr(lib, f"{entry}_{dt}")
    # device scratch is sized per trajectory (today: the CD-KF pushforward cache), so chunks just offset into it
    d.N = 1
    scratch_row = int(lib.cdk_scratch_bytes(ctypes.byref(d), entry.encode())) if N > 0 else 0
    d.N = N
    if scratch_row:
        if scratch is None or scratch.numel() < N * scratch_row:
            scratch = torch.empty((N * scratch_row,), dtype=torch.uint8, device=dev)
        keep.append(scratch)
    bounds = [(N * c) // nchunks for c in range(nchunks + 1)]
    rng_offset0 = int(d.rng_offset)
    if nchunks > 1:
        h2d.wait_stream(cur)  # staged device buffers were allocated on `cur`
        for cs in comp:
            cs.wait_stream(cur)
    if host_out:
        d2h.wait_stream(cur)
    for c in range(nchunks):
        lo, hi = bounds[c], bounds[c + 1]
        if hi == lo:
            continue
        ks = comp[c % COMPUTE_STREAMS] if nchunks > 1 else cur  # the stream this chunk's kernel runs on
        if staged:
            with torch.cuda.stream(h2d):
                for ht, dtens in staged.values():
                    dtens[lo:hi].copy_(ht[lo:hi], non_blocking=True)
            ks.wait_stream(h2d)
        d.N = hi - lo
        d.rng_offset = rng_offset0 + lo
        in_ptrs = (ctypes.c_void_p * L.NUM_IN)()
        for slot in range(L.NUM_IN):
            in_ptrs[slot] = None
        for slot, t in dev_in.items():
            if t.numel() > 0:
                _, batched, row, _ = metas[slot]
                in_ptrs[slot] = t.data_ptr() + (lo * row * esz if batched else 0)
        out_ptrs = (ctypes.c_void_p * L.NUM_OUT)()
        for slot in range(L.NUM_OUT):
            out_ptrs[slot] = None
        for slot, t in out.items():
            if t.numel() > 0:
                out_ptrs[slot] = t.data_ptr() + lo * (t.numel() // N) * t.element_size()
        if scratch_row:
            out_ptrs[L.OUT_SCRATCH] = scratch.data_ptr() + lo * scratch_row
        rc = fn(ctypes.byref(d), in_ptrs, out_ptrs, ctypes.c_void_p(ks.cuda_stream))
        if rc != 0:
            raise L.CdkError(f"{entry}_{dt} failed with code {rc}: {lib.cdk_last_error().decode()}")
        if host_out:
            d2h.wait_stream(ks)
            with torch.cuda.stream(d2h):
                for slot, t in out.items():
                    hout[slot][lo:hi].copy_(t[lo:hi], non_blocking=True)
    if nchunks > 1:
        for cs in comp:
            cur.wait_stream(cs)  # the caller's stream sees the finished outputs
    if nchunks > 1 or host_out:
        for t in keep + list(out.values()):
            for st in [h2d, d2h] + (comp if nchunks > 1 else []):
                t.record_stream(st)
    global _last_status
    if host_out:
        d2h.synchronize()
        _last_status = hout[L.OUT_STATUS]
        if RAISE_ON_MAX_STEPS and N > 0 and bool((hout[L.OUT_STATUS] == 2).any()):
            bad = int((hout[L.OUT_STATUS] == 2).sum())
            raise MaxStepsReached(f"{entry}: the maximum number of solver steps (max_steps={int(d.max_steps)}) was reached "
                                  f"in {bad} of {N} trajectories; increase diffeqsolve_settings['max_steps'] or dt0")
        if scratch_row:
            hout[L.OUT_SCRATCH] = scratch
        return hout
    _last_status = status
    # staged inputs / scratch were allocated on this stream: the caching allocator keeps them valid until the kernel
    # has consumed them (stream-ordered reuse), so dropping `keep` here is safe.
    del keep
    if scratch_row:
        out[L.OUT_SCRATCH] = scratch
    return out


def _out_shape(slot, N, K, n, scross_rows=None, n_theta=0):
    return {
        L.OUT_GRAD: (N, L.GRAD_COLS_L63),
        L.OUT_LL: (N,), L.OUT_FM: (N, K, n), L.OUT_FP: (N, K, n, n), L.OUT_PM: (N, K, n), L.OUT_PP: (N, K, n, n),
        L.OUT_LLCUM: (N, K), L.OUT_SM: (N, K, n), L.OUT_SP: (N, K, n, n),
        L.OUT_SCROSS: (N, max(K - 1, 0) if scross_rows is None else scross_rows, n, n), L.OUT_STATUS: (N,),
    }[slot]


def ll_sum(ll: torch.Tensor) -> torch.Tensor:
    """Deterministic on-device sum of per-trajectory log-likelihoods -> float64 scalar tensor
    (`vmap(marginal_log_prob)(...).sum()`, src/ssm_temissions.py:555-567)."""
    lib = L.lib()
    out = torch.empty((1,), dtype=torch.float64, device=ll.device)
    fn = lib.cdk_ll_sum_f64 if ll.dtype == torch.float64 else lib.cdk_ll_sum_f32
    stream = torch.cuda.current_stream(ll.device).cuda_stream
    L.check(fn(ctypes.c_void_p(ll.data_ptr()), ll.numel(), ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(stream)),
            "cdk_ll_sum")
    return out


# ---- diffeqsolve_settings -> {solver, dt0, max_steps} -----------------------------------------------------------------
def parse_settings(settings: Optional[dict], sde: bool = False) -> dict:
    """Map the reference's `diffeqsolve_settings` dict (forwarded verbatim to diffrax, src/utils/diffrax_utils.py:40-57)
    onto the fixed-step solver registry.  Unsupported settings are rejected loudly."""
    settings = dict(settings or {})
    solver = settings.pop("solver", None)
    if solver is None:
        name = "heun" if sde else "dopri5"  # diffrax_utils.py:121-127
    elif isinstance(solver, str):
        name = solver.lower()
    else:
        name = type(solver).__name__.lower()  # works for diffrax solver instances and cd_dynamax_b200.solvers
    if name not in L.SOLVERS:
        raise NotImplementedError(f"solver {name!r} is not in the fixed-step registry {sorted(L.SOLVERS)}")
    ctrl = settings.pop("stepsize_controller", None)
    if ctrl is not None and type(ctrl).__name__ != "ConstantStepSize":
        raise NotImplementedError("only diffrax.ConstantStepSize is supported (adaptive PID controllers are not)")
    settings.pop("adjoint", None)  # gradient checkpointing strategy: irrelevant without autodiff
    settings.pop("tol_vbt", None)
    settings.pop("debug", None)
    dt0 = float(settings.pop("dt0", 0.01))
    max_steps = int(settings.pop("max_steps", 1e5))
    if settings:
        raise NotImplementedError(f"unsupported diffeqsolve_settings: {sorted(settings)}")
    return {"solver": L.SOLVERS[name], "dt0": dt0, "max_steps": max_steps}
