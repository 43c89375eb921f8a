"""The kernels' stepping rule (StepClock, csrc/cdk_common.cuh) compiled for the host and run on the time grids of
test_gpu_time_grids: substep counts against the oracle, full-step flags against the rule restated in NumPy."""
import os
import subprocess

import numpy as np
import pytest

from cd_dynamax_b200 import build
from oracle import cd_oracle as o
from tests import test_gpu_time_grids as tg

# stdin: one gap per line, "t0 t1 dt0" as hexadecimal floats; stdout: "<substeps> <full flag of each substep, or ->"
SRC = r"""
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "cdk_common.cuh"

template <typename T>
static void run() {
  char a[64], b[64], c[64], flags[4097];
  while (scanf("%63s %63s %63s", a, b, c) == 3) {
    cdk::StepClock<T> clk(T(strtod(a, 0)), T(strtod(b, 0)), T(strtod(c, 0)));
    while (clk.running() && clk.n < 4096) {
      flags[clk.n] = clk.full() ? '1' : '0';
      clk.advance();
    }
    flags[clk.n] = 0;
    printf("%d %s\n", clk.n, clk.n ? flags : "-");
  }
}

int main(int argc, char** argv) {
  if (argc > 1 && !strcmp(argv[1], "f32")) run<float>();
  else run<double>();
  return 0;
}
"""


@pytest.fixture(scope="module")
def step_rule(tmp_path_factory):
    """-> run(t0, t1, dt0, dtype) -> (substep counts, full flags as '0'/'1' strings), from the host build of the header."""
    nvcc = build._nvcc()
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    d = tmp_path_factory.mktemp("step_rule")
    src, exe = d / "step_rule.cu", d / "step_rule"
    src.write_text(SRC)
    subprocess.run([nvcc] + build.NVCC_FLAGS + [str(src), "-o", str(exe)], check=True, capture_output=True)

    def run(t0, t1, dt0, dtype):
        t0, t1 = np.asarray(t0, dtype).ravel(), np.asarray(t1, dtype).ravel()
        lines = "".join(f"{float(a).hex()} {float(b).hex()} {float(dtype(dt0)).hex()}\n" for a, b in zip(t0, t1))
        out = subprocess.run([str(exe), "f32" if dtype == np.float32 else "f64"], input=lines, capture_output=True,
                             text=True, check=True).stdout.split("\n")[:-1]
        counts = np.array([int(ln.split()[0]) for ln in out])
        flags = [ln.split()[1].strip("-") for ln in out]
        return counts, flags
    return run


def full_flags(t0, t1, dt0, dtype):
    """Whether each substep has the nominal length dt0 (kf_warp's one-product step): the first if t0 + dt0 < t1, a later
    one if not tprev + dt0 > t1 - tol."""
    t0, t1 = np.asarray(t0, dtype).ravel(), np.asarray(t1, dtype).ravel()
    dt0, tol = dtype(dt0), dtype(o._tol_for(dtype))
    tprev, tnext, full = t0.copy(), np.minimum(t0 + dt0, t1), t0 + dt0 < t1
    flags = [""] * t0.size
    while (act := tprev < t1).any():
        for i in np.nonzero(act)[0]:
            flags[i] += "1" if full[i] else "0"
        tprev = np.where(act, tnext, tprev)
        cand = tprev + dt0
        full = ~(cand > t1 - tol)
        tnext = np.where(full, cand, t1)
    return flags


def _grids():
    g = {f"regular:{kind}@{t0:g}:{dt0:.4g}": (tg.regular_grid(tg.N_VAL, tg.K_VAL, kind, t0), dt0, np.float64)
         for kind, t0, _, dt0 in tg.REGULAR}
    for dt0 in (0.0025, 0.01):
        g[f"edge:{dt0}"] = (tg.edge_grid(tg.N_VAL, tg.K_VAL, dt0), dt0, np.float64)
    g["degenerate"] = (tg.degenerate_grid(tg.N_VAL, tg.K_VAL, 0.0025), 0.0025, np.float64)
    g["long"] = (tg.long_grid(45, 5, 0.001), 0.001, np.float64)
    dt32 = float(np.float32(0.0025))
    g["fp32:regular"] = ((np.arange(24 * 20, dtype=np.float32) * np.float32(0.01)).reshape(24, 20), dt32, np.float32)
    g["fp32:long"] = (tg.long_grid(45, 4, 0.0025, np.float32), dt32, np.float32)
    return g


GRIDS = _grids()


@pytest.mark.parametrize("grid", sorted(GRIDS))
def test_step_rule_matches_the_oracle(step_rule, grid):
    t, dt0, dtype = GRIDS[grid]
    t0, t1 = t[:, :-1], t[:, 1:]
    counts, flags = step_rule(t0, t1, dt0, dtype)
    assert np.array_equal(counts, o.substep_counts(t0, t1, dtype(dt0), dtype).ravel()), grid
    assert flags == full_flags(t0, t1, dt0, dtype), grid
