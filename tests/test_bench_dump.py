"""CPU: bench.py --dump-outputs writes the same seeded sample of trajectories for every field, within its byte budget."""
import os

import numpy as np
import torch

import bench
from cd_dynamax_b200.types import PosteriorGSSMFiltered


def _post(N, K):
    row = torch.arange(N, dtype=torch.float64)  # every entry of a trajectory holds its index
    return PosteriorGSSMFiltered(row, row[:, None, None].expand(N, K, 3), row[:, None, None, None].expand(N, K, 3, 3),
                                 row[:, None, None].expand(N, K, 3), row[:, None, None, None].expand(N, K, 3, 3))


def test_dump_outputs_samples_rows_within_the_budget(tmp_path, monkeypatch):
    N, K = 500, 20
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * (1 + 24 * K) * 8)  # room for 100 of the 500 trajectories
    post = _post(N, K)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), post, post.marginal_loglik.sum()[None])
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(f + ".npy" for f in PosteriorGSSMFiltered._fields + ("ll_sum",))
    rows = np.load(tmp_path / "a" / "marginal_loglik.npy")
    assert rows.shape == (100,) and len(np.unique(rows)) == 100 and np.all(np.diff(rows) > 0)
    total = 0
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b), f  # same sample from run to run
        total += a.nbytes
        if f != "ll_sum.npy":
            assert a.shape[:2] == ((100, K) if a.ndim > 1 else (100,)), f
            assert np.all(a == rows.reshape((-1,) + (1,) * (a.ndim - 1))), f  # the same trajectories in every field
    assert total <= bench.DUMP_BYTES + 8
    assert np.load(tmp_path / "a" / "ll_sum.npy")[0] == N * (N - 1) / 2


def test_dump_outputs_keeps_a_small_batch_whole(tmp_path):
    post = _post(7, 3)
    bench.dump_outputs(str(tmp_path), post, post.marginal_loglik.sum()[None])
    assert np.array_equal(np.load(tmp_path / "filtered_means.npy"), post.filtered_means.numpy())
