"""bench.py --dump-outputs on the host: the size cap, the seeded path sample and the row layout of the files."""
import os

import numpy as np

import bench
from path_optimizer_b200 import workloads
from path_optimizer_b200.abi import STATE_DTYPE


def _dump(tmp_path, batch):
    total, B = int(batch["offsets"][-1]), len(batch["n_points"])
    states = np.zeros(total, dtype=STATE_DTYPE)
    for k, f in enumerate(STATE_DTYPE.names):
        states[f] = np.arange(total) * 10 + k
    frenet = np.arange(total * 3, dtype=np.float64)
    bench.dump_outputs(str(tmp_path), batch["n_points"], states, frenet, np.arange(B, dtype=np.int32),
                       np.arange(B, dtype=np.int32) + 7)
    return {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}


def _check_rows(out, batch):
    off = batch["offsets"]
    paths = out["paths"].astype(np.int64)
    rows = np.concatenate([np.arange(off[p], off[p + 1]) for p in paths])
    assert np.array_equal(out["states"], rows[:, None] * 10.0 + np.arange(len(STATE_DTYPE.names)))
    assert np.array_equal(out["frenet"], rows[:, None] * 3.0 + np.arange(3))
    B = len(batch["n_points"])
    assert np.array_equal(out["status"], np.arange(B)) and np.array_equal(out["iters"], np.arange(B) + 7)


def test_small_batch_is_dumped_whole(tmp_path):
    batch = workloads.build(2)
    out = _dump(tmp_path, batch)
    assert set(out) == {"status", "iters", "paths", "states", "frenet"}
    assert all(a.dtype == np.float64 for a in out.values())
    assert np.array_equal(out["paths"], np.arange(len(batch["n_points"])))
    _check_rows(out, batch)


def test_large_batch_is_a_seeded_sample_under_the_cap(tmp_path):
    batch = workloads.build(5)
    out = _dump(tmp_path / "a", batch)
    size = sum(os.path.getsize(os.path.join(tmp_path / "a", f)) for f in os.listdir(tmp_path / "a"))
    assert size <= bench.DUMP_LIMIT_BYTES
    assert 0 < len(out["paths"]) < len(batch["n_points"]) and np.all(np.diff(out["paths"]) > 0)
    _check_rows(out, batch)
    assert np.array_equal(_dump(tmp_path / "b", batch)["paths"], out["paths"])
