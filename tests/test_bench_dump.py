"""bench.py --dump-outputs: what it writes, within its size limit, the same sample on every run."""
import os

import numpy as np
import torch

import bench
from roadsurf_b200 import lib


def _dump(directory, npoints, limit, with_state=False):
    g = torch.Generator().manual_seed(3)
    out = torch.randn((lib.O_NVAR, 25, npoints + 31), generator=g, dtype=torch.float64)
    status = torch.randint(0, 512, (npoints + 31,), generator=g, dtype=torch.int32)
    state = torch.randn((lib.state_nplanes(15), npoints + 31), generator=g, dtype=torch.float64) if with_state else None
    bench.dump_outputs(str(directory), out, status, npoints, state=state, limit=limit)
    return out, status, state, {f[:-4]: np.load(os.path.join(directory, f)) for f in os.listdir(directory)}


def test_small_batches_are_written_whole(tmp_path):
    out, status, _, d = _dump(tmp_path, 100, bench.DUMP_LIMIT_BYTES)
    assert set(d) == set(lib.O_NAMES) | {"status", "point_index"}
    assert all(a.dtype == np.float64 for a in d.values())
    assert np.array_equal(d["point_index"], np.arange(100))
    for v, name in enumerate(lib.O_NAMES):
        assert np.array_equal(d[name], out[v, :, :100].numpy().T)
    assert np.array_equal(d["status"], status[:100].numpy())


def test_large_batches_are_sampled_within_the_limit_the_same_way_every_run(tmp_path):
    limit = 200_000
    out, status, state, a = _dump(tmp_path / "a", 5000, limit, with_state=True)
    _, _, _, b = _dump(tmp_path / "b", 5000, limit, with_state=True)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= limit
    idx = a["point_index"].astype(np.int64)
    assert 0 < len(idx) < 5000 and (np.diff(idx) > 0).all() and idx[-1] < 5000
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert np.array_equal(a["TsurfOut"], out[0][:, idx].numpy().T)
    assert np.array_equal(a["status"], status[idx].numpy())
    assert np.array_equal(a["state"], state[:, idx].numpy().T)
