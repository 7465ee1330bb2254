"""bench.py --dump-outputs on CPU: file names, dtypes, the size cap and the seeded row sample."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_writes_every_tensor(tmp_path):
    torch.manual_seed(0)
    out = {"traj": torch.randn(6, 5, 3), "offroad": torch.rand(6, 5) > 0.5, "coll": torch.arange(6, dtype=torch.int64),
           "x1": None, "aux_info": {"cond_feat": torch.randn(6, 4).double(), "names": ["a"] * 6}}
    bench.dump_outputs(str(tmp_path), out)
    assert sorted(os.listdir(tmp_path)) == ["aux_info.cond_feat.npy", "coll.npy", "offroad.npy", "traj.npy"]
    traj, off = np.load(tmp_path / "traj.npy"), np.load(tmp_path / "offroad.npy")
    coll, cond = np.load(tmp_path / "coll.npy"), np.load(tmp_path / "aux_info.cond_feat.npy")
    assert traj.dtype == np.float32 and np.array_equal(traj, out["traj"].numpy())
    assert off.dtype == np.float32 and np.array_equal(off, out["offroad"].float().numpy())
    assert coll.dtype == np.float64 and np.array_equal(coll, np.arange(6))
    assert cond.dtype == np.float64 and np.array_equal(cond, out["aux_info"]["cond_feat"].numpy())


def test_dump_outputs_samples_the_same_rows_under_the_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    rows = torch.arange(1000, dtype=torch.float32)
    out = {"a": rows[:, None].expand(1000, 3).contiguous(), "b": rows.clone()}      # 16 000 bytes: a quarter of the rows is kept
    for d in ("one", "two"):
        bench.dump_outputs(str(tmp_path / d), out)
    a, b = np.load(tmp_path / "one" / "a.npy"), np.load(tmp_path / "one" / "b.npy")
    assert a.nbytes + b.nbytes <= 4000 and b.shape == (250,)
    assert np.array_equal(a[:, 0], b) and np.all(np.diff(b) > 0)
    assert np.array_equal(b, np.load(tmp_path / "two" / "b.npy"))
