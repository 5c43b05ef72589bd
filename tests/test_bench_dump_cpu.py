"""bench.py --dump-outputs: every array is written exactly as float32 / float64, and a dump above the size limit keeps the same seeded
rows of every array."""
import numpy as np
import torch

import bench


def test_dump_outputs_exact_dtypes(tmp_path):
    B = 37
    rng = np.random.default_rng(1)
    arrays = dict(action=torch.from_numpy(rng.integers(-2**31, 2**31 - 1, B, dtype=np.int32)),
                  value=torch.from_numpy(rng.standard_normal(B).astype(np.float32)),
                  terminated=torch.from_numpy(rng.integers(0, 2, B, dtype=np.uint8)),
                  short=torch.from_numpy(rng.integers(-2**15, 2**15 - 1, (B, 8), dtype=np.int16)),
                  flag=torch.from_numpy(rng.random(B) < 0.5))
    bench.dump_outputs(str(tmp_path / "d"), arrays, prefix="rank1_")
    for name, t in arrays.items():
        got = np.load(tmp_path / "d" / f"rank1_{name}.npy")
        assert got.dtype == (np.float64 if name == "action" else np.float32), name
        assert got.shape == tuple(t.shape) and (got == t.numpy()).all(), name


def test_dump_outputs_samples_rows_above_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4000)
    B = 1000
    idx = torch.arange(B, dtype=torch.int32)
    arrays = dict(index=idx, logits=torch.arange(B * 2, dtype=torch.float32).reshape(B, 2))
    bench.dump_outputs(str(tmp_path), arrays)
    index, logits = np.load(tmp_path / "index.npy"), np.load(tmp_path / "logits.npy")
    assert index.nbytes + logits.nbytes <= 4000 and len(index) == len(logits) > 0
    assert (np.diff(index) > 0).all() and (logits[:, 0] == 2 * index).all()  # same rows, in order, in both arrays
    bench.dump_outputs(str(tmp_path / "again"), arrays)
    assert (np.load(tmp_path / "again" / "index.npy") == index).all()  # fixed seed: the same sample every run
