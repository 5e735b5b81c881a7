"""CPU-only checks of bench.py's --dump-outputs writer: one .npy per output, float32 for floating tensors, float64 for ids,
and a bounded total size."""
import os

import numpy as np
import pytest
import torch

import bench


def test_write_outputs_dtypes_and_names(tmp_path):
    ids = torch.tensor([[3, 2 ** 40 + 1]], dtype=torch.int64)
    bench.write_outputs(str(tmp_path / "out"), {"loss": torch.tensor(1.25), "param.w": torch.ones(2, 3, dtype=torch.float16),
                                                "top10_ids": ids})
    assert sorted(os.listdir(tmp_path / "out")) == ["loss.npy", "param.w.npy", "top10_ids.npy"]
    loss = np.load(tmp_path / "out" / "loss.npy")
    assert loss.dtype == np.float32 and loss.shape == () and loss == 1.25
    assert np.load(tmp_path / "out" / "param.w.npy").dtype == np.float32
    got = np.load(tmp_path / "out" / "top10_ids.npy")
    assert got.dtype == np.float64 and (got.astype(np.int64) == ids.numpy()).all()


def test_write_outputs_refuses_more_than_the_limit(tmp_path):
    with pytest.raises(RuntimeError, match="limit"):
        bench.write_outputs(str(tmp_path / "out"), {"big": torch.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1)})
    assert not (tmp_path / "out").exists()
