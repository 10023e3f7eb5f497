"""bench.py --dump-outputs: what it saves of a step's result, and that the same arguments save the same cells."""
from types import SimpleNamespace

import numpy as np
import torch

import bench


def fake_result(c, b, n, dtype):
    g = torch.Generator().manual_seed(3)
    power = torch.rand((c, b, n), generator=g, dtype=dtype)
    total = power.double().sum((1, 2))
    info = -torch.log2(power.double() / total[:, None, None]).to(dtype)
    return SimpleNamespace(frequency_hz=np.linspace(1.0, 300.0, b), power=power, info=info,
                           band_power=power.double().sum(-1), total_power=total,
                           band_entropy_bits=torch.rand((c, b), generator=g, dtype=torch.float64),
                           entropy_bits=lambda: torch.ones(c, dtype=torch.float64))


def test_sample_is_fixed_and_within_budget():
    # the headline shape: 8 channels x 60 bands x 2^24 samples, fp32 and fp64 planes
    for item in (4, 8):
        shape = (8, 60, 1 << 24)
        idx = bench.plane_sample_index(shape, item)
        assert np.array_equal(idx, bench.plane_sample_index(shape, item))
        assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < np.prod(shape)
        per_band = 8 * 60 * 8 * 2 + 8 * 8 * 2 + 60 * 8
        assert 2 * len(idx) * item + per_band <= 64 << 20
        assert len(idx) > 0.99 * bench.DUMP_PLANE_BYTES // item
    assert bench.plane_sample_index((2, 3, 1024), 4) is None


def test_dump_whole_and_sampled(tmp_path, monkeypatch):
    for dtype, np_dtype in ((torch.float32, np.float32), (torch.float64, np.float64)):
        r = fake_result(2, 3, 512, dtype)
        out = bench.dump_outputs(torch, r, str(tmp_path / "whole"))
        assert out["planes"] == "whole"
        for name in ("power", "info"):
            a = np.load(tmp_path / "whole" / f"{name}.npy")
            assert a.dtype == np_dtype and np.array_equal(a, getattr(r, name).numpy())
        for name in ("band_power", "total_power", "band_entropy_bits", "frequency_hz", "entropy_bits"):
            assert np.load(tmp_path / "whole" / f"{name}.npy").dtype == np.float64
        assert sorted(p.name for p in (tmp_path / "whole").iterdir()) == out["files"]

        monkeypatch.setattr(bench, "DUMP_PLANE_BYTES", 1024)
        out = bench.dump_outputs(torch, r, str(tmp_path / "sampled"))
        idx = bench.plane_sample_index(r.power.shape, r.power.element_size())
        assert idx is not None and str(len(idx)) in out["planes"]
        for name in ("power", "info"):
            a = np.load(tmp_path / "sampled" / f"{name}.npy")
            assert a.dtype == np_dtype and np.array_equal(a, getattr(r, name).numpy().reshape(-1)[idx])
        assert np.array_equal(np.load(tmp_path / "sampled" / "band_power.npy"), r.band_power.numpy())
        monkeypatch.undo()
