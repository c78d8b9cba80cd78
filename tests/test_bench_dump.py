"""bench.py --dump-outputs: which part of a step's output it writes (host-side logic, no GPU)."""
import numpy as np
import torch

import bench


def test_dump_outputs_is_a_seeded_sample_within_the_cap(tmp_path):
    # the default bench size: 4096 streams x 4096 output samples per step is more than the cap
    y = torch.randn((4096, 4200, 2), generator=torch.Generator().manual_seed(1))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch, y, 4096)
    got = np.load(tmp_path / "a" / "output.npy")
    ids = np.load(tmp_path / "a" / "output_streams.npy")
    assert got.dtype == np.float32 and ids.dtype == np.float64
    assert 0 < len(ids) < 4096 and got.shape == (len(ids), 4096, 2)
    assert np.array_equal(got, y[ids.astype(np.int64), :4096].numpy())
    assert np.array_equal(ids, np.load(tmp_path / "b" / "output_streams.npy"))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20
    # an output within the cap is written whole
    small = torch.randn((3, 10, 2))
    bench.dump_outputs(str(tmp_path / "c"), torch, small, 7)
    assert np.array_equal(np.load(tmp_path / "c" / "output.npy"), small[:, :7].numpy())
    assert np.array_equal(np.load(tmp_path / "c" / "output_streams.npy"), [0.0, 1.0, 2.0])
