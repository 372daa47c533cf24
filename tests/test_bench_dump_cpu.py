"""CPU: bench.py --dump-outputs writes float arrays under its size budget, and the same sample of an oversized output every run."""
import os

import numpy as np
import torch


def test_dump_outputs_writes_small_arrays_whole(tmp_path):
    import bench
    arrays = {'pred_wp': torch.randn(2, 6, 4, 2), 'pred_speed': torch.randn(2, 1, dtype=torch.float64),
              'mu_branches': torch.randn(2, 6, 2, dtype=torch.float16)}
    bench.dump_outputs(arrays, str(tmp_path / 'out'))
    assert sorted(os.listdir(tmp_path / 'out')) == sorted(k + '.npy' for k in arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / 'out' / (k + '.npy'))
        assert got.dtype == (np.float64 if v.dtype == torch.float64 else np.float32)
        assert np.array_equal(got, v.double().numpy())


def test_dump_outputs_samples_oversized_arrays_the_same_way_every_run(tmp_path):
    import bench
    big = torch.arange(100000, dtype=torch.float32).view(10, 100, 100)
    arrays = {'big': big, 'small': torch.ones(3)}
    budget = 64 << 10
    for d in ('a', 'b'):
        bench.dump_outputs(arrays, str(tmp_path / d), budget=budget)
    a, b = np.load(tmp_path / 'a' / 'big.npy'), np.load(tmp_path / 'b' / 'big.npy')
    assert sum(os.path.getsize(tmp_path / 'a' / f) - 128 for f in os.listdir(tmp_path / 'a')) <= budget
    assert np.array_equal(a, b) and a.size > 0
    assert np.all(np.diff(a) > 0)                                      # distinct elements, in flat order
    assert np.array_equal(np.load(tmp_path / 'a' / 'small.npy'), np.ones(3, np.float32))
