"""CPU tests of bench.py's command line: --dump-outputs writes a fixed, bounded sample of what the timed step returned."""
import os
import sys

import numpy as np
import pytest
import torch

import bench


def test_dump_outputs_writes_a_fixed_bounded_sample(tmp_path):
    numel = 8 * 128 * 10 * 352 * 400                       # the grid of one headline step
    idx = bench.grid_sample_index(numel)
    assert np.array_equal(idx, bench.grid_sample_index(numel))
    assert idx.size == bench.DUMP_GRID_SAMPLES and idx.min() >= 0 and idx.max() < numel and np.all(np.diff(idx) >= 0)
    rows = bench.voxel_sample_rows(3, 21_000)
    assert np.array_equal(rows, bench.voxel_sample_rows(3, 21_000)) and np.all(np.diff(rows) > 0) and rows[-1] < 21_000
    assert np.array_equal(bench.voxel_sample_rows(3, 100), np.arange(100))
    assert idx.size * 4 + 8 * rows.size * (128 * 4 + 4 * 8) < 64 << 20       # 8 frames: the dump stays below 64 MB

    class Path:       # voxel_features() of PointPath: (N_f,128) features, (N_f,4) [frame, ix, iy, iz]
        def __init__(self, n):
            self.v = [torch.randn((k, 128)) for k in n]

        def voxel_features(self, f):
            return self.v[f], torch.full((self.v[f].shape[0], 4), f, dtype=torch.int64)

    grid = torch.randn((2, 128, 3, 4, 5))
    counts = torch.tensor([[7, 9, 0, 3], [9000, 9500, 1, 2]], dtype=torch.int32)
    path = Path([7, 9000])
    bench.dump_outputs(str(tmp_path / 'out'), path, grid, counts)
    out = {n[:-4]: np.load(tmp_path / 'out' / n) for n in os.listdir(tmp_path / 'out')}
    assert sorted(out) == ['counts', 'grid_sample', 'voxel_features', 'voxel_index']
    assert out['counts'].dtype == np.float64 and np.array_equal(out['counts'], counts.numpy())
    assert out['grid_sample'].dtype == np.float32
    assert np.array_equal(out['grid_sample'], grid.numpy().reshape(-1)[bench.grid_sample_index(grid.numel())])
    want = np.concatenate([path.v[0].numpy(), path.v[1].numpy()[bench.voxel_sample_rows(1, 9000)]])
    assert out['voxel_features'].dtype == np.float32 and np.array_equal(out['voxel_features'], want)
    assert out['voxel_index'].dtype == np.float64 and out['voxel_index'].shape == (7 + bench.DUMP_VOXEL_ROWS, 4)


@pytest.mark.parametrize('argv', [['--steps', '0'], ['--warmup', '-1'], ['--workload', 'train', '--dump-outputs', 'x'],
                                  ['--impl', 'reference', '--dump-outputs', 'x']])
def test_bench_rejects_arguments_it_cannot_honour(monkeypatch, argv):
    monkeypatch.setattr(sys, 'argv', ['bench.py'] + argv)
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
