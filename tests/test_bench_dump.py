"""CPU: bench.py --dump-outputs (what it writes, its size bound, a fixed sample of large outputs) and its argument checks."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from conftest import ROOT


def test_dump_keeps_small_outputs_whole_and_samples_large_ones_the_same_way(tmp_path):
    codes = torch.randn(4, 25, 67, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    verts = torch.arange(64 * 25 * 50 * 3, dtype=torch.float32).reshape(64, 25, 50, 3)    # frame f holds 150 f .. 150 f + 149
    max_bytes = 100_000
    for d in ('a', 'b'):
        bench.dump_outputs(dict(codes=codes, vertices=verts), str(tmp_path / d), max_bytes=max_bytes)
    assert sorted(os.listdir(tmp_path / 'a')) == ['codes.npy', 'vertices.npy']
    c, v = np.load(tmp_path / 'a' / 'codes.npy'), np.load(tmp_path / 'a' / 'vertices.npy')
    assert c.dtype == np.float32 and np.array_equal(c, codes.float().numpy())
    frames = v[:, 0, 0] / 150
    assert v.dtype == np.float32 and v.shape[1:] == (50, 3) and 0 < len(frames) < 64 * 25
    assert np.all(np.diff(frames) > 0) and np.array_equal(v, verts.reshape(-1, 50, 3).numpy()[frames.astype(int)])
    assert c.nbytes + v.nbytes <= max_bytes
    for f in ('codes.npy', 'vertices.npy'):
        assert (tmp_path / 'a' / f).read_bytes() == (tmp_path / 'b' / f).read_bytes()


@pytest.mark.parametrize('argv, msg', [(['--steps', '0'], '--steps must be at least 1'),
                                       (['--impl', 'reference', '--dump-outputs', 'out'], '--dump-outputs')])
def test_bench_rejects_arguments_it_cannot_honour(argv, msg):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + argv, capture_output=True, text=True)
    assert r.returncode == 2 and msg in r.stderr, r.stderr


def test_dump_refuses_an_output_whose_single_matrix_exceeds_its_share(tmp_path):
    with pytest.raises(AssertionError, match='larger than its'):
        bench.dump_outputs(dict(vertices=torch.zeros(2, 100, 3)), str(tmp_path), max_bytes=1000)


@pytest.mark.gpu
def test_bench_dump_outputs_end_to_end(built_lib, tmp_path):
    """The wiring in main(): the last timed step's codes and vertices of one 10 s clip (latency1) land in DIR."""
    d = tmp_path / 'dump'
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'latency1', '--steps', '1', '--warmup',
                        '1', '--no-cpu-baseline', '--dump-outputs', str(d)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(d)) == ['codes.npy', 'vertices.npy']
    c, v = np.load(d / 'codes.npy'), np.load(d / 'vertices.npy')
    assert c.shape == (1, 250, 67) and v.shape == (1, 250, 5023, 3) and c.dtype == v.dtype == np.float32
    assert np.isfinite(c).all() and np.isfinite(v).all() and np.abs(v).max() > 0
    assert sum(os.path.getsize(d / f) for f in os.listdir(d)) < 64e6
