"""bench.py --dump-outputs: the outputs of the last timed step as float32 .npy files, at most 64 MB in all (a seeded sample of
environments above that)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')


def _arrays(n):
    return {'state': torch.arange(n * 6, dtype=torch.float32).reshape(n, 6), 'obs': torch.zeros((n, 0)),
            'term': (torch.arange(n) % 2).to(torch.uint8)[:, None], 'camera0_rgb': torch.rand((n, 4, 5, 3), generator=torch.Generator().manual_seed(0))}


def test_dump_outputs_writes_every_row_as_float32(tmp_path):
    arrays = _arrays(100)
    bench.dump_outputs(str(tmp_path), arrays, 100)
    assert sorted(os.listdir(tmp_path)) == ['camera0_rgb.npy', 'env_index.npy', 'state.npy', 'term.npy']   # zero-width obs skipped
    assert np.array_equal(np.load(tmp_path / 'env_index.npy'), np.arange(100.0))
    for name in ('state', 'term', 'camera0_rgb'):
        got = np.load(tmp_path / (name + '.npy'))
        assert got.dtype == np.float32 and np.array_equal(got, arrays[name].float().numpy()), name


def test_dump_outputs_samples_the_same_rows_above_the_limit(tmp_path, monkeypatch):
    arrays = _arrays(100)
    row = 4 * (6 + 1 + 60) + 8
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 128 * 4 + 10 * row)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), arrays, 100)
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= bench.DUMP_LIMIT
    idx = np.load(tmp_path / 'a' / 'env_index.npy')
    assert len(idx) == 10 and len(set(idx)) == 10 and np.array_equal(idx, np.load(tmp_path / 'b' / 'env_index.npy'))
    rows = idx.astype(np.int64)
    for name in ('state', 'term', 'camera0_rgb'):
        assert np.array_equal(np.load(tmp_path / 'a' / (name + '.npy')), arrays[name][rows].float().numpy()), name


def _bench_dump(tmp_path, name, steps):
    out = tmp_path / name
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--config', 'basic_env', '--envs', '64', '--steps', str(steps), '--warmup', '3',
           '--preroll', '2', '--no-cpu-baseline', '--dump-outputs', str(out)]
    r = subprocess.run(cmd, cwd=str(tmp_path), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])['steps'] == steps
    return out, {f[:-4]: np.load(out / f) for f in os.listdir(out)}


@pytest.mark.gpu
def test_bench_dumps_the_outputs_of_its_last_timed_step(tmp_path):
    out, got = _bench_dump(tmp_path, 'a', 3)
    _, again = _bench_dump(tmp_path, 'b', 3)
    _, later = _bench_dump(tmp_path, 'c', 4)
    assert sorted(again) == sorted(got) and all(np.array_equal(again[k], got[k]) for k in got)   # same arguments, same outputs
    assert not np.allclose(later['state'], got['state'])                                        # one more timed step, another state
    assert sorted(os.listdir(out)) == ['camera0_depth.npy', 'camera0_rgb.npy', 'env_index.npy', 'obs.npy', 'state.npy']
    assert np.array_equal(np.load(out / 'env_index.npy'), np.arange(64.0))
    shapes = {'obs': (64, 3), 'camera0_rgb': (64, 50, 50, 3), 'camera0_depth': (64, 50, 50)}
    for name, shape in shapes.items():
        a = np.load(out / (name + '.npy'))
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all(), name
    st = np.load(out / 'state.npy')
    assert st.dtype == np.float32 and st.shape[0] == 64 and np.isfinite(st).all()
