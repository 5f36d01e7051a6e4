"""bench.py --dump-outputs: what the last timed step returned, in a form two builds can be compared on."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fake_step(n_pairs, kpts, seed=0):
    g = torch.Generator().manual_seed(seed)
    outs = []
    for i in range(n_pairs):
        n = kpts - 3 * i
        counts = torch.tensor([n, n - 1, 5 * n, 5 * n, 1, 1, 0x100, 0], dtype=torch.int32)
        outs.append({'n_kept_dev': counts,
                     'matches0': torch.randint(-1, n - 1, (kpts,), generator=g, dtype=torch.int64),
                     'mscores0': torch.rand(kpts, generator=g)})
    return outs


def _load(path):
    return {name[:-4]: np.load(os.path.join(path, name)) for name in sorted(os.listdir(path))}


def _split(dump, name):
    return np.split(dump[name], np.cumsum(dump['counts'][:, 0].astype(int))[:-1])


def test_dump_layout(tmp_path):
    outs = _fake_step(5, 64)
    bench.dump_outputs(str(tmp_path), outs, 64)
    got = _load(str(tmp_path))
    assert sorted(got) == ['counts', 'matches0', 'matching_scores0', 'pair_index']
    assert all(np.isfinite(v).all() for v in got.values())
    assert got['counts'].shape == (5, 8) and got['counts'].dtype == np.float64
    n_total = sum(int(o['n_kept_dev'][0]) for o in outs)
    assert got['matches0'].shape == (n_total,) and got['matches0'].dtype == np.float64
    assert got['matching_scores0'].shape == (n_total,) and got['matching_scores0'].dtype == np.float32
    assert np.array_equal(got['pair_index'], np.arange(5.0))
    for o, c, m, sc in zip(outs, got['counts'], _split(got, 'matches0'), _split(got, 'matching_scores0')):
        n = int(o['n_kept_dev'][0])
        assert np.array_equal(c, o['n_kept_dev'].numpy())
        assert np.array_equal(m, o['matches0'][:n].numpy())
        assert np.array_equal(sc, o['mscores0'][:n].numpy())


def test_dump_samples_pairs_over_the_limit(tmp_path, monkeypatch):
    per_pair = 9 * 8 + 64 * 12
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 4 * 128 + 3 * per_pair + 10)
    outs = _fake_step(10, 64)
    bench.dump_outputs(str(tmp_path / 'a'), outs, 64)
    bench.dump_outputs(str(tmp_path / 'b'), outs, 64)
    a, b = _load(str(tmp_path / 'a')), _load(str(tmp_path / 'b'))
    assert sum(os.path.getsize(os.path.join(tmp_path, 'a', f)) for f in os.listdir(tmp_path / 'a')) <= bench.DUMP_LIMIT_BYTES
    idx = a['pair_index'].astype(int)
    assert len(idx) == 3 and np.all(np.diff(idx) > 0)
    for name in a:                                     # the sample is fixed
        assert np.array_equal(a[name], b[name])
    for row, i in enumerate(idx):
        assert np.array_equal(a['counts'][row], outs[i]['n_kept_dev'].numpy())


@pytest.mark.gpu
def test_dump_repeats_across_runs(tmp_path):
    """Same arguments, two processes: same inputs, so the same counts and matches (scores up to fp32 atomics)."""
    steps = 2
    lines, dumps = [], []
    for run in ('a', 'b'):
        cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', str(steps), '--warmup', '3',
               '--kpts', '512', '--pairs-per-step', '4', '--streams', '2', '--pool', '6', '--no-e2e',
               '--no-cpu-baseline', '--dump-outputs', str(tmp_path / run)]
        r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
        dumps.append(_load(str(tmp_path / run)))
    a, b = dumps
    assert lines[0]['steps'] == steps and lines[0]['gpu_launches'] > 0
    assert a['counts'].shape == (4, 8) and all(np.isfinite(v).all() for d in dumps for v in d.values())
    assert np.array_equal(a['counts'][:, :6], b['counts'][:, :6])
    assert (a['counts'][:, 0] > 0).all() and not (a['counts'][:, 6].astype(np.int64) & 0xff).any()
    assert a['matches0'].shape == (int(a['counts'][:, 0].sum()),) == b['matches0'].shape
    assert (a['matches0'] == b['matches0']).mean() >= 0.999
    assert np.allclose(a['matching_scores0'], b['matching_scores0'], rtol=1e-4, atol=1e-6)
