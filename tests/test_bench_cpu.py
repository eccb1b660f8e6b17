"""Host logic of bench.py: the timed region runs exactly --steps steps and keeps what the last one returned, and
--dump-outputs writes it as float32 / float64 .npy files within the size limit."""
import os

import numpy as np
import pytest
import torch

import bench


def test_command_line_sets_the_steps_and_rejects_what_cannot_be_honoured(monkeypatch):
    monkeypatch.setattr('sys.argv', ['bench.py', '--steps', '3', '--warmup', '0', '--dump-outputs', 'out'])
    args = bench.parse()
    assert (args.steps, args.warmup, args.dump_outputs) == (3, 0, 'out')
    for argv in (['--steps', '0'], ['--steps', '-2'], ['--impl', 'reference', '--dump-outputs', 'out']):
        monkeypatch.setattr('sys.argv', ['bench.py'] + argv)
        with pytest.raises(SystemExit) as e:
            bench.parse()
        assert e.value.code == 2, argv


def test_timed_region_keeps_the_last_timed_step():
    calls = []

    def step(i):
        calls.append(i)
        return (torch.tensor([float(i)]),)

    bench.run_timed(step, lambda i: (torch.tensor([-1.0]),), 7, lambda: None, lambda: None, lambda: None, lambda: 8, lambda: None)
    assert calls == list(range(7))
    assert float(bench.run_timed.last[0]) == 6.0


def test_dump_outputs_writes_winners_and_samples_past_the_limit(tmp_path, monkeypatch):
    g = torch.Generator().manual_seed(0)
    best = torch.randn(1000, generator=g)
    idx = torch.randint(-1, 3172, (1000,), generator=g, dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / 'all'), best, idx)
    b, i = np.load(tmp_path / 'all' / 'best_score.npy'), np.load(tmp_path / 'all' / 'best_index.npy')
    assert b.dtype == np.float32 and i.dtype == np.float64
    assert np.array_equal(b, best.numpy()) and np.array_equal(i, idx.numpy())
    assert sorted(os.listdir(tmp_path / 'all')) == ['best_index.npy', 'best_score.npy']
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 4096 + 20 * 100)
    for d in ('s1', 's2'):
        bench.dump_outputs(str(tmp_path / d), best, idx)
    files = sorted(os.listdir(tmp_path / 's1'))
    assert files == ['best_index.npy', 'best_score.npy', 'sample_rows.npy']
    assert sum(os.path.getsize(tmp_path / 's1' / f) for f in files) <= bench.DUMP_LIMIT
    rows = np.load(tmp_path / 's1' / 'sample_rows.npy').astype(np.int64)
    assert len(rows) == 100 and np.array_equal(rows, np.load(tmp_path / 's2' / 'sample_rows.npy'))
    assert np.array_equal(np.load(tmp_path / 's1' / 'best_score.npy'), best.numpy()[rows])
    assert np.array_equal(np.load(tmp_path / 's1' / 'best_index.npy'), idx.numpy()[rows])
