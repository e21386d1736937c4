"""bench.py --dump-outputs: the arrays it writes, their types, and the fixed sample that stands in for a large array."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_writes_the_step_and_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, 'DUMP_MAX_ELEMS', 1000)
    step = {'loss': 0.25, 'train_loss': 0.125, 'epe': 0.0, 'bad3': 0.0, 'blocks': [3], 'reset': False}
    disp = torch.rand(2, 8, 16, 1)                       # 256 elements: written whole
    weights = torch.arange(5000, dtype=torch.float32)    # above the cap: a seeded sample
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), step, disp, weights)
    names = sorted(os.listdir(tmp_path / 'a'))
    assert names == ['blocks.npy', 'disparity.npy', 'loss.npy', 'train_loss.npy', 'weights.npy']
    load = lambda d, n: np.load(str(tmp_path / d / n))
    assert load('a', 'loss.npy').dtype == np.float64 and load('a', 'loss.npy').tolist() == [0.25]
    assert load('a', 'train_loss.npy').tolist() == [0.125] and load('a', 'blocks.npy').tolist() == [3.0]
    assert load('a', 'disparity.npy').dtype == np.float32 and np.array_equal(load('a', 'disparity.npy'), disp.numpy())
    w = load('a', 'weights.npy')
    assert w.dtype == np.float32 and w.shape == (1000,)
    assert np.all(np.diff(w) > 0)                        # distinct elements in ascending index order
    for n in names:
        assert np.array_equal(load('a', n), load('b', n)), n
