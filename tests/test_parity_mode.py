"""B200OCL_MODE=parity: the host-side random decisions consume the reference's generators call for call
(VERDICT r01 item 9).  CPU tests against the draws of the unmodified reference classes on the same inputs,
recorded in tests/golden/parity.npz by tests/golden/make_golden.py (image tensors as sha256 digests)."""
import hashlib
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch


@pytest.fixture()
def ref(golden_dir):
    from b200ocl import memory
    memory.set_mode(True, 'cpu')
    memory.ClassBalancedRandomSampling.reset()
    yield np.load(os.path.join(golden_dir, 'parity.npz'), allow_pickle=False)
    memory.set_mode(False)
    memory.ClassBalancedRandomSampling.reset()


def _digest(t):
    return np.frombuffer(hashlib.sha256(t.contiguous().numpy().tobytes()).digest(), np.uint8)


def _sample(mine, n, excl, seed):
    torch.manual_seed(seed)
    return mine.sample_indices(n, excl_indices=excl)


@pytest.mark.parametrize('n_cls,mem', [(10, 200), (100, 1000)])
def test_sampler_incremental_stream_identical(ref, n_cls, mem):
    from b200ocl.memory import ClassBalancedRandomSampling as Mine
    tag = 'inc%d' % n_cls
    rs = np.random.RandomState(3)
    labels = rs.randint(0, n_cls, mem).astype(np.int64)
    buf_y = torch.zeros(mem, dtype=torch.int64)
    # fill phase in batches of 10, as ASER_update does (aser_update.py:28-35)
    for s in range(0, mem, 10):
        Mine.update_cache(buf_y, n_cls, new_y=labels[s:s + 10], ind=np.arange(s, s + 10))
        buf_y[s:s + 10] = torch.from_numpy(labels[s:s + 10])
    assert ref[tag + '_keys'].tolist() == list(Mine.class_index_cache.keys())
    for step in range(25):
        m1 = _sample(Mine, 1, None, 100 + step)
        assert np.array_equal(ref['%s_r1_%d' % (tag, step)], m1)
        m2 = _sample(Mine, 2, m1.tolist(), 200 + step)
        assert np.array_equal(ref['%s_r2_%d' % (tag, step)], m2)
        # replacement of a few slots (aser_update.py:108-112)
        slots = rs.choice(mem, 4, replace=False)
        ny = rs.randint(0, n_cls, 4).astype(np.int64)
        Mine.update_cache(buf_y, n_cls, new_y=ny, ind=slots)
        buf_y[torch.from_numpy(slots)] = torch.from_numpy(ny)
        assert np.array_equal(ref['%s_num_%d' % (tag, step)], Mine.class_num_cache)


def test_sampler_rebuild_stream_identical(ref):
    from b200ocl.memory import ClassBalancedRandomSampling as Mine
    rs = np.random.RandomState(4)
    labels = rs.randint(0, 20, 300).astype(np.int64)
    Mine.update_cache(torch.from_numpy(labels), 20, labels_host=labels)
    assert ref['rebuild_keys'].tolist() == list(Mine.class_index_cache.keys())
    for step in range(10):
        m = _sample(Mine, 3, None, step)
        assert np.array_equal(ref['rebuild_r_%d' % step], m)
        m2 = _sample(Mine, 3, m.tolist(), 50 + step)
        assert np.array_equal(ref['rebuild_r2_%d' % step], m2)


def test_reservoir_stream_identical(ref):
    from b200ocl.memory import Buffer
    from b200ocl import registry
    params = SimpleNamespace(data='cifar10', cuda=False, mem_size=50, update='random', retrieve='random',
                             eps_mem_batch=10, buffer_tracker=False)
    mine = Buffer(None, params)
    rs = np.random.RandomState(0)
    for step in range(30):
        x = torch.from_numpy(rs.rand(10, 3, 32, 32).astype(np.float32))
        y = torch.from_numpy(rs.randint(0, 10, 10).astype(np.int64))
        torch.manual_seed(step)
        b = mine.update(x, y)
        assert ref['reservoir_ret_%d' % step].tolist() == list(b)
        assert np.array_equal(ref['reservoir_label'][step], mine.buffer_label.numpy())
        assert mine.buffer_img.shape == (50, 3, 32, 32) and mine.buffer_img.dtype == torch.float32
        assert np.array_equal(ref['reservoir_img_sha256'][step], _digest(mine.buffer_img))
        assert ref['reservoir_n_seen'][step] == mine.n_seen_so_far


def test_stream_order_identical(ref):
    from b200ocl.learners import StreamFeeder
    rs = np.random.RandomState(1)
    x = rs.randint(0, 256, (57, 32, 32, 3)).astype(np.uint8)
    y = rs.randint(0, 10, 57).astype(np.int64)
    torch.manual_seed(11)
    mine = list(StreamFeeder(x, y, 10, 'cpu'))
    after_mine = torch.rand(1)
    assert len(mine) == len(ref['stream_label']) == 5
    for ry, rx_sha, (mx, my, myh) in zip(ref['stream_label'], ref['stream_img_sha256'], mine):
        assert np.array_equal(ry, my.numpy()) and np.array_equal(ry, myh)
        assert list(mx.shape) == ref['stream_img_shape'].tolist() and mx.dtype == torch.float32
        assert np.array_equal(rx_sha, _digest(mx))
    assert np.array_equal(ref['stream_rand_after'], after_mine.numpy())   # the default generator ends in the same state
