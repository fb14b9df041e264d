"""Checkpoint state that lives on the host: the replay buffer and numpy's global random stream (the engine's full
state dict needs CUDA and is covered by tests/test_resume_gpu.py)."""
import io

import numpy as np
import torch

from rorl_b200.buffers.transition_buffer.nested_replay_memory import NestedMemoryArray
from rorl_b200.buffers.transition_buffer.replay_memory import Transition
from rorl_b200.utility.rng_state import numpy_state, set_numpy_state

S, A = 5, 3


def _push(buf, rng, lens, cut=None):
    """Push trajectories of the given lengths; with `cut`, stop that many steps into the last one (a pending partial
    trajectory).  Scalar and array fields are mixed as a rollout loop hands them over."""
    for j, Tn in enumerate(lens):
        last_s, last_a, last_r = np.zeros((1, S)), np.zeros((1, A)), np.zeros((1, 1))
        s = rng.standard_normal((1, S))
        for t in range(Tn):
            if cut is not None and j == len(lens) - 1 and t == cut:
                return
            a = np.tanh(rng.standard_normal((1, A)))
            ns = rng.standard_normal((1, S))
            r = float(rng.standard_normal())
            done = t == Tn - 1
            buf.mem_push(Transition(state=s, last_state=last_s, last_action=last_a, action=a, next_state=ns, reward=r, logp=None,
                                    mask=1, done=done, timeout=done, start=(t == 0), reward_input=last_r))
            last_s, last_a, last_r, s = s, a, np.array([[r]]), ns


def _roundtrip(obj):
    f = io.BytesIO()
    torch.save(obj, f)
    f.seek(0)
    return torch.load(f, weights_only=True)


def _assert_same(a, b):
    assert a.trajectory_start == b.trajectory_start
    assert a.trajectory_length == b.trajectory_length
    assert (a.ptr, a.transition_count) == (b.ptr, b.transition_count)
    assert a.ind_range == b.ind_range
    for s, n in zip(a.trajectory_start, a.trajectory_length):      # every row the sampler can read
        assert np.array_equal(a.memory_buffer[s:s + n], b.memory_buffer[s:s + n])
    assert len(a.memory) == len(b.memory)
    for ta, tb in zip(a.memory, b.memory):
        for fa, fb in zip(ta, tb):
            assert (fa is None) == (fb is None)
            if fa is not None:
                assert np.array_equal(np.asarray(fa, dtype=np.float64), np.asarray(fb, dtype=np.float64))


def test_replay_state_roundtrip_through_eviction_and_wraparound():
    cap, lens = 300, [37, 52, 23, 61, 44, 30, 58, 41]
    straight = NestedMemoryArray(cap, 64, additional_history_len=4)
    saved = NestedMemoryArray(cap, 64, additional_history_len=4)
    r1, r2 = np.random.RandomState(7), np.random.RandomState(7)
    _push(straight, r1, lens[:5], cut=17)
    _push(saved, r2, lens[:5], cut=17)
    sd = _roundtrip(saved.state_dict())
    assert sd['pending']['steps'] == 17
    resumed = NestedMemoryArray(cap, 64, additional_history_len=4)
    resumed.load_state_dict(sd)
    _assert_same(straight, resumed)
    # finish the pending trajectory, then keep pushing until the oldest trajectories are evicted and the pointer wraps
    wrapped = False
    for k in range(6):
        more = [lens[(k + 3) % len(lens)]] * 2
        _push(straight, np.random.RandomState(100 + k), more)
        _push(resumed, np.random.RandomState(100 + k), more)
        wrapped = wrapped or straight.ptr < straight.trajectory_start[0]
        _assert_same(straight, resumed)
    assert wrapped and straight.trajectory_start[0] > 0, 'no eviction / wrap-around happened'
    # the sampler draws the same plan from both
    np.random.seed(5)
    pa = straight.plan_trajs(200, nest_stack_trajs=True)
    np.random.seed(5)
    pb = resumed.plan_trajs(200, nest_stack_trajs=True)
    assert np.array_equal(pa.entries, pb.entries) and np.array_equal(pa.lens, pb.lens)


def test_replay_state_refuses_other_layout():
    a = NestedMemoryArray(300, 64)
    _push(a, np.random.RandomState(1), [20])
    b = NestedMemoryArray(400, 64)
    try:
        b.load_state_dict(a.state_dict())
    except ValueError as e:
        assert 'max_transition_num' in str(e)
    else:
        raise AssertionError('a buffer of another capacity was accepted')
    assert b.memory_buffer is None and b.trajectory_length == []


def test_empty_replay_state_roundtrip():
    a = NestedMemoryArray(300, 64)
    b = NestedMemoryArray(300, 64)
    b.load_state_dict(_roundtrip(a.state_dict()))
    assert b.memory_buffer is None and b.ptr == 0 and b.memory == []


def test_numpy_rng_state_roundtrip():
    np.random.seed(1234)
    np.random.standard_normal(3)               # leave a cached Gaussian behind (has_gauss = 1)
    np.random.random_sample(5)
    sd = _roundtrip(numpy_state())
    assert sd['keys'].dtype == torch.int64 and sd['keys'].numel() == 624
    want = (np.random.permutation(50), np.random.standard_normal(7), np.random.randint(0, 1000, 9))
    np.random.seed(99)
    set_numpy_state(sd)
    got = (np.random.permutation(50), np.random.standard_normal(7), np.random.randint(0, 1000, 9))
    for w, g in zip(want, got):
        assert np.array_equal(w, g)
