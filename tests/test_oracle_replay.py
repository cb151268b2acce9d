"""Pin the replay oracle: against CPython's ``random`` and against golden vectors produced by the
unmodified reference (tests/golden/make_golden.py)."""
import os
import random
import zlib

import numpy as np
import pytest

from conftest import GOLDEN
from oracle.mt19937 import MT19937, twist_segmented, twist_sequential
from oracle.replay_oracle import (ReplayOracle, StateBufferOracle, decode_frame_tag,
                                  indexed_episode_stream)


def crc(a):
    return np.uint32(zlib.crc32(np.ascontiguousarray(a).tobytes()))


def test_mt19937_kat_survey_a5():
    # SURVEY §8 a5 known-answer vectors (CPython 3 semantics)
    random.seed(123)
    g = MT19937.from_python(random)
    assert [g.randint(4, 999999) for _ in range(6)] == [54911, 280683, 91425, 806313, 427027, 279505]
    random.seed(123)
    g = MT19937.from_python(random)
    assert [g.randint(4, 9999) for _ in range(5)] == [861, 4389, 1432, 6676, 4371]


@pytest.mark.parametrize("seed", [0, 1, 7, 2 ** 40 + 3])
def test_mt19937_matches_cpython_stream(seed):
    r = random.Random(seed)
    g = MT19937.from_python(r)
    for hi in (5, 9999, 999999, 2 ** 31):
        assert [g.randint(4, hi) for _ in range(700)] == [r.randint(4, hi) for _ in range(700)]
    # and the state can be handed back
    g.to_python(r)
    assert r.getrandbits(32) == g.genrand_uint32()


def test_twist_segmented_equals_sequential():
    for seed in range(5):
        st = np.array(random.Random(seed).getstate()[1][:624], dtype=np.uint32)
        assert (twist_sequential(st) == twist_segmented(st)).all()


def _build(case, g):
    size, steps, batch, seed, nmb = [int(x) for x in g[case + "/cfg"]]
    tp = float(g[case + "/terminal_p"])
    mem = ReplayOracle(size, batch_size=batch)
    for (a, r, s, t) in indexed_episode_stream(steps, seed=seed, terminal_p=tp):
        mem.add(a, r, s, t)
    return mem, size, steps, batch, seed, nmb


def test_replay_oracle_matches_reference_golden():
    g = np.load(os.path.join(GOLDEN, "replay_golden.npz"))
    for case in g["names"]:
        mem, size, steps, batch, seed, nmb = _build(case, g)
        assert [mem.count, mem.current] == list(g[case + "/count_current"])
        rng = MT19937(g[case + "/mt_before"])
        for i in range(nmb):
            idx = mem.sample_indexes(rng)
            assert (idx == g[case + "/indexes"][i]).all(), case
            pre, a, r, post, t = mem.gather(idx)
            assert crc(pre) == g[case + "/pre_crc"][i] and crc(post) == g[case + "/post_crc"][i]
            assert (a == g[case + "/actions"][i]).all() and a.dtype == np.uint8
            assert (r == g[case + "/rewards"][i]).all() and r.dtype == np.int64
            assert (t == g[case + "/terminals"][i]).all() and t.dtype == np.bool_
        assert rng.state625() == [int(x) for x in g[case + "/mt_after"]], "stream position after sampling"
        assert (pre[0] == g[case + "/last_pre_sample0"]).all()
        assert (mem.getState(-1) == g[case + "/getState_m1"]).all()
        assert (mem.getState(2) == g[case + "/getState_2"]).all()


def test_state_buffer_oracle_matches_reference_golden():
    g = np.load(os.path.join(GOLDEN, "replay_golden.npz"))
    buf = StateBufferOracle()
    for (_, _, s, _) in indexed_episode_stream(10, seed=21):
        buf.add(s)
    assert (decode_frame_tag(buf.getState()) == g["statebuffer/row0_tags"]).all()
    assert crc(buf.getStateMinibatch()) == g["statebuffer/crc"]
    buf.reset()
    assert not buf.getStateMinibatch().any()


def test_replay_oracle_live_against_reference_file():
    """The oracle's minibatches equal those the unmodified reference replay_memory.py drew from the same adds and
    the same `random` stream (tests/golden/make_golden.py::live_case)."""
    g = np.load(os.path.join(GOLDEN, "replay_live_golden.npz"))
    mem = ReplayOracle(500)
    for (a, r, s, t) in indexed_episode_stream(1300, seed=3, terminal_p=0.03):
        mem.add(a, r, s, t)
    random.seed(99)
    assert list(random.getstate()[1]) == [int(x) for x in g["mt_before"]]
    rng = MT19937.from_python(random)
    for i in range(20):
        op, oa, orr, oq, ot = mem.getMinibatch(rng)
        assert crc(op) == g["pre_crc"][i] and crc(oq) == g["post_crc"][i], i
        assert (oa == g["actions"][i]).all() and (orr == g["rewards"][i]).all() and (ot == g["terminals"][i]).all()
    assert rng.state625() == [int(x) for x in g["mt_after"]]
