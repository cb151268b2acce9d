"""Generate tests/golden/replay_golden.npz and replay_live_golden.npz by running the UNMODIFIED files
src/replay_memory.py and src/state_buffer.py of the original simple_dqn project:

    python tests/golden/make_golden.py <simple_dqn checkout>

The only accommodation is the numpy shim of SURVEY §8(c): numpy >= 2 removed the
ability to use the abstract ``np.integer`` as a dtype (replay_memory.py:11), so the
module's ``np`` name is rebound to a namespace whose ``integer`` is ``np.int64``
(what ``np.integer`` meant on the reference's numpy).  The reference source is not edited.
"""
import os
import random
import sys
import types
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.replay_oracle import indexed_episode_stream, decode_frame_tag  # noqa: E402

# (name, ring size, env steps added, batch, terminal_p, python seed, minibatches)
CASES = [
    ("small_unwrapped", 97, 60, 32, 0.02, 11, 4),
    ("small_wrapped", 97, 250, 32, 0.02, 12, 4),
    ("terminal_heavy", 300, 700, 32, 0.20, 13, 4),
    ("batch256", 2000, 4100, 256, 0.01, 14, 2),
    ("minimal_count", 50, 6, 1, 0.0, 15, 3),
    ("exact_fill", 128, 128, 32, 0.05, 16, 3),
]


def load_reference(ref_src):
    sys.path.insert(0, ref_src)
    import replay_memory
    import state_buffer
    shim = types.SimpleNamespace(**{k: getattr(np, k) for k in dir(np) if not k.startswith("__")})
    shim.integer = np.int64
    replay_memory.np = shim
    return replay_memory, state_buffer


def crc(a):
    return np.uint32(zlib.crc32(np.ascontiguousarray(a).tobytes()))


def live_case(replay_memory):
    """A ring of 500 wrapped by 1300 adds and 20 minibatches from random.seed(99), in the order the replay oracle
    draws them (tests/test_oracle_replay.py::test_replay_oracle_live_against_reference_file)."""
    args = types.SimpleNamespace(screen_height=84, screen_width=84, history_length=4, batch_size=32)
    mem = replay_memory.ReplayMemory(500, args)
    for (a, r, s, t) in indexed_episode_stream(1300, seed=3, terminal_p=0.03):
        mem.add(a, r, s, t)
    random.seed(99)
    out = {"mt_before": np.array(random.getstate()[1], dtype=np.uint32)}
    rows = {k: [] for k in ("pre_crc", "post_crc", "actions", "rewards", "terminals")}
    for _ in range(20):
        pre, a, r, post, t = mem.getMinibatch()
        rows["pre_crc"].append(crc(pre)); rows["post_crc"].append(crc(post))
        rows["actions"].append(a.copy()); rows["rewards"].append(r.copy()); rows["terminals"].append(t.copy())
    out.update({k: np.stack(v) for k, v in rows.items()})
    out["mt_after"] = np.array(random.getstate()[1], dtype=np.uint32)
    return out


def main(ref_src):
    replay_memory, state_buffer = load_reference(ref_src)
    out = {}
    names = []
    for (name, size, steps, batch, tp, seed, nmb) in CASES:
        args = types.SimpleNamespace(screen_height=84, screen_width=84, history_length=4, batch_size=batch)
        mem = replay_memory.ReplayMemory(size, args)
        for (a, r, s, t) in indexed_episode_stream(steps, seed=seed, terminal_p=tp):
            mem.add(a, r, s, t)
        random.seed(seed)
        state_before = random.getstate()[1]
        idx, acts, rews, terms, pre_crc, post_crc = [], [], [], [], [], []
        for _ in range(nmb):
            pre, a, r, post, t = mem.getMinibatch()
            idx.append(decode_frame_tag(post[:, 3]) % size if size < steps else decode_frame_tag(post[:, 3]))
            acts.append(a.copy()); rews.append(r.copy()); terms.append(t.copy())
            pre_crc.append(crc(pre)); post_crc.append(crc(post))
        state_after = random.getstate()[1]
        names.append(name)
        out[name + "/cfg"] = np.array([size, steps, batch, seed, nmb], dtype=np.int64)
        out[name + "/terminal_p"] = np.float64(tp)
        out[name + "/count_current"] = np.array([mem.count, mem.current], dtype=np.int64)
        out[name + "/mt_before"] = np.array(state_before, dtype=np.uint32)
        out[name + "/mt_after"] = np.array(state_after, dtype=np.uint32)
        out[name + "/indexes"] = np.stack(idx)
        out[name + "/actions"] = np.stack(acts)
        out[name + "/rewards"] = np.stack(rews)
        out[name + "/terminals"] = np.stack(terms)
        out[name + "/pre_crc"] = np.array(pre_crc, dtype=np.uint32)
        out[name + "/post_crc"] = np.array(post_crc, dtype=np.uint32)
        out[name + "/last_pre_sample0"] = pre[0].copy()          # a few raw bytes, not only CRCs
        out[name + "/getState_m1"] = mem.getState(-1).copy()     # wrap-around / negative index path
        out[name + "/getState_2"] = mem.getState(2).copy()       # slow list path (index < 3)

    # state_buffer.py: 10 adds, snapshot of row 0 and the full-batch CRC
    args = types.SimpleNamespace(screen_height=84, screen_width=84, history_length=4, batch_size=32)
    buf = state_buffer.StateBuffer(args)
    for (_, _, s, _) in indexed_episode_stream(10, seed=21):
        buf.add(s)
    out["statebuffer/row0_tags"] = decode_frame_tag(buf.getState())
    out["statebuffer/crc"] = crc(buf.getStateMinibatch())
    out["names"] = np.array(names)
    path = os.path.join(HERE, "replay_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")
    path = os.path.join(HERE, "replay_live_golden.npz")
    np.savez_compressed(path, **live_case(replay_memory))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_golden.py <simple_dqn checkout>")
    main(os.path.join(sys.argv[1], "src"))
