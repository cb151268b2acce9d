"""Generate tests/golden/snapshot_breakout_77.npz and snapshot_layouts.json from the original simple_dqn
project's shipped checkpoints (its snapshots/*.pkl):

    python tests/golden/make_snapshot_fixture.py <simple_dqn checkout>

What is kept (data only — no source of the original project):
  * breakout_77.pkl (pre-1.0 ``layer_params_states`` layout): the fp32 W and RMSProp state of conv1-3 and fc2
    bit for bit, and of fc1 the rows of the FC1_UNITS hidden units that carry most of the Q-values on the KAT
    input of SURVEY §8(c) (RandomState(1234) states), bit for bit, every other fc1 row zero.  A zero fc1 row
    is a dead ReLU unit: no Q contribution, no gradient, no update, so the sampled network is a complete trained
    network in the trained regime (|Q| ~ 4) that fits in a small file.  ``fc1_units`` names the rows kept and
    ``q_kat`` holds the fp32 Q-values the numpy oracle computes from the sampled weights on the KAT input;
  * of breakout_77, seaquest_178, pong_141 and space_invaders_126 (both layouts; 4, 18, 3 and 6 actions): the fc2
    W and RMSProp state columns of the same units, ``<name>/W4`` and ``<name>/S4``;
  * seaquest_178.pkl (neon 1.3.0 layout): the pickle's SKELETON — every key, type string and config
    dict of the 9-entry layer list with the arrays replaced by (shape, dtype, crc32) — so that tests can
    rebuild a byte-faithful 1.3.0-layout checkpoint around any weights and check that the product's
    writer emits the same structure; likewise breakout_77.pkl's skeleton for the pre-1.0 layout.  The CRCs
    are those of the full arrays of both files.
"""
import json
import os
import pickle
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import dqn_oracle as O  # noqa: E402

# 12 units: Q stays in the trained regime, and the sampled network is well conditioned for the 5-step training
# test (with 8, one unit's pre-activation sits near zero there and fp32 rounding decides the ReLU)
FC1_UNITS = 12
GAMES = {"breakout_77": 4, "seaquest_178": 18, "pong_141": 3, "space_invaders_126": 6}


def crc(a):
    return int(zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xffffffff)


def skeleton(obj):
    """The structure of a checkpoint with every ndarray replaced by a descriptor."""
    if isinstance(obj, np.ndarray):
        return {"__ndarray__": True, "shape": list(obj.shape), "dtype": str(obj.dtype), "crc32": crc(obj)}
    if isinstance(obj, dict):
        return {str(k): skeleton(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return {"__seq__": type(obj).__name__, "items": [skeleton(v) for v in obj]}
    if isinstance(obj, (np.integer,)):
        return int(obj)
    if isinstance(obj, (np.floating,)):
        return float(obj)
    if isinstance(obj, bytes):
        return obj.decode("latin1")
    return obj


def kat_states():
    return np.random.RandomState(1234).randint(0, 256, (32, 4, 84, 84)).astype(np.uint8)


def main(snap):
    ws, ss = O.load_snapshot(os.path.join(snap, "breakout_77.pkl"))
    ws = [np.asarray(w, np.float32) for w in ws]
    ss = [np.asarray(s, np.float32) for s in ss]
    q, acts = O.forward(ws, kat_states(), keep=True)
    assert np.allclose(q[0], [4.052785, 3.199721, 5.557730, 4.043888], atol=2e-5)   # SURVEY §8(c) KAT
    # each unit's share of the Q-values on the KAT input: mean activation x norm of its fc2 column
    share = acts["h4"].mean(0) * np.linalg.norm(ws[4], axis=0)
    units = np.sort(np.argsort(-share, kind="stable")[:FC1_UNITS])
    keep = np.zeros(ws[3].shape[0], bool)
    keep[units] = True
    ws[3][~keep] = 0
    ss[3][~keep] = 0
    out = {"q_kat": O.forward(ws, kat_states()).astype(np.float32), "fc1_units": units.astype(np.int64)}
    for i, (w, s) in enumerate(zip(ws, ss)):
        out["W%d" % i] = w
        out["S%d" % i] = s
    for name, actions in GAMES.items():
        gw, gs = O.load_snapshot(os.path.join(snap, name + ".pkl"))
        assert gw[4].shape == (actions, 512)
        out[name + "/W4"] = np.ascontiguousarray(np.asarray(gw[4], np.float32)[:, units])
        out[name + "/S4"] = np.ascontiguousarray(np.asarray(gs[4], np.float32)[:, units])
    np.savez_compressed(os.path.join(HERE, "snapshot_breakout_77.npz"), **out)

    with open(os.path.join(snap, "breakout_77.pkl"), "rb") as f:
        old = pickle.load(f, encoding="latin1")
    with open(os.path.join(snap, "seaquest_178.pkl"), "rb") as f:
        new = pickle.load(f, encoding="latin1")
    new = dict(new)
    new["backend"] = {k: v for k, v in new["backend"].items() if k != "rng_state"}   # 0.8 MB of RNG words: dropped
    meta = {"breakout_77": {"layout": "pre-1.0 layer_params_states", "skeleton": skeleton(old)},
            "seaquest_178": {"layout": "neon 1.3.0", "skeleton": skeleton(new),
                             "note": "backend.rng_state (NervanaGPU RNG words) omitted from the skeleton"}}
    with open(os.path.join(HERE, "snapshot_layouts.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    print("wrote", os.path.getsize(os.path.join(HERE, "snapshot_breakout_77.npz")), "bytes of weights")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_snapshot_fixture.py <simple_dqn checkout>")
    main(os.path.join(sys.argv[1], "snapshots"))
