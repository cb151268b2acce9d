"""The reference's own control loop (src/agent.py + src/statistics.py through src/main.py's schedule) as a test
of the drop-in boundary — BASELINE configs[0] (replay 10k, batch 32, history 4) and the periodic target sync of
configs[2], on the deterministic synthetic environment (ALE is not installed).

CPU tests (here): tests/golden/agent_loop_golden.npz holds the traces of the mechanically converted reference
Agent + Statistics driving the UNMODIFIED reference replay_memory.py / state_buffer.py and the numpy DQN oracle
(tests/golden/make_agent_golden.py); this repository's restatement of the loop (tests/agent_loop.py) on the oracle
classes reproduces those golden traces: every action, the `random` stream position at every phase boundary, the replay
    cursor, every cost and Q row — so the restatement IS the reference loop, and ReplayOracle / StateBufferOracle
    are the reference's replay / state buffer, as far as the loop can tell.
GPU test: tests/test_gpu_agent_loop.py runs the restatement on the product classes."""
import os

import numpy as np
import pytest

import agent_loop as AL
from conftest import GOLDEN
from synthetic_env import SyntheticEnvironment

CASES = {
    # BASELINE configs[0]: replay 10k, batch 32, history 4, A = 4 (Breakout); 920 env steps, 150 updates, 3 target syncs/epoch
    "breakout10k": dict(num_actions=4, env_seed=3,
                        cfg=dict(random_steps=200, train_steps=300, test_steps=60, target_steps=120,
                                 exploration_decay_steps=250)),
    # A = 6 (Pong), --train_repeat 2, a ring small enough to wrap (replay 400 < 500 env steps), periodic target syncs
    "pong_repeat2": dict(num_actions=6, env_seed=5,
                         cfg=dict(train_repeat=2, target_steps=80, random_steps=100, train_steps=160, test_steps=40,
                                  epochs=2, exploration_decay_steps=150, random_seed=4242, replay_size=400)),
}


def golden(name):
    g = np.load(os.path.join(GOLDEN, "agent_loop_golden.npz"))
    return {k.split("/", 1)[1]: g[k] for k in g.files if k.startswith(name + "/")}


def assert_same_trace(tr, ref, exact_numbers):
    for k in ("actions", "rewards", "terminals", "rng_crc", "mem_cursor"):
        assert (tr[k] == ref[k]).all(), k
    assert np.array_equal(tr["rates"], ref["rates"])
    assert tr["costs"].shape == ref["costs"].shape and tr["q_rows"].shape == ref["q_rows"].shape
    if exact_numbers:
        assert (tr["costs"] == ref["costs"]).all() and (tr["q_rows"] == ref["q_rows"]).all()
    else:   # another host CPU may pick other BLAS kernels: same decisions, numbers to fp32 round-off
        assert np.allclose(tr["costs"], ref["costs"], rtol=1e-4)
        assert np.abs(tr["q_rows"] - ref["q_rows"]).max() <= 1e-4 * np.abs(ref["q_rows"]).max()
    # columns: steps, nr_games, average_reward, min, max, meanq, meancost, weight_updates
    assert np.allclose(tr["phase_rows"], ref["phase_rows"], rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("name", list(CASES))
def test_restated_loop_on_oracle_classes_reproduces_golden(name):
    spec = CASES[name]
    cfg = AL.loop_config(**spec["cfg"])
    OracleReplay, OracleStateBuffer, OracleDQN = AL.oracle_classes()
    env = SyntheticEnvironment(spec["num_actions"], seed=spec["env_seed"])
    tr = AL.run_restated_loop(env, OracleReplay(cfg.replay_size, cfg), OracleDQN(env.numActions(), cfg),
                              OracleStateBuffer(cfg), cfg)
    ref = golden(name)
    assert_same_trace(tr.arrays(), ref, exact_numbers=False)
    assert len(ref["actions"]) == cfg.random_steps + cfg.epochs * (cfg.train_steps + cfg.test_steps)
    assert len(ref["costs"]) == cfg.epochs * cfg.train_repeat * (cfg.train_steps // cfg.train_frequency)


def test_synthetic_environment_is_deterministic_and_action_independent():
    a, b = SyntheticEnvironment(4, seed=3), SyntheticEnvironment(4, seed=3)
    ra, rb, term = [], [], 0
    for t in range(300):
        ra.append(a.act(t % 4)); rb.append(b.act(3 - t % 4))
        assert (a.getScreen() == b.getScreen()).all() and a.isTerminal() == b.isTerminal()
        term += a.isTerminal()
    assert ra == rb and 1 <= term <= 10 and min(ra) < -1 and max(ra) > 1
    assert a.getScreen().shape == (84, 84) and a.getScreen().dtype == np.uint8
