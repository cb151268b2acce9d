"""Generate tests/golden/agent_loop_golden.npz: traces of the REFERENCE's own control loop (src/agent.py +
src/statistics.py, mechanically converted to Python 3 in a temp dir) driving the reference's unmodified
replay_memory.py / state_buffer.py and the numpy DQN oracle through the schedule of src/main.py:130-162, on the
deterministic synthetic environment:

    python tests/golden/make_agent_golden.py <simple_dqn checkout>

Cases: "breakout10k" = BASELINE configs[0] shape (replay 10k, batch 32, history 4, A = 4, train_repeat 1);
"pong_repeat2" = A = 6 with --train_repeat 2 and target syncs every 120 steps (configs[2]'s periodic
update_target_network, scaled)."""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import agent_loop as AL  # noqa: E402
import ref_convert as RC  # noqa: E402
from synthetic_env import SyntheticEnvironment  # noqa: E402

from test_agent_loop import CASES  # noqa: E402  (one definition of the cases: the tests own it)


def run_case(name, spec, tmp):
    cfg = AL.loop_config(**spec["cfg"])
    RefReplay, RefStateBuffer = RC.load_reference_replay_and_statebuffer()
    Agent, Statistics = RC.load_agent_and_statistics(tmp, RefStateBuffer, tag=name)
    _, _, OracleDQN = AL.oracle_classes()
    env = SyntheticEnvironment(spec["num_actions"], seed=spec["env_seed"])
    mem = RefReplay(cfg.replay_size, cfg)
    net = OracleDQN(env.numActions(), cfg)
    return cfg, AL.run_reference_loop(Agent, Statistics, env, mem, net, cfg, os.path.join(tmp, name + ".csv"))


def top2_gap(q_rows):
    s = np.sort(q_rows, axis=1)
    return (s[:, -1] - s[:, -2]) / np.abs(q_rows).max(axis=1)


def main():
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        assert RC.convert(tmp) == {"agent.py": 7, "statistics.py": 6}      # the whole py2 -> py3 conversion: 13 lines
        for name, spec in CASES.items():
            cfg, tr = run_case(name, spec, tmp)
            arr = tr.arrays()
            for k, v in arr.items():
                out["%s/%s" % (name, k)] = v
            gap = top2_gap(arr["q_rows"])
            out[name + "/min_rel_gap"] = np.float64(gap.min())
            print("%s: %d steps, %d updates, %d predicts, min relative top-2 Q gap %.3e (median %.3e), last cost %.6g"
                  % (name, len(arr["actions"]), len(arr["costs"]), len(arr["q_rows"]), gap.min(), np.median(gap),
                     arr["costs"][-1]))
    np.savez_compressed(os.path.join(HERE, "agent_loop_golden.npz"), **out)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_agent_golden.py <simple_dqn checkout>")
    RC.REFERENCE_SRC = os.path.join(sys.argv[1], "src")
    main()
