"""§8 a17 / f2: the reference's shipped checkpoints through the PRODUCT on the device.

tests/golden/snapshot_breakout_77.npz holds the fp32 W and RMSProp state of the reference's breakout_77.pkl bit for
bit, with fc1 sampled to its 12 most active units (generator: tests/golden/make_snapshot_fixture.py), and the fc2
columns of those units from four shipped snapshots; snapshot_layouts.json holds the structure of both pickle layouts
found in snapshots/.  The tests rebuild a checkpoint file in EACH layout around those weights, load it with
DeepQNetwork.load_weights (src/deepqnetwork.py:188-189) and hold the device to the fixture's Q-value known answer;
then train on the trained weights (every other GPU test runs on Xavier weights) and round-trip through
save_weights (:191-192)."""
import json
import os
import pickle

import numpy as np
import pytest

from conftest import GOLDEN
from helpers import make_args, random_minibatch, rel_l2
from oracle import dqn_oracle as O

pytestmark = pytest.mark.gpu
MODES = ["fp32", "tcgen05"]
KAT_Q0 = [4.393127, 3.402484, 5.425210, 4.558548]          # breakout_77 weights, fc1 sampled
KAT_Q31 = [0.011635, -0.392340, 1.878573, 0.668184]


from ckpt_helpers import fixture as _fixture, game_fixture, write_checkpoint as _write_checkpoint


def _net(mode, **kw):
    from simple_dqn_b200 import DeepQNetwork
    return DeepQNetwork(4, make_args(**kw), math_mode=mode)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("layout", ["pre-1.0", "neon-1.3.0"])
def test_load_reference_layouts_and_q_kat(tmp_path, mode, layout):
    ws, ss, q_kat = _fixture()
    path = str(tmp_path / "ckpt.pkl")
    _write_checkpoint(path, layout, ws, ss)
    net = _net(mode, random_seed=5)
    net.load_weights(path)
    w1, s1 = net.get_weights()
    for l in range(5):
        assert (w1[l] == ws[l]).all() and (s1[l] == ss[l]).all(), l           # weights AND optimizer state, bit for bit
    states = np.random.RandomState(1234).randint(0, 256, (32, 4, 84, 84)).astype(np.uint8)
    q = net.predict(states)
    assert np.allclose(q[0], KAT_Q0, atol=2e-5 * 5.6) and np.allclose(q[31], KAT_Q31, atol=2e-5 * 5.6), (q[0], q[31])
    assert np.abs(q - q_kat).max() <= 1e-3 * np.abs(q_kat).max()             # north_star's bar; measured ~1e-5
    assert np.abs(q - q_kat).max() <= 5e-5 * np.abs(q_kat).max(), np.abs(q - q_kat).max() / np.abs(q_kat).max()


@pytest.mark.parametrize("mode", MODES)
def test_train_on_trained_weights(mode):
    """One step and a 5-step trajectory starting from the reference's trained (W, S): the regime the published
    runs spend their time in (large Q, saturated second moments), unlike Xavier x 3."""
    from simple_dqn_b200 import Stream
    ws, ss, _ = _fixture()
    from simple_dqn_b200 import DeepQNetwork
    net = DeepQNetwork(4, make_args(), math_mode=mode, stream=Stream())
    net.set_weights(ws, ss)
    net.update_target_network()
    net.keep_grads(True)
    orc = O.DQNOracle(4, weights=ws, states=ss)
    for i in range(5):
        mb = random_minibatch(32, 4, 70 + i, terminal_p=0.05, reward_range=(-1, 2))
        net.train(mb, 0)
        ref_cost = float(orc.train(mb))
        cost = float(net.last_costs(1)[0])
        assert abs(cost - ref_cost) <= 1e-3 * abs(ref_cost), (i, cost, ref_cost)
        if i == 0:
            preq, postq = net.last_q()
            assert np.abs(preq - orc.last["preq"]).max() <= 1e-3 * np.abs(orc.last["preq"]).max()
            assert np.abs(postq - orc.last["postq"]).max() <= 1e-3 * np.abs(orc.last["postq"]).max()
            for l, (g, r) in enumerate(zip(net.get_grads(), orc.last["grads"])):
                assert rel_l2(g, r) <= 2e-3, (l, rel_l2(g, r))
    w1 = net.get_weights(with_states=False)
    for l in range(5):
        assert rel_l2(w1[l] - ws[l], orc.weights[l] - ws[l]) <= 2e-2, (l, rel_l2(w1[l] - ws[l], orc.weights[l] - ws[l]))


@pytest.mark.parametrize("layout", ["pre-1.0", "neon-1.3.0"])
def test_save_weights_structure_matches_reference_layout(tmp_path, layout):
    """What save_weights writes has the reference layout's keys, nesting and type strings (skeleton compare)."""
    ws, ss, _ = _fixture()
    net = _net("fp32")
    net.set_weights(ws, ss)
    path = str(tmp_path / "out.pkl")
    net.save_weights(path, layout=layout)
    d = pickle.load(open(path, "rb"))
    meta = json.load(open(os.path.join(GOLDEN, "snapshot_layouts.json")))
    skel = meta["breakout_77" if layout == "pre-1.0" else "seaquest_178"]["skeleton"]

    def same_shape(a, sk, where):
        if isinstance(sk, dict) and sk.get("__ndarray__"):
            assert isinstance(a, np.ndarray) and a.dtype == np.float32, where
        elif isinstance(sk, dict) and "__seq__" in sk:
            assert isinstance(a, (list, tuple)) and len(a) == len(sk["items"]), where
            for i, (x, y) in enumerate(zip(a, sk["items"])):
                same_shape(x, y, where + "[%d]" % i)
        elif isinstance(sk, dict):
            assert isinstance(a, dict), where
            want = set(sk) - {"init"}                     # the snapshot's era drew Gaussian(0.01); today's code Xavier
            assert want <= set(a), (where, want - set(a))
            for k in want:
                same_shape(a[k], sk[k], where + "." + k)
        elif isinstance(sk, str) and where.endswith(".type") and "backend" not in where:
            assert a == sk, (where, a, sk)

    if layout == "pre-1.0":
        same_shape(d, skel, "ckpt")
    else:
        same_shape({k: v for k, v in d.items() if k != "backend"}, {k: v for k, v in skel.items() if k != "backend"},
                   "ckpt")
    for (w, s), l in zip(zip(ws, ss), d["layer_params_states"] if layout == "pre-1.0" else
                         [l for l in d["model"]["config"]["layers"] if "params" in l]):
        assert (l["params"]["W"] == w).all() and (l["states"][0] == s).all()


@pytest.mark.parametrize("name,actions", [("breakout_77", 4), ("seaquest_178", 18), ("pong_141", 3),
                                          ("space_invaders_126", 6)])
def test_live_reference_snapshots(tmp_path, name, actions):
    """Each shipped snapshot's layout and action count through load_weights: the fixture's conv and fc1 layers with
    that snapshot's fc2 columns of the fixture's fc1 units."""
    from simple_dqn_b200 import DeepQNetwork
    path = str(tmp_path / ("%s.pkl" % name))
    layout = "pre-1.0" if name in ("breakout_77", "pong_141") else "neon-1.3.0"
    _write_checkpoint(path, layout, *game_fixture(name))
    net = DeepQNetwork(actions, make_args(), math_mode="tcgen05")
    net.load_weights(path)
    ws, ss = O.load_snapshot(path)
    assert ws[4].shape == (actions, 512)
    states = np.random.RandomState(1234).randint(0, 256, (32, 4, 84, 84)).astype(np.uint8)
    ref = O.forward(ws, states)
    assert np.abs(net.predict(states) - ref).max() <= 1e-3 * np.abs(ref).max()
