"""Cross-check the numpy Nature-DQN oracle against an independent torch-CPU autograd
implementation, and against the Q-value KAT of the shipped breakout_77 snapshot (tests/golden).
The Neon arithmetic itself cannot be run anywhere (parity unpinned — see oracle/__init__.py)."""
import json
import os

import numpy as np
import torch

from ckpt_helpers import fixture
from conftest import GOLDEN
from oracle import dqn_oracle as O


def torch_forward(ws, x):
    h = x.float() / 255
    for li, (r, s, k, st) in enumerate(O.CONV_GEOM):
        c = h.shape[1]
        w = ws[li].reshape(c, r, s, k).permute(3, 0, 1, 2)       # CRSK → KCRS
        h = torch.relu(torch.nn.functional.conv2d(h, w, stride=st))
    h = torch.relu(h.flatten(1) @ ws[3].T)
    return h @ ws[4].T


def _batch(n, a, seed):
    rs = np.random.RandomState(seed)
    pre = rs.randint(0, 256, (n, 4, 84, 84)).astype(np.uint8)
    post = rs.randint(0, 256, (n, 4, 84, 84)).astype(np.uint8)
    return pre, rs.randint(0, a, n).astype(np.uint8), rs.randint(-3, 4, n).astype(np.int64), post, rs.rand(n) < 0.3


def test_shapes_and_param_count():
    shp = O.layer_shapes(4)
    assert shp == [(256, 32), (512, 64), (576, 64), (512, 3136), (4, 512)]
    assert sum(a * b for a, b in shp) == 1685504          # SURVEY §8 a7


def test_forward_backward_match_torch_autograd():
    ws = O.xavier_init(6, seed=3)
    pre, *_ = _batch(8, 6, 0)
    q, acts = O.forward(ws, pre, keep=True)
    tw = [torch.tensor(w, requires_grad=True) for w in ws]
    tq = torch_forward(tw, torch.tensor(pre))
    assert np.abs(tq.detach().numpy() - q).max() <= 1e-5 * np.abs(q).max()
    d = np.random.RandomState(1).randn(8, 6).astype(np.float32)
    tq.backward(torch.tensor(d))
    for g, t in zip(O.backward(ws, acts, d), tw):
        ref = t.grad.numpy()
        # L2 metric: a single ReLU-mask flip at a ~0 pre-activation is a legitimate fp32 difference
        assert np.linalg.norm(g - ref) <= 1e-4 * np.linalg.norm(ref)


def test_train_step_semantics():
    """cost before clip, terminal branch, reward clip, RMSProp with g = dW / N (deepqnetwork.py:133-165)."""
    n, a = 8, 4
    net = O.DQNOracle(a, batch_size=n, seed=5)
    w0 = [w.copy() for w in net.weights]
    mb = _batch(n, a, 2)
    cost = net.train(mb)
    pre, act, rew, post, term = mb
    postq = O.forward(w0, post)
    preq = O.forward(w0, pre)
    r = np.clip(rew, -1, 1)
    y = np.where(term, r, r + 0.99 * postq.max(1))
    delta = preq[np.arange(n), act] - y
    assert np.isclose(cost, np.mean(delta ** 2 / 2), rtol=1e-5)
    assert np.allclose(net.last["deltas"][np.arange(n), act], np.clip(delta, -1, 1), atol=1e-6)
    assert np.count_nonzero(net.last["deltas"]) <= n
    g = net.last["grads"][4] / n
    s = 0.05 * g * g
    assert np.allclose(net.weights[4], w0[4] - 0.00025 * g / (np.sqrt(s + 1e-6) + 1e-6), atol=1e-7)
    assert net.train_iterations == 1
    # target net untouched until update_target_network
    assert all((t == w).all() for t, w in zip(net.target_weights, w0))
    net.update_target_network()
    assert all((t == w).all() for t, w in zip(net.target_weights, net.weights))


def test_snapshot_kat_breakout_77():
    """breakout_77 with fc1 sampled (tests/golden/make_snapshot_fixture.py); the full network's KAT of SURVEY §8(c)
    was asserted when the fixture was made."""
    ws, ss, _ = fixture()
    assert [w.shape for w in ws] == O.layer_shapes(4) == [s.shape for s in ss]
    states = np.random.RandomState(1234).randint(0, 256, (32, 4, 84, 84)).astype(np.uint8)
    q = O.forward(ws, states)
    assert np.allclose(q[0], [4.393127, 3.402484, 5.425210, 4.558548], atol=2e-5)
    assert np.allclose(q[31], [0.011635, -0.392340, 1.878573, 0.668184], atol=2e-5)
    meta = json.load(open(os.path.join(GOLDEN, "snapshot_layouts.json")))
    sk = meta["seaquest_178"]["skeleton"]["model"]["config"]["layers"]["items"]     # neon-1.3.0 layout
    assert [tuple(l["params"]["W"]["shape"]) for l in sk if "params" in l] == O.layer_shapes(18)
