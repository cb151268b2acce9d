"""CPU half of the checkpoint tests: the committed snapshot fixture is what the reference ships (checked against
the CRCs of the reference's arrays), both rebuilt checkpoint layouts parse, and the numpy oracle reproduces the
fixture's Q-value KAT from them.  The device half is tests/test_gpu_checkpoint.py."""
import json
import os
import zlib

import numpy as np
import pytest

from ckpt_helpers import fixture, write_checkpoint
from conftest import GOLDEN
from oracle import dqn_oracle as O


@pytest.mark.parametrize("layout", ["pre-1.0", "neon-1.3.0"])
def test_rebuilt_checkpoints_parse_and_reproduce_the_kat(tmp_path, layout):
    ws, ss, q_kat = fixture()
    path = str(tmp_path / "c.pkl")
    d = write_checkpoint(path, layout, ws, ss)
    if layout == "neon-1.3.0":
        assert d["neon_version"] == "1.3.0+344372b" and len(d["model"]["config"]["layers"]) == 9
    w2, s2 = O.load_snapshot(path)
    assert all((a == b).all() for a, b in zip(w2, ws)) and all((a == b).all() for a, b in zip(s2, ss))
    states = np.random.RandomState(1234).randint(0, 256, (32, 4, 84, 84)).astype(np.uint8)
    q = O.forward(w2, states)
    assert np.allclose(q[0], [4.393127, 3.402484, 5.425210, 4.558548], atol=2e-5)
    assert (q == q_kat).all()


def test_fixture_is_the_reference_snapshot_bit_for_bit():
    """conv1-3 and fc2 are breakout_77's arrays (CRC32 of the reference's arrays, recorded in the layout skeleton);
    fc1 keeps only the rows of the sampled units, and fc2's columns of them are also stored on their own."""
    ws, ss, _ = fixture()
    g = np.load(os.path.join(GOLDEN, "snapshot_breakout_77.npz"))
    meta = json.load(open(os.path.join(GOLDEN, "snapshot_layouts.json")))
    sk = meta["breakout_77"]["skeleton"]["layer_params_states"]["items"]
    for l in (0, 1, 2, 4):
        assert ws[l].dtype == np.float32 and ss[l].dtype == np.float32
        assert (zlib.crc32(ws[l].tobytes()) & 0xffffffff) == sk[l]["params"]["W"]["crc32"], l
        assert (zlib.crc32(ss[l].tobytes()) & 0xffffffff) == sk[l]["states"]["items"][0]["crc32"], l
    units = g["fc1_units"]
    dead = np.ones(ws[3].shape[0], bool)
    dead[units] = False
    assert len(units) == 12 and not ws[3][dead].any() and not ss[3][dead].any()
    assert (ws[3][units] != 0).all(axis=1).any() and (ss[3][units] > 0).all()
    assert (g["breakout_77/W4"] == ws[4][:, units]).all() and (g["breakout_77/S4"] == ss[4][:, units]).all()
    for name, actions in (("seaquest_178", 18), ("pong_141", 3), ("space_invaders_126", 6)):
        assert g[name + "/W4"].shape == g[name + "/S4"].shape == (actions, len(units))
