"""Checkpoint fixtures shared by the CPU and GPU tests: the reference's snapshot weights (data, fc1 sampled — see
tests/golden/make_snapshot_fixture.py) and a writer that rebuilds a checkpoint FILE with the reference's own pickle
structure around them."""
import json
import os
import pickle

import numpy as np

from conftest import GOLDEN


def fixture():
    g = np.load(os.path.join(GOLDEN, "snapshot_breakout_77.npz"))
    return [g["W%d" % i] for i in range(5)], [g["S%d" % i] for i in range(5)], g["q_kat"]


def game_fixture(name):
    """(W, S) of the breakout fixture with fc2 replaced by snapshot `name`'s fc2 columns of the kept fc1 units."""
    g = np.load(os.path.join(GOLDEN, "snapshot_breakout_77.npz"))
    ws, ss, _ = fixture()
    w4, s4 = g[name + "/W4"], g[name + "/S4"]
    ws[4] = np.zeros((w4.shape[0], ws[4].shape[1]), np.float32)
    ss[4] = np.zeros_like(ws[4])
    ws[4][:, g["fc1_units"]] = w4
    ss[4][:, g["fc1_units"]] = s4
    return ws, ss


def rebuild(skel, arrays):
    """Inverse of make_snapshot_fixture.skeleton(): arrays are consumed in traversal order."""
    if isinstance(skel, dict):
        if skel.get("__ndarray__"):
            a = next(arrays)
            # only fc2 (the one layer with 512 columns) may have another number of rows: the action count
            assert list(a.shape) == skel["shape"] or (skel["shape"][1:] == [512] and a.shape[1:] == (512,)), \
                (a.shape, skel["shape"])
            return a
        if "__seq__" in skel:
            items = [rebuild(v, arrays) for v in skel["items"]]
            return tuple(items) if skel["__seq__"] == "tuple" else items
        return {k: rebuild(v, arrays) for k, v in skel.items()}
    return skel


def write_checkpoint(path, layout, ws, ss):
    """A checkpoint file with the reference's own structure (keys, nesting, type strings) around (ws, ss)."""
    meta = json.load(open(os.path.join(GOLDEN, "snapshot_layouts.json")))
    skel = meta["breakout_77" if layout == "pre-1.0" else "seaquest_178"]["skeleton"]
    order = []
    if layout == "pre-1.0":
        for w, s in zip(ws, ss):            # dict traversal order of the skeleton: params before states
            order += [w, s]
        d = rebuild(skel, iter(order))
    else:
        # json sorted the keys: inside a layer dict "params" precedes "states"
        for w, s in zip(ws, ss):
            order += [w, s]
        d = rebuild(skel, iter(order))
        d["model"]["config"]["layers"][-1]["config"]["nout"] = int(ws[4].shape[0])
    with open(path, "wb") as f:
        pickle.dump(d, f, protocol=2)
    return d


