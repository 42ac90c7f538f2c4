"""Logger writes the reference's on-disk layout (SURVEY.md 8f rank 4); checked against arrays recorded from the reference's
own Logger (tests/golden/logger_reference.npz, made by tests/golden/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest

from gym_pybullet_drones_b200.utils import Logger


def test_logger_layout_and_roundtrip(tmp_path):
    lg = Logger(logging_freq_hz=48, output_folder=str(tmp_path), num_drones=2)
    rng = np.random.default_rng(0)
    states = rng.normal(size=(5, 2, 20)); ctrls = rng.normal(size=(5, 2, 12))
    for t in range(5):
        if t % 2:
            lg.log_all(t / 48, states[t], ctrls[t])
        else:
            for j in range(2):
                lg.log(drone=j, timestamp=t / 48, state=states[t, j], control=ctrls[t, j])
    path = lg.save()
    d = np.load(path)
    assert d["timestamps"].shape == (2, 5) and d["states"].shape == (2, 16, 5) and d["controls"].shape == (2, 12, 5)
    want = np.concatenate([states[..., 0:3], states[..., 10:13], states[..., 7:10], states[..., 13:20]], axis=-1)   # Logger.py:117
    assert np.array_equal(d["states"], want.transpose(1, 2, 0)) and np.array_equal(d["controls"], ctrls.transpose(1, 2, 0))
    assert os.path.isdir(lg.save_as_csv("x"))
    with pytest.raises(ValueError):
        lg.log(drone=3, timestamp=0, state=states[0, 0])


def test_logger_matches_reference_logger(golden, tmp_path):
    """The reference's Logger fed the same entries, one drone at a time, holds the same arrays."""
    g = golden("logger_reference")
    nd = g["state"].shape[1]
    lg = Logger(logging_freq_hz=48, output_folder=str(tmp_path), num_drones=nd)
    for t in range(len(g["timestamp"])):
        for j in range(nd):
            lg.log(drone=j, timestamp=g["timestamp"][t], state=g["state"][t, j], control=g["control"][t, j])
    ts, st, ct = lg._trimmed()
    assert np.array_equal(ts, g["timestamps"]) and np.array_equal(st, g["states"]) and np.array_equal(ct, g["controls"])
