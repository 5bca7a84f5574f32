"""CPU: the host side of the event log -- EnvView's get_data filters and B200VecEnv's argument check."""
import numpy as np
import pytest

from nmmo_b200.config import SPEC


def _rows():
    # [id, ent_id, tick, event, type, level, number, gold, target]
    S = SPEC
    return np.array([
        [1, 1, 1, S["EV_DRINK_WATER"], 0, 0, 0, 0, 0],
        [2, 1, 1, S["EV_SCORE_HIT"], 1, 0, 7, 0, -3],
        [3, 2, 1, S["EV_GO_FARTHEST"], 0, 0, 4, 0, 0],
        [4, 2, 2, S["EV_SCORE_HIT"], 0, 0, 5, 0, 4],
        [5, 3, 2, S["EV_LOOT_GOLD"], 0, 0, 0, 9, 4],
        [6, 1, 3, S["EV_EARN_GOLD"], 0, 0, 0, 12, 0],
    ], np.int32)


def test_get_data_filters():
    from nmmo_b200.env import EventLogView
    rows = _rows()
    log = EventLogView(rows, tick=3)
    assert np.array_equal(log.get_data(), rows)
    assert np.array_equal(log.get_data(event_code=SPEC["EV_SCORE_HIT"]), rows[[1, 3]])
    assert np.array_equal(log.get_data(agents=[1]), rows[[0, 1, 5]])
    assert np.array_equal(log.get_data(agents=[2, 3]), rows[[2, 3, 4]])
    assert np.array_equal(log.get_data(tick=2), rows[[3, 4]])
    assert np.array_equal(log.get_data(tick=-1), rows[[5]])
    assert np.array_equal(log.get_data(event_code=SPEC["EV_SCORE_HIT"], agents=[2], tick=2), rows[[3]])
    assert log.get_data(agents=[]).shape == (0, 9)
    assert log.get_data(event_code=SPEC["EV_LEVEL_UP"]).shape == (0, 9)
    assert log.attr_to_col["target_ent"] == 8 and log.attr_to_col["gold"] == 7 and log.attr_to_col["damage"] == 6


def test_vecenv_rejects_negative_cap():
    from nmmo_b200.vecenv import B200VecEnv
    with pytest.raises(ValueError, match="event_log_cap"):
        B200VecEnv(num_envs=2, event_log_cap=-1)
