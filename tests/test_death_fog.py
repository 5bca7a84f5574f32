"""Death fog (DESIGN.md 7): env.death_fog_tick -> NC_DEATH_FOG, the C ABI's refusals, and the fog oracle
(tests/fog_oracle.py) against a Python transcription of Player.update's fog block and, without fog, against the oracle."""
import ctypes as C
from argparse import Namespace

import numpy as np
import pytest

from nmmo_b200.config import SPEC, default_env_args, make_config
from util import build_world

EV_EAT, EV_DRINK, EV_KILL = SPEC["EV_EAT_FOOD"], SPEC["EV_DRINK_WATER"], SPEC["EV_PLAYER_KILL"]


def fog_damage(cfg, tick, row, col):
    """Player.update's fog block [UPSTREAM nmmo/entity/player.py]: the damage a player at (row, col) receives in the step
    that starts at `tick`, or None when the fog does not touch it."""
    fog = int(cfg[SPEC["NC_DEATH_FOG"]])
    if fog < 0 or tick < fog:
        return None
    half = int(cfg[SPEC["NC_MAP_CENTER"]]) // 2
    cent = int(cfg[SPEC["NC_MAP_BORDER"]]) + half
    dist = max(abs(row - cent), abs(col - cent))
    if dist <= int(cfg[SPEC["NC_DEATH_FOG_FINAL_SIZE"]]):
        return None
    time_dmg = int(cfg[SPEC["NC_DEATH_FOG_SPEED"]]) * (tick - fog + 1)
    return max(0, dist - half + time_dmg)


def test_make_config_maps_death_fog_tick():
    for tick, want in ((None, -1), (0, 0), (256, 256), (np.int64(7), 7)):
        cfg, _ = make_config(default_env_args(death_fog_tick=tick))
        assert int(cfg[SPEC["NC_DEATH_FOG"]]) == want, tick
        assert int(cfg[SPEC["NC_DEATH_FOG_SPEED"]]) == 1 and int(cfg[SPEC["NC_DEATH_FOG_FINAL_SIZE"]]) == 8
    # an env namespace without the key (older configs) has no fog
    ns = vars(default_env_args())
    del ns["death_fog_tick"]
    assert int(make_config(Namespace(**ns))[0][SPEC["NC_DEATH_FOG"]]) == -1
    for bad in (-5, 1.5, "x", True, 2**31):
        with pytest.raises(ValueError, match="death_fog_tick"):
            make_config(default_env_args(death_fog_tick=bad))
    # speed and final size are engine constants: only raw overrides reach them
    cfg, _ = make_config(default_env_args(death_fog_tick=3), NC_DEATH_FOG_SPEED=2, NC_DEATH_FOG_FINAL_SIZE=0)
    assert cfg[SPEC["NC_DEATH_FOG"]] == 3 and cfg[SPEC["NC_DEATH_FOG_SPEED"]] == 2 and cfg[SPEC["NC_DEATH_FOG_FINAL_SIZE"]] == 0


def test_the_std_kernels_fold_the_fog_off():
    from util import std_cfg_table
    table = std_cfg_table()
    assert table[SPEC["NC_DEATH_FOG"]] == -1
    assert table[SPEC["NC_DEATH_FOG_SPEED"]] == 1 and table[SPEC["NC_DEATH_FOG_FINAL_SIZE"]] == 8
    cfg, _ = make_config(default_env_args(death_fog_tick=0))
    assert cfg[SPEC["NC_DEATH_FOG"]] != table[SPEC["NC_DEATH_FOG"]], "a fog-on handle must not match the std table"


def test_c_abi_refuses_bad_fog_entries():
    """nmmo_create checks the fog entries before it touches CUDA (C callers do not pass through make_config)."""
    from nmmo_b200 import lib
    L = lib.load()
    cfg, fcfg, maps, tab, emb = build_world(task_dim=64, NC_N_PLAYERS=16, NC_N_NPCS=32, NC_MAP_CENTER=32)
    for key, val in (("NC_DEATH_FOG", -2), ("NC_DEATH_FOG_SPEED", -1), ("NC_DEATH_FOG_FINAL_SIZE", -3)):
        bad = cfg.copy()
        bad[SPEC[key]] = val
        h = C.c_void_p()
        rc = L.nmmo_create(bad.ctypes.data_as(C.c_void_p), len(bad), fcfg.ctypes.data_as(C.c_void_p), len(fcfg), 2, 0, 0,
                           maps.ctypes.data_as(C.c_void_p), len(maps), tab.ctypes.data_as(C.c_void_p),
                           emb.ctypes.data_as(C.c_void_p), len(tab), C.byref(h))
        assert rc == -1 and b"DEATH_FOG" in L.nmmo_last_error(), (key, rc)
        assert not h.value


def _items_by_owner(items, P):
    owners = items[:, SPEC["IS_OWNER"]][items[:, SPEC["IS_TYPE"]] != 0]
    return np.bincount(owners[owners > 0], minlength=P + 1)[1:]


@pytest.mark.parametrize("agent,over", [("takeru", {}), ("neurips23_start_kit", {"NC_ALLOW_OCCUPIED": 1})])
def test_oracle_fog_matches_the_transcription(agent, over):
    """No NPCs and no player attacks, no depletion: every hit a player takes is the fog's.  Each tick, each alive
    player's EA_DAMAGE and EA_DMG_RECEIVED increment equal fog_damage() at the position it started the step on."""
    from fog_oracle import FogOracleEnv
    w = build_world(agent=agent, task_dim=64, NC_N_PLAYERS=16, NC_N_NPCS=0, NC_MAP_CENTER=32, NC_HORIZON=200,
                    NC_RES_DEPLETION=0, NC_WEAPON_DROP_THR=1 << 30, NC_DEATH_FOG=20, NC_DEATH_FOG_FINAL_SIZE=3, **over)
    cfg = w[0]
    A, D, DR, H, HR = SPEC["EA_ROW"], SPEC["EA_DAMAGE"], SPEC["EA_DMG_RECEIVED"], SPEC["EA_HEALTH"], SPEC["EA_HEALTH_RESTORE"]
    ST, FOOD = SPEC["EA_STATUS"], SPEC["EA_FOOD"]
    hurt = fog_kills = fog_kills_with_items = 0
    for seed in (3, 4):
        o = FogOracleEnv(*w)
        o.reset(seed)
        P = o.P
        for t in range(120):
            ent0, items0, _ = o.snapshot()
            tick0, done0 = o.tick, o.episode_done
            acts = o.sample_actions(50 + t)
            acts[:, SPEC["AC_ATTACK_STYLE"]] = -1         # no attacks
            o.step(acts)
            if done0:
                continue                                  # that step was the automatic reset
            ent1, items1, _ = o.snapshot()
            owned0, owned1 = _items_by_owner(items0, P), _items_by_owner(items1, P)
            rows = np.concatenate([o.log_rows(p) for p in range(P)])
            rows = rows[rows[:, 2] == o.tick]
            assert not (rows[:, 3] == EV_KILL).any(), "the fog gives no kill credit"
            for p in range(P):
                if ent0[p, ST] != SPEC["ES_ALIVE"]:
                    continue
                dmg = fog_damage(cfg, tick0, int(ent0[p, A]), int(ent0[p, A + 1]))
                want = 0 if dmg is None else dmg         # inside the final square (or before the onset): never hurt
                assert ent1[p, D] == want, (seed, t, p, int(ent1[p, D]), want)
                assert ent1[p, DR] - ent0[p, DR] == want, (seed, t, p)
                hurt += want > 0
                if want >= ent0[p, H]:                       # killed by the fog
                    fog_kills += 1
                    fog_kills_with_items += owned0[p] > 0
                    assert ent1[p, ST] == SPEC["ES_DEAD_THIS_TICK"] and ent1[p, H] == 0
                    assert owned1[p] == 0, "a fog-killed player keeps no items"
                    mine = rows[rows[:, 1] == p + 1]
                    assert not np.isin(mine[:, 3], (EV_EAT, EV_DRINK)).any(), "a fog-killed player does not eat or drink"
                    assert ent1[p, HR] == ent0[p, HR] and ent1[p, FOOD] == ent0[p, FOOD]
                else:
                    assert ent1[p, ST] == SPEC["ES_ALIVE"]
        o.close()
    assert hurt > 100 and fog_kills >= 16 and fog_kills_with_items >= 4, (hurt, fog_kills, fog_kills_with_items)


def test_oracle_fog_off_is_untouched():
    """NC_DEATH_FOG = -1: nobody is hurt without NPCs and attacks."""
    from fog_oracle import FogOracleEnv
    w = build_world(task_dim=64, NC_N_PLAYERS=16, NC_N_NPCS=0, NC_MAP_CENTER=32, NC_HORIZON=100, NC_RES_DEPLETION=0)
    o = FogOracleEnv(*w)
    o.reset(5)
    for t in range(60):
        acts = o.sample_actions(t)
        acts[:, SPEC["AC_ATTACK_STYLE"]] = -1
        o.step(acts)
        ent, _, _ = o.snapshot()
        assert not ent[:o.P, SPEC["EA_DMG_RECEIVED"]].any()
    o.close()


def test_fog_oracle_without_fog_is_the_oracle():
    """The fog oracle is oracle/nmmo_oracle.c plus the fog: with the fog off it steps exactly what the oracle steps
    (records, rewards, flags, infos, tables, event log), through automatic resets."""
    from fog_oracle import FogOracleEnv
    from oracle.oracle import OracleEnv
    for agent, over in (("takeru", {}), ("neurips23_start_kit", {"NC_ALLOW_OCCUPIED": 1})):
        w = build_world(agent=agent, task_dim=64, NC_N_PLAYERS=16, NC_N_NPCS=32, NC_MAP_CENTER=32, NC_HORIZON=90,
                        NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3, NC_WEAPON_DROP_THR=1 << 30, **over)
        a, b = OracleEnv(*w), FogOracleEnv(*w)
        a.reset(7); b.reset(7)
        done = 0
        for t in range(200):
            for name in ("obs", "rewards", "terminated", "truncated", "mask", "info_valid", "episode_done", "tick"):
                x, y = getattr(a, name), getattr(b, name)
                assert np.array_equal(x, y), (agent, t, name)
            assert np.array_equal(a.info.view(np.uint32), b.info.view(np.uint32)), (agent, t)
            for x, y in zip(a.snapshot(), b.snapshot()):
                assert np.array_equal(x, y), (agent, t)
            for p in range(a.P):
                assert np.array_equal(a.log_rows(p), b.log_rows(p)), (agent, t, p)
            done += a.episode_done
            acts = a.sample_actions(t)
            a.step(acts); b.step(acts)
        assert done >= 1
        a.close(); b.close()
