"""CPU: host-side logic -- config vector, record layout, emulation views, C ABI surface."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from nmmo_b200.config import SPEC, ObsLayout, default_env_args, default_wrapper_args, make_config
from nmmo_b200.emulation import UnflattenContext, unpack_batched_obs
from nmmo_b200.tasks import default_curriculum, make_task_table
from util import SMALL, build_world

ROOT = Path(__file__).resolve().parent.parent


def test_spec_enums_parse():
    assert SPEC["EA_N_OBS"] == 31 and SPEC["IA_N_OBS"] == 16 and SPEC["AC_N"] == 12      # takeru/policy.py:120-161,223-241,293-307
    assert SPEC["EA_ID"] == 0 and SPEC["EA_NPC_TYPE"] == 1 and SPEC["IA_TYPE"] == 1 and SPEC["IA_EQUIPPED"] == 14
    assert SPEC["NM_UNIQ_WORDS"] * 32 >= SPEC["NM_N_EVENT"] * SPEC["IT_N"] * SPEC["NM_UNIQ_LEVELS"]


def test_config_mirrors_reference_defaults():
    cfg, fcfg = make_config(agent="takeru")
    assert cfg[SPEC["NC_N_PLAYERS"]] == 128 and cfg[SPEC["NC_N_NPCS"]] == 256 and cfg[SPEC["NC_HORIZON"]] == 1024   # config.yaml:76-78
    assert cfg[SPEC["NC_MAP_SIZE"]] == 160 and cfg[SPEC["NC_TASK_DIM"]] == 2048                                      # config.yaml:80,84
    assert cfg[SPEC["NC_EARLY_STOP_N"]] == 0 and cfg[SPEC["NC_DISABLE_GIVE"]] == 1 and fcfg[SPEC["NF_EXPLORE_W"]] == 0.01   # config.yaml:137-139
    assert cfg[SPEC["NC_RES_RESILIENT_N"]] == 0                                                                      # config.yaml:132
    cfg2, fcfg2 = make_config(agent="neurips23_start_kit")
    assert cfg2[SPEC["NC_EARLY_STOP_N"]] == 8 and fcfg2[SPEC["NF_HEAL_W"]] == 0.03 and cfg2[SPEC["NC_RES_RESILIENT_N"]] == 26
    cfg3, _ = make_config(default_env_args(num_agents=64, spawn_immunity=5), default_wrapper_args("takeru"), "takeru")
    assert cfg3[SPEC["NC_N_PLAYERS"]] == 64 and cfg3[SPEC["NC_SPAWN_IMMUNITY"]] == 5 and cfg3[SPEC["NC_ITEM_CAP"]] == 64 * 12


def test_hybrid_agent_uses_yaofeng_wrapper():
    a, fa = make_config(agent="hybrid")
    b, fb = make_config(agent="yaofeng")
    assert np.array_equal(a, b) and np.array_equal(fa, fb) and a[SPEC["NC_WRAPPER"]] == SPEC["NW_YAOFENG"]      # agent_zoo/hybrid.py:4
    assert fa[SPEC["NF_HP_W"]] == 0.03 and fa[SPEC["NF_BONUS_SCALE"]] == 0.1 and a[SPEC["NC_NO_DANGEROUS_NPC"]] == 1   # config.yaml:151-159


def test_layout_matches_survey_accounting():
    cfg, _ = make_config(agent="takeru")
    L = ObsLayout(cfg)
    # SURVEY.md 8(d): Tile 1350 + Entity 6200 + Inventory 384 + Market 12288 + Task 4096 + ids 4 + masks 946
    assert L.m_end == 946 and L.alg_bytes == 1350 + 6200 + 384 + 12288 + 4096 + 4 + 946
    assert L.stride % 128 == 0 and L.stride >= L.alg_bytes
    for off in (L.o_ids, L.o_entity, L.o_inventory, L.o_market, L.o_task, L.o_tile):
        assert off % 16 == 0
    assert L.action_dims == [3, 101, 385, 13, 13, 101, 99, 101, 5, 13, 99, 13]          # takeru/policy.py:310-322


def test_unpack_batched_obs_views_oracle_record():
    from oracle.oracle import OracleEnv
    world = build_world(task_dim=64, **SMALL, NC_RES_DEPLETION=1)
    o = OracleEnv(*world)
    o.reset(4)
    for _ in range(30):
        o.step(o.sample_actions(1))
    cfg = world[0]
    ctx = UnflattenContext(cfg)
    flat = o.obs
    nested = unpack_batched_obs(flat, ctx)
    ent, items, mp = o.snapshot()
    alive = np.flatnonzero(o.mask & (1 - o.terminated))
    assert len(alive) > 0
    for p in alive:
        assert nested["AgentId"][p, 0] == p + 1 and nested["CurrentTick"][p, 0] == o.tick
        r, c = ent[p, SPEC["EA_ROW"]], ent[p, SPEC["EA_COL"]]
        tile = nested["Tile"][p]
        assert tile.shape == (225, 3) and tile[112, 0] == r and tile[112, 1] == c        # centre of the 15x15 window, baseline_policy.py:96-97
        assert np.array_equal(tile[:, 2], mp[r - 7:r + 8, c - 7:c + 8].ravel())
        e = nested["Entity"][p]
        me = e[e[:, 0] == p + 1]
        assert len(me) == 1 and np.array_equal(me[0], ent[p, :31])                       # takeru/policy.py:177-182
        assert nested["Task"][p].dtype == np.float16
        assert nested["ActionTargets"]["Move"]["Direction"][p].shape == (5,)
    import torch
    t = unpack_batched_obs(torch.from_numpy(flat), ctx)
    assert torch.equal(t["Entity"], torch.from_numpy(nested["Entity"]))
    assert t["Task"].dtype == torch.float16 and t["Market"].shape[1:] == (ctx.layout.n_mkt, 16)


def test_task_table_is_device_evaluable():
    tab, emb = make_task_table(default_curriculum(), 64)
    assert tab.shape[1] == SPEC["NM_TASK_COLS"] and emb.dtype == np.uint16 and emb.shape == (tab.shape[0], 64)
    from nmmo_b200.tasks import PRED, STATE_PREDICATES, practice_skill_with_tool, task_row
    state = [PRED[n] for n in STATE_PREDICATES]
    assert np.isin(tab[:, 7], (0, 1, 2)).all() and np.isin(tab[tab[:, 7] != 0][:, 5], state).all()
    # manual_curriculum.py:119-122: 0.3 * EquipItem(tool) + 0.7 * GainExperience(skill, exp)
    row = practice_skill_with_tool("FISHING", 30)
    assert row[0] == SPEC["TP_EQUIP_ITEM"] and row[1] == SPEC["IT_ROD"] and row[5] == SPEC["TP_GAIN_EXPERIENCE"]
    assert row[6] == SPEC["SK_FISHING"] and row[8] == 30 and row[7] == 2 and (row[10], row[11]) == (300, 700)
    with pytest.raises(ValueError):
        task_row("TICK_GE", 10, pred2="COUNT_EVENT", q0=1, combine=1)       # event-driven second predicate
    assert (tab[:, 0] > 0).all() and (tab[:, 0] < SPEC["TP_N"]).all()


def _header_functions():
    text = (ROOT / "include" / "nmmo_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nmmo_\w+)\s*\(", text)))


def test_c_abi_exports_every_declared_symbol():
    from nmmo_b200 import lib
    L = lib.load()
    names = _header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), f"include/nmmo_b200.h declares {n} but libnmmo_b200.so does not export it"
    assert set(lib.EXPORTS) == set(names)


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from nmmo_b200 import lib
    L = lib.load()
    world = build_world(task_dim=64, **SMALL)
    cfg, fcfg, maps, tab, emb = world
    h = C.c_void_p()
    rc = L.nmmo_create(cfg.ctypes.data_as(C.c_void_p), len(cfg), fcfg.ctypes.data_as(C.c_void_p), len(fcfg), 2, 0, 0,
                       maps.ctypes.data_as(C.c_void_p), len(maps), tab.ctypes.data_as(C.c_void_p),
                       emb.ctypes.data_as(C.c_void_p), len(tab), C.byref(h))
    assert rc == -2 and b"no CPU fallback" in L.nmmo_last_error()
    with pytest.raises(lib.NmmoError):
        lib.Simulator(cfg, fcfg, 2, maps, tab, emb)


def test_pack_actions_u8_layout():
    """12 bytes per agent for nmmo_step_host_u8 (include/nmmo_b200.h): byte k = head k, the high bits of the one wide
    head (Buy.MarketItem, head 2) in bits 2..7 of byte 0; numpy and torch packers agree."""
    import torch
    from nmmo_b200.lib import pack_actions_u8
    rng = np.random.default_rng(0)
    dims = ObsLayout(make_config()[0]).action_dims
    a = np.stack([rng.integers(0, n, size=(5, 7)) for n in dims], -1).astype(np.int32)
    a[0, 0] = -1                                            # "no action" entries stay out of range after packing
    pk = pack_actions_u8(a)
    assert pk.dtype == np.uint8 and pk.shape == a.shape
    back = pk.astype(np.int32)
    buy = back[..., 2] | ((back[..., 0] >> 2) << 8)
    style = back[..., 0] & 3
    ok = a[..., 2] >= 0
    assert np.array_equal(buy[ok], a[..., 2][ok]) and np.array_equal(style[1:], a[1:, :, 0])
    for k in (1, 3, 4, 5, 6, 7, 8, 9, 10, 11):
        assert np.array_equal(back[1:, :, k], a[1:, :, k])
    assert buy[0, 0] >= dims[2] and style[0, 0] == 3 and (back[0, 0, 1:] == 255).all()
    assert np.array_equal(pack_actions_u8(torch.from_numpy(a)).numpy(), pk)


def test_std_cfg_table_matches_the_python_defaults():
    """nm_cfg_std_value (csrc/nmmo_device.cuh): the engine defaults the *_std kernel instantiations fold to immediates must be
    the values nmmo_b200/config.py produces; entries the reference's Config or wrappers set stay run-time."""
    from util import std_cfg_table
    table = std_cfg_table()
    assert len(table) > 60
    for agent in ("takeru", "neurips23_start_kit", "yaofeng"):
        cfg, _ = make_config(agent=agent)
        for i, v in table.items():
            assert int(cfg[i]) == v, (agent, i, v, int(cfg[i]))
    runtime = {"NC_N_PLAYERS", "NC_N_NPCS", "NC_MAP_CENTER", "NC_MAP_SIZE", "NC_ITEM_CAP", "NC_HORIZON", "NC_RES_RESILIENT_N",
               "NC_SPAWN_IMMUNITY", "NC_WRAPPER", "NC_EARLY_STOP_N", "NC_EVAL_MODE", "NC_USE_CUSTOM_REWARD",
               "NC_CLIP_UNIQUE", "NC_DISABLE_GIVE", "NC_NO_DANGEROUS_NPC", "NC_SPAWN_PATCH", "NC_TEAM_SIZE", "NC_SAMPLE_MOVE_PCT"}
    assert not ({SPEC[n] for n in runtime} & set(table)), "an entry the reference sets per run must not be folded"
    assert set(table) | {SPEC[n] for n in runtime} == set(range(SPEC["NC_COUNT"]))
