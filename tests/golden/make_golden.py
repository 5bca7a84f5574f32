#!/usr/bin/env python
"""Golden vectors for the in-tree part of the hot path, produced by running the REFERENCE's own code.

What is pinned.  The reference's stat / reward wrapper stack
    reinforcement_learning/stat_wrapper.py      BaseStatWrapper.step, _process_stats_and_early_stop,
                                                process_event_log, count_unique_events
    agent_zoo/takeru/reward_wrapper.py          RewardWrapper.observation / reward_terminated_truncated_info
    agent_zoo/neurips23_start_kit/reward_wrapper.py   same + RewardWrapper.action
    agent_zoo/yaofeng/reward_wrapper.py         same (hp / exp / defense / attack / gold bonuses, dangerous-NPC mask)
is imported UNMODIFIED from the reference checkout named by $NMMO_REFERENCE (only the missing
third-party modules pettingzoo and nmmo are replaced by minimal stubs: a BaseParallelWrapper that stores `env`, the EventCode
constants, the item class lists) and driven through whole episodes by a fake `nmmo.Env` that
replays an engine trajectory.  Its outputs -- reward, terminated, truncated, episode info dict and
the edited ActionTargets masks -- are stored; tests/test_golden.py requires the CPU oracle's wrapper
part to reproduce them bit for bit, and the GPU tests require the CUDA path to equal the oracle.

What is NOT pinned.  The engine trajectory itself comes from oracle/nmmo_oracle.c (the nmmo 2.1
engine is not available here), so these vectors pin rows a-4..a-10 of SURVEY.md section 8, not a-3/a-16.

Run with a checkout of the reference baselines repository:  NMMO_REFERENCE=<checkout> python tests/golden/make_golden.py
"""
from __future__ import annotations

import sys
import types
from argparse import Namespace
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from nmmo_b200.config import SPEC, ObsLayout  # noqa: E402
from util import reference_file  # noqa: E402

REF = reference_file()

INFO_KEYS = {  # episode-info key -> column of the nm_info record (include/nmmo_spec.h)
    "length": "IN_LENGTH", "return": "IN_RETURN",
    "stats/cod/attacked": "IN_COD_ATTACKED", "stats/cod/starved": "IN_COD_STARVED", "stats/cod/dehydrated": "IN_COD_DEHYDRATED",
    "stats/task/completed": "IN_TASK_COMPLETED", "stats/task/pcnt_2_reward_signal": "IN_TASK_2_REWARD_SIGNAL",
    "stats/task/pcnt_0p2_max_progress": "IN_TASK_0P2_MAX_PROGRESS",
    "stats/achieved/max_combat_level": "IN_MAX_COMBAT_LEVEL", "stats/achieved/max_harvest_skill_ammo": "IN_MAX_HARVEST_AMMO",
    "stats/achieved/max_harvest_skill_consum": "IN_MAX_HARVEST_CONSUM",
    "stats/achieved/max_progress_to_center": "IN_MAX_PROGRESS_TO_CENTER", "stats/achieved/earned_gold": "IN_EARNED_GOLD",
    "stats/achieved/max_damage": "IN_MAX_DAMAGE", "stats/achieved/max_armor_level": "IN_MAXLVL_ARMOR",
    "stats/achieved/max_weapon_level": "IN_MAXLVL_WEAPON", "stats/achieved/max_tool_level": "IN_MAXLVL_TOOL",
    "stats/achieved/max_ammo_level": "IN_MAXLVL_AMMO", "stats/achieved/max_consumable_level": "IN_MAXLVL_CONSUMABLE",
    "stats/achieved/agent_kill_count": "IN_AGENT_KILLS", "stats/achieved/npc_kill_count": "IN_NPC_KILLS",
    "stats/achieved/unique_events": "IN_UNIQUE_EVENTS",
    "stats/event/eat_food": "IN_EV_EAT_FOOD", "stats/event/drink_water": "IN_EV_DRINK_WATER",
    "stats/event/score_hit": "IN_EV_SCORE_HIT", "stats/event/player_kill": "IN_EV_PLAYER_KILL",
    "stats/event/consume_item": "IN_EV_CONSUME_ITEM", "stats/event/harvest_item": "IN_EV_HARVEST_ITEM",
    "stats/event/list_item": "IN_EV_LIST_ITEM", "stats/event/buy_item": "IN_EV_BUY_ITEM",
    "stats/event/equip_armor": "IN_EQUIP_ARMOR", "stats/event/equip_weapon": "IN_EQUIP_WEAPON",
    "stats/event/equip_tool": "IN_EQUIP_TOOL", "stats/event/equip_ammo": "IN_EQUIP_AMMO",
    "stats/event/harvest_weapon": "IN_HARVEST_WEAPON",
}
MASK_PATHS = ["Attack.Style", "Attack.Target", "Buy.MarketItem", "Destroy.InventoryItem", "Give.InventoryItem",
              "Give.Target", "GiveGold.Price", "GiveGold.Target", "Move.Direction", "Sell.InventoryItem",
              "Sell.Price", "Use.InventoryItem"]
ACTION_KEYS = [("Attack", "Style"), ("Attack", "Target"), ("Buy", "MarketItem"), ("Destroy", "InventoryItem"),
               ("Give", "InventoryItem"), ("Give", "Target"), ("GiveGold", "Price"), ("GiveGold", "Target"),
               ("Move", "Direction"), ("Sell", "InventoryItem"), ("Sell", "Price"), ("Use", "InventoryItem")]


def install_stubs():
    """Minimal stand-ins for the two third-party packages the reference modules import."""
    def mod(name):
        m = types.ModuleType(name)
        sys.modules[name] = m
        return m

    for n in ("pettingzoo", "pettingzoo.utils", "pettingzoo.utils.wrappers", "pettingzoo.utils.wrappers.base_parallel"):
        mod(n)

    class BaseParallelWrapper:
        def __init__(self, env):
            self.env = env

    sys.modules["pettingzoo.utils.wrappers.base_parallel"].BaseParallelWrapper = BaseParallelWrapper
    nmmo = mod("nmmo"); lib = mod("nmmo.lib"); ec = mod("nmmo.lib.event_code"); systems = mod("nmmo.systems"); item = mod("nmmo.systems.item")
    nmmo.lib = lib; lib.event_code = ec; nmmo.systems = systems; systems.item = item
    entity = mod("nmmo.entity"); ent_entity = mod("nmmo.entity.entity"); nmmo.entity = entity; entity.entity = ent_entity
    # EntityState.State.attr_name_to_col (yaofeng/reward_wrapper.py:7): observed column order of include/nmmo_spec.h
    cols = {k[3:].lower(): v for k, v in SPEC.items() if k.startswith("EA_") and isinstance(v, int) and v < SPEC["EA_N_OBS"] and k != "EA_N_OBS"}
    ent_entity.EntityState = type("EntityState", (), {"State": type("State", (), {"attr_name_to_col": cols})})
    ec.EventCode = type("EventCode", (), {k[3:]: v for k, v in SPEC.items() if k.startswith("EV_")})

    def cls(name):
        return type(name.title(), (), {"ITEM_TYPE_ID": SPEC["IT_" + name]})

    item.ARMOR = [cls(n) for n in ("HAT", "TOP", "BOTTOM")]
    item.WEAPON = [cls(n) for n in ("SPEAR", "BOW", "WAND")]
    item.TOOL = [cls(n) for n in ("ROD", "GLOVES", "PICKAXE", "AXE", "CHISEL")]
    item.AMMUNITION = [cls(n) for n in ("WHETSTONE", "ARROW", "RUNES")]
    item.CONSUMABLE = [cls(n) for n in ("RATION", "POTION")]


class _Val:
    def __init__(self, v):
        self.val = int(v)


class FakePlayer:
    """The attributes BaseStatWrapper reads from realm.players[id] (stat_wrapper.py:136-175)."""

    def __init__(self, row):
        S = SPEC
        self.damage = _Val(row[S["EA_DAMAGE"]]); self.food = _Val(row[S["EA_FOOD"]]); self.water = _Val(row[S["EA_WATER"]])
        self.attack_level = int(max(row[S["EA_MELEE_LEVEL"]], row[S["EA_RANGE_LEVEL"]], row[S["EA_MAGE_LEVEL"]]))
        for name in ("prospecting", "carving", "alchemy", "fishing", "herbalism"):
            setattr(self, name + "_level", _Val(row[S["EA_" + name.upper() + "_LEVEL"]]))
        self.resources = Namespace(health_restore=int(row[S["EA_HEALTH_RESTORE"]]))
        # read by agent_zoo/yaofeng/reward_wrapper.py:88-121
        self.health = _Val(row[S["EA_HEALTH"]]); self.gold = _Val(row[S["EA_GOLD"]])
        for name in ("melee", "range", "mage", "fishing", "herbalism", "prospecting", "carving", "alchemy"):
            setattr(self, name + "_exp", _Val(row[S["EA_" + name.upper() + "_EXP"]]))
        self.history = Namespace(damage_received=int(row[S["EA_DMG_RECEIVED"]]), damage_inflicted=int(row[S["EA_DMG_INFLICTED"]]))
        self.inventory = None      # filled in by FakeEnv._sync (needs the item table)


class FakePlayers(dict):
    dead_this_tick = {}


class FakeEventLog:
    attr_to_col = {"event": 3, "type": 4, "item_type": 4, "combat_style": 4, "skill": 4, "level": 5, "number": 6,
                   "distance": 6, "damage": 6, "quantity": 6, "gold": 7, "price": 7, "target_ent": 8}

    def __init__(self, env):
        self.env = env

    def get_data(self, agents=None, tick=None):
        rows = [self.env.oracle.log_rows(a - 1) for a in agents]
        log = np.concatenate(rows) if rows else np.zeros((0, 9), np.int32)
        if tick == -1:
            log = log[log[:, 2] == self.env.realm.tick]
        return log


class FakeTask:
    def __init__(self, completed, signals, max_progress, tid):
        self.completed = bool(completed); self.reward_signal_count = int(signals); self._max_progress = float(max_progress)
        self.spec_name = f"task_{tid}"


class FakeEnv:
    """nmmo.Env stand-in replaying the oracle's engine trajectory (raw, pre-wrapper quantities)."""

    def __init__(self, oracle, raw_oracle, actions, cfg):
        self.oracle, self.raw, self.actions, self.cfg = oracle, raw_oracle, actions, cfg
        self.P = int(cfg[SPEC["NC_N_PLAYERS"]])
        self.L = ObsLayout(cfg)
        self.possible_agents = list(range(1, self.P + 1))
        self.agents = list(self.possible_agents)
        self.realm = Namespace(tick=0, players=FakePlayers(), event_log=FakeEventLog(self))
        self.agent_task_map = {}
        self.config = Namespace(COMBAT_SPAWN_IMMUNITY=int(cfg[SPEC["NC_SPAWN_IMMUNITY"]]))
        self.t = 0

    def _masks(self, p):
        rec = self.raw.obs[p]
        out = {}
        for path in MASK_PATHS:
            a, b = path.split(".")
            o, n = self.L.masks[path]
            out.setdefault(a, {})[b] = rec[o:o + n].copy().view(np.int8)
        return out

    def _obs(self, p):
        """The parts of the engine observation the wrappers read: ActionTargets and the Entity block."""
        rec = self.raw.obs[p]
        ent = rec[self.L.o_entity:self.L.o_entity + self.L.n_ent * 62].copy().view(np.int16).reshape(self.L.n_ent, 31)
        return {"ActionTargets": self._masks(p), "Entity": ent}

    def _sync(self):
        ent, _, _ = self.oracle.snapshot()
        st = ent[:self.P, SPEC["EA_STATUS"]]
        self.realm.tick = self.oracle.tick
        ent, items, _ = self.oracle.snapshot()
        self.realm.players = FakePlayers({p + 1: FakePlayer(ent[p]) for p in range(self.P) if st[p] == 1})
        for a, pl in self.realm.players.items():      # Equipment.{melee,range,mage}_defense: sums over equipped items
            d = 0
            for col in ("EA_EQ_HAT", "EA_EQ_TOP", "EA_EQ_BOTTOM", "EA_EQ_HELD", "EA_EQ_AMMO"):
                it = int(ent[a - 1][SPEC[col]])
                if it:
                    typ, lvl = int(items[it - 1][SPEC["IS_TYPE"]]), int(items[it - 1][SPEC["IS_LEVEL"]])
                    if SPEC["IT_HAT"] <= typ <= SPEC["IT_BOTTOM"]:
                        d += int(self.cfg[SPEC["NC_ARMOR_BASE"]]) + lvl * int(self.cfg[SPEC["NC_ARMOR_LEVEL"]])
                    elif SPEC["IT_ROD"] <= typ <= SPEC["IT_CHISEL"]:
                        d += int(self.cfg[SPEC["NC_TOOL_BASE"]]) + lvl * int(self.cfg[SPEC["NC_TOOL_LEVEL"]])
            pl.inventory = Namespace(equipment=Namespace(melee_defense=d, range_defense=d, mage_defense=d))
        self.realm.players.dead_this_tick = {p + 1: FakePlayer(ent[p]) for p in range(self.P) if st[p] == 2}
        tid, comp, sig, mp = self.oracle.task_state()
        self.agent_task_map = {p + 1: [FakeTask(comp[p], sig[p], mp[p], tid[p])] for p in range(self.P)}
        return st

    def reset(self, **kw):
        st = self._sync()
        self.agents = [p + 1 for p in range(self.P) if st[p] == 1]
        return {a: self._obs(a - 1) for a in self.agents}, {a: {} for a in self.agents}

    def step(self, action):
        flat = self.actions[self.t]
        for a, d in action.items():      # what the wrapper passes down is what was recorded
            for k, (x, y) in enumerate(ACTION_KEYS):
                assert int(d[x][y]) == int(flat[a - 1, k])
        self.oracle.step(flat); self.raw.step(flat)
        self.t += 1
        st = self._sync()
        horizon = self.realm.tick >= int(self.cfg[SPEC["NC_HORIZON"]])
        current = [p + 1 for p in range(self.P) if st[p] in (1, 2)]
        env_rew = self.oracle.env_rewards
        obs = {a: self._obs(a - 1) for a in current}
        rewards = {a: float(env_rew[a - 1]) for a in current}
        terms = {a: bool(st[a - 1] == 2) for a in current}
        truncs = {a: bool(horizon and st[a - 1] == 1) for a in current}
        infos = {a: {"task": {}} for a in current}
        self.agents = [] if horizon else current
        return obs, rewards, terms, truncs, infos


def pack_masks(L, obs_agent, out):
    for path in MASK_PATHS:
        a, b = path.split(".")
        o, n = L.masks[path]
        out[o:o + n] = obs_agent["ActionTargets"][a][b].view(np.uint8)


def run_case(name, agent, ticks, seed, wrapper_over=None, **engine_over):
    from util import SMALL, build_world
    from oracle.oracle import OracleEnv
    world = build_world(agent=agent, task_dim=64, wrapper_over=wrapper_over, **SMALL, **engine_over)
    cfg, fcfg = world[0], world[1]
    raw_cfg = cfg.copy(); raw_cfg[SPEC["NC_WRAPPER"]] = SPEC["NW_BASE"]
    oracle = OracleEnv(cfg, fcfg, *world[2:])
    raw = OracleEnv(raw_cfg, fcfg, *world[2:])
    P = oracle.P
    L = ObsLayout(cfg)
    # pass 1: record the actions of the episode (sampled from the wrapped masks)
    rec = OracleEnv(cfg, fcfg, *world[2:])
    rec.reset(seed)
    actions = []
    for t in range(ticks):
        a = rec.sample_actions(1000 + seed)
        actions.append(a)
        rec.step(a)
        if rec.episode_done:
            break
    T = len(actions)
    # pass 2: the reference wrapper on top of the replayed trajectory
    oracle.reset(seed); raw.reset(seed)
    if agent in ("takeru", "neurips23_start_kit", "yaofeng"):
        # the module file itself, unmodified; loaded by path because the package __init__ also
        # imports the policy (pufferlib), which is irrelevant here
        import importlib.util
        spec = importlib.util.spec_from_file_location(f"ref_{agent}_reward_wrapper", REF / "agent_zoo" / agent / "reward_wrapper.py")
        module = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(module)
        RewardWrapper = module.RewardWrapper
    else:
        from reinforcement_learning.stat_wrapper import BaseStatWrapper as RewardWrapper
    from nmmo_b200.config import default_wrapper_args
    kw = vars(default_wrapper_args(agent, **(wrapper_over or {})))
    env = FakeEnv(oracle, raw, actions, cfg)
    wrapper = RewardWrapper(env, **kw)
    obs, _ = wrapper.reset()
    rew = np.zeros((T, P), np.float32); term = np.zeros((T, P), np.uint8); trunc = np.zeros((T, P), np.uint8)
    present = np.zeros((T, P), np.uint8); masks = np.zeros((T + 1, P, L.m_end), np.uint8)
    info = np.full((T, P, SPEC["IN_N"]), np.nan, np.float32); info_valid = np.zeros((T, P), np.uint8)
    done_tick = -1
    for a, o in obs.items():
        pack_masks(L, o, masks[0, a - 1])
    for t in range(T):
        act = {a: {} for a in env.agents}
        for a in env.agents:
            for k, (x, y) in enumerate(ACTION_KEYS):
                act[a].setdefault(x, {})[y] = int(actions[t][a - 1, k])
        obs, rewards, terms, truncs, infos = wrapper.step(act)
        for a in obs:
            p = a - 1
            present[t, p] = 1
            rew[t, p] = np.float32(rewards[a]); term[t, p] = terms[a]; trunc[t, p] = truncs[a]
            pack_masks(L, obs[a], masks[t + 1, p])
            inf = infos[a]
            if "stats" in inf:
                info_valid[t, p] = 1
                row = info[t, p]
                row[:] = np.nan
                flat = {"length": inf["length"], "return": inf["return"]}
                flat.update({"stats/" + k: v for k, v in inf["stats"].items()})
                for k, col in INFO_KEYS.items():
                    if k in flat:
                        row[SPEC[col]] = np.float32(flat[k])
                (spec_name, (mp, sig)), = inf["curriculum"].items()
                row[SPEC["IN_CURR_MAX_PROGRESS"]] = np.float32(mp); row[SPEC["IN_CURR_REWARD_SIGNALS"]] = np.float32(sig)
                row[SPEC["IN_TASK_ID"]] = np.float32(int(spec_name.split("_")[1]))
            if inf.get("episode_done"):
                done_tick = t
        if done_tick >= 0:
            break
    out = HERE / f"{name}.npz"
    np.savez_compressed(out, agent=agent, seed=seed, ticks=T, engine_over=np.array(sorted(engine_over.items()), dtype=object),
                        wrapper_over=np.array(sorted((wrapper_over or {}).items()), dtype=object),
                        actions=np.stack(actions).astype(np.int16), rew=rew, term=term, trunc=trunc, present=present,
                        masks=np.packbits(masks, axis=-1), mask_len=L.m_end, info=info, info_valid=info_valid, done_tick=done_tick)
    print(f"{name}: {T} ticks, {int(info_valid.sum())} episode infos, done at {done_tick}, {out.stat().st_size} bytes")


def main():
    assert REF is not None, "set NMMO_REFERENCE to a checkout of the reference baselines repository"
    install_stubs()
    sys.path.insert(0, str(REF))
    run_case("takeru_small", "takeru", 140, 3, NC_HORIZON=120, NC_RES_DEPLETION=2, NC_SPAWN_IMMUNITY=3, NC_WEAPON_DROP_THR=1 << 30)
    run_case("start_kit_small", "neurips23_start_kit", 140, 5, NC_HORIZON=100, NC_RES_DEPLETION=2, NC_SPAWN_IMMUNITY=3)
    run_case("takeru_eval_nocustom", "takeru", 90, 7, wrapper_over={"eval_mode": True, "use_custom_reward": False, "early_stop_agent_num": 4},
             NC_HORIZON=80, NC_RES_DEPLETION=3)
    run_case("start_kit_nocustom_prefix", "neurips23_start_kit", 80, 11, wrapper_over={"use_custom_reward": False, "early_stop_agent_num": 12},
             NC_HORIZON=70, NC_RES_DEPLETION=3)
    run_case("yaofeng_eval", "yaofeng", 120, 13, wrapper_over={"eval_mode": True, "early_stop_agent_num": 0, "donot_attack_dangerous_npc": False,
                                                               "disable_give": False, "custom_bonus_scale": 1.0},
             NC_HORIZON=100, NC_RES_DEPLETION=2, NC_SPAWN_IMMUNITY=2)
    # slow starvation + fast item drops: combat, equipment (defense bonus), gold and exp all move
    run_case("yaofeng_small", "yaofeng", 200, 9, wrapper_over={"attack_bonus_weight": 0.005, "early_stop_agent_num": 2},
             NC_HORIZON=180, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3, NC_WEAPON_DROP_THR=1 << 30)


if __name__ == "__main__":
    main()
