"""Engine configuration: the reference's ``Config(env_args)`` + wrapper kwargs -> flat vectors.

Mirrors /root/reference/reinforcement_learning/environment.py:14-49 (the ten config mixins and
the ``self.set`` overrides) and the ``env`` / ``reward_wrapper`` blocks of
/root/reference/config.yaml:75-139.  Engine defaults that live in the un-vendored ``nmmo``
package (``nmmo/core/config.py``) are restated here and tagged [UPSTREAM]; see DESIGN.md.

The result is the ``int32[NC_COUNT]`` / ``float64[NF_COUNT]`` pair that ``include/nmmo_spec.h``
describes and both the CUDA library and the CPU oracle consume.
"""
from __future__ import annotations

import math
import re
from argparse import Namespace
from pathlib import Path
from typing import Dict, Tuple

import numpy as np

_SPEC = Path(__file__).resolve().parent.parent / "include" / "nmmo_spec.h"


def _parse_enums(text: str) -> Dict[str, int]:
    """Read every ``enum { ... }`` of nmmo_spec.h so Python never duplicates an index."""
    out: Dict[str, int] = {}
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    for body in re.findall(r"enum\s+\w*\s*\{(.*?)\};", text, flags=re.S):
        val = -1
        for item in body.split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, expr = [s.strip() for s in item.split("=", 1)]
                val = int(eval(expr, {}, out))  # noqa: S307 - our own header, simple int exprs
            else:
                name = item
                val += 1
            out[name] = val
    for name, expr in re.findall(r"#define\s+(NM_\w+)\s+(\d+)\s*$", text, flags=re.M):
        out[name] = int(expr)
    return out


SPEC = _parse_enums(_SPEC.read_text())
globals().update(SPEC)  # NC_*, EA_*, IA_*, ... as module attributes

WRAPPERS = {"base": SPEC["NW_BASE"], "takeru": SPEC["NW_TAKERU"], "neurips23_start_kit": SPEC["NW_START_KIT"],
            "yaofeng": SPEC["NW_YAOFENG"],
            "hybrid": SPEC["NW_YAOFENG"]}      # agent_zoo/hybrid.py: takeru's policy with yaofeng's RewardWrapper


def default_exp_threshold(base_exp: int, max_level: int):
    """[UPSTREAM] nmmo/core/config.py default_exp_threshold."""
    add = [round(base_exp * math.sqrt(lvl)) for lvl in range(1, max_level + 1)]
    return [sum(add[:lvl]) for lvl in range(max_level)]


def _thr(p: float) -> int:
    """probability -> u32 threshold, stored as the int32 bit pattern."""
    u = min(int(p * 4294967296.0), 0xFFFFFFFF)
    return int(np.uint32(u).view(np.int32))


def default_env_args(**over) -> Namespace:
    """``env`` block of config.yaml:75-86."""
    d = dict(num_agents=128, num_npcs=256, max_episode_length=1024, maps_path="maps/train/",
             map_size=128, num_maps=256, map_force_generation=False, death_fog_tick=None,
             task_size=2048, spawn_immunity=20, resilient_population=0.2,
             curriculum_file_path=None)
    d.update(over)
    return Namespace(**d)


def default_wrapper_args(agent: str = "takeru", **over) -> Namespace:
    """``reward_wrapper`` block of config.yaml:98-106 with the per-agent overrides :128-139."""
    d = dict(eval_mode=False, early_stop_agent_num=8, use_custom_reward=True)
    if agent == "takeru":
        d.update(early_stop_agent_num=0, explore_bonus_weight=0.01, clip_unique_event=3, disable_give=True)
    elif agent == "neurips23_start_kit":
        d.update(heal_bonus_weight=0.03, explore_bonus_weight=0.01, clip_unique_event=3)
    elif agent in ("yaofeng", "hybrid"):      # config.yaml:117-125, :151-159; constructor defaults agent_zoo/yaofeng/reward_wrapper.py:13-29
        d.update(hp_bonus_weight=0.03, exp_bonus_weight=0.002, defense_bonus_weight=0.04, attack_bonus_weight=0.0,
                 gold_bonus_weight=0.001, custom_bonus_scale=0.1, disable_give=True, donot_attack_dangerous_npc=True)
    d.update(over)
    return Namespace(**d)


def death_fog_onset(tick) -> int:
    """``env.death_fog_tick`` (environment.py:36-39 -> PLAYER_DEATH_FOG) as NC_DEATH_FOG: None -> -1 (no fog), an int
    >= 0 -> the first tick of the fog.  Anything else is refused here, before a handle is created."""
    if tick is None:
        return -1
    if isinstance(tick, (bool, np.bool_)) or not isinstance(tick, (int, np.integer)) or tick < 0 or tick > 2**31 - 1:
        raise ValueError(f"death_fog_tick must be None or an int >= 0, got {tick!r}")
    return int(tick)


def make_config(env_args: Namespace = None, wrapper_args: Namespace = None, agent: str = "takeru",
                **engine_over) -> Tuple[np.ndarray, np.ndarray]:
    """Build (cfg int32, fcfg float64).  ``engine_over`` overrides raw NC_* entries (tests)."""
    if env_args is None:
        env_args = default_env_args(resilient_population=0 if agent in ("takeru", "yaofeng", "hybrid") else 0.2)
    if wrapper_args is None:
        wrapper_args = default_wrapper_args(agent)
    S = SPEC
    c = np.zeros(S["NC_COUNT"], np.int32)
    f = np.zeros(S["NF_COUNT"], np.float64)
    P = int(env_args.num_agents)
    border = 16
    c[S["NC_N_PLAYERS"]] = P
    c[S["NC_N_NPCS"]] = int(env_args.num_npcs)
    c[S["NC_HORIZON"]] = int(env_args.max_episode_length)
    c[S["NC_MAP_CENTER"]] = int(env_args.map_size)
    c[S["NC_MAP_BORDER"]] = border
    c[S["NC_MAP_SIZE"]] = int(env_args.map_size) + 2 * border
    c[S["NC_N_ENT_OBS"]] = 100
    c[S["NC_N_MKT_OBS"]] = 384
    c[S["NC_N_INV"]] = 12
    c[S["NC_N_PRICE"]] = 99
    c[S["NC_VISION"]] = 7
    c[S["NC_TASK_DIM"]] = int(env_args.task_size)
    c[S["NC_NPC_VISION"]] = 5
    base = 100
    c[S["NC_RES_BASE"]] = base
    c[S["NC_RES_DEPLETION"]] = 5
    c[S["NC_RES_STARVATION"]] = 10
    c[S["NC_RES_DEHYDRATION"]] = 10
    c[S["NC_RES_REGEN_THRESH"]] = int(math.floor(0.5 * base))
    c[S["NC_RES_HEALTH_RESTORE"]] = int(math.floor(0.1 * base))
    c[S["NC_RES_HARVEST_RESTORE"]] = int(math.floor(1.0 * base))
    c[S["NC_RES_RESILIENT_N"]] = int(round(float(env_args.resilient_population) * P))
    c[S["NC_SPAWN_IMMUNITY"]] = int(env_args.spawn_immunity)
    c[S["NC_REACH"]] = 3
    c[S["NC_FREEZE_TIME"]] = 3
    c[S["NC_WEAK_NUM"]], c[S["NC_WEAK_DEN"]] = 3, 2
    c[S["NC_MINDMG_NUM"]], c[S["NC_MINDMG_DEN"]] = 1, 4
    c[S["NC_LEVEL_MAX"]] = 10
    c[S["NC_XP_COMBAT"]], c[S["NC_XP_AMMO"]], c[S["NC_XP_CONSUMABLE"]] = 6, 15, 30
    c[S["NC_BASE_DAMAGE"]], c[S["NC_LEVEL_DAMAGE"]] = 10, 5
    c[S["NC_BASE_DEFENSE"]], c[S["NC_LEVEL_DEFENSE"]] = 0, 5
    for i, v in enumerate(default_exp_threshold(30, 10)):
        c[S["NC_EXP_THRESH0"] + i] = v
    c[S["NC_NPC_SPAWN_ATTEMPTS"]] = 25
    c[S["NC_NPC_AGGR_PCT"]], c[S["NC_NPC_NEUT_PCT"]], c[S["NC_NPC_PASS_PCT"]] = 80, 50, 0
    c[S["NC_NPC_LEVEL_MIN"]], c[S["NC_NPC_LEVEL_MAX"]] = 1, 10
    c[S["NC_NPC_BASE_DEFENSE"]], c[S["NC_NPC_LEVEL_DEFENSE"]] = 0, 15
    c[S["NC_NPC_BASE_DAMAGE"]], c[S["NC_NPC_LEVEL_DAMAGE"]] = 15, 15
    c[S["NC_WEAPON_DROP_THR"]] = _thr(0.025)
    c[S["NC_WEAPON_BASE"]], c[S["NC_WEAPON_LEVEL"]] = 5, 5
    c[S["NC_AMMO_BASE"]], c[S["NC_AMMO_LEVEL"]] = 5, 10
    c[S["NC_TOOL_BASE"]], c[S["NC_TOOL_LEVEL"]] = 15, 0
    c[S["NC_ARMOR_BASE"]], c[S["NC_ARMOR_LEVEL"]] = 0, 3
    c[S["NC_RESTORE_BASE"]], c[S["NC_RESTORE_LEVEL"]] = 50, 5
    c[S["NC_RESPAWN_FOILAGE"]] = _thr(0.025)
    c[S["NC_RESPAWN_ORE"]] = _thr(0.10)
    c[S["NC_RESPAWN_TREE"]] = _thr(0.105)
    c[S["NC_RESPAWN_CRYSTAL"]] = _thr(0.10)
    c[S["NC_RESPAWN_HERB"]] = _thr(0.02)
    c[S["NC_RESPAWN_FISH"]] = _thr(0.02)
    c[S["NC_BASE_GOLD"]] = 1
    c[S["NC_LISTING_DURATION"]] = 3
    c[S["NC_ALLOW_OCCUPIED"]] = 0
    c[S["NC_DEATH_FOG"]] = death_fog_onset(getattr(env_args, "death_fog_tick", None))
    c[S["NC_DEATH_FOG_SPEED"]] = 1
    c[S["NC_DEATH_FOG_FINAL_SIZE"]] = 8
    c[S["NC_WRAPPER"]] = WRAPPERS.get(agent, S["NW_BASE"])
    c[S["NC_EARLY_STOP_N"]] = int(getattr(wrapper_args, "early_stop_agent_num", 0))
    c[S["NC_EVAL_MODE"]] = int(bool(getattr(wrapper_args, "eval_mode", False)))
    c[S["NC_USE_CUSTOM_REWARD"]] = int(bool(getattr(wrapper_args, "use_custom_reward", True)))
    c[S["NC_CLIP_UNIQUE"]] = int(getattr(wrapper_args, "clip_unique_event", 3))
    c[S["NC_DISABLE_GIVE"]] = int(bool(getattr(wrapper_args, "disable_give", False)))
    c[S["NC_ITEM_CAP"]] = P * 12
    f[S["NF_EXPLORE_W"]] = float(getattr(wrapper_args, "explore_bonus_weight", 0.0))
    f[S["NF_HEAL_W"]] = float(getattr(wrapper_args, "heal_bonus_weight", 0.0))
    c[S["NC_NO_DANGEROUS_NPC"]] = int(bool(getattr(wrapper_args, "donot_attack_dangerous_npc", False)))
    for key, arg, dflt in (("NF_HP_W", "hp_bonus_weight", 0.0), ("NF_EXP_W", "exp_bonus_weight", 0.0),
                           ("NF_DEFENSE_W", "defense_bonus_weight", 0.0), ("NF_ATTACK_W", "attack_bonus_weight", 0.0),
                           ("NF_GOLD_W", "gold_bonus_weight", 0.0), ("NF_BONUS_SCALE", "custom_bonus_scale", 1.0)):
        f[S[key]] = float(getattr(wrapper_args, arg, dflt))
    for k, v in engine_over.items():
        c[S[k]] = v
    c[S["NC_MAP_SIZE"]] = c[S["NC_MAP_CENTER"]] + 2 * c[S["NC_MAP_BORDER"]]
    c[S["NC_ITEM_CAP"]] = c[S["NC_N_PLAYERS"]] * c[S["NC_N_INV"]]
    return c, f


class ObsLayout:
    """Python mirror of ``nm_obs_layout_init`` (include/nmmo_spec.h)."""

    def __init__(self, cfg: np.ndarray):
        S = SPEC
        a16 = lambda x: (x + 15) & ~15  # noqa: E731
        self.n_ent = int(cfg[S["NC_N_ENT_OBS"]]); self.n_mkt = int(cfg[S["NC_N_MKT_OBS"]])
        self.n_inv = int(cfg[S["NC_N_INV"]]); self.n_price = int(cfg[S["NC_N_PRICE"]])
        self.task_dim = int(cfg[S["NC_TASK_DIM"]]); self.win = 2 * int(cfg[S["NC_VISION"]]) + 1
        o = 0
        self.masks = {}
        for name, n in (("Attack.Style", 3), ("Attack.Target", self.n_ent + 1), ("Buy.MarketItem", self.n_mkt + 1),
                        ("Destroy.InventoryItem", self.n_inv + 1), ("Give.InventoryItem", self.n_inv + 1),
                        ("Give.Target", self.n_ent + 1), ("GiveGold.Price", self.n_price),
                        ("GiveGold.Target", self.n_ent + 1), ("Move.Direction", 5),
                        ("Sell.InventoryItem", self.n_inv + 1), ("Sell.Price", self.n_price),
                        ("Use.InventoryItem", self.n_inv + 1)):
            self.masks[name] = (o, n)
            o += n
        self.m_end = o
        alg = o
        o = a16(o)
        self.o_ids = o; o += 4; alg += 4; o = a16(o)
        self.o_entity = o; o += self.n_ent * 31 * 2; alg += self.n_ent * 31 * 2; o = a16(o)
        self.o_inventory = o; o += self.n_inv * 16 * 2; alg += self.n_inv * 16 * 2; o = a16(o)
        self.o_market = o; o += self.n_mkt * 16 * 2; alg += self.n_mkt * 16 * 2; o = a16(o)
        self.o_task = o; o += self.task_dim * 2; alg += self.task_dim * 2; o = a16(o)
        self.o_tile = o; o += self.win * self.win * 3 * 2; alg += self.win * self.win * 3 * 2
        self.stride = (o + 127) & ~127
        self.alg_bytes = alg
        self.action_dims = [n for (_, n) in self.masks.values()]
