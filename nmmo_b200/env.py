"""Per-environment PettingZoo-parallel view of one simulated env (parity / debugging boundary).

Mirrors what the reference's wrappers see of ``nmmo.Env``: ``reset(seed=) -> (obs, info)``,
``step({agent_id: nested action dict}) -> (obs, rewards, terminated, truncated, infos)``,
``agents`` / ``possible_agents`` with 1-based ids (/root/reference/train_helper.py:147,
/root/reference/reinforcement_learning/stat_wrapper.py:48-97).  The values already include the
RewardWrapper hooks, i.e. this is the env *as wrapped by* ``make_env_creator``
(/root/reference/reinforcement_learning/environment.py:55-74) minus the pufferlib flattening.
Everything is copied to the host: use B200VecEnv for rollouts.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Dict

import numpy as np

from .config import SPEC
from .emulation import UnflattenContext, unpack_batched_obs
from .vecenv import info_record_to_dict

class _Val:
    def __init__(self, v):
        self.val = int(v)


class PlayerView:
    """The attributes the reference's wrappers read from ``realm.players[id]``
    (stat_wrapper.py:136-175, yaofeng/reward_wrapper.py:88-121, start_kit/reward_wrapper.py:69)."""

    def __init__(self, row, defense):
        S = SPEC
        for name in ("damage", "food", "water", "health", "gold"):
            setattr(self, name, _Val(row[S["EA_" + name.upper()]]))
        self.attack_level = int(max(row[S["EA_MELEE_LEVEL"]], row[S["EA_RANGE_LEVEL"]], row[S["EA_MAGE_LEVEL"]]))
        for name in ("melee", "range", "mage", "fishing", "herbalism", "prospecting", "carving", "alchemy"):
            setattr(self, name + "_level", _Val(row[S["EA_" + name.upper() + "_LEVEL"]]))
            setattr(self, name + "_exp", _Val(row[S["EA_" + name.upper() + "_EXP"]]))
        self.resources = SimpleNamespace(health_restore=int(row[S["EA_HEALTH_RESTORE"]]))
        self.history = SimpleNamespace(damage_received=int(row[S["EA_DMG_RECEIVED"]]), damage_inflicted=int(row[S["EA_DMG_INFLICTED"]]))
        eq = SimpleNamespace(melee_defense=defense, range_defense=defense, mage_defense=defense)
        self.inventory = SimpleNamespace(equipment=eq)
        self.pos = (int(row[S["EA_ROW"]]), int(row[S["EA_COL"]]))


class _Players(dict):
    dead_this_tick = {}


class TaskView:
    """``env.agent_task_map[id][0]`` as stat_wrapper.py:155-159 reads it."""

    def __init__(self, tid, completed, signals, max_progress):
        self.completed = bool(completed); self.reward_signal_count = int(signals); self._max_progress = float(max_progress)
        self.spec_name = f"task_{int(tid)}"
        self.progress_info = {"max_progress": float(max_progress), "completed_tick": int(completed) if completed else None}


class EventLogView:
    """``realm.event_log`` of the reference (nmmo/lib/event_log.py EventLogger) over the episode's rows: int32
    [n, 9] = [id, ent_id, tick, event, type, level, number, gold, target_ent], id the running row number.  Each tick's
    rows are ordered by agent, then by the order the agent's events happened in."""

    attr_to_col = {"event": 3, "type": 4, "item_type": 4, "combat_style": 4, "skill": 4, "level": 5, "number": 6,
                   "distance": 6, "damage": 6, "quantity": 6, "gold": 7, "price": 7, "target_ent": 8}

    def __init__(self, rows: np.ndarray, tick: int):
        self._rows, self._tick = rows, int(tick)

    def get_data(self, event_code=None, agents=None, tick=None) -> np.ndarray:
        """Rows of event `event_code` (an EventCode), of the agents (ent ids) in `agents`, at tick `tick` (-1: the
        current tick); None keeps every row on that axis."""
        log = self._rows
        if event_code is not None:
            log = log[log[:, 3] == int(event_code)]
        if agents is not None:
            log = log[np.isin(log[:, 1], np.asarray(list(agents), np.int64))]
        if tick is not None:
            log = log[log[:, 2] == (self._tick if int(tick) == -1 else int(tick))]
        return log


ACTION_KEYS = [("Attack", "Style"), ("Attack", "Target"), ("Buy", "MarketItem"), ("Destroy", "InventoryItem"),
               ("Give", "InventoryItem"), ("Give", "Target"), ("GiveGold", "Price"), ("GiveGold", "Target"),
               ("Move", "Direction"), ("Sell", "InventoryItem"), ("Sell", "Price"), ("Use", "InventoryItem")]


class EnvView:
    def __init__(self, sim, env_index: int = 0):
        self.sim, self.k = sim, int(env_index)
        self.P = sim.P
        self.ctx = UnflattenContext(sim.cfg)
        self.possible_agents = list(range(1, self.P + 1))
        self.agents = []
        self.max_num_agents = self.P
        self.config = SimpleNamespace(COMBAT_SPAWN_IMMUNITY=int(sim.cfg[SPEC["NC_SPAWN_IMMUNITY"]]), PLAYER_N=self.P,
                                      HORIZON=int(sim.cfg[SPEC["NC_HORIZON"]]))      # yaofeng/reward_wrapper.py:33
        # the episode's event log, accumulated on the host from the device rows of every step (realm.event_log)
        sim.set_event_log(True)
        self._log = np.zeros((0, 9), np.int32)
        self._log_done = False      # the env finished its episode: the next step resets it and starts a new log

    def _slice(self, t):
        return t[self.k * self.P:(self.k + 1) * self.P].cpu().numpy()

    def _obs(self, present):
        flat = self._slice(self.sim.obs)
        nested = unpack_batched_obs(flat, self.ctx)

        def pick(x, p):
            return {k: pick(v, p) for k, v in x.items()} if isinstance(x, dict) else x[p]

        return {p + 1: pick(nested, p) for p in range(self.P) if present[p]}

    def reset(self, seed=0, new_task=None, **kw):
        """``new_task`` = row of the task table every agent of this env gets for the episode: the task swap
        SyllabusTaskWrapper.reset does through ``make_task_fn`` (/root/reference/syllabus_wrapper.py:129-150).
        Without it the tasks are drawn from the table as on every other reset."""
        mask = np.zeros(self.sim.E, np.uint8); mask[self.k] = 1
        seeds = np.zeros(self.sim.E, np.uint64); seeds[self.k] = seed
        task_ids = None
        if new_task is not None:
            task_ids = np.zeros((self.sim.E, self.P), np.int32); task_ids[self.k] = int(new_task)
        self.sim.reset(seeds, task_ids=task_ids, env_mask=mask)
        self._log = np.zeros((0, 9), np.int32)
        self._log_done = False
        present = self._slice(self.sim.mask).astype(bool)
        self.agents = [p + 1 for p in range(self.P) if present[p]]
        return self._obs(present), {a: {} for a in self.agents}

    def step(self, actions: Dict[int, Dict]):
        if self.sim.E != 1:
            raise RuntimeError("EnvView.step drives the whole simulator; create it with n_envs=1")
        import torch
        flat = np.zeros((1, self.P, 12), np.int32)
        for a, d in actions.items():
            for k, (x, y) in enumerate(ACTION_KEYS):
                flat[0, a - 1, k] = int(d.get(x, {}).get(y, 0))
        self.sim.actions.copy_(torch.from_numpy(flat))
        self.sim.step()
        present = self._slice(self.sim.mask).astype(bool)
        rew, term, trunc = self._slice(self.sim.rewards), self._slice(self.sim.terminated), self._slice(self.sim.truncated)
        iv, info = self._slice(self.sim.info_valid), self._slice(self.sim.info)
        done = bool(self.sim.episode_done[self.k].item())
        self._append_events()
        self._log_done = done
        ids = [p + 1 for p in range(self.P) if present[p]]
        infos = {a: (info_record_to_dict(info[a - 1]) if iv[a - 1] else {}) for a in ids}
        if done and ids:
            infos[ids[-1]]["episode_done"] = True
        self.agents = [] if done else [a for a in ids if not term[a - 1]]
        return (self._obs(present), {a: float(rew[a - 1]) for a in ids}, {a: bool(term[a - 1]) for a in ids},
                {a: bool(trunc[a - 1]) for a in ids}, infos)

    def _append_events(self):
        rows, cnt = self.sim.events(self.k, self.k + 1)
        n = int(cnt.item())
        if n > rows.shape[0]:
            rows, _ = self.sim.events(self.k, self.k + 1, out=rows.new_empty((n, 9)))
        new = rows[:n].cpu().numpy()
        new[:, 0] = np.arange(1, n + 1) + (0 if self._log_done else len(self._log))
        self._log = new if self._log_done else np.concatenate([self._log, new])

    @property
    def tick(self):
        return int(self.sim.snapshot(self.k)[3][0])

    @property
    def realm(self):
        """``env.realm`` as the wrappers use it: ``tick``, ``players[id]``, ``players.dead_this_tick``
        (stat_wrapper.py:136,140) and ``event_log.get_data`` (stat_wrapper.py:123): the episode's player events,
        exported from the device after every step (Simulator.events) and kept on the host until the next reset."""
        ent, items, _, sc = self.sim.snapshot(self.k)
        cfg = self.sim.cfg

        def defense(row):
            d = 0
            for col in ("EA_EQ_HAT", "EA_EQ_TOP", "EA_EQ_BOTTOM", "EA_EQ_HELD", "EA_EQ_AMMO"):
                it = int(row[SPEC[col]])
                if it:
                    typ, lvl = int(items[it - 1][SPEC["IS_TYPE"]]), int(items[it - 1][SPEC["IS_LEVEL"]])
                    if SPEC["IT_HAT"] <= typ <= SPEC["IT_BOTTOM"]:
                        d += int(cfg[SPEC["NC_ARMOR_BASE"]]) + lvl * int(cfg[SPEC["NC_ARMOR_LEVEL"]])
                    elif SPEC["IT_ROD"] <= typ <= SPEC["IT_CHISEL"]:
                        d += int(cfg[SPEC["NC_TOOL_BASE"]]) + lvl * int(cfg[SPEC["NC_TOOL_LEVEL"]])
            return d

        st = ent[:self.P, SPEC["EA_STATUS"]]
        players = _Players({p + 1: PlayerView(ent[p], defense(ent[p])) for p in range(self.P) if st[p] == SPEC["ES_ALIVE"]})
        players.dead_this_tick = {p + 1: PlayerView(ent[p], 0) for p in range(self.P) if st[p] == SPEC["ES_DEAD_THIS_TICK"]}
        return SimpleNamespace(tick=int(sc[0]), players=players, event_log=EventLogView(self._log, int(sc[0])))

    @property
    def agent_task_map(self):
        tid, comp, sig, mp = self.sim.task_state(self.k)
        return {p + 1: [TaskView(tid[p], comp[p], sig[p], mp[p])] for p in range(self.P)}
