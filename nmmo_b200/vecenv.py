"""Vector-env backend with the pufferlib vectorisation contract, backed by the CUDA simulator.

This is the reference's own plugin seam: ``clean_pufferl.create`` builds
``vectorization(env_creator, env_kwargs, num_envs, envs_per_worker, envs_per_batch, env_pool,
mask_agents)`` and then only uses ``async_reset / recv / send / close`` plus a few attributes
(/root/reference/reinforcement_learning/clean_pufferl.py:106-118,151,158,175,293,357,563;
selected in /root/reference/train.py:117-125).  ``B200VecEnv`` has that shape, reads the same
``env_kwargs`` (``{"env": Namespace, "reward_wrapper": Namespace}``, train_helper.py:55) and returns
CUDA tensors, so the rollout loop can skip its ``.cpu()`` / ``.to(device)`` copies
(clean_pufferl.py:302-345).  It replaces, in one piece, pufferlib's Serial/Multiprocessing pool,
``PettingZooPufferEnv``, the RewardWrapper/BaseStatWrapper stack and ``nmmo.Env``.
"""
from __future__ import annotations

from argparse import Namespace
from typing import Dict, List, Optional

import numpy as np

from .config import SPEC, make_config, default_env_args, default_wrapper_args
from .emulation import UnflattenContext
from .lib import Simulator
from .mapgen import generate_maps
from .tasks import default_curriculum, make_task_table

INFO_NAMES = {
    "IN_LENGTH": "length", "IN_RETURN": "return",
    "IN_COD_ATTACKED": "stats/cod/attacked", "IN_COD_STARVED": "stats/cod/starved", "IN_COD_DEHYDRATED": "stats/cod/dehydrated",
    "IN_TASK_COMPLETED": "stats/task/completed", "IN_TASK_2_REWARD_SIGNAL": "stats/task/pcnt_2_reward_signal",
    "IN_TASK_0P2_MAX_PROGRESS": "stats/task/pcnt_0p2_max_progress",
    "IN_MAX_COMBAT_LEVEL": "stats/achieved/max_combat_level", "IN_MAX_HARVEST_AMMO": "stats/achieved/max_harvest_skill_ammo",
    "IN_MAX_HARVEST_CONSUM": "stats/achieved/max_harvest_skill_consum",
    "IN_MAX_PROGRESS_TO_CENTER": "stats/achieved/max_progress_to_center", "IN_EARNED_GOLD": "stats/achieved/earned_gold",
    "IN_MAX_DAMAGE": "stats/achieved/max_damage", "IN_MAXLVL_ARMOR": "stats/achieved/max_armor_level",
    "IN_MAXLVL_WEAPON": "stats/achieved/max_weapon_level", "IN_MAXLVL_TOOL": "stats/achieved/max_tool_level",
    "IN_MAXLVL_AMMO": "stats/achieved/max_ammo_level", "IN_MAXLVL_CONSUMABLE": "stats/achieved/max_consumable_level",
    "IN_AGENT_KILLS": "stats/achieved/agent_kill_count", "IN_NPC_KILLS": "stats/achieved/npc_kill_count",
    "IN_UNIQUE_EVENTS": "stats/achieved/unique_events",
    "IN_EV_EAT_FOOD": "stats/event/eat_food", "IN_EV_DRINK_WATER": "stats/event/drink_water",
    "IN_EV_SCORE_HIT": "stats/event/score_hit", "IN_EV_PLAYER_KILL": "stats/event/player_kill",
    "IN_EV_CONSUME_ITEM": "stats/event/consume_item", "IN_EV_HARVEST_ITEM": "stats/event/harvest_item",
    "IN_EV_LIST_ITEM": "stats/event/list_item", "IN_EV_BUY_ITEM": "stats/event/buy_item",
    "IN_EQUIP_ARMOR": "stats/event/equip_armor", "IN_EQUIP_WEAPON": "stats/event/equip_weapon",
    "IN_EQUIP_TOOL": "stats/event/equip_tool", "IN_EQUIP_AMMO": "stats/event/equip_ammo",
    "IN_HARVEST_WEAPON": "stats/event/harvest_weapon",
}


def info_record_to_dict(row: np.ndarray, episode_done: bool = False, stat_prefix: Optional[str] = None,
                        task_names: Optional[List[str]] = None) -> Dict:
    """nm_info float record -> the dict BaseStatWrapper emits (stat_wrapper.py:132-185).  Keys whose
    record entry is NaN are absent, exactly like the achieved/max_*_level keys of the reference."""
    info: Dict = {"stats": {}}
    for col, key in INFO_NAMES.items():
        v = float(row[SPEC[col]])
        if v != v:
            continue
        if key.startswith("stats/"):
            info["stats"][key[len("stats/"):]] = v
        else:
            info[key] = v
    info["length"] = int(info["length"])
    tid = int(row[SPEC["IN_TASK_ID"]])
    # curriculum[spec_name] = (max_progress, reward_signal_count), stat_wrapper.py:159
    name = task_names[tid] if task_names is not None and 0 <= tid < len(task_names) else f"task_{tid}"
    info["curriculum"] = {name: (float(row[SPEC["IN_CURR_MAX_PROGRESS"]]), int(row[SPEC["IN_CURR_REWARD_SIGNALS"]]))}
    if episode_done:
        info["episode_done"] = True
    if stat_prefix:
        info = {stat_prefix: info}
    return info


class _Space:
    def __init__(self, shape, dtype, nvec=None):
        self.shape, self.dtype, self.nvec = tuple(shape), dtype, nvec


class DriverEnv:
    """What clean_pufferl / the policies read from ``pool.driver_env`` (clean_pufferl.py:151,
    agent_zoo/takeru/policy.py:27)."""

    def __init__(self, cfg, ctx: UnflattenContext, action_dims):
        self.unflatten_context = ctx
        self.obs_sz = ctx.obs_sz
        self.observation_space = _Space((ctx.obs_sz,), np.uint8)
        self.action_space = _Space((len(action_dims),), np.int32, nvec=np.asarray(action_dims))
        self.single_observation_space = self.observation_space
        self.single_action_space = self.action_space
        self.possible_agents = list(range(1, int(cfg[SPEC["NC_N_PLAYERS"]]) + 1))
        self.config = cfg


class _BatchedSimulator(Simulator):
    """Simulator of an env pool: the calls that touch the whole handle first make the current stream wait for every batch
    stream, so they never run while a batch's step is in flight (nmmo_reset reads and writes back the scalars of every
    env).  The other whole-handle calls (snapshot, inject_rng, stats, check, task_state) synchronise the device."""

    batch_streams = ()

    def join_batches(self):
        cur = self.torch.cuda.current_stream(self.device)
        for st in self.batch_streams:
            cur.wait_stream(st)

    def reset(self, *args, **kwargs):
        self.join_batches()
        return super().reset(*args, **kwargs)

    def step(self, actions=None):
        self.join_batches()
        return super().step(actions)

    def step_host(self, *args, **kwargs):
        self.join_batches()
        return super().step_host(*args, **kwargs)

    def save_envs(self, *args, **kwargs):
        self.join_batches()
        return super().save_envs(*args, **kwargs)

    def load_envs(self, *args, **kwargs):
        self.join_batches()
        return super().load_envs(*args, **kwargs)

    def set_event_log(self, *args, **kwargs):
        self.join_batches()
        return super().set_event_log(*args, **kwargs)


class B200VecEnv:
    def __init__(self, env_creator=None, env_args=None, env_kwargs: Optional[Dict] = None, num_envs: int = 1,
                 envs_per_worker: int = 1, envs_per_batch: Optional[int] = None, env_pool: bool = False,
                 mask_agents: bool = True, agent: str = "takeru", device: int = 0, env_base: int = 0,
                 maps: Optional[np.ndarray] = None, task_rows=None, map_seed: int = 2023, collect_infos="async",
                 task_embed: Optional[np.ndarray] = None, info_cap: int = 16384, curriculum: Optional[str] = None,
                 task_names: Optional[List[str]] = None, event_log_cap: int = 0):
        """collect_infos: "async" (default) -- finished-agent info records are compacted on the device, copied to
        pinned host memory on a side stream and handed out by the NEXT recv() (no host sync in the loop; call
        drain_infos() after the last step); True -- gathered synchronously inside recv() (exact tick, one host sync
        per step); False -- never (use stats()).

        envs_per_batch: b envs per recv()/send() (default num_envs: one lock-step tick per call).  b must divide num_envs;
        the pool then holds K = num_envs / b batches of contiguous envs, batch k = envs [k*b, (k+1)*b), handed out in
        the fixed order 0, 1, ..., K-1, 0, ... whatever env_pool says; each batch steps on its own CUDA stream while the
        caller works on the batch it was handed.  recv() returns the batch's B = b * agents_per_env rows, with env_id
        the batch's global agent slots (the LSTM-state index of clean_pufferl.py:313-314); batch_env_range is its
        (lo, hi).  send() takes the actions of those B rows.

        event_log_cap: 0 (default) leaves the event log off.  n > 0 switches it on: every send() also exports the
        stepped batch's player events, as rows of the reference's event log, into a device buffer of n rows per batch,
        and events() hands out the rows of the batch the last recv() returned (DESIGN.md 2.4)."""
        if int(event_log_cap) < 0:
            raise ValueError(f"event_log_cap must be >= 0 (0 = event log off), got {event_log_cap}")
        # env_creator / env_args / envs_per_worker are accepted for signature compatibility
        self.num_envs = int(num_envs)
        b = self.num_envs if envs_per_batch is None else int(envs_per_batch)
        if self.num_envs < 1 or not 1 <= b <= self.num_envs or self.num_envs % b:
            raise ValueError(f"envs_per_batch must divide num_envs with 1 <= envs_per_batch <= num_envs (got {b} of {self.num_envs}); "
                             "batches hold contiguous envs of equal size, e.g. 15 envs in batches of 5, or 18 in batches of 6")
        self.envs_per_batch = b
        self.num_batches = self.num_envs // b
        self.env_pool = bool(env_pool)      # the batch order is round-robin either way (a legal "first ready" order)
        env_kwargs = env_kwargs or {}
        env_ns = env_kwargs.get("env") or default_env_args(resilient_population=0 if agent in ("takeru", "yaofeng", "hybrid") else 0.2)
        wrap_ns = env_kwargs.get("reward_wrapper") or default_wrapper_args(agent)
        if isinstance(env_ns, dict):
            env_ns = Namespace(**env_ns)
        if isinstance(wrap_ns, dict):
            wrap_ns = Namespace(**wrap_ns)
        self.cfg, self.fcfg = make_config(env_ns, wrap_ns, agent)
        # num_maps is honoured as given (takeru 1280, yaofeng 1024: config.yaml:131,113); generation costs ~2 ms per map
        n_maps = max(1, int(getattr(env_ns, "num_maps", 64))) if maps is None else len(maps)
        self.maps = generate_maps(self.cfg, map_seed, n_maps) if maps is None else maps
        # curriculum: a table translated from the reference's own spec sources (nmmo_b200/curriculum.py): "heldout" (the 63
        # evaluation tasks with their real 2048-d embeddings, evaluate.py:20,52), "sample_eval", "manual" (training specs)
        if curriculum is not None:
            from .curriculum import load_table
            tab = load_table(curriculum)
            task_rows, task_names = tab["rows"], tab["names"]
            if tab["embed"] is not None and tab["embed"].shape[1] == int(self.cfg[SPEC["NC_TASK_DIM"]]):
                task_embed = tab["embed"]
        self.task_names = list(task_names) if task_names is not None else None
        rows = task_rows if task_rows is not None else default_curriculum()
        self.task_table, self.task_embed = make_task_table(rows, int(self.cfg[SPEC["NC_TASK_DIM"]]), seed=3)
        if task_embed is not None:      # real embeddings (e.g. nmmo_b200.curriculum.load_heldout): fp16 bit patterns [T, task_dim]
            te = np.ascontiguousarray(task_embed)
            self.task_embed = te.view(np.uint16) if te.dtype == np.float16 else te.astype(np.uint16)
            assert self.task_embed.shape == (self.task_table.shape[0], int(self.cfg[SPEC["NC_TASK_DIM"]]))
        sim_cls = Simulator if self.num_batches == 1 else _BatchedSimulator
        self.sim = sim_cls(self.cfg, self.fcfg, self.num_envs, self.maps, self.task_table, self.task_embed,
                           device=device, env_base=env_base)
        self.agents_per_env = self.sim.P
        self.stat_prefix = getattr(wrap_ns, "stat_prefix", None)
        self.collect_infos = collect_infos
        ctx = UnflattenContext(self.cfg)
        self.driver_env = DriverEnv(self.cfg, ctx, ctx.layout.action_dims)
        self.single_observation_space = self.driver_env.observation_space
        self.single_action_space = self.driver_env.action_space
        self.mask_agents = mask_agents
        self.multi_envs = None           # replay path (train_helper.py:133) is out of scope
        import torch
        self._torch = torch
        self.env_id = torch.arange(self.num_envs * self.agents_per_env, device=self.sim.obs.device)
        self._pending = False
        self.last_info_slots = []
        self.env_base = int(env_base)
        self._info_cap = int(min(info_cap, b * self.agents_per_env))
        self._next_batch = 0
        self.batch_env_range = (0, self.num_envs)      # envs [lo, hi) of the batch the last recv() returned
        if self.num_batches > 1:
            dev = self.sim.obs.device
            self._streams = [torch.cuda.Stream(device=dev) for _ in range(self.num_batches)]
            self._sent = [torch.cuda.Event() for _ in range(self.num_batches)]       # actions of batch k are ready
            self._stepped = [torch.cuda.Event() for _ in range(self.num_batches)]    # batch k's outputs are ready
            self.sim.batch_streams = self._streams
        self._info_q = None              # in-flight async gather: (event, n, idx, rows, done)
        self._info_stream = None
        self._recv_batch = 0
        self._ev = None                  # event log on: per batch (rows int32 [event_log_cap, 9], count int32 [1])
        if event_log_cap:
            self.sim.set_event_log(True)
            dev = self.sim.obs.device
            self._ev = [(torch.empty((int(event_log_cap), 9), dtype=torch.int32, device=dev),
                         torch.zeros(1, dtype=torch.int32, device=dev)) for _ in range(self.num_batches)]

    # ---- pufferlib pool contract -------------------------------------------------------
    def async_reset(self, seed: int = 0):
        # seeds derive from the GLOBAL env index (INTEGRATION.md section 5): two shards of a job reproduce the
        # trajectories of one handle holding all the envs
        from .dist import global_seeds
        self.sim.reset(global_seeds(int(seed), self.env_base, self.num_envs))
        self._export_all_events()
        self._info_q = None
        self._pending = True
        self._next_batch = 0

    def reset_envs(self, env_indices, seeds, new_tasks=None):
        """Reset some envs, optionally assigning each a task (one table row for all of its agents): the
        curriculum hook of /root/reference/syllabus_wrapper.py:129-150 for a batch of envs."""
        E, P = self.num_envs, self.agents_per_env
        mask = np.zeros(E, np.uint8); sd = np.zeros(E, np.uint64)
        mask[np.asarray(env_indices)] = 1; sd[np.asarray(env_indices)] = np.asarray(seeds, np.uint64)
        task_ids = None
        if new_tasks is not None:
            task_ids = np.zeros((E, P), np.int32)
            task_ids[np.asarray(env_indices)] = np.asarray(new_tasks, np.int32).reshape(-1, 1)
        self.sim.reset(sd, task_ids=task_ids, env_mask=mask)
        self._export_all_events()
        self._pending = True

    def save_envs(self, env_indices):
        """Saved state of envs `env_indices` -> uint8 CUDA tensor [n, sim.state_bytes] (DESIGN.md 2.3).  Call it where
        reset_envs may be called; a batch in flight finishes first.  A checkpoint of the whole pool is
        ``torch.save(pool.save_envs(range(pool.num_envs)), path)`` next to the trainer's own checkpoint."""
        return self.sim.save_envs(env_indices)

    def load_envs(self, env_indices, states):
        """Put saved states (rows of save_envs, from this pool or another one of the same world) into envs
        `env_indices`, where reset_envs may be called.  Like reset_envs it leaves the outputs pending: the restored envs'
        observations, rewards, flags and masks appear in their batch's next recv(), and so do the infos of the tick
        they were saved at, which are handed out again."""
        self.sim.load_envs(env_indices, states)
        self._export_all_events()
        self._pending = True

    def events(self):
        """(rows int32 CUDA [event_log_cap, 9], count int32 CUDA [1]): the player events of the step whose outputs the
        last recv() returned, for that batch's envs (none for envs reset or loaded since), as Simulator.events lays them
        out: rows [env, ent_id, tick, event, type, level, number, gold, target] by env, agent and order of occurrence,
        count[0] the number of rows (only the first event_log_cap are kept).  Views of the batch's buffer, ready on the
        caller's stream with no host sync, and rewritten by the batch's next send()."""
        if self._ev is None:
            raise RuntimeError("the event log is off: create the pool with event_log_cap > 0")
        return self._ev[self._recv_batch]

    def _export_all_events(self):
        """After a reset or load: every batch's rows again describe the envs as they now stand (reset and loaded envs
        have no events).  Runs on the current stream, which the sim call has made wait for every batch stream."""
        if self._ev is not None:
            b = self.envs_per_batch
            for k, (rows, cnt) in enumerate(self._ev):
                self.sim.events(k * b, (k + 1) * b, out=rows, count=cnt)

    def sim_env_base(self) -> int:
        return self.env_base

    def _infos_from(self, idx, rows, done):
        infos: List[Dict] = []
        last = {}
        for k, a in enumerate(idx):
            last[int(a) // self.agents_per_env] = k
        for k, a in enumerate(idx):
            e = int(a) // self.agents_per_env
            infos.append(info_record_to_dict(rows[k], episode_done=bool(done[e]) and last[e] == k, stat_prefix=self.stat_prefix,
                                             task_names=self.task_names))
        return infos

    def _enqueue_infos(self, s0: int, s1: int):
        """Compact the finished-agent records of slots [s0, s1) (this tick's, or the batch's) on the device (fixed
        capacity, no size read-back) and start their copy to pinned host memory on a side stream."""
        t, s = self._torch, self.sim
        cap = self._info_cap
        if self._info_stream is None:
            self._info_stream = t.cuda.Stream(device=s.obs.device)
            self._info_host = [(t.empty(1, dtype=t.int64).pin_memory(), t.empty(cap, dtype=t.int64).pin_memory(),
                                t.empty((cap, s.info.shape[1]), dtype=t.float32).pin_memory(),
                                t.empty(self.num_envs, dtype=t.uint8).pin_memory()) for _ in range(2)]
            self._info_flip = 0
        valid = s.info_valid[s0:s1]
        n_d = valid.sum(dtype=t.int64).reshape(1)
        idx_d = t.nonzero_static(valid, size=cap, fill_value=0).flatten()
        if s0:
            idx_d += s0
        rows_d = s.info[idx_d]
        done_d = s.episode_done.clone()
        ev = t.cuda.Event()
        cur = t.cuda.current_stream(s.obs.device)
        self._info_stream.wait_stream(cur)
        h = self._info_host[self._info_flip]; self._info_flip ^= 1
        with t.cuda.stream(self._info_stream):
            h[0].copy_(n_d, non_blocking=True); h[1].copy_(idx_d, non_blocking=True)
            h[2].copy_(rows_d, non_blocking=True); h[3].copy_(done_d, non_blocking=True)
            for x in (n_d, idx_d, rows_d, done_d):
                x.record_stream(self._info_stream)
            ev.record(self._info_stream)
        self._info_q = (ev, h, valid.clone(), s0)

    def drain_infos(self):
        """Infos of the in-flight asynchronous gather (the last step's), if any."""
        q, self._info_q = self._info_q, None
        self.last_info_slots = []
        if q is None:
            return []
        ev, h, valid_d, s0 = q
        ev.synchronize()           # recorded a whole tick ago on a side stream: normally already complete
        n = int(h[0][0])
        if n > self._info_cap:
            # more agents finished in one tick than the staging holds (every env truncating at the horizon together):
            # gather them synchronously.  Their records are still intact: a slot cannot finish again in the tick
            # that resets its env.  (An env pool's batch may be stepping again: wait for it first.)
            if self.num_batches > 1:
                self.sim.join_batches()
            idx_d = valid_d.nonzero().flatten() + s0
            idx, rows = idx_d.cpu().numpy(), self.sim.info[idx_d].cpu().numpy()
        else:
            idx, rows = h[1][:n].numpy().copy(), h[2][:n].numpy()
        self.last_info_slots = idx
        return self._infos_from(idx, rows, h[3].numpy())

    def recv(self):
        """-> (obs uint8 [B, obs_sz], reward f32 [B], terminated u8 [B], truncated u8 [B], infos,
        env_id [B], mask u8 [B]) -- all CUDA tensors except `infos` (list of dicts).

        The returned tensors are views of the handle's own buffers, and the NEXT step decodes the actions' target
        indices by reading entity / item ids back from this very observation buffer (csrc/nmmo_step.cu, action decode):
        treat `obs` as read-only.  A consumer that edits observations in place must work on a copy
        (`recv_copy=True` at construction is not offered on purpose: 13 GB per tick)."""
        s = self.sim
        if not self._pending:
            raise RuntimeError("recv() without a preceding async_reset()/send(): the outputs on the device were already handed out")
        P, b, k = self.agents_per_env, self.envs_per_batch, self._next_batch
        lo, hi = k * b, (k + 1) * b
        self.batch_env_range = (lo, hi)
        self._recv_batch = k
        s0, s1 = lo * P, hi * P
        if self.num_batches > 1:
            # the caller's stream waits for the batch's last step; the host does not
            self._torch.cuda.current_stream(s.obs.device).wait_event(self._stepped[k])
        infos: List[Dict] = []
        self.last_info_slots = []        # flat agent slot (env * agents_per_env + agent) of each entry of `infos`
        if self.collect_infos == "async":
            infos = self.drain_infos()   # the previous recv()'s records (their copy ran underneath that step)
            self._enqueue_infos(s0, s1)
        elif self.collect_infos:
            # only this batch's flags: the other batches' still hold their last step, whose infos were handed out then
            valid = s.info_valid[s0:s1].nonzero().flatten()
            if valid.numel():
                if s0:
                    valid += s0
                idx = valid.cpu().numpy()
                self.last_info_slots = idx
                infos = self._infos_from(idx, s.info[valid].cpu().numpy(), s.episode_done.cpu().numpy())
        self._pending = False
        if self.num_batches == 1:
            return s.obs, s.rewards, s.terminated, s.truncated, infos, self.env_id, s.mask
        return (s.obs[s0:s1], s.rewards[s0:s1], s.terminated[s0:s1], s.truncated[s0:s1], infos, self.env_id[s0:s1],
                s.mask[s0:s1])

    def send(self, actions):
        """actions: [B, 12] for the B = envs_per_batch * agents_per_env slots the last recv() returned."""
        t = self._torch
        a = actions if t.is_tensor(actions) else t.as_tensor(np.asarray(actions))
        a = a.to(device=self.sim.obs.device, dtype=t.int32).reshape(self.envs_per_batch, self.agents_per_env, 12).contiguous()
        if self.num_batches == 1:
            self.sim.step(a)
            if self._ev is not None:
                self.sim.events(0, self.num_envs, out=self._ev[0][0], count=self._ev[0][1])
        else:
            k = self._next_batch
            lo, hi = self.batch_env_range
            st = self._streams[k]
            self._sent[k].record(t.cuda.current_stream(self.sim.obs.device))
            st.wait_event(self._sent[k])
            with t.cuda.stream(st):
                self.sim.step_envs(lo, hi, a)
                if self._ev is not None:
                    self.sim.events(lo, hi, out=self._ev[k][0], count=self._ev[k][1])
                self._stepped[k].record(st)
            a.record_stream(st)      # the caching allocator must not hand `a` out again before the step has read it
            self._next_batch = (k + 1) % self.num_batches
        self._pending = True

    def close(self):
        self.sim.close()

    # ---- extras --------------------------------------------------------------------------
    def stats(self, clear: bool = False) -> Dict[str, float]:
        """Means of the finished-agent infos since the last clear (clean_pufferl.py:381-390)."""
        if self.num_batches > 1:
            self.sim.join_batches()
        self.sim.check()             # a dropped event makes these means wrong: fail instead of reporting them
        sums, counts, counters = self.sim.stats(clear)
        out = {}
        for col, key in INFO_NAMES.items():
            n = counts[SPEC[col]]
            if n > 0:
                out[key] = sums[SPEC[col]] / n
        out["agent_steps"] = float(counters[1]); out["slot_steps"] = float(counters[0]); out["episodes"] = float(counters[2])
        return out
