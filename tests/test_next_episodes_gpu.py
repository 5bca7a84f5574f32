"""GPU: pending next-episode values (DESIGN.md 2.5).  An env's automatic reset takes the seed, map and tasks written for
it, and derives the fields with no entry exactly as before.  The oracle side resets its env at the same tick with
Oracle.reset(seed, map_id, task_ids), the values the device should have used, and the two must agree bit for bit."""
import re
from pathlib import Path

import numpy as np
import pytest

from util import SMALL, build_world, run_parity

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1
SC_TICK, SC_EPISODE = 0, 5      # env scalars of a snapshot (nm_scalar, csrc/nmmo_device.cuh)


def _spec(name):
    from nmmo_b200.config import SPEC
    return SPEC[name]


def mix64(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def next_seed(seed):
    """The seed of the episode after one with seed `seed` (nmmo_step.cu, automatic reset)."""
    return mix64((seed + 0x632BE59BD9B4E019) & M64)


class AutoOracle:
    """An oracle env whose automatic reset takes the entry the device env holds: `pending` = [flags, seed, map, tasks[P]]."""

    def __init__(self, o, n_maps, n_tasks, team):
        self.o, self.n_maps, self.n_tasks, self.team = o, n_maps, n_tasks, max(1, team)
        self.flags, self.seed_v, self.map_v, self.task_v = 0, 0, 0, np.zeros(o.P, np.int32)
        self.resets = self.plain_resets = 0      # automatic resets; those with nothing pending
        self.just_reset = False
        self.rejected = 0

    def __getattr__(self, name):
        return getattr(self.o, name)

    def reset(self, seed, map_id=-1, task_ids=None):
        self.seed = int(seed)
        self.o.reset(seed, map_id, task_ids)

    def write(self, flags, seed=None, map_id=None, tasks=None):
        self.flags |= flags
        if seed is not None:
            self.seed_v = int(seed)
        if map_id is not None:
            self.map_v = int(map_id)
        if tasks is not None:
            self.task_v = np.asarray(tasks, np.int32).copy()

    def step(self, actions):
        self.just_reset = False
        if not self.o.episode_done:
            self.o.step(actions)
            return
        f = self.flags
        self.plain_resets += f == 0
        seed = self.seed_v if f & _spec("NM_NEXT_SEED") else next_seed(self.seed)
        map_id = -1
        if f & _spec("NM_NEXT_MAP"):
            if 0 <= self.map_v < self.n_maps:
                map_id = self.map_v
            else:
                self.rejected += 1
        tasks = None
        if f & _spec("NM_NEXT_TASKS"):
            self.o.reset(seed, map_id, None)          # the draws, for the teams whose entry is out of range
            drawn = self.o.task_state()[0].astype(np.int32)
            tasks = drawn.copy()
            for lead in range(0, self.o.P, self.team):
                t = int(self.task_v[lead])
                if 0 <= t < self.n_tasks:
                    tasks[lead:lead + self.team] = t
                else:
                    self.rejected += 1
        self.seed = seed
        self.o.reset(seed, map_id, tasks)
        self.flags = 0
        self.resets += 1
        self.just_reset = True


KINDS = ("seed", "map", "tasks", "all", "none")


class Entries:
    """on_tick hook of run_parity: writes entries of every kind at different ticks through Simulator.set_next, checks after
    each automatic reset that the env's flags read 0 and its value arrays kept what was written."""

    def __init__(self, sim, oracles, seed=0, bad=False, per_agent=False):
        self.rng = np.random.default_rng(seed)
        self.sim, self.oracles, self.bad, self.per_agent = sim, oracles, bad, per_agent
        self.kinds = set()
        sim.set_next_episodes(True)

    def __call__(self, t, sim, oracles):
        import torch
        torch.cuda.synchronize()
        flags = sim.next_flags.cpu().numpy()
        d_seed = sim.next_seed.cpu().numpy().view(np.uint64)
        d_map, d_task = sim.next_map.cpu().numpy(), sim.next_task.cpu().numpy()
        for e, o in enumerate(oracles):
            assert flags[e] == o.flags, f"tick {t} env {e}: flags {flags[e]} vs {o.flags}"
            if o.just_reset:
                assert flags[e] == 0
                assert int(d_seed[e]) == o.seed_v and int(d_map[e]) == o.map_v and np.array_equal(d_task[e], o.task_v), \
                    f"tick {t} env {e}: the reset changed the value arrays"
            if o.flags or (t + 3 * e) % 5:
                continue
            if e == len(oracles) - 1 and o.resets % 2 == 0:
                continue          # the last env runs every other episode with nothing pending
            kind = KINDS[(t // 5 + e) % len(KINDS)]
            self.kinds.add(kind)
            if kind == "none":
                continue
            P = o.P
            seed = int(self.rng.integers(0, 1 << 62)) * 2 + 1 if kind in ("seed", "all") else None
            hi_m, hi_t = o.n_maps + (3 if self.bad else 0), o.n_tasks + (5 if self.bad else 0)
            map_id = int(self.rng.integers(0, hi_m)) if kind in ("map", "all") else None
            tasks = None
            if kind in ("tasks", "all"):
                tasks = self.rng.integers(0, hi_t, size=P) if self.per_agent else np.full(P, self.rng.integers(0, hi_t))
            if self.bad:      # out-of-range entries go in as CUDA tensors: those are not checked on the host
                dev = sim.next_flags.device
                sim.set_next(torch.tensor([e], device=dev),
                             seeds=None if seed is None else torch.tensor([seed], dtype=torch.int64, device=dev),
                             maps=None if map_id is None else torch.tensor([map_id], dtype=torch.int32, device=dev),
                             tasks=None if tasks is None else torch.as_tensor(tasks[None], dtype=torch.int32, device=dev))
            else:
                sim.set_next([e], seeds=None if seed is None else np.array([seed], np.uint64),
                             maps=None if map_id is None else [map_id],
                             tasks=None if tasks is None else (tasks[None] if self.per_agent else tasks[:1]))
            bits = (_spec("NM_NEXT_SEED") if seed is not None else 0) | (_spec("NM_NEXT_MAP") if map_id is not None else 0) | \
                   (_spec("NM_NEXT_TASKS") if tasks is not None else 0)
            o.write(bits, seed, map_id, tasks)


def _sim(w, E):
    from nmmo_b200.lib import Simulator
    return Simulator(*w[:2], E, *w[2:])


def _oracles(w, E):
    from oracle.oracle import OracleEnv
    team = int(w[0][_spec("NC_TEAM_SIZE")])
    return [AutoOracle(OracleEnv(*w), len(w[2]), len(w[3]), team) for _ in range(E)]


def _parity(w, E, want_step, ticks, seeds, bad=False, per_agent=False, min_resets=3, check_state_every=8):
    sim, oracles = _sim(w, E), _oracles(w, E)
    assert sim.kernel_names()[0] == want_step, sim.kernel_names()
    hook = Entries(sim, oracles, seed=int(seeds[0]), bad=bad, per_agent=per_agent)
    run_parity(sim, oracles, seeds=seeds, ticks=ticks, check_state_every=check_state_every, on_tick=hook)
    assert min(o.resets for o in oracles) >= min_resets, [o.resets for o in oracles]
    assert hook.kinds >= {"seed", "map", "tasks", "all"}, hook.kinds
    assert sum(o.plain_resets for o in oracles) > 0, "no automatic reset with nothing pending"
    return sim, oracles


def _small(**over):
    return build_world(task_dim=64, **SMALL, NC_HORIZON=24, **over)


@pytest.mark.parametrize("variant,env,want", [
    ("four", {"NMMO_B200_ENVS_PER_CTA": "4"}, "nmmo_step4_kernel"),
    ("three", {"NMMO_B200_ENVS_PER_CTA": "3"}, "nmmo_step3_kernel"),
    ("two", {"NMMO_B200_ENVS_PER_CTA": "2"}, "nmmo_step_kernel"),
    ("one", {"NMMO_B200_ENVS_PER_CTA": "1"}, "nmmo_step_kernel"),
    ("big", {"NMMO_B200_FORCE_BIG": "1"}, "nmmo_step_big_kernel")])
def test_step_variants_against_oracle(monkeypatch, variant, env, want):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    sim, _ = _parity(_small(), 6, want, ticks=110, seeds=np.arange(6) + 5)
    sim.check()
    sim.close()


def _std_world(workload=None, horizon=16):
    from bench import world
    cfg, fcfg, maps, tab, emb = world(n_maps=3) if workload is None else world(workload=workload, n_maps=3)
    cfg = cfg.copy()
    cfg[_spec("NC_HORIZON")] = horizon
    return cfg, fcfg, maps, tab, emb


def test_default_shape_std_kernels_against_oracle():
    sim, _ = _parity(_std_world(), 4, "nmmo_step4_std_kernel", ticks=70, seeds=np.arange(4) + 31, check_state_every=16)
    sim.close()


def test_config5_big_std_kernel_against_oracle():
    sim, _ = _parity(_std_world("config5", horizon=8), 2, "nmmo_step_big_std_kernel", ticks=40, seeds=np.arange(2) + 9,
                     check_state_every=20)
    sim.close()


def test_teams_take_the_leaders_entry():
    w = _small(NC_TEAM_SIZE=4)
    sim, oracles = _parity(w, 4, "nmmo_step4_kernel", ticks=110, seeds=np.arange(4) + 13, per_agent=True)
    sim.close()


def test_out_of_range_entries():
    from nmmo_b200.lib import NmmoError
    w = _small()
    sim, oracles = _parity(w, 4, "nmmo_step4_kernel", ticks=110, seeds=np.arange(4) + 21, bad=True)
    rejected = sum(o.rejected for o in oracles)
    assert rejected > 0
    assert int(sim.stats()[2][5]) == rejected
    with pytest.raises(NmmoError, match="next-episode entr.*out of range"):
        sim.check()
    # host inputs out of range: ValueError, nothing written
    import torch
    before = [x.clone() for x in (sim.next_flags, sim.next_seed, sim.next_map, sim.next_task)]
    for kw in ({"maps": [len(w[2])]}, {"tasks": [len(w[3])]}, {"tasks": [-1]}, {"seeds": [-5]}):
        with pytest.raises(ValueError):
            sim.set_next([1], **kw)
    with pytest.raises(ValueError):
        sim.set_next([4], maps=[0])
    with pytest.raises(ValueError):
        sim.set_next([0, 1], tasks=np.zeros((2, 3), np.int32))
    for x, y in zip(before, (sim.next_flags, sim.next_seed, sim.next_map, sim.next_task)):
        assert torch.equal(x, y)
    sim.stats(clear=True)
    sim.check()
    sim.close()


def _outputs(sim):
    import torch
    torch.cuda.synchronize()
    return {n: getattr(sim, n).cpu().numpy().copy() for n in
            ("obs", "rewards", "terminated", "truncated", "mask", "info", "info_valid", "episode_done", "task_id")}


def _assert_same(a, b, tag):
    for n in a:
        x, y = a[n], b[n]
        if x.dtype == np.float32:
            x, y = x.view(np.uint32), y.view(np.uint32)
        assert np.array_equal(x, y), f"{tag}: {n} differ"


@pytest.mark.parametrize("shape", ["generic", "std"])
def test_nothing_pending_changes_nothing(shape):
    w = _small() if shape == "generic" else _std_world(horizon=20)
    a, b = _sim(w, 4), _sim(w, 4)
    a.set_next_episodes(True)
    assert b.next_flags is None
    for s in (a, b):
        s.set_autosample(5)
        s.reset(np.arange(4) + 40)
    assert a.kernel_names() == b.kernel_names()
    assert a.kernel_names()[0].endswith("_std_kernel") == (shape == "std")
    for t in range(70):
        _assert_same(_outputs(a), _outputs(b), f"tick {t}")
        a.step(); b.step()
    assert int(a.stats()[2][2]) >= 8 and int(a.stats()[2][2]) == int(b.stats()[2][2])
    a.set_next_episodes(False)
    assert a.next_flags is None
    a.close(); b.close()


def test_level_replay():
    """An env whose automatic reset took seed s, stepped with recorded actions, equals an env of another handle reset
    with seed s and stepped with the same actions."""
    import torch
    w = _small()
    a, b = _sim(w, 2), _sim(w, 2)
    a.set_autosample(3)
    a.reset([7, 8])
    a.set_next_episodes(True)
    s = 0xDEADBEEF12345
    a.set_next([0], seeds=[s])
    while True:
        done = bool(a.episode_done[0].item())
        a.step()
        if done:
            break
    assert int(a.next_flags[0].item()) == 0 and int(a.snapshot(0)[3][SC_TICK]) == 0
    b.reset([s, 9])
    for t in range(60):
        oa, ob = _outputs(a), _outputs(b)
        for o in (oa, ob):      # a record is defined where info_valid is set (a reset leaves the last episode's rows)
            o["info"][o["info_valid"] == 0] = 0
        for n in oa:
            k = oa[n].shape[0] // 2
            x, y = oa[n][:k], ob[n][:k]
            if x.dtype == np.float32:
                x, y = x.view(np.uint32), y.view(np.uint32)
            assert np.array_equal(x, y), f"tick {t}: {n} of the replayed level differ"
        if oa["episode_done"][0]:
            break
        x = a.actions.clone()
        y = torch.zeros_like(x)
        y[0] = x[0]
        a.step(x); b.step(y)
    a.close(); b.close()


def test_step_host_consumes_entries():
    from nmmo_b200.lib import pack_actions_u8
    import torch
    w = _small()
    a, b = _sim(w, 4), _sim(w, 4)
    for s in (a, b):
        s.set_autosample(2)
        s.reset(np.arange(4) + 60)
        s.set_next_episodes(True)
        s.set_next([0, 1, 2, 3], seeds=np.arange(4, dtype=np.uint64) + 1000, maps=[1, 2, 3, 0], tasks=[5, 6, 7, 8])
    for t in range(60):
        _assert_same(_outputs(a), _outputs(b), f"tick {t}")
        x = a.actions.clone()
        a.step(x)
        b.step_host(pack_actions_u8(x.cpu().numpy()))
    assert int(a.stats()[2][2]) >= 4
    assert int(a.next_flags.sum().item()) == 0 and int(b.next_flags.sum().item()) == 0
    a.close(); b.close()


def test_state_blobs_and_loads():
    import torch
    w = _small()
    a, b = _sim(w, 3), _sim(w, 3)
    for s in (a, b):
        s.set_autosample(4)
        s.reset(np.arange(3) + 70)
        for _ in range(10):
            s.step()
    a.set_next_episodes(True)
    a.set_next([0, 2], seeds=[11, 12], maps=[1, 1], tasks=[[3] * a.P, [4] * a.P])
    assert torch.equal(a.save_envs([0, 1, 2]), b.save_envs([0, 1, 2]))
    pend = [x.clone() for x in (a.next_flags, a.next_seed, a.next_map, a.next_task)]
    a.load_envs([0, 2], b.save_envs([1, 1]))
    for x, y in zip(pend, (a.next_flags, a.next_seed, a.next_map, a.next_task)):
        assert torch.equal(x, y)
    a.reset(np.arange(3))
    for x, y in zip(pend, (a.next_flags, a.next_seed, a.next_map, a.next_task)):
        assert torch.equal(x, y)
    a.close(); b.close()


def test_set_next_with_cuda_inputs_does_not_sync():
    import torch
    w = _small()
    s = _sim(w, 4)
    s.reset(np.arange(4))
    s.set_next_episodes(True)
    dev = s.next_flags.device
    ids = torch.tensor([1, 3], device=dev)
    seeds = torch.tensor([5, 6], dtype=torch.int64, device=dev)
    maps = torch.tensor([0, 2], dtype=torch.int32, device=dev)
    tasks = torch.tensor([4, 9], dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        s.set_next(ids, seeds=seeds, maps=maps, tasks=tasks)
        s.set_next(ids, tasks=tasks[:, None].expand(2, s.P).contiguous())
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert s.next_flags.cpu().tolist() == [0, 7, 0, 7]
    assert s.next_task[3].cpu().tolist() == [9] * s.P and s.next_map.cpu().tolist()[3] == 2
    s.close()


# ---- env pools ---------------------------------------------------------------------------------------------------------
def _pool_pair(collect_infos="async"):
    from test_env_pool_gpu import _pools, _small_env
    return _pools(_small_env(horizon=24), 4, 2, collect_infos=collect_infos)


def _entry_for(e, n):
    """The entry env e gets at its n-th tick (None: nothing)."""
    if (n + e) % 4:
        return None
    return dict(seeds=[1000 * e + n], maps=[(n // 4 + e) % 4], tasks=[(7 * n + e) % 50])


def test_env_pool_equals_lock_step():
    from test_env_pool_gpu import _same_outputs
    lock, pool = _pool_pair()
    ticks = np.zeros(4, int)
    for r in range(90):
        lock.recv()
        for e in range(4):
            x = _entry_for(e, r)
            if x:
                lock.set_next_episodes([e], **x)
        lock.send(lock.sim.actions)
        for _ in range(pool.num_batches):
            pool.recv()
            lo, hi = pool.batch_env_range
            for e in range(lo, hi):
                x = _entry_for(e, ticks[e])
                if x:
                    pool.set_next_episodes([e], **x)
                ticks[e] += 1
            if r:      # (before the first send() after a reset no batch is stepping: every env is accepted)
                with pytest.raises(ValueError, match="not in the batch"):
                    pool.set_next_episodes([2 if lo == 0 else 0], seeds=[1])
            pool.send(pool.sim.actions[lo:hi])
        _same_outputs(lock, pool, f"round {r}")
    assert int(pool.sim.stats()[2][2]) >= 8
    assert int(pool.sim.stats()[2][2]) == int(lock.sim.stats()[2][2])
    lock.close(); pool.close()


def _task_of(pool, info):
    body = info[pool.stat_prefix] if pool.stat_prefix else info
    return int(re.fullmatch(r"task_(\d+)", next(iter(body["curriculum"]))).group(1))


@pytest.mark.parametrize("collect_infos", ["async", True])
@pytest.mark.parametrize("batch", [4, 2])
def test_task_feed(collect_infos, batch):
    from nmmo_b200.task_feed import TaskFeed
    from nmmo_b200.vecenv import B200VecEnv
    from test_env_pool_gpu import _small_env
    E = 4
    pool = B200VecEnv(env_kwargs={"env": _small_env(horizon=20)}, num_envs=E, envs_per_batch=batch, env_pool=batch < E,
                      collect_infos=collect_infos)
    pool.sim.set_autosample(6)
    n_tasks = pool.task_table.shape[0]
    counter = [0]

    def sample(k):
        out = (np.arange(k) + counter[0]) % n_tasks
        counter[0] += k
        return out

    assigned = {e: [] for e in range(E)}          # every task handed to env e, in order
    orig_reset, orig_next = pool.reset_envs, pool.set_next_episodes

    def reset_envs(envs, seeds, new_tasks=None):
        for e, t in zip(envs, new_tasks):
            assigned[int(e)].append(int(t))
        return orig_reset(envs, seeds, new_tasks)

    def set_next(envs, tasks=None, **kw):
        for e, t in zip(envs, tasks):
            assigned[int(e)].append(int(t))
        return orig_next(envs, tasks=tasks, **kw)

    pool.reset_envs, pool.set_next_episodes = reset_envs, set_next
    reported = {e: [] for e in range(E)}

    def update(env, task, infos):
        assert infos and all(_task_of(pool, i) == task for i in infos), (env, task, [_task_of(pool, i) for i in infos])
        reported[env].append(task)

    feed = TaskFeed(pool, sample, update)
    feed.start(3)
    for _ in range(120 * pool.num_batches):
        feed.recv()
        lo, hi = pool.batch_env_range
        feed.send(pool.sim.actions[lo:hi])
    import torch
    torch.cuda.synchronize()
    for e in range(E):
        n = len(reported[e])
        episodes = int(pool.sim.snapshot(e)[3][SC_EPISODE])      # automatic resets since the start
        assert n >= 4 and episodes - 1 <= n <= episodes + 1, (e, n, episodes)
        # every episode ran the next task handed to the env: no seed-drawn fallback, nothing reported twice
        assert reported[e] == assigned[e][:n], (e, reported[e], assigned[e])
    assert int(pool.sim.stats()[2][5]) == 0
    pool.close()


def test_weighted_draw_snippet():
    """INTEGRATION.md's weighted-draw snippet, with all the weight on two rows: every episode after the first runs one
    of them."""
    import torch
    from test_env_pool_gpu import _small_env
    from nmmo_b200.vecenv import B200VecEnv
    text = (Path(__file__).resolve().parent.parent / "INTEGRATION.md").read_text()
    snippet = next(b for b in re.findall(r"```python\n(.*?)```", text, flags=re.S) if "refill_weighted" in b)
    pool = B200VecEnv(env_kwargs={"env": _small_env(horizon=20)}, num_envs=4, collect_infos=True)
    pool.sim.set_autosample(8)
    pool.async_reset(1)
    weights = np.zeros(pool.task_table.shape[0])
    weights[[3, 17]] = [0.4, 0.6]
    torch.manual_seed(0)
    ns = {"pool": pool, "weights": weights}
    exec(snippet, ns)
    first = pool.sim.task_id.view(4, -1)[:, 0].cpu().numpy().copy()
    seen = set()
    for _ in range(150):
        pool.recv()
        ns["refill_weighted"](*pool.batch_env_range)
        pool.send(pool.sim.actions)
        torch.cuda.synchronize()
        ep = [int(pool.sim.snapshot(e)[3][SC_EPISODE]) for e in range(4)]
        tid = pool.sim.task_id.view(4, -1)[:, 0].cpu().numpy()
        for e in range(4):
            if ep[e]:
                seen.add(int(tid[e]))
    assert seen == {3, 17}, (seen, first)
    pool.close()
