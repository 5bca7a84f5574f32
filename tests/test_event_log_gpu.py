"""GPU: the event log (DESIGN.md 2.4) -- every player event of a step as a row of the reference's event log.

The CPU oracle keeps the reference's per-player log (oracle_log_rows); its rows of the current tick, laid out by env and
agent, must equal the device's rows exactly, in order, every tick, for every kernel variant.  Switching the log on must
change nothing else the simulator produces.
"""
import collections

import numpy as np
import pytest

from util import SMALL, build_world, run_parity

pytestmark = pytest.mark.gpu

TARGETED = (11, 12, 26, 35)      # SCORE_HIT, PLAYER_KILL, LOOT_ITEM, LOOT_GOLD: the events with a target
OUTS = ("obs", "rewards", "terminated", "truncated", "mask", "info", "info_valid", "episode_done", "actions")


def _rich(agent="takeru", horizon=400, **over):
    # test_small_world_rich_interactions: slow starvation keeps agents alive for items, market, combat and level-ups
    return build_world(agent=agent, task_dim=64, **SMALL, NC_HORIZON=horizon, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3,
                       NC_WEAPON_DROP_THR=1 << 30, **over)


def _sim(w, E, log=True):
    from nmmo_b200.lib import Simulator
    sim = Simulator(*w[:2], E, *w[2:])
    if log:
        sim.set_event_log(True)
    return sim


def _oracles(w, E):
    from oracle.oracle import OracleEnv
    return [OracleEnv(*w) for _ in range(E)]


def gpu_rows(sim, lo=0, hi=None):
    import torch
    rows, cnt = sim.events(lo, hi)
    torch.cuda.synchronize()
    n = int(cnt.item())
    assert n <= rows.shape[0]
    return rows[:n].cpu().numpy()


def oracle_rows(oracles, lo=0):
    """The oracles' rows of their current tick, env column = lo + index, by env then agent then record order."""
    out = [np.zeros((0, 9), np.int32)]
    for e, o in enumerate(oracles):
        for p in range(o.P):
            r = o.log_rows(p)
            r = r[r[:, 2] == o.tick].copy()
            r[:, 0] = lo + e
            out.append(r)
    return np.concatenate(out)


def assert_rows(g, o, tag):
    if g.shape == o.shape and np.array_equal(g, o):
        return
    n = min(len(g), len(o))
    bad = np.flatnonzero((g[:n] != o[:n]).any(axis=1))
    k = int(bad[0]) if len(bad) else n
    raise AssertionError(f"{tag}: {len(g)} device rows, {len(o)} oracle rows; first difference at row {k}: "
                         f"device {g[k].tolist() if k < len(g) else None} oracle {o[k].tolist() if k < len(o) else None}")


class Parity:
    """on_tick hook of run_parity: device rows == oracle rows; tallies what the run produced."""

    def __init__(self):
        self.codes, self.targets, self.rows = collections.Counter(), set(), 0

    def __call__(self, t, sim, oracles):
        g = gpu_rows(sim)
        assert_rows(g, oracle_rows(oracles), f"tick {t}")
        self.rows += len(g)
        self.codes.update(g[:, 3].tolist())
        tg = g[np.isin(g[:, 3], TARGETED)]
        assert (tg[:, 8] != 0).all(), "a targeted event without its target"
        assert (g[~np.isin(g[:, 3], TARGETED), 8] == 0).all()
        self.targets.update(np.sign(tg[:, 8]).tolist())


def test_oracle_parity_every_code():
    """Three worlds, every tick, exact rows in order; together they produce all 17 event codes, with player and NPC
    targets.  The start-kit world allows shared tiles: Give and GiveGold need the giver on the target's tile."""
    from nmmo_b200.config import ObsLayout, SPEC
    seen = Parity()
    for w, seeds, ticks, act in (
            (_rich(), np.arange(4) + 5, 420, None),
            (_rich(agent="neurips23_start_kit", NC_ALLOW_OCCUPIED=1), np.arange(4) + 5, 420, None),
            (build_world(task_dim=64, **SMALL, NC_HORIZON=120, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=2,
                         NC_WEAPON_DROP_THR=1 << 30), np.arange(4) + 31, 125, "adversarial")):
        sim, oracles = _sim(w, 4), _oracles(w, 4)
        action_fn = None
        if act == "adversarial":      # test_adversarial_actions: every head uniform over [-2, width + 2)
            dims, rng = np.asarray(ObsLayout(w[0]).action_dims), np.random.default_rng(5)
            action_fn = lambda t, obs: rng.integers(-2, dims[None, None, :] + 2, size=(4, sim.P, 12))
        stats = run_parity(sim, oracles, seeds=seeds, ticks=ticks, action_fn=action_fn, check_state_every=0, on_tick=seen)
        assert stats["episodes_done"] >= 1
        sim.close()
    codes = {v for k, v in SPEC.items() if k.startswith("EV_")}
    assert len(codes) == 17 and set(seen.codes) == codes, f"missing codes {sorted(codes - set(seen.codes))}"
    assert seen.targets == {-1, 1}, "both player and NPC targets must occur"


def _variant_rows(monkeypatch, env, ticks=200, E=9):
    """Rows of every tick of a default-shape run with the built-in sampler (horizon 80: two automatic resets)."""
    import torch
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    try:
        from bench import world
        from nmmo_b200.config import SPEC
        cfg, fcfg, maps, tab, emb = world(n_maps=2)
        cfg = cfg.copy()
        cfg[SPEC["NC_HORIZON"]] = 80
        sim = _sim((cfg, fcfg, maps, tab, emb), E)
        names = sim.kernel_names()[0]
        sim.reset(np.arange(E) + 3)
        out = []
        for t in range(ticks):
            sim.sample_actions(17)
            sim.step()
            out.append(gpu_rows(sim))
        torch.cuda.synchronize()
        sim.close()
    finally:
        for k in env:
            monkeypatch.delenv(k)
    return names, out


def test_kernel_variants_agree(monkeypatch):
    names, ref = _variant_rows(monkeypatch, {})
    assert names == "nmmo_step4_std_kernel"
    assert sum(len(r) for r in ref) > 1000
    for env, want in (({"NMMO_B200_NO_STD_STEP": "1"}, "nmmo_step4_kernel"),
                      ({"NMMO_B200_ENVS_PER_CTA": "4"}, "nmmo_step4_std_kernel"),
                      ({"NMMO_B200_ENVS_PER_CTA": "3"}, "nmmo_step3_std_kernel"),
                      ({"NMMO_B200_ENVS_PER_CTA": "2"}, "nmmo_step_kernel"),
                      ({"NMMO_B200_ENVS_PER_CTA": "1"}, "nmmo_step_kernel")):
        got_names, rows = _variant_rows(monkeypatch, env)
        assert got_names == want, (env, got_names)
        for t, (a, b) in enumerate(zip(ref, rows)):
            assert_rows(b, a, f"{env} tick {t}")


def test_big_family_against_oracle(monkeypatch):
    from bench import world
    from nmmo_b200.config import SPEC
    monkeypatch.setenv("NMMO_B200_FORCE_BIG", "1")
    w = _rich()
    sim, oracles = _sim(w, 3), _oracles(w, 3)
    monkeypatch.delenv("NMMO_B200_FORCE_BIG")
    assert sim.kernel_names()[0] == "nmmo_step_big_kernel"
    seen = Parity()
    run_parity(sim, oracles, seeds=np.arange(3) + 5, ticks=150, check_state_every=0, on_tick=seen)
    assert seen.rows > 500
    sim.close()
    # the config-5 std kernels (bench.py --workload config5), horizon 24: the run passes an automatic reset
    cfg, fcfg, maps, tab, emb = world(workload="config5", n_maps=2)
    cfg = cfg.copy()
    cfg[SPEC["NC_HORIZON"]] = 24
    w5 = (cfg, fcfg, maps, tab, emb)
    sim, oracles = _sim(w5, 3), _oracles(w5, 3)
    assert sim.kernel_names() == ("nmmo_step_big_std_kernel", "nmmo_obs_big_std_kernel")
    seen = Parity()
    stats = run_parity(sim, oracles, seeds=np.arange(3) + 21, ticks=48, action_seed=1, check_state_every=0, on_tick=seen)
    assert stats["episodes_done"] >= 3 and seen.rows > 1000
    assert sim.kernel_names() == ("nmmo_step_big_std_kernel", "nmmo_obs_big_std_kernel")
    sim.close()


def test_logging_changes_nothing_else():
    import torch
    w = build_world(task_dim=64, **SMALL, NC_HORIZON=70, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3)
    E = 5
    on, off = _sim(w, E, log=True), _sim(w, E, log=False)
    for s in (on, off):
        s.reset(np.arange(E) + 40)
    for t in range(80):
        for s in (on, off):
            s.sample_actions(5)
            s.step()
        torch.cuda.synchronize()
        for name in OUTS:
            x, y = getattr(on, name), getattr(off, name)
            if x.dtype == torch.float32:
                x, y = x.view(torch.int32), y.view(torch.int32)
            assert torch.equal(x, y), f"tick {t}: {name} differ"
        if t % 10 == 9:
            for e in range(E):
                for a, b in zip(on.snapshot(e), off.snapshot(e)):
                    assert np.array_equal(a, b), f"tick {t} env {e}: tables differ"
                for a, b in zip(on.task_state(e), off.task_state(e)):
                    assert np.array_equal(a, b), f"tick {t} env {e}: task state differs"
    for a, b in zip(on.stats(), off.stats()):
        assert np.array_equal(a, b), "stats differ"
    assert on.stats()[2][2] >= E, "every env must finish an episode"
    on.close(); off.close()


@pytest.mark.parametrize("b", [2, 4])
def test_env_pool_batches_equal_lock_step(b):
    import torch
    from test_env_pool_gpu import _small_env
    from nmmo_b200.vecenv import B200VecEnv
    E, cap = 8, 4096
    lock = B200VecEnv(env_kwargs={"env": _small_env()}, num_envs=E, event_log_cap=cap)
    pool = B200VecEnv(env_kwargs={"env": _small_env()}, num_envs=E, envs_per_batch=b, env_pool=True, event_log_cap=cap)
    for p in (lock, pool):
        p.sim.set_autosample(11)
        p.async_reset(3)

    def host(rows_cnt):
        rows, cnt = rows_cnt
        torch.cuda.synchronize()
        n = int(cnt.item())
        assert n <= cap
        return rows[:n].cpu().numpy()

    total = 0
    for r in range(90):
        lock.recv()
        ref = host(lock.events())
        lock.send(lock.sim.actions)
        for _ in range(pool.num_batches):
            pool.recv()
            lo, hi = pool.batch_env_range
            got = host(pool.events())
            assert_rows(got, ref[(ref[:, 0] >= lo) & (ref[:, 0] < hi)], f"round {r} batch [{lo}, {hi})")
            total += len(got)
            pool.send(pool.sim.actions[lo:hi])
    assert total > 1000
    assert int(pool.sim.stats()[2][2]) >= E, "every env must have reset"
    lock.close(); pool.close()


def test_semantics():
    import torch
    w = build_world(task_dim=64, **SMALL, NC_HORIZON=200, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3)
    E = 4
    sim, twin = _sim(w, E), _sim(w, E)
    for s in (sim, twin):
        s.reset(np.arange(E) + 9)
    for t in range(30):
        for s in (sim, twin):
            s.sample_actions(2)
            s.step()
        assert_rows(gpu_rows(twin), gpu_rows(sim), f"identical runs, tick {t}")
    full = gpu_rows(sim)
    assert all((full[:, 0] == e).any() for e in range(E))

    # a small cap: the true count, the first cap rows, and nothing written beyond them
    cap = len(full) // 3
    buf = torch.full((cap + 4, 9), -777, dtype=torch.int32, device=sim.obs.device)
    rows, cnt = sim.events(out=buf[:cap])
    torch.cuda.synchronize()
    assert int(cnt.item()) == len(full)
    assert np.array_equal(rows.cpu().numpy(), full[:cap])
    assert (buf[cap:] == -777).all()
    _, cnt = sim.events(out=buf[:0])
    assert int(cnt.item()) == len(full)
    # a sub-range
    assert_rows(gpu_rows(sim, 1, 3), full[(full[:, 0] >= 1) & (full[:, 0] < 3)], "range [1, 3)")

    # reset and load clear the affected envs' events, and only theirs
    mask = np.zeros(E, np.uint8); mask[1] = 1
    sim.reset(np.arange(E) + 100, env_mask=mask)
    assert_rows(gpu_rows(sim), full[full[:, 0] != 1], "after reset of env 1")
    saved = sim.save_envs([3])
    sim.load_envs([2], saved)
    assert_rows(gpu_rows(sim), full[(full[:, 0] != 1) & (full[:, 0] != 2)], "after load into env 2")
    sim.set_event_log(True)      # on again: every count zeroed
    assert len(gpu_rows(sim)) == 0
    sim.close(); twin.close()


def test_refusals():
    import ctypes as C
    import torch
    from nmmo_b200.lib import NmmoError
    w = build_world(task_dim=64, **SMALL, NC_HORIZON=50)
    sim = _sim(w, 3, log=False)
    sim.reset(np.arange(3))
    with pytest.raises(NmmoError, match=r"error -4: the event log is off"):
        sim.events()
    sim.set_event_log(True)
    rows = torch.zeros((64, 9), dtype=torch.int32, device=sim.obs.device)
    cnt = torch.zeros(2, dtype=torch.int32, device=sim.obs.device)
    L, h, st = sim.L, sim.h, sim._stream()
    p = lambda x, off=0: C.c_void_p(x.data_ptr() + off)
    for lo, hi in ((1, 1), (2, 1), (-1, 2), (0, 4)):
        assert L.nmmo_events(h, lo, hi, p(rows), 64, p(cnt), st) == -1
        assert b"0 <= env_lo < env_hi <= E" in L.nmmo_last_error()
    assert L.nmmo_events(h, 0, 3, p(rows), -1, p(cnt), st) == -1
    assert b"cap must be >= 0" in L.nmmo_last_error()
    assert L.nmmo_events(h, 0, 3, p(rows, 2), 8, p(cnt), st) == -1
    assert b"4-byte aligned" in L.nmmo_last_error()
    assert L.nmmo_events(h, 0, 3, p(rows), 8, p(cnt, 1), st) == -1
    assert b"4-byte aligned" in L.nmmo_last_error()
    assert L.nmmo_events(h, 0, 3, None, 8, p(cnt), st) == -1
    assert b"null argument" in L.nmmo_last_error()
    assert L.nmmo_events(h, 0, 3, None, 0, p(cnt), st) == 0
    assert L.nmmo_events(None, 0, 3, p(rows), 8, p(cnt), st) == -1
    with pytest.raises(ValueError):
        sim.events(out=torch.zeros((4, 8), dtype=torch.int32, device=sim.obs.device))
    sim.set_event_log(False)
    with pytest.raises(NmmoError, match="event log is off"):
        sim.events()
    sim.close()


def test_env_view_event_log():
    """EnvView.realm.event_log.get_data over a whole episode equals the oracle's log, for every agent and with the
    event_code, agents and tick=-1 filters; column 0 is the running row id."""
    from nmmo_b200.env import ACTION_KEYS, EnvView
    from nmmo_b200.config import SPEC
    w = _rich(horizon=120)
    sim, (o,) = _sim(w, 1, log=False), _oracles(w, 1)
    view = EnvView(sim, 0)
    view.reset(seed=13)
    o.reset(13)
    assert len(view.realm.event_log.get_data()) == 0
    for t in range(130):
        acts = o.sample_actions(4)
        nested = {p + 1: {} for p in range(o.P)}
        for p in range(o.P):
            for k, (x, y) in enumerate(ACTION_KEYS):
                nested[p + 1].setdefault(x, {})[y] = int(acts[p, k])
        view.step(nested)
        o.step(acts)
        done = bool(sim.episode_done[0].item())
        log = view.realm.event_log
        data = log.get_data()
        assert np.array_equal(data[:, 0], np.arange(1, len(data) + 1)), "column 0 is the running row id"
        if t % 10 == 9 or done:
            for p in range(o.P):
                assert np.array_equal(log.get_data(agents=[p + 1])[:, 1:], o.log_rows(p)[:, 1:]), f"tick {t} agent {p + 1}"
        now = log.get_data(tick=-1)
        assert (now[:, 2] == o.tick).all()
        assert len(now) == sum(int((o.log_rows(p)[:, 2] == o.tick).sum()) for p in range(o.P))
        for code in (SPEC["EV_SCORE_HIT"], SPEC["EV_DRINK_WATER"]):
            sel = log.get_data(event_code=code, agents=[1, 2, 3])
            want = np.concatenate([o.log_rows(p) for p in range(3)])
            assert len(sel) == int((want[:, 3] == code).sum()) and (sel[:, 3] == code).all() and (sel[:, 1] <= 3).all()
        if done:
            break
    assert done and len(data) > 100, (t, len(data))
    sim.close()
