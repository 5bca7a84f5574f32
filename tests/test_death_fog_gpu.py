"""GPU: the death fog (DESIGN.md 7) against the fog oracle (tests/fog_oracle.py), bit for bit, in every generic
step-kernel variant.

A fog-on handle runs the generic kernels (the *_std ones fold the fog off).  The worlds starve slowly so that players
hold and list items when the fog kills them: their items are destroyed inside the id-ordered part of players.update, so
the rows they free are the ones a higher-id player's harvest drop of the same tick allocates.  The runs pass an episode
ended by the fog, the automatic reset, and the fog of the next episode.
"""
import numpy as np
import pytest

from test_death_fog import _items_by_owner, fog_damage
from test_event_log_gpu import assert_rows, gpu_rows, oracle_rows
from util import SMALL, build_world, run_parity

pytestmark = pytest.mark.gpu

BIG_STD = ("nmmo_step_big_std_kernel", "nmmo_obs_big_std_kernel")
BIG_GENERIC = ("nmmo_step_big_kernel", "nmmo_obs_big_kernel")


def _spec(name):
    from nmmo_b200.config import SPEC
    return SPEC[name]


def _fog_world(agent="takeru", onset=40, final=2, **over):
    # the event log tests' rich world (slow starvation: agents harvest, list and fight) with the fog from `onset`
    return build_world(agent=agent, task_dim=64, **SMALL, NC_HORIZON=200, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3,
                       NC_WEAPON_DROP_THR=1 << 30, NC_DEATH_FOG_FINAL_SIZE=final, env_over={"death_fog_tick": onset}, **over)


def _sim(w, E, log=True):
    from nmmo_b200.lib import Simulator
    sim = Simulator(*w[:2], E, *w[2:])
    if log:
        sim.set_event_log(True)
    return sim


def _oracles(w, E):
    from fog_oracle import FogOracleEnv
    return [FogOracleEnv(*w) for _ in range(E)]


class FogCheck:
    """on_tick hook of run_parity: device event rows == oracle rows, and a tally, from the oracles' snapshots, of the
    players the fog killed this tick (phase 2 runs on the health and position the step started with)."""

    def __init__(self, cfg, log=True):
        self.cfg, self.log = cfg, log
        self.prev, self.episode = {}, {}
        self.hurt = self.kills = self.kills_with_items = self.kills_before_drop = 0
        self.kill_episodes = set()      # (env, episode) pairs with a fog kill
        self.early_ends = 0             # episodes that ended before the horizon

    def __call__(self, t, sim, oracles):
        if self.log:
            assert_rows(gpu_rows(sim), oracle_rows(oracles), f"tick {t}")
        ST, H, R = _spec("EA_STATUS"), _spec("EA_HEALTH"), _spec("EA_ROW")
        for e, o in enumerate(oracles):
            ent, items, _ = o.snapshot()
            prev = self.prev.get(e)
            self.prev[e] = (ent, items, o.tick, o.episode_done)
            if o.episode_done and o.tick < int(self.cfg[_spec("NC_HORIZON")]):
                self.early_ends += 1
            if prev is None:
                continue
            ent0, items0, tick0, done0 = prev
            if done0:                   # this step was the automatic reset
                self.episode[e] = self.episode.get(e, 0) + 1
                continue
            P = o.P
            rows = np.concatenate([o.log_rows(p) for p in range(P)])
            rows = rows[rows[:, 2] == o.tick]
            owned0 = _items_by_owner(items0, P)
            for p in np.flatnonzero(ent0[:P, ST] == _spec("ES_ALIVE")):
                dmg = fog_damage(self.cfg, tick0, int(ent0[p, R]), int(ent0[p, R + 1]))
                if not dmg:
                    continue
                self.hurt += 1
                if dmg < ent0[p, H]:
                    continue
                self.kills += 1
                self.kill_episodes.add((e, self.episode.get(e, 0)))
                assert ent[p, ST] == _spec("ES_DEAD_THIS_TICK"), (t, e, p)
                kill_rows = rows[(rows[:, 3] == _spec("EV_PLAYER_KILL")) & (rows[:, 8] == p + 1)]
                assert len(kill_rows) == 0, f"tick {t} env {e}: a PLAYER_KILL row for the fog's victim {p + 1}"
                if owned0[p]:
                    self.kills_with_items += 1
                    later = (rows[:, 3] == _spec("EV_HARVEST_ITEM")) & (rows[:, 1] > p + 1)
                    self.kills_before_drop += bool(later.any())

    def assert_covered(self, min_kills_with_items=1, min_before_drop=1):
        assert self.hurt > 50 and self.kills > 10, (self.hurt, self.kills)
        assert self.kills_with_items >= min_kills_with_items, self.kills_with_items
        assert self.kills_before_drop >= min_before_drop, "no fog kill of an item holder met a higher id's harvest drop"
        envs = {}
        for e, ep in self.kill_episodes:
            envs.setdefault(e, set()).add(ep)
        assert any(len(s) >= 2 for s in envs.values()), "no env met the fog again after its automatic reset"
        assert self.early_ends >= 1, "no episode was ended by deaths"


def _parity(w, E, want_step, seeds, ticks=220, log=True):
    sim, oracles = _sim(w, E, log=log), _oracles(w, E)
    assert sim.kernel_names()[0] == want_step, sim.kernel_names()
    check = FogCheck(w[0], log=log)
    stats = run_parity(sim, oracles, seeds=seeds, ticks=ticks, check_state_every=8, on_tick=check)
    assert stats["episodes_done"] >= E
    sim.close()
    return check


@pytest.mark.parametrize("variant,env,want", [
    ("four", {"NMMO_B200_ENVS_PER_CTA": "4"}, "nmmo_step4_kernel"),
    ("three", {"NMMO_B200_ENVS_PER_CTA": "3"}, "nmmo_step3_kernel"),
    ("two", {"NMMO_B200_ENVS_PER_CTA": "2"}, "nmmo_step_kernel"),
    ("one", {"NMMO_B200_ENVS_PER_CTA": "1"}, "nmmo_step_kernel"),
    ("big", {"NMMO_B200_FORCE_BIG": "1"}, "nmmo_step_big_kernel")])
def test_step_variants_against_oracle(monkeypatch, variant, env, want):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    w = _fog_world()
    check = _parity(w, 6, want, seeds=np.arange(6) + 5)
    check.assert_covered()


@pytest.mark.parametrize("agent,over", [("neurips23_start_kit", {"NC_ALLOW_OCCUPIED": 1}), ("yaofeng", {})])
def test_wrappers_against_oracle(agent, over):
    w = _fog_world(agent=agent, **over)
    check = _parity(w, 6, "nmmo_step4_kernel", seeds=np.arange(6) + 17)
    check.assert_covered()


def test_config5_shape_against_oracle():
    """The config-5 shape (1024 players, clustered spawn near the centre) with the fog on from tick 0: at the default
    speed the fog would not reach the patch within an episode, so it runs 24 times faster."""
    from bench import world
    cfg, fcfg, maps, tab, emb = world(workload="config5", n_maps=2)
    cfg = cfg.copy()
    cfg[_spec("NC_HORIZON")] = 28
    assert _kernel_names((cfg, fcfg, maps, tab, emb)) == BIG_STD
    cfg[_spec("NC_DEATH_FOG")] = 0
    cfg[_spec("NC_DEATH_FOG_SPEED")] = 24
    w5 = (cfg, fcfg, maps, tab, emb)
    sim, oracles = _sim(w5, 2), _oracles(w5, 2)
    assert sim.kernel_names() == BIG_GENERIC
    check = FogCheck(cfg)
    stats = run_parity(sim, oracles, seeds=np.arange(2) + 21, ticks=60, action_seed=1, check_state_every=10, on_tick=check)
    assert stats["episodes_done"] >= 2
    assert check.kills > 100 and check.kills_with_items >= 1, (check.kills, check.kills_with_items)
    sim.close()


def _kernel_names(w):
    sim = _sim(w, 2, log=False)
    names = sim.kernel_names()
    sim.close()
    return names


def test_kernel_selection():
    from bench import world
    cfg, fcfg, maps, tab, emb = world(n_maps=2)
    assert _kernel_names((cfg, fcfg, maps, tab, emb)) == ("nmmo_step4_std_kernel", "nmmo_obs_std_kernel")
    for onset in (0, 128):
        on = cfg.copy()
        on[_spec("NC_DEATH_FOG")] = onset
        assert _kernel_names((on, fcfg, maps, tab, emb)) == ("nmmo_step4_kernel", "nmmo_obs_kernel")
    cfg5, fcfg5, maps5, tab5, emb5 = world(workload="config5", n_maps=1)
    on = cfg5.copy()
    on[_spec("NC_DEATH_FOG")] = 0
    assert _kernel_names((on, fcfg5, maps5, tab5, emb5)) == BIG_GENERIC


def test_state_blob_mid_fog():
    """An env saved while the fog is closing in, loaded into another slot of another handle, continues exactly like the
    uninterrupted env (through its fog deaths and automatic reset); a handle without the fog refuses the blob."""
    import torch
    from test_env_state_gpu import _assert_outputs, _outputs
    from nmmo_b200.lib import NmmoError
    w = _fog_world(onset=20)
    a = _sim(w, 4, log=False)
    a.set_autosample(7)
    a.reset(np.arange(4) + 3)
    for _ in range(30):
        a.step(a.actions)
    blob = a.save_envs([1])
    acts, outs = [], []
    for t in range(90):
        acts.append(a.actions.clone())
        a.step(acts[-1])
        outs.append(_outputs(a, [1]))
    assert int(a.stats()[2][2]) >= 1, "no automatic reset after the save"
    b = _sim(w, 4, log=False)
    b.set_autosample(9)
    b.reset(np.arange(4) + 50)
    for _ in range(5):
        b.step(b.actions)
    b.load_envs([3], blob)
    for t in range(90):
        x = b.actions.clone()
        x[3] = acts[t][1]
        b.step(x)
        _assert_outputs(outs[t], _outputs(b, [3]), f"tick {t} after the load", skip=("actions",))
    torch.cuda.synchronize()
    off = list(w)
    off[0] = w[0].copy()
    off[0][_spec("NC_DEATH_FOG")] = -1
    c = _sim(tuple(off), 2, log=False)
    c.reset(np.arange(2))
    with pytest.raises(NmmoError, match="digest mismatch"):
        c.load_envs([0], blob)
    a.close(); b.close(); c.close()


def test_env_pool_equals_lock_step():
    """B200VecEnv(envs_per_batch=2) with death_fog_tick in its env namespace gives what the lock-step pool gives."""
    from test_env_pool_gpu import _pools, _run_equal, _small_env
    ns = _small_env(horizon=80)
    ns.death_fog_tick = 20
    lock, pool = _pools(ns, 4, 2)
    assert lock.sim.kernel_names()[0] == "nmmo_step4_kernel" and int(lock.cfg[_spec("NC_DEATH_FOG")]) == 20
    _run_equal(lock, pool, 200)
    hurt = max(int(lock.sim.snapshot(e)[0][:lock.agents_per_env, _spec("EA_DMG_RECEIVED")].max()) for e in range(4))
    assert hurt > 0
    lock.close(); pool.close()
