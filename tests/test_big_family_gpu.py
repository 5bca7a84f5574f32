"""GPU parity of the big kernel family (nmmo_step_big_kernel / nmmo_obs_big_kernel) vs the CPU oracle, bit-exact.

BASELINE.json configs[4] ("stress: 1024 agents per env on larger map, nearest-entity obs and collision-heavy Move";
SURVEY.md 8(d) config 5: NPC_N x8, map centre 512, all agents spawned inside a 32x32 patch, Move-biased actions
p = 0.9).  The reference only scales the knobs it passes to nmmo.Env (/root/reference/config.yaml:76-80:
num_agents, num_npcs, map_size); the clustered spawn and the Move bias are workload knobs of this repo
(NC_SPAWN_PATCH, NC_SAMPLE_MOVE_PCT) that the oracle implements too.

The big family is selected by the shape (more than 256 players / 512 entities / a 255^2 map); the environment
variable NMMO_B200_FORCE_BIG=1 also runs it on small shapes, which is how the rich small-world scenarios of
test_parity_gpu.py (items, market, combat, kills, every wrapper) are replayed through it here.
"""
import numpy as np
import pytest

from util import SMALL, build_world, run_parity

pytestmark = pytest.mark.gpu


def _make(world, E):
    from nmmo_b200.lib import Simulator
    from oracle.oracle import OracleEnv
    cfg, fcfg, maps, tab, emb = world
    sim = Simulator(cfg, fcfg, E, maps, tab, emb)
    return sim, [OracleEnv(cfg, fcfg, maps, tab, emb) for _ in range(E)]


@pytest.fixture
def force_big(monkeypatch):
    monkeypatch.setenv("NMMO_B200_FORCE_BIG", "1")


def test_big_family_small_world_episode(force_big):
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=96)
    sim, oracles = _make(world, 5)
    stats = run_parity(sim, oracles, seeds=np.arange(5) + 11, ticks=210)
    assert stats["episodes_done"] >= 5
    sim.close()


@pytest.mark.parametrize("agent", ["takeru", "neurips23_start_kit", "yaofeng"])
def test_big_family_rich_interactions(force_big, agent):
    world = build_world(agent=agent, task_dim=64, **SMALL, NC_HORIZON=300, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3,
                        NC_WEAPON_DROP_THR=1 << 30)
    sim, oracles = _make(world, 4)
    stats = run_parity(sim, oracles, seeds=np.arange(4) + 5, ticks=320)
    assert stats["infos"] > 0
    sim.close()


def test_big_family_default_config(force_big):
    world = build_world()
    sim, oracles = _make(world, 2)
    run_parity(sim, oracles, seeds=np.array([1, 2]), ticks=120, check_state_every=40)
    sim.close()


def test_big_family_item_heavy(force_big):
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=260, NC_RES_DEPLETION=0, NC_SPAWN_IMMUNITY=3,
                        NC_WEAPON_DROP_THR=-1, NC_NPC_AGGR_PCT=200, NC_NPC_NEUT_PCT=200)
    sim, oracles = _make(world, 3)
    stats = run_parity(sim, oracles, seeds=np.arange(3) + 41, ticks=270)
    assert stats["infos"] > 0
    sim.close()


def test_big_family_respawn_scan_fallback(force_big, monkeypatch):
    monkeypatch.setenv("NMMO_B200_NO_DEPL_LIST", "1")
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=120, NC_RES_DEPLETION=1)
    sim, oracles = _make(world, 3)
    run_parity(sim, oracles, seeds=np.arange(3) + 61, ticks=100, check_state_every=10)
    sim.close()


@pytest.mark.parametrize("P,N,center,E,over", [
    (300, 500, 96, 2, dict(NC_RES_DEPLETION=2)),                                   # just past the small family's limits
    (512, 1024, 96, 2, dict(NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=2, NC_SPAWN_PATCH=24, NC_SAMPLE_MOVE_PCT=90)),
    (1000, 2000, 256, 1, dict(NC_RES_DEPLETION=3, NC_SPAWN_IMMUNITY=4)),           # ring spawn on a 288^2 map, ragged sizes
])
def test_big_family_shapes(P, N, center, E, over):
    world = build_world(task_dim=64, NC_N_PLAYERS=P, NC_N_NPCS=N, NC_MAP_CENTER=center, NC_HORIZON=60, **over)
    sim, oracles = _make(world, E)
    stats = run_parity(sim, oracles, seeds=np.arange(E) + 500 + P, ticks=70, check_state_every=20)
    assert stats["infos"] > 0
    sim.close()


def config5_stress_world():
    """The configs[4] table shape with a 64-d task block and a folded engine default changed (NC_RES_DEPLETION): neither
    is the std record layout / engine table, so a handle of this world runs the generic big kernels."""
    return build_world(task_dim=64, n_maps=2, NC_N_PLAYERS=1024, NC_N_NPCS=2048, NC_MAP_CENTER=512, NC_HORIZON=48,
                       NC_SPAWN_PATCH=32, NC_SAMPLE_MOVE_PCT=90, NC_SPAWN_IMMUNITY=5, NC_RES_DEPLETION=4)


def test_config5_stress_shape():
    """The generic big kernels (nmmo_step_big_kernel / nmmo_obs_big_kernel) at the configs[4] table shape: 1024 players,
    2048 NPCs, 544^2 map (centre 512 + 2 x 16 border), all players spawned in a 32x32 patch, Move chosen with p = 0.9 by
    the built-in sampler, spawn immunity short enough that the crowd fights.  Every observation, mask, reward, flag and
    (every 10 ticks) the full state against the oracle.  The 64-d task block and NC_RES_DEPLETION = 4 keep this world off
    the compile-time-shape kernels that `bench.py --workload config5` runs; tests/test_config5_std_gpu.py checks those."""
    sim, oracles = _make(config5_stress_world(), 2)
    assert sim.kernel_names() == ("nmmo_step_big_kernel", "nmmo_obs_big_kernel")
    moved = []

    def watch(t, sim_, oracles_):
        if t in (0, 40):
            ent = oracles_[0].snapshot()[0]
            moved.append(ent[:1024, 2:4].copy())

    stats = run_parity(sim, oracles, seeds=np.array([3, 4]), ticks=56, check_state_every=10, on_tick=watch)
    assert stats["episodes_done"] >= 2            # ran through the horizon and the automatic reset
    assert (moved[0] != moved[1]).any(axis=1).sum() > 100, "the crowd must actually move"
    sim.close()


def test_config5_limits():
    from nmmo_b200.lib import NmmoError
    for over in (dict(NC_N_PLAYERS=1032, NC_N_NPCS=16, NC_MAP_CENTER=512),       # more players than threads
                 dict(NC_N_PLAYERS=300, NC_N_NPCS=20, NC_MAP_CENTER=64),         # ring spawn: two players per tile
                 dict(NC_N_PLAYERS=1024, NC_N_NPCS=2056, NC_MAP_CENTER=512),     # too many NPCs
                 dict(NC_N_PLAYERS=1024, NC_N_NPCS=1024, NC_MAP_CENTER=512, NC_SPAWN_PATCH=31)):      # patch too small
        world = build_world(task_dim=64, n_maps=1, **over)
        with pytest.raises(NmmoError):
            _make(world, 1)


def test_big_family_injected_draws_and_team_tasks(force_big):
    """Recorded-draw injection (NPC wander, respawn, spawn, reset permutation) and team / named-target tasks through
    the big family: same keys and same task rows on both sides, bit-exact episodes."""
    from nmmo_b200.config import SPEC as S
    from nmmo_b200.tasks import EVENT, TF_RELATIVE_TARGET, TF_TEAM, default_curriculum, make_task_table, task_row
    rows = default_curriculum()[:12] + [task_row("ALL_MEMBERS_WITHIN_RANGE", 6, 0, 0, TF_TEAM), task_row("ALL_DEAD", 1, 0, 0, TF_TEAM | TF_RELATIVE_TARGET),
                                        task_row("CAN_SEE_GROUP", -1, 0, 0, TF_RELATIVE_TARGET), task_row("COUNT_EVENT", EVENT["EAT_FOOD"], 6, 0, TF_TEAM)]
    cfg, fcfg, maps, _, _ = build_world(task_dim=64, **SMALL, NC_HORIZON=120, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=2, NC_TEAM_SIZE=4)
    tab, emb = make_task_table(rows, 64, seed=5)
    sim, oracles = _make((cfg, fcfg, maps, tab, emb), 3)
    assert sim.kernel_names() == ("nmmo_step_big_kernel", "nmmo_obs_big_kernel")
    rng = np.random.default_rng(2)
    P, R, Sz = int(cfg[S["NC_N_PLAYERS"]]), int(cfg[S["NC_N_PLAYERS"]] + cfg[S["NC_N_NPCS"]]), int(cfg[S["NC_MAP_SIZE"]])
    for e, o in enumerate(oracles):
        keys, vals = [], []
        for t in range(100):
            for row in rng.choice(np.arange(P, R), 6, replace=False):
                keys.append((t << 36) | (S["RS_NPC_DECIDE"] << 32) | (int(row) << 8)); vals.append(int(rng.integers(0, 2 ** 32)))
            for i in rng.choice(Sz * Sz, 30, replace=False):
                keys.append((t << 36) | (S["RS_RESPAWN"] << 32) | (int(i) << 8)); vals.append(int(rng.integers(0, 2 ** 28)))
            for att in range(25):
                for k in range(6):
                    keys.append((t << 36) | (S["RS_NPC_SPAWN"] << 32) | (att << 8) | k); vals.append(int(rng.integers(0, 2 ** 32)))
        for i in range(1, P):
            keys.append((S["RS_SPAWN_PERM"] << 32) | (i << 8)); vals.append(int(rng.integers(0, 2 ** 32)))
        keys = np.array(keys, np.uint64); vals = np.array(vals, np.uint32)
        o.inject_rng(keys, vals); sim.inject_rng(e, keys, vals)
    stats = run_parity(sim, oracles, seeds=np.arange(3) + 90, ticks=130)
    assert stats["infos"] > 0
    sim.close()
