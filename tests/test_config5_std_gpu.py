"""The compile-time-shape big kernels (nmmo_step_big_std_kernel / nmmo_obs_big_std_kernel), the pair that
`bench.py --workload config5` times, against the CPU oracle and against the generic big kernels.

nmmo_create selects the std pair only for the configs[4] shape (StdShape5 in csrc/nmmo_device.cuh), the default record
layout and every engine default the kernels fold in (nm_cfg_std_value); a handle with injected draws or the phase
profiler on launches the generic pair instead.  So the worlds here come from bench.world(workload="config5"), only the
run-time horizon is changed, nothing is injected, and every GPU test asserts the kernel names when the handle is created
and again at the end.  The CPU test at the bottom fails on any machine when a config or workload edit moves the benchmark
off the std pair.
"""
import re

import numpy as np
import pytest

from bench import world
from nmmo_b200.config import SPEC, ObsLayout, make_config
from util import DEVICE_HEADER, run_parity, std_cfg_table

BIG_STD = ("nmmo_step_big_std_kernel", "nmmo_obs_big_std_kernel")
BIG_GENERIC = ("nmmo_step_big_kernel", "nmmo_obs_big_kernel")
SEED = 1          # bench.py's default --seed: the built-in policy's draws


def _config5(horizon=None):
    cfg, fcfg, maps, tab, emb = world(workload="config5", n_maps=2)
    if horizon is not None:
        assert SPEC["NC_HORIZON"] not in std_cfg_table()
        cfg = cfg.copy()
        cfg[SPEC["NC_HORIZON"]] = horizon
    return cfg, fcfg, maps, tab, emb


def _make(w, E):
    from nmmo_b200.lib import Simulator
    from oracle.oracle import OracleEnv
    sim = Simulator(*w[:2], E, *w[2:])
    assert sim.kernel_names() == BIG_STD
    return sim, [OracleEnv(*w) for _ in range(E)]


def _kernel_names(w):
    from nmmo_b200.lib import Simulator
    sim = Simulator(*w[:2], 1, *w[2:])
    names = sim.kernel_names()
    sim.close()
    return names


@pytest.mark.gpu
def test_kernel_selection(monkeypatch):
    from test_big_family_gpu import config5_stress_world
    c5 = _config5()
    assert _kernel_names(c5) == BIG_STD
    assert _kernel_names(world(n_maps=2)) == ("nmmo_step4_std_kernel", "nmmo_obs_std_kernel")
    # the world of test_config5_stress_shape: the same table shape, but not the std layout and engine table
    assert _kernel_names(config5_stress_world()) == BIG_GENERIC
    monkeypatch.setenv("NMMO_B200_NO_STD_STEP", "1")
    assert _kernel_names(c5) == BIG_GENERIC


@pytest.mark.gpu
def test_std_kernels_match_oracle():
    """Three envs through two automatic resets: the sampler kernel's Move-biased actions against the oracle's, every
    output every tick and the full state every 16 ticks, bit for bit."""
    E, P = 3, 1024
    sim, oracles = _make(_config5(horizon=96), E)
    ea_pos = slice(SPEC["EA_ROW"], SPEC["EA_COL"] + 1)
    seen = dict(done=set(), died=0, items=0, moved=0)
    start = []

    def watch(t, sim_, oracles_):
        for e, o in enumerate(oracles_):
            if o.episode_done:
                seen["done"].add(e)
            else:
                seen["died"] += int(o.terminated.sum())
            if t % 16 == 0:
                items = o.snapshot()[1]
                seen["items"] = max(seen["items"], int((items[:, SPEC["IS_TYPE"]] != 0).sum()))
        if t in (0, 40):
            pos = oracles_[0].snapshot()[0][:P, ea_pos]
            if t == 0:
                start.append(pos.copy())
            else:
                seen["moved"] = int(((pos != start[0]).any(axis=1) & (oracles_[0].mask != 0)).sum())

    stats = run_parity(sim, oracles, seeds=np.arange(E) + 21, ticks=200, action_seed=SEED, check_state_every=16,
                       on_tick=watch)
    assert seen["done"] == set(range(E)), "every env must finish an episode"
    assert stats["infos"] > 0
    assert seen["died"] > 0, "agents must die before the horizon"
    assert seen["items"] > 0, "the item table must hold live rows"
    assert seen["moved"] > 100, "the crowd must actually move"
    assert sim.kernel_names() == BIG_STD
    sim.close()


@pytest.mark.gpu
def test_fused_sampler_matches_sampler_kernel_and_oracle():
    """The benchmark's mode: the big std observation kernel writes the next actions itself (set_autosample into
    sim.actions before the reset), with the Move bias of NC_SAMPLE_MOVE_PCT = 90."""
    import torch
    E = 2
    w = _config5()
    sim, oracles = _make(w, E)
    sim.set_autosample(SEED, sim.actions)
    scratch = torch.zeros_like(sim.actions)
    o_move = ObsLayout(w[0]).masks["Move.Direction"][0]
    pct = int(w[0][SPEC["NC_SAMPLE_MOVE_PCT"]])
    assert pct == 90
    fused = {}
    n = dict(eligible=0, moved=0)

    def check(t, sim_, oracles_):
        a = sim.actions.cpu().numpy()
        sim.sample_actions(SEED, out=scratch)
        assert np.array_equal(a, scratch.cpu().numpy()), f"tick {t}: fused sampler differs from the sampler kernel"
        for e, o in enumerate(oracles_):
            assert np.array_equal(a[e], o.sample_actions(SEED + e)), f"tick {t} env {e}: oracle sampler differs"
        # alive agents with at least one valid direction other than Stay: Move != Stay with p = NC_SAMPLE_MOVE_PCT %
        can_move = (sim.obs[:, o_move:o_move + 4] != 0).any(dim=1) & (sim.mask != 0)
        elig = can_move.cpu().numpy()
        n["eligible"] += int(elig.sum())
        n["moved"] += int((a.reshape(-1, 12)[elig, SPEC["AC_MOVE_DIR"]] != 4).sum())
        fused[t] = a

    run_parity(sim, oracles, seeds=np.arange(E) + SEED, ticks=80, check_state_every=16, action_fn=lambda t, g_obs: fused[t],
               on_tick=check)
    assert n["eligible"] > 50000
    assert abs(n["moved"] / n["eligible"] - pct / 100) < 0.03, n
    assert sim.kernel_names() == BIG_STD
    sim.set_autosample(0, enable=False)
    sim.close()


def _same_outputs(a, b, tag):
    import torch
    for name in ("obs", "rewards", "terminated", "truncated", "mask", "info", "info_valid", "episode_done", "actions"):
        x, y = getattr(a, name), getattr(b, name)
        assert torch.equal(x.view(torch.uint8), y.view(torch.uint8)), f"{tag}: {name} differ"


@pytest.mark.gpu
def test_std_equals_generic_over_a_benchmark_episode(monkeypatch):
    """Eight envs at the benchmark's own horizon (1024) with the built-in policy, past the automatic reset: the late
    episode (levels, respawns, a thinned population) that the oracle run does not reach cheaply."""
    from nmmo_b200.lib import Simulator
    E, T = 8, 1100
    w = _config5()
    assert int(w[0][SPEC["NC_HORIZON"]]) == 1024
    std = Simulator(*w[:2], E, *w[2:])
    monkeypatch.setenv("NMMO_B200_NO_STD_STEP", "1")      # read by nmmo_create: disables both big std kernels
    gen = Simulator(*w[:2], E, *w[2:])
    monkeypatch.delenv("NMMO_B200_NO_STD_STEP")
    assert std.kernel_names() == BIG_STD and gen.kernel_names() == BIG_GENERIC
    seeds = np.arange(E) + SEED
    for s in (std, gen):
        s.set_autosample(SEED, s.actions)
        s.reset(seeds)
    for t in range(T + 1):
        _same_outputs(std, gen, f"tick {t}")
        if t % 128 == 0 or t == T:
            for e in range(E):
                for name, x, y in zip(("entities", "items", "map", "scalars"), std.snapshot(e), gen.snapshot(e)):
                    assert np.array_equal(x, y), f"tick {t} env {e}: {name} differ"
        if t < T:
            std.step()
            gen.step()
    (s_sums, s_counts, s_ctr), (g_sums, g_counts, g_ctr) = std.stats(), gen.stats()
    assert np.array_equal(s_ctr, g_ctr) and np.array_equal(s_counts, g_counts)
    # float atomics into double running sums: the order of the adds may differ
    np.testing.assert_allclose(s_sums, g_sums, rtol=1e-9)
    assert int(s_ctr[2]) >= E, "every env must pass the automatic reset"
    assert std.kernel_names() == BIG_STD and gen.kernel_names() == BIG_GENERIC
    for s in (std, gen):
        s.set_autosample(0, enable=False)
        s.close()


@pytest.mark.gpu
def test_env_pool_on_std_kernels():
    """B200VecEnv at the configs[4] shape in batches of two envs: the range launches of the big std pair (act_env_lo,
    [env_lo, env_hi)) against the lock-step pool, bit for bit, across episode resets."""
    from nmmo_b200.config import default_env_args
    from test_env_pool_gpu import _pools, _run_equal
    env = default_env_args(num_agents=1024, num_npcs=2048, map_size=512, num_maps=2, max_episode_length=40,
                           resilient_population=0)
    lock, pool = _pools(env, 4, 2, seed=7)
    assert lock.sim.kernel_names() == BIG_STD and pool.sim.kernel_names() == BIG_STD
    _run_equal(lock, pool, 100)
    assert lock.sim.kernel_names() == BIG_STD and pool.sim.kernel_names() == BIG_STD
    lock.close(); pool.close()


def test_config5_workload_is_the_std_shape():
    """bench.py's config-5 world has exactly the shape, record layout and folded engine defaults that select the big std
    kernels; the small family's limit (NM_STEP_THREADS players) puts it in the big family."""
    text = DEVICE_HEADER.read_text()
    shape = text[text.index("struct StdShape5 {"):]
    shape = {k: int(v) for k, v in re.findall(r"(\w+) = (\d+)", shape[:shape.index("};")])}
    cfg = world(workload="config5", n_maps=2)[0]
    for i, v in std_cfg_table().items():
        assert int(cfg[i]) == v, (i, v, int(cfg[i]))
    P, N = int(cfg[SPEC["NC_N_PLAYERS"]]), int(cfg[SPEC["NC_N_NPCS"]])
    assert (P, N, P + N) == (shape["P"], shape["N"], shape["R"])
    assert int(cfg[SPEC["NC_MAP_SIZE"]]) == shape["S"] and int(cfg[SPEC["NC_ITEM_CAP"]]) == shape["CAP"]
    assert int(cfg[SPEC["NC_N_INV"]]) == shape["NINV"] and int(cfg[SPEC["NC_VISION"]]) == shape["VIS"]
    assert P > int(re.search(r"#define NM_STEP_THREADS (\d+)", text).group(1))
    # nm_std_layout(): the section sizes it is built from, and the layout the Python mirror computes from them
    std = text[text.index("constexpr nm_obs_layout nm_std_layout()"):]
    counts = {k: int(v) for k, v in re.findall(r"L\.(\w+) = (\d+);", std[:std.index("int o = 0;")])}
    L = ObsLayout(cfg)
    assert counts == {k: getattr(L, k) for k in counts}
    assert vars(L) == vars(ObsLayout(make_config()[0]))
