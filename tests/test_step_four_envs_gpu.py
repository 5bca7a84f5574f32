"""GPU: the step kernel with four environments per CTA (nmmo_step4_kernel / nmmo_step4_std_kernel) computes what the
three-per-CTA kernel computes, at env counts that leave the last CTA one to three environments short, through the
device step and the two-range host step, and matches the CPU oracle."""
import numpy as np
import pytest

from util import SMALL, build_world, run_parity

pytestmark = pytest.mark.gpu


def _sim(monkeypatch, world, E, epc, **env):
    from nmmo_b200.lib import Simulator
    cfg, fcfg, maps, tab, emb = world
    monkeypatch.setenv("NMMO_B200_ENVS_PER_CTA", str(epc))
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    try:
        sim = Simulator(cfg, fcfg, E, maps, tab, emb)
    finally:
        monkeypatch.delenv("NMMO_B200_ENVS_PER_CTA")
        for k in env:
            monkeypatch.delenv(k)
    assert sim.kernel_names()[0].startswith(f"nmmo_step{epc}_"), sim.kernel_names()
    return sim


def _outputs(sim):
    return [x.cpu().numpy() for x in (sim.rewards, sim.terminated, sim.truncated, sim.mask, sim.info, sim.info_valid,
                                      sim.episode_done)]


def _same_state(a, b, E, tag):
    for e in range(E):
        for x, y in zip(a.snapshot(e), b.snapshot(e)):
            assert np.array_equal(x, y), f"{tag} env {e}: tables differ"


@pytest.mark.parametrize("E", [9, 10, 11, 12])
def test_four_envs_per_cta_equal_three(monkeypatch, E):
    # 200 ticks over a 60-tick horizon: every env finishes episodes and resets inside the window
    import torch
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=60, NC_RES_DEPLETION=1)
    a, b = _sim(monkeypatch, world, E, 3), _sim(monkeypatch, world, E, 4)
    seeds = np.arange(E) + 21
    a.reset(seeds); b.reset(seeds)
    for t in range(200):
        a.sample_actions(5)
        b.actions.copy_(a.actions)
        a.step(); b.step()
        torch.cuda.synchronize()
        assert np.array_equal(a.obs.cpu().numpy(), b.obs.cpu().numpy()), f"tick {t}: records differ"
        for x, y in zip(_outputs(a), _outputs(b)):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), f"tick {t}: outputs differ"
        if t % 20 == 19:
            _same_state(a, b, E, f"tick {t}")
    assert int(b.stats()[2][2]) >= E, "every env must have reset at least once"
    a.close(); b.close()


def test_four_envs_per_cta_default_shape(monkeypatch):
    # the reference's default shape (128 players, 256 NPCs, 160^2 map), 4k + 1 envs, across an episode reset
    import torch
    world = build_world(NC_HORIZON=100)
    E = 9
    a, b = _sim(monkeypatch, world, E, 3), _sim(monkeypatch, world, E, 4)
    seeds = np.arange(E) + 5
    a.reset(seeds); b.reset(seeds)
    for t in range(210):
        a.sample_actions(8)
        b.actions.copy_(a.actions)
        a.step(); b.step()
        torch.cuda.synchronize()
        for x, y in zip(_outputs(a), _outputs(b)):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), f"tick {t}: outputs differ"
        if t % 15 == 14:
            assert np.array_equal(a.obs.cpu().numpy(), b.obs.cpu().numpy()), f"tick {t}: records differ"
            _same_state(a, b, E, f"tick {t}")
    a.close(); b.close()


def test_four_envs_per_cta_host_step_in_two_ranges(monkeypatch):
    # nmmo_step_host_u8 copies and steps two env ranges; the cut falls on a CTA boundary (17 envs: 4 + 13, last CTA one env)
    import torch
    from nmmo_b200.lib import pack_actions_u8
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=30)
    E = 17
    a = _sim(monkeypatch, world, E, 3)
    b = _sim(monkeypatch, world, E, 4, NMMO_B200_H2D_SPLIT_MIN="4")
    seeds = list(range(3, 3 + E))
    a.reset(seeds); b.reset(seeds)
    for t in range(45):
        a.sample_actions(6)
        torch.cuda.synchronize()
        packed = pack_actions_u8(a.actions).cpu().numpy()
        a.step()
        rew, term, trunc, mask, obs = b.step_host(packed, want_obs=True)
        torch.cuda.synchronize()
        assert np.array_equal(obs, a.obs.cpu().numpy()), f"tick {t}"
        assert np.array_equal(rew, a.rewards.cpu().numpy()) and np.array_equal(mask, a.mask.cpu().numpy()), f"tick {t}"
        assert np.array_equal(term, a.terminated.cpu().numpy()) and np.array_equal(trunc, a.truncated.cpu().numpy()), f"tick {t}"
    a.close(); b.close()


def test_four_envs_per_cta_matches_oracle(monkeypatch):
    from oracle.oracle import OracleEnv
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=60, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3)
    E = 7
    sim = _sim(monkeypatch, world, E, 4)
    oracles = [OracleEnv(*world) for _ in range(E)]
    stats = run_parity(sim, oracles, seeds=np.arange(E) + 3, ticks=130)
    assert stats["episodes_done"] >= E
    sim.close()
