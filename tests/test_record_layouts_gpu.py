"""GPU parity at record layouts away from the reference's: every vision radius and record width nmmo_create accepts,
through both kernel families, the fused sampler, the dense writer, the host-buffer calls, the compact rollout and the
forager -- and the layouts the kernels cannot write, which nmmo_create refuses.

The reference's layout (vision 7, 100 entity / 384 market / 12 inventory rows, 99 prices) never truncates anything in
a small world and keeps the observation kernel on its fast tile path; these layouts reach the slow tile paths
(vision <= 3 and >= 8), the all-rows visibility scan (vision >= 9), Entity / Market / Inventory truncation, mask heads
whose no-op sits on a 32-entry word boundary, and a Buy head wider than the byte-packed host path's low byte."""
import numpy as np
import pytest

from nmmo_b200.config import SPEC, ObsLayout
from util import (LONG_LIVED, MARKET_FILLING, RECORD_LAYOUTS, SMALL, build_world, fill_market, layout_world, random_layouts,
                  run_parity)

pytestmark = pytest.mark.gpu
S = SPEC
TICKS = 120          # horizon 100: every case crosses an automatic reset


def _make(world, E):
    from nmmo_b200.lib import Simulator
    from oracle.oracle import OracleEnv
    return Simulator(*world[:2], E, *world[2:]), [OracleEnv(*world) for _ in range(E)]


def _sim(world, E):
    from nmmo_b200.lib import Simulator
    return Simulator(*world[:2], E, *world[2:])


def _parity(world, E=3, ticks=TICKS, seed=0, **kw):
    sim, oracles = _make(world, E)
    stats = run_parity(sim, oracles, seeds=np.arange(E) + 100 + seed, ticks=ticks, check_state_every=20, **kw)
    sim.close()
    return stats


@pytest.mark.parametrize("vision", [0, 1, 3, 4, 5, 8, 9, 15])
def test_vision_sweep(vision):
    # 0..3 and 8.. take the observation kernel's per-group tile loop, 4..7 its fast path; from 9 on the visibility
    # search scans every row instead of 16-tile cells; 15 is the widest window that stays inside the map
    world = build_world(task_dim=64, **SMALL, NC_VISION=vision, NC_HORIZON=100, **LONG_LIVED)
    _parity(world, seed=vision)


@pytest.mark.parametrize("name", list(RECORD_LAYOUTS))
def test_record_layouts(name):
    world = layout_world(RECORD_LAYOUTS[name], NC_HORIZON=100, **LONG_LIVED)
    seen = []

    def watch(t, sim, oracles):
        L = ObsLayout(sim.cfg)
        obs = oracles[0].obs
        ent = obs[:, L.o_entity:L.o_entity + L.n_ent * 62].view(np.int16).reshape(-1, L.n_ent, 31)[:, :, 0]
        seen.append(int((ent != 0).sum(1).max()))

    _parity(world, on_tick=watch)
    if name == "many_entities":
        assert max(seen) > 32, f"agents must see more than one mask word of entities (saw {max(seen)})"


@pytest.mark.parametrize("layout", random_layouts(8), ids=lambda lay: "ent{}_mkt{}_inv{}_price{}_vis{}_task{}".format(*lay[:6]))
def test_random_layouts(layout):
    _parity(layout_world(layout, NC_HORIZON=100, **LONG_LIVED), ticks=110, seed=layout[0])


def _market_filler(oracles, L, rng, stats):
    bo = L.masks["Buy.MarketItem"][0]

    def act(t, obs):
        acts = fill_market(np.stack([o.sample_actions(7 + e) for e, o in enumerate(oracles)]), obs, L, rng)
        for e, o in enumerate(oracles):
            items = o.snapshot()[1]
            n_listed = int(((items[:, S["IS_TYPE"]] > 0) & (items[:, S["IS_PRICE"]] > 0)).sum())
            stats["full"] += n_listed >= L.n_mkt
            k = acts[e, :, 2]
            shown = k < L.n_mkt
            stats["truncated_buys"] += int(n_listed > L.n_mkt) * int((obs[e, shown, bo + k[shown]] == 1).sum())
        return acts

    return act


def test_market_overflow():
    # a Buy index is a row of the truncated Market block the agent was shown, not a listing of the whole table: the
    # step kernel decodes it from the record, the observation kernel writes the first n_mkt listings
    world = layout_world(RECORD_LAYOUTS["truncating"], NC_HORIZON=200, **MARKET_FILLING)
    sim, oracles = _make(world, 3)
    stats = dict(full=0, truncated_buys=0)
    act = _market_filler(oracles, ObsLayout(world[0]), np.random.default_rng(1), stats)
    run_parity(sim, oracles, seeds=np.arange(3) + 41, ticks=90, action_fn=act, check_state_every=15)
    sim.close()
    assert stats["full"] > 0, "the market never filled its rows"
    assert stats["truncated_buys"] > 0, "no valid Buy against a truncated market"


PATH_LAYOUTS = list(RECORD_LAYOUTS)


@pytest.mark.parametrize("name", PATH_LAYOUTS)
def test_big_family(name, monkeypatch):
    monkeypatch.setenv("NMMO_B200_FORCE_BIG", "1")
    world = layout_world(RECORD_LAYOUTS[name], NC_HORIZON=100, **LONG_LIVED)
    sim, oracles = _make(world, 3)
    assert all("big" in k for k in sim.kernel_names()), sim.kernel_names()
    run_parity(sim, oracles, seeds=np.arange(3) + 7, ticks=TICKS, check_state_every=20)
    sim.close()


@pytest.mark.parametrize("name", PATH_LAYOUTS)
def test_fused_sampler_matches_sampler_kernel(name):
    import torch
    world = layout_world(RECORD_LAYOUTS[name], NC_HORIZON=60, **LONG_LIVED)
    sim, oracles = _make(world, 3)
    auto = torch.zeros_like(sim.actions)
    sim.set_autosample(77, auto)
    sim.reset(np.arange(3) + 9)
    for o, s in zip(oracles, np.arange(3) + 9):
        o.reset(int(s))
    for t in range(70):                                     # crosses an episode boundary (auto-reset)
        sim.sample_actions(77)
        torch.cuda.synchronize()
        a = sim.actions.cpu().numpy()
        assert np.array_equal(a, auto.cpu().numpy()), f"tick {t}: fused sampler differs from the sampler kernel"
        for e, o in enumerate(oracles):
            assert np.array_equal(a[e], o.sample_actions(77 + e)), f"tick {t} env {e}: oracle sampler differs"
            o.step(a[e])
        sim.step()
    sim.set_autosample(0, enable=False)
    sim.close()


@pytest.mark.parametrize("name", PATH_LAYOUTS)
def test_dense_and_incremental_writers_agree(name):
    import torch
    # listings come and go (3-tick listings, most agents selling): the incremental writer's Market rows grow and shrink
    world = layout_world(RECORD_LAYOUTS[name], NC_HORIZON=60, NC_WEAPON_DROP_THR=-1, **LONG_LIVED)
    L = ObsLayout(world[0])
    rng = np.random.default_rng(4)
    a, b = _sim(world, 3), _sim(world, 3)
    b.set_obs_full(True)
    a.reset([7, 8, 9]); b.reset([7, 8, 9])
    for t in range(70):
        a.sample_actions(2)
        torch.cuda.synchronize()
        assert torch.equal(a.obs, b.obs), f"tick {t}"
        assert torch.equal(a.mask, b.mask) and torch.equal(a.rewards, b.rewards), f"tick {t}"
        acts = torch.from_numpy(fill_market(a.actions.cpu().numpy(), a.obs.cpu().numpy().reshape(3, a.P, -1), L, rng))
        a.actions.copy_(acts); b.actions.copy_(acts)
        a.step(); b.step()
    a.close(); b.close()


@pytest.mark.parametrize("name", PATH_LAYOUTS)
def test_step_host_equals_device_step(name):
    import torch
    from nmmo_b200.lib import pack_actions_u8
    world = layout_world(RECORD_LAYOUTS[name], NC_HORIZON=50, NC_WEAPON_DROP_THR=-1, **LONG_LIVED)
    L = ObsLayout(world[0])
    bo = L.masks["Buy.MarketItem"][0]
    rng = np.random.default_rng(6)
    a, b, c, d = _sim(world, 2), _sim(world, 2), _sim(world, 2), _sim(world, 2)
    for s in (a, b, c, d):
        s.reset([1, 2])
    planted = 0
    for t in range(50):
        a.sample_actions(4)
        torch.cuda.synchronize()
        obs_now = a.obs.cpu().numpy().reshape(2, a.P, -1)
        acts = fill_market(a.actions.cpu().numpy(), obs_now, L, rng)
        # Buy index 256 + k from an agent that may buy row k: row 256 + k of a wide Market block is always empty (the
        # item table has at most 192 rows), so carried whole the index is a no-op; with its bits 8.. dropped on the
        # way it would buy row k
        for e in range(2):
            can = np.argwhere(obs_now[e, :, bo:bo + max(0, L.n_mkt - 256)] == 1)
            if len(can):
                p, k = can[0]
                acts[e, p, 2] = 256 + k; planted += 1
        a.actions.copy_(torch.from_numpy(acts))
        a.step()
        packed = pack_actions_u8(acts)
        for other, host_acts in ((b, acts), (c, acts.astype(np.int16)), (d, packed)):      # int32, int16 and byte-packed calls
            rew, term, trunc, mask, obs = other.step_host(host_acts, want_obs=True)
            torch.cuda.synchronize()
            assert np.array_equal(obs, a.obs.cpu().numpy()), f"tick {t} {host_acts.dtype}"
            assert np.array_equal(rew, a.rewards.cpu().numpy()) and np.array_equal(mask, a.mask.cpu().numpy())
            assert np.array_equal(term, a.terminated.cpu().numpy()) and np.array_equal(trunc, a.truncated.cpu().numpy())
    if L.n_mkt > 256:
        assert int(world[0][S["NC_ITEM_CAP"]]) <= 256
        assert planted > 0, "no agent could buy a listed row: the wide Buy field was never put to the test"
    a.close(); b.close(); c.close(); d.close()


def test_compact_rollout_reassembles_the_plain_one():
    # Market and Task are cut out of the stored rows and re-assembled by expand(): 8 market rows, a 24-entry task
    import torch
    from nmmo_b200.rollout import DeviceRollout
    world = layout_world(RECORD_LAYOUTS["truncating"], NC_HORIZON=40, NC_RES_DEPLETION=0, NC_SPAWN_IMMUNITY=3,
                         NC_WEAPON_DROP_THR=-1, NC_LISTING_DURATION=400)
    L = ObsLayout(world[0])
    E = 4
    sim = _sim(world, E)
    n = E * sim.P
    plain = DeviceRollout(2000, n, sim.stride)
    comp = DeviceRollout(2000, n, sim.stride, compact=DeviceRollout.compact_for(sim, max_steps=40))
    assert comp.row_stride == sim.stride - L.n_mkt * 32 - L.task_dim * 2
    sim.reset(np.arange(E, dtype=np.uint64) + 3)
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    rng = np.random.default_rng(3)
    for step in range(1, 40):
        val = torch.randn(n, device="cuda", generator=g); lp = -torch.rand(n, device="cuda", generator=g)
        d = (sim.terminated | sim.truncated).float()
        plain.store(sim.obs, val, sim.actions, lp, sim.rewards, d, sim.mask, step)
        comp.store(sim.obs, val, sim.actions, lp, sim.rewards, d, sim.mask, step, task_id=sim.task_id)
        sim.sample_actions(5)
        torch.cuda.synchronize()
        acts = fill_market(sim.actions.cpu().numpy(), sim.obs.cpu().numpy().reshape(E, sim.P, -1), L, rng)
        sim.actions.copy_(torch.from_numpy(acts))
        sim.step()
    rows = plain.ptr
    assert rows == comp.ptr and rows > 1500
    assert torch.equal(comp.expand(n=rows), plain.obs[:rows])
    mkt = plain.obs[:rows, L.o_market:L.o_market + L.n_mkt * 32]
    assert int(mkt.to(torch.int32).sum()) > 0, "no listing reached the Market block"
    plain.close(); comp.close(); sim.close()


def _forager_world(vision):
    from nmmo_b200.mapgen import generate_maps
    cfg, fcfg, maps, tab, emb = build_world(task_dim=64, NC_N_PLAYERS=32, NC_N_NPCS=32, NC_MAP_CENTER=48, NC_HORIZON=200,
                                            NC_VISION=vision)
    return cfg, fcfg, generate_maps(cfg, 11, 3, terrain="fine"), tab, emb


@pytest.mark.parametrize("vision", [2, 4, 7])
def test_forager_matches_numpy(vision):
    import torch
    from forager_ref import forage_actions
    world = _forager_world(vision)
    sim = _sim(world, 2)
    sim.reset(np.arange(2, dtype=np.uint64) + 2)
    P = sim.P
    for t in range(40):
        sim.forage_actions(7)
        torch.cuda.synchronize()
        a = sim.actions.cpu().numpy()
        obs = sim.obs.cpu().numpy().reshape(2, P, -1); mask = sim.mask.cpu().numpy().reshape(2, P)
        for e in range(2):
            tick = int(sim.snapshot(e)[3][0])
            ref = forage_actions(world[0], obs[e], mask[e], tick, 7, env_global=e)
            assert np.array_equal(a[e], ref), f"tick {t} env {e}: rows {np.flatnonzero((a[e] != ref).any(1))[:4]}"
        sim.step()
    sim.close()


def test_forager_refuses_windows_beyond_256_tiles():
    from nmmo_b200.lib import NmmoError
    sim = _sim(_forager_world(8), 2)        # 17 x 17 tiles
    sim.reset(np.arange(2, dtype=np.uint64) + 2)
    with pytest.raises(NmmoError, match="256 tiles"):
        sim.forage_actions(7)
    sim.close()


@pytest.mark.parametrize("over", [dict(NC_VISION=16), dict(NC_VISION=17), dict(NC_VISION=-1), dict(task_dim=12),
                                  dict(task_dim=100), dict(task_dim=0), dict(NC_N_ENT_OBS=0), dict(NC_N_MKT_OBS=0),
                                  dict(NC_N_INV=0), dict(NC_N_PRICE=0)],
                         ids=lambda o: "{}={}".format(*next(iter(o.items()))))
def test_layouts_the_kernels_cannot_write_are_refused(over):
    # only creates handles: stepping such a layout would read tiles outside the map (vision), load the Task block
    # misaligned and leave its tail unwritten (task_dim), or index an empty table (zero widths)
    from nmmo_b200.lib import NmmoError
    kw = dict(task_dim=64, **SMALL)
    kw.update(over)
    world = build_world(**kw)
    with pytest.raises(NmmoError, match="error -3"):
        _sim(world, 2).close()
