"""Shared parity harness: drive the CUDA simulator and the CPU oracle with identical inputs."""
from __future__ import annotations

import os
from pathlib import Path

import numpy as np

from nmmo_b200.config import SPEC, ObsLayout, make_config
from nmmo_b200.mapgen import generate_maps
from nmmo_b200.tasks import default_curriculum, make_task_table

SMALL = dict(NC_N_PLAYERS=16, NC_N_NPCS=32, NC_MAP_CENTER=32)
DEVICE_HEADER = Path(__file__).resolve().parent.parent / "nmmo_b200" / "csrc" / "nmmo_device.cuh"


def std_cfg_table():
    """nm_cfg_std_value (csrc/nmmo_device.cuh) as {config index: value}: the engine defaults that the *_std kernel
    instantiations fold into immediates."""
    import re
    text = DEVICE_HEADER.read_text()
    body = text[text.index("constexpr int nm_cfg_std_value"):text.index("default: return NM_CFG_RUNTIME")]
    return {SPEC[name] + int(off or 0): int(val) for name, off, val in re.findall(r"case (NC_\w+)(?: \+ (\d+))?: return (-?\d+);", body)}


def reference_file(*parts):
    """A path in the checkout of the reference baselines repository (Meeso1/nmmo) named by $NMMO_REFERENCE, or None
    when that variable is unset or the path does not exist there."""
    root = os.environ.get("NMMO_REFERENCE")
    path = Path(root, *parts) if root else None
    return path if path is not None and path.exists() else None


def build_world(agent="takeru", n_maps=4, map_seed=7, task_dim=None, env_over=None, wrapper_over=None, **engine_over):
    from nmmo_b200.config import default_env_args, default_wrapper_args
    env_args = default_env_args(resilient_population=0 if agent in ("takeru", "yaofeng") else 0.2, **(env_over or {}))
    if task_dim is not None:
        env_args.task_size = task_dim
    wrap = default_wrapper_args(agent, **(wrapper_over or {}))
    cfg, fcfg = make_config(env_args, wrap, agent, **engine_over)
    maps = generate_maps(cfg, map_seed, n_maps)
    tab, emb = make_task_table(default_curriculum(), int(cfg[SPEC["NC_TASK_DIM"]]), seed=3)
    return cfg, fcfg, maps, tab, emb


# Record layouts away from the reference's (100 entities, 384 market rows, 12 inventory rows, 99 prices, vision 7):
# name -> (N_ENT_OBS, N_MKT_OBS, N_INV, N_PRICE, VISION, task_dim, world shape).  Widths of 31 / 32 / 33 mask entries
# put a head's no-op on either side of a 32-entry mask word; "many entities" lets an agent see more than 32 entities.
RECORD_LAYOUTS = {
    "minimal": (1, 1, 1, 1, 3, 8, SMALL),
    "truncating": (8, 8, 4, 5, 5, 24, SMALL),
    "word_edges": (31, 31, 16, 31, 7, 64, SMALL),
    "word_edges_plus_1": (32, 63, 15, 32, 8, 64, SMALL),
    "many_entities": (255, 16, 4, 4, 9, 16, dict(NC_N_PLAYERS=64, NC_N_NPCS=64, NC_MAP_CENTER=24)),
    "wide_buy": (60, 600, 12, 80, 4, 64, SMALL),
}
# agents that live long enough to pick up, list and buy items
LONG_LIVED = dict(NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=3)
# with fill_market's actions, a world whose market outgrows a few rows: nobody starves, every harvest drops a weapon,
# listings stay up for 400 ticks, NPCs are passive
MARKET_FILLING = dict(NC_LISTING_DURATION=400, NC_RES_DEPLETION=0, NC_SPAWN_IMMUNITY=3, NC_WEAPON_DROP_THR=-1,
                      NC_NPC_AGGR_PCT=200, NC_NPC_NEUT_PCT=200)


def fill_market(acts, obs, L, rng):
    """Edit random valid actions acts [E, P, 12] in place, given the records obs [E, P, stride] they were drawn from:
    most agents list their first sellable item at a random price, nobody destroys or uses items, and only one agent in
    four buys -- uniform-random play never lists more than a few items at a time; this outgrows a small Market block."""
    so, sn = L.masks["Sell.InventoryItem"]
    for e in range(acts.shape[0]):
        for p in range(acts.shape[1]):
            sellable = np.flatnonzero(obs[e, p, so:so + sn - 1])
            if len(sellable) and rng.random() < 0.9:
                acts[e, p, 9] = sellable[0]; acts[e, p, 10] = rng.integers(0, L.n_price)
            acts[e, p, 3] = acts[e, p, 11] = L.n_inv
            if p % 4:
                acts[e, p, 2] = L.n_mkt
    return acts


def random_layouts(n, seed=2024):
    """n record layouts drawn uniformly within what nmmo_create accepts: every width >= 1, N_ENT_OBS <= 255,
    N_INV <= 16, N_PRICE <= 256, VISION < MAP_BORDER (16), TASK_DIM a multiple of 8, the twelve mask heads <= 1024."""
    rng = np.random.default_rng(seed)
    cfg = np.zeros(SPEC["NC_COUNT"], np.int32)
    out = []
    while len(out) < n:
        n_ent, n_mkt, n_inv = int(rng.integers(1, 256)), int(rng.integers(1, 1000)), int(rng.integers(1, 17))
        n_price, vision, task_dim = int(rng.integers(1, 257)), int(rng.integers(0, 16)), 8 * int(rng.integers(1, 65))
        for k, v in zip(("NC_N_ENT_OBS", "NC_N_MKT_OBS", "NC_N_INV", "NC_N_PRICE"), (n_ent, n_mkt, n_inv, n_price)):
            cfg[SPEC[k]] = v
        if ObsLayout(cfg).m_end <= 1024:
            out.append((n_ent, n_mkt, n_inv, n_price, vision, task_dim, SMALL))
    return out


def layout_world(layout, **engine_over):
    n_ent, n_mkt, n_inv, n_price, vision, task_dim, shape = layout
    return build_world(task_dim=task_dim, **shape, NC_N_ENT_OBS=n_ent, NC_N_MKT_OBS=n_mkt, NC_N_INV=n_inv,
                       NC_N_PRICE=n_price, NC_VISION=vision, **engine_over)


def describe_obs_mismatch(cfg, a, b):
    """Human-readable location of the first differing byte between two obs records."""
    L = ObsLayout(cfg)
    idx = int(np.flatnonzero(a != b)[0])
    for name, (o, n) in L.masks.items():
        if o <= idx < o + n:
            return f"mask {name}[{idx - o}] gpu={a[idx]} oracle={b[idx]}"
    sections = [("ids", L.o_ids, 4, 2), ("Entity", L.o_entity, L.n_ent * 62, 62), ("Inventory", L.o_inventory, L.n_inv * 32, 32),
                ("Market", L.o_market, L.n_mkt * 32, 32), ("Task", L.o_task, L.task_dim * 2, 2), ("Tile", L.o_tile, L.win * L.win * 6, 6)]
    for name, o, n, rowb in sections:
        if o <= idx < o + n:
            row, col = (idx - o) // rowb, ((idx - o) % rowb) // 2
            ra = a[o + row * rowb:o + (row + 1) * rowb].view(np.int16)
            rb = b[o + row * rowb:o + (row + 1) * rowb].view(np.int16)
            return f"{name} row {row} col {col}: gpu={ra.tolist()} oracle={rb.tolist()}"
    return f"padding byte {idx}"


def run_parity(sim, oracles, seeds, ticks, action_seed=99, map_ids=None, task_ids=None, check_state_every=16,
               action_fn=None, on_tick=None):
    """Step `sim` (E envs) and the E oracle envs in lockstep; assert bit-exact outputs every tick."""
    import torch
    E, P = sim.E, sim.P
    cfg = sim.cfg
    sim.reset(seeds, map_ids=map_ids, task_ids=task_ids)
    for e, o in enumerate(oracles):
        o.reset(int(seeds[e]), -1 if map_ids is None else int(map_ids[e]), None if task_ids is None else task_ids[e])
    n_infos = 0
    n_done = 0
    for t in range(ticks + 1):
        torch.cuda.synchronize()
        g_obs = sim.obs.cpu().numpy().reshape(E, P, -1)
        g_rew = sim.rewards.cpu().numpy().reshape(E, P); g_term = sim.terminated.cpu().numpy().reshape(E, P)
        g_trunc = sim.truncated.cpu().numpy().reshape(E, P); g_mask = sim.mask.cpu().numpy().reshape(E, P)
        g_info = sim.info.cpu().numpy().reshape(E, P, -1); g_iv = sim.info_valid.cpu().numpy().reshape(E, P)
        g_done = sim.episode_done.cpu().numpy()
        for e, o in enumerate(oracles):
            tag = f"tick {t} env {e}"
            o_obs = o.obs
            if not np.array_equal(g_obs[e], o_obs):
                bad = np.flatnonzero((g_obs[e] != o_obs).any(axis=1))
                p = int(bad[0])
                raise AssertionError(f"{tag} agent row {p}: obs differ ({len(bad)} agents): " + describe_obs_mismatch(cfg, g_obs[e, p], o_obs[p]))
            assert np.array_equal(g_mask[e], o.mask), f"{tag}: mask {g_mask[e]} vs {o.mask}"
            assert np.array_equal(g_term[e], o.terminated), f"{tag}: terminated"
            assert np.array_equal(g_trunc[e], o.truncated), f"{tag}: truncated"
            assert np.array_equal(g_rew[e].view(np.uint32), o.rewards.view(np.uint32)), \
                f"{tag}: rewards {g_rew[e][g_rew[e] != o.rewards]} vs {o.rewards[g_rew[e] != o.rewards]}"
            assert np.array_equal(g_iv[e], o.info_valid), f"{tag}: info_valid"
            assert bool(g_done[e]) == o.episode_done, f"{tag}: episode_done"
            if o.info_valid.any():
                v = o.info_valid.astype(bool)
                gi, oi = g_info[e][v], o.info[v]
                same = (gi == oi) | (np.isnan(gi) & np.isnan(oi))
                if not same.all():
                    r, k = np.argwhere(~same)[0]
                    names = [n for n, _ in sorted(((n, i) for n, i in SPEC.items() if n.startswith("IN_") and n != "IN_N"), key=lambda x: x[1])]
                    raise AssertionError(f"{tag}: info {names[k]} gpu={gi[r, k]} oracle={oi[r, k]}")
                n_infos += int(v.sum())
            n_done += int(o.episode_done)
            if check_state_every and t % check_state_every == 0:
                ge, gi_, gm, gsc = sim.snapshot(e)
                oe, oi_, om = o.snapshot()
                assert np.array_equal(gm, om), f"{tag}: map differs at {np.argwhere(gm != om)[:4].tolist()}"
                if not np.array_equal(gi_, oi_):
                    r = int(np.flatnonzero((gi_ != oi_).any(axis=1))[0])
                    raise AssertionError(f"{tag}: item row {r} gpu={gi_[r].tolist()} oracle={oi_[r].tolist()}")
                if not np.array_equal(ge, oe):
                    r = int(np.flatnonzero((ge != oe).any(axis=1))[0])
                    cols = np.flatnonzero(ge[r] != oe[r]).tolist()
                    raise AssertionError(f"{tag}: entity row {r} cols {cols} gpu={ge[r][cols].tolist()} oracle={oe[r][cols].tolist()}")
                assert gsc[SPEC["NC_N_PLAYERS"] * 0 + 7] == 0, f"{tag}: device error flag {gsc[7]}"
        if on_tick is not None:
            on_tick(t, sim, oracles)
        if t == ticks:
            break
        if action_fn is None:
            sim.sample_actions(action_seed)
            torch.cuda.synchronize()
            acts = sim.actions.cpu().numpy()
            for e, o in enumerate(oracles):
                oa = o.sample_actions(action_seed + e)
                assert np.array_equal(acts[e], oa), f"tick {t} env {e}: sampled actions differ"
        else:
            acts = action_fn(t, g_obs).astype(np.int32)
            sim.actions.copy_(torch.from_numpy(acts))
        sim.step()
        for e, o in enumerate(oracles):
            o.step(acts[e])
    return dict(infos=n_infos, episodes_done=n_done)
