"""The oracle's own records at record layouts away from the reference's, checked in numpy against its state snapshot:
the GPU is judged against these records (tests/test_record_layouts_gpu.py), so they must be right at every width."""
import numpy as np
import pytest

from nmmo_b200.config import SPEC, ObsLayout
from util import LONG_LIVED, MARKET_FILLING, RECORD_LAYOUTS, fill_market, layout_world, random_layouts

S = SPEC
CASES = dict(RECORD_LAYOUTS)
CASES.update({"vision_0": (100, 384, 12, 99, 0, 64, RECORD_LAYOUTS["minimal"][6]),
              "vision_15": (100, 384, 12, 99, 15, 64, RECORD_LAYOUTS["minimal"][6])})
CASES.update({f"random_{i}": lay for i, lay in enumerate(random_layouts(8))})
ITEM_COLS = ((S["IA_TYPE"], S["IS_TYPE"]), (S["IA_OWNER"], S["IS_OWNER"]), (S["IA_LEVEL"], S["IS_LEVEL"]),
             (S["IA_QUANTITY"], S["IS_QUANTITY"]), (S["IA_EQUIPPED"], S["IS_EQUIPPED"]), (S["IA_LISTED_PRICE"], S["IS_PRICE"]))


def _item_rows(items, rows):
    """Expected Inventory / Market rows of item-table rows `rows`: the table's own columns (id = row + 1)."""
    out = np.zeros((len(rows), 16), np.int16)
    out[:, S["IA_ID"]] = rows + 1
    for ia, is_ in ITEM_COLS:
        out[:, ia] = items[rows, is_]
    return out


def check_records(o):
    L, obs = o.L, o.obs
    ent, items, mp = o.snapshot()
    vis = L.win // 2
    alive = np.flatnonzero(ent[:, S["EA_STATUS"]] == S["ES_ALIVE"])
    used = items[:, S["IS_TYPE"]] > 0
    all_listed = np.flatnonzero(used & (items[:, S["IS_PRICE"]] > 0))
    listed = all_listed[:L.n_mkt]
    ia_cols = [ia for ia, _ in ITEM_COLS] + [S["IA_ID"]]
    # the takeru / yaofeng wrappers' disable_give: only GiveGold.Price 0 stays offered
    no_give = o.cfg[S["NC_DISABLE_GIVE"]] and o.cfg[S["NC_WRAPPER"]] in (S["NW_TAKERU"], S["NW_YAOFENG"])
    seen = dict(ent=0, inv=0, listed=len(all_listed))
    for p in range(o.P):
        rec = obs[p]
        if ent[p, S["EA_STATUS"]] != S["ES_ALIVE"]:
            assert not rec.any(), f"agent {p}: the record of an absent agent is not zero"
            continue
        me = ent[p]
        r0, c0 = int(me[S["EA_ROW"]]), int(me[S["EA_COL"]])
        ids = rec[L.o_ids:L.o_ids + 4].view(np.int16)
        assert ids[0] == me[S["EA_ID"]] and ids[1] == o.tick
        # Tile: the (2 vis + 1)^2 window around the agent, row-major, (row, col, material)
        tiles = rec[L.o_tile:L.o_tile + L.win * L.win * 6].view(np.int16).reshape(L.win, L.win, 3)
        rr, cc = np.meshgrid(np.arange(r0 - vis, r0 + vis + 1), np.arange(c0 - vis, c0 + vis + 1), indexing="ij")
        assert np.array_equal(tiles[..., 0], rr) and np.array_equal(tiles[..., 1], cc), f"agent {p}: tile coordinates"
        assert np.array_equal(tiles[..., 2], mp[rr, cc]), f"agent {p}: tile window is not the map slice"
        # Entity: the first n_ent alive table rows inside the window, in table order, then zero rows
        near = alive[(np.abs(ent[alive, S["EA_ROW"]] - r0) <= vis) & (np.abs(ent[alive, S["EA_COL"]] - c0) <= vis)][:L.n_ent]
        eo = rec[L.o_entity:L.o_entity + L.n_ent * 62].view(np.int16).reshape(L.n_ent, 31)
        assert np.array_equal(eo[:len(near)], ent[near, :31]), f"agent {p}: Entity rows"
        assert not eo[len(near):].any(), f"agent {p}: Entity rows past the visible ones"
        assert p in near or len(near) == L.n_ent, f"agent {p} does not see itself"
        # Inventory: the first n_inv items the agent owns, in table order
        own = np.flatnonzero(used & (items[:, S["IS_OWNER"]] == me[S["EA_ID"]]))[:L.n_inv]
        io = rec[L.o_inventory:L.o_inventory + L.n_inv * 32].view(np.int16).reshape(L.n_inv, 16)
        assert np.array_equal(io[:len(own)][:, ia_cols], _item_rows(items, own)[:, ia_cols]), f"agent {p}: Inventory rows"
        assert not io[len(own):].any(), f"agent {p}: Inventory rows past the owned ones"
        # Market: the first n_mkt listed items, in table order
        mo = rec[L.o_market:L.o_market + L.n_mkt * 32].view(np.int16).reshape(L.n_mkt, 16)
        assert np.array_equal(mo[:len(listed)][:, ia_cols], _item_rows(items, listed)[:, ia_cols]), f"agent {p}: Market rows"
        assert not mo[len(listed):].any(), f"agent {p}: Market rows past the listed ones"
        # masks: every head where ObsLayout puts it, no-ops last, nothing beyond the last head
        m = rec[:L.m_end].view(np.int8)
        head = {name: m[off:off + n] for name, (off, n) in L.masks.items()}
        assert head["Attack.Style"].tolist() == [1, 1, 1] and head["Sell.Price"].all() and head["GiveGold.Price"][0] == 1
        for name in ("Buy.MarketItem", "Destroy.InventoryItem", "Give.InventoryItem", "Give.Target", "GiveGold.Target",
                     "Sell.InventoryItem", "Use.InventoryItem"):
            assert head[name][-1] == 1, f"agent {p}: {name} no-op"
        assert not head["Buy.MarketItem"][len(listed):-1].any(), f"agent {p}: Buy entries past the listed rows"
        for name in ("Destroy.InventoryItem", "Give.InventoryItem", "Sell.InventoryItem", "Use.InventoryItem"):
            assert not head[name][len(own):-1].any(), f"agent {p}: {name} entries past the owned items"
        for name in ("Attack.Target", "Give.Target", "GiveGold.Target"):
            assert not head[name][len(near):-1].any(), f"agent {p}: {name} entries past the visible rows"
        gold = 0 if no_give else int(me[S["EA_GOLD"]])
        assert np.array_equal(head["GiveGold.Price"][1:], (np.arange(1, L.n_price) < gold).astype(np.int8))
        assert not rec[L.m_end:L.o_ids].any()
        seen["ent"] = max(seen["ent"], len(near)); seen["inv"] = max(seen["inv"], len(own))
    return seen


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_records_follow_the_layout(name):
    from oracle.oracle import OracleEnv
    lay = CASES[name]
    world = layout_world(lay, NC_HORIZON=200, **LONG_LIVED)
    L = ObsLayout(world[0])
    assert L.m_end <= 1024
    assert [n for _, n in L.masks.values()] == [3, lay[0] + 1, lay[1] + 1, lay[2] + 1, lay[2] + 1, lay[0] + 1, lay[3],
                                                 lay[0] + 1, 5, lay[2] + 1, lay[3], lay[2] + 1]
    o = OracleEnv(*world)
    assert o.obs.shape[1] == L.stride
    o.reset(17)
    peak = dict(ent=0, inv=0, listed=0)
    for t in range(61):
        if t % 6 == 0:
            peak = {k: max(v, s) for (k, v), s in zip(peak.items(), check_records(o).values())}
        o.step(o.sample_actions(5))
    # agents saw each other (at vision 0 only the agent itself is on its tile): the Entity checks compared something
    assert peak["ent"] >= (min(2, lay[0]) if lay[4] else 1), peak


def test_oracle_records_of_a_truncated_market():
    """More listings than Market rows: the records show the first n_mkt listings of the item table, in table order,
    and offer Buy only on those rows."""
    from oracle.oracle import OracleEnv
    world = layout_world(RECORD_LAYOUTS["truncating"], NC_HORIZON=200, **MARKET_FILLING)
    L = ObsLayout(world[0])
    envs = [OracleEnv(*world) for _ in range(2)]
    for e, o in enumerate(envs):
        o.reset(41 + e)
    rng = np.random.default_rng(1)
    over = 0
    for t in range(91):
        if t % 3 == 0:
            over += sum(check_records(o)["listed"] > L.n_mkt for o in envs)
        obs = np.stack([o.obs for o in envs])
        acts = fill_market(np.stack([o.sample_actions(7 + e) for e, o in enumerate(envs)]), obs, L, rng)
        for e, o in enumerate(envs):
            o.step(acts[e])
    assert over >= 10, f"the item table held more than {L.n_mkt} listings on only {over} checked env-ticks"


def test_widest_accepted_window_stays_inside_the_map():
    """nmmo_create accepts VISION up to MAP_BORDER - 1: players spawn on the ring MAP_BORDER .. MAP_BORDER + MAP_CENTER,
    whose far side is MAP_BORDER tiles from the edge, so one more tile of vision would read past the map."""
    from oracle.oracle import OracleEnv
    world = layout_world((100, 384, 12, 99, 15, 64, RECORD_LAYOUTS["minimal"][6]), NC_HORIZON=50)
    o = OracleEnv(*world)
    o.reset(3)
    b, Sz = int(world[0][S["NC_MAP_BORDER"]]), o.Sz
    pos = o.snapshot()[0][:o.P][:, [S["EA_ROW"], S["EA_COL"]]]
    assert pos.min() == b and pos.max() == Sz - b
    assert pos.max() + int(world[0][S["NC_VISION"]]) == Sz - 1
