"""The reference's real curricula -> device task tables (nmmo_b200/curriculum.py), and team-task semantics on the oracle.

The spec modules and the embedding pickles live in the reference baselines repository; the translated tables are
committed under nmmo_b200/data/ (tools/make_task_tables.py).  Tests that need a checkout of the reference (named by
$NMMO_REFERENCE) skip without it.
"""
import textwrap

import numpy as np
import pytest

from nmmo_b200.config import SPEC
from nmmo_b200.curriculum import (Unsupported, load_spec_module, load_spec_pickle, load_table, spec_name, spec_to_row, translate)
from nmmo_b200.tasks import EVENT, ITEM, PRED, SKILL, TF_RELATIVE_TARGET, TF_TEAM, task_row
from util import SMALL, build_world, reference_file

REF = reference_file("neurips23_evaluation")
needs_ref = pytest.mark.skipif(REF is None, reason="no reference checkout: set NMMO_REFERENCE")


def test_committed_tables():
    h = load_table("heldout")
    assert h["rows"].shape == (63, SPEC["NM_TASK_COLS"]) and h["embed"].shape == (63, 2048) and h["embed"].dtype == np.float16
    assert h["unsupported"] == [] and len(set(h["names"])) == 63
    assert h["names"][0] == "Task_TickGE_(num_tick:1024)_reward_to:agent" and h["rows"][0].tolist()[:2] == [PRED["TICK_GE"], 1024]
    assert np.isfinite(h["embed"].astype(np.float32)).all() and np.abs(h["embed"].astype(np.float32)).max() > 0.1
    # spot checks against the source (heldout_evaluation_task.py:43-50, :112-119)
    r = dict(zip(h["names"], h["rows"].tolist()))
    assert r["Task_DefeatEntity_(agent_type:npc_level:3_num_agent:20)_reward_to:agent"][:4] == [PRED["DEFEAT_ENTITY"], 0, 3, 20]
    assert r["Task_FullyArmed_(combat_style:Mage_level:3_num_agent:1)_reward_to:agent"][:3] == [PRED["FULLY_ARMED"], SKILL["MAGE"], 3]
    assert r["Task_CountEvent_(event:EARN_GOLD_N:20)_reward_to:agent"][:3] == [PRED["COUNT_EVENT"], EVENT["EARN_GOLD"], 20]
    s = load_table("sample_eval")
    assert s["rows"].shape[0] == 24 and s["embed"].shape == (24, 2048) and s["unsupported"] == []
    m = load_table("manual")
    assert m["rows"].shape[0] > 1000 and m["unsupported"] == [] and m["embed"] is None
    # composites of manual_curriculum.py:119-122 and :201-202
    i = m["names"].index("Task_PracticeSkillWithTool_(skill:Fishing_exp:50)_reward_to:agent")
    assert m["rows"][i].tolist() == task_row("EQUIP_ITEM", ITEM["ROD"], 1, pred2="GAIN_EXPERIENCE", q0=SKILL["FISHING"], q1=50, combine=2, wa=300, wb=700)
    i = m["names"].index("Task_PracticeInventoryManagement_(space:4_num_tick:200)_reward_to:agent")
    assert m["rows"][i].tolist() == task_row("INVENTORY_SPACE_GE", 4, pred2="TICK_GE", q0=200, combine=1)
    # named targets are resolved on the device relative to the assignee's team
    i = m["names"].index("Task_CanSeeGroup_(target:left_team)_reward_to:agent")
    assert m["rows"][i].tolist() == task_row("CAN_SEE_GROUP", -1, 0, 0, TF_RELATIVE_TARGET)
    assert m["weights"].max() == 100.0                         # sampling_weight of the most essential events (:66-72)


@needs_ref
def test_spec_module_and_pickle_agree_and_match_the_committed_table():
    py = load_spec_module(REF / "heldout_evaluation_task.py")
    pk = load_spec_pickle(REF / "heldout_task_with_embedding.pkl")
    assert [spec_name(s) for s in py] == [spec_name(s) for s in pk]
    rows_py, names, _, _, bad_py = translate(py)
    rows_pk, _, _, emb, bad_pk = translate(pk)
    assert bad_py == [] and bad_pk == [] and np.array_equal(rows_py, rows_pk)
    h = load_table("heldout")
    assert np.array_equal(h["rows"], rows_py) and h["names"] == names
    assert np.array_equal(h["embed"].view(np.uint16), emb.view(np.uint16))
    # spot checks against the source (heldout_evaluation_task.py:43-50, :112-119)
    r = dict(zip(names, rows_py.tolist()))
    assert r["Task_DefeatEntity_(agent_type:npc_level:3_num_agent:20)_reward_to:agent"][:4] == [PRED["DEFEAT_ENTITY"], 0, 3, 20]
    assert r["Task_FullyArmed_(combat_style:Mage_level:3_num_agent:1)_reward_to:agent"][:3] == [PRED["FULLY_ARMED"], SKILL["MAGE"], 3]
    assert r["Task_CountEvent_(event:EARN_GOLD_N:20)_reward_to:agent"][:3] == [PRED["COUNT_EVENT"], EVENT["EARN_GOLD"], 20]


def test_unsupported_specs_are_reported_by_name(tmp_path):
    src = tmp_path / "my_curriculum.py"
    src.write_text(textwrap.dedent('''
        import nmmo.systems.skill as Skill
        from nmmo.task.base_predicates import AttainSkill, TickGE, CanSeeGroup, AllDead, AllMembersWithinRange, HoardGold
        from nmmo.task.task_spec import TaskSpec
        def Weird(gs, subject, a):
            return TickGE(gs, subject, a) * TickGE(gs, subject, a) * HoardGold(gs, subject, a)
        def Formation(gs, subject, dist, num_tick):
            return AllMembersWithinRange(gs, subject, dist) * TickGE(gs, subject, num_tick)
        curriculum = [
            TaskSpec(eval_fn=AttainSkill, eval_fn_kwargs={"skill": Skill.Melee, "level": 3, "num_agent": 3}),
            TaskSpec(eval_fn=Weird, eval_fn_kwargs={"a": 5}),
            TaskSpec(eval_fn=lambda gs, subject: 1.0, eval_fn_kwargs={}),
            TaskSpec(eval_fn=Formation, eval_fn_kwargs={"dist": 3, "num_tick": 100}, reward_to="team"),
            TaskSpec(eval_fn=AllDead, eval_fn_kwargs={"target": "left_team_leader"}, reward_to="team"),
            TaskSpec(eval_fn=CanSeeGroup, eval_fn_kwargs={"target": "right_team"}, reward_to="team"),
        ]
    '''))
    specs = load_spec_module(src)
    rows, names, _, _, bad = translate(specs)
    assert len(rows) == 3 and len(bad) == 3
    assert "num_agent=3" in bad[0][1] and "AttainSkill" in bad[0][0] and "Weird" in bad[1][0]
    assert rows[0].tolist() == task_row("ALL_MEMBERS_WITHIN_RANGE", 3, 0, 0, TF_TEAM, pred2="TICK_GE", q0=100, combine=1)
    assert rows[1].tolist() == task_row("ALL_DEAD", -1, 1, 0, TF_TEAM | TF_RELATIVE_TARGET)
    assert rows[2].tolist() == task_row("CAN_SEE_GROUP", 1, 0, 0, TF_TEAM | TF_RELATIVE_TARGET)
    with pytest.raises(Unsupported):
        spec_to_row(specs[0])


def _team_world(team_size, rows):
    from nmmo_b200.tasks import make_task_table
    cfg, fcfg, maps, _, _ = build_world(task_dim=64, **SMALL, NC_HORIZON=80, NC_RES_DEPLETION=1, NC_TEAM_SIZE=team_size)
    tab, emb = make_task_table(rows, 64, seed=1)
    return cfg, fcfg, maps, tab, emb


def test_team_task_semantics_on_the_oracle():
    from oracle.oracle import OracleEnv
    rows = [task_row("ALL_MEMBERS_WITHIN_RANGE", 6, 0, 0, TF_TEAM), task_row("ALL_DEAD", 1, 0, 0, TF_TEAM | TF_RELATIVE_TARGET),
            task_row("STAY_ALIVE", 0, 0, 0, TF_TEAM), task_row("DISTANCE_TRAVELED", 12, 0, 0, TF_TEAM),
            task_row("COUNT_EVENT", EVENT["DRINK_WATER"], 6, 0, TF_TEAM)]
    world = _team_world(4, rows)
    o = OracleEnv(*world)
    o.reset(5)
    tid = o.task_state()[0]
    assert all(len(set(tid[t * 4:(t + 1) * 4].tolist())) == 1 for t in range(4)), "one task per team"
    P = o.P
    S = SPEC
    for t in range(60):
        o.step(o.sample_actions(3))
        ent = o.snapshot()[0]
        alive = (ent[:P, S["EA_STATUS"]] == 1) & (ent[:P, S["EA_HEALTH"]] > 0)
        tid, completed, signals, maxprog = o.task_state()
        # members of a team that are alive and hold an uncompleted team task report the same progress
        for team in range(4):
            m = [p for p in range(team * 4, team * 4 + 4) if alive[p]]
            if len(m) > 1 and not any(completed[p] for p in m):
                assert len({round(float(maxprog[p]), 12) for p in m}) == 1
        if o.episode_done:
            break
    # direct check of one predicate against the state: AllDead over the right-hand team = fraction of its members dead
    o2 = OracleEnv(*_team_world(4, [rows[1]])); o2.reset(9)
    for t in range(70):
        o2.step(o2.sample_actions(4))
        if o2.episode_done:
            break
        ent = o2.snapshot()[0]
        alive = (ent[:P, S["EA_STATUS"]] == 1) & (ent[:P, S["EA_HEALTH"]] > 0)
        _, completed, _, maxprog = o2.task_state()
        for p in range(P):
            if alive[p] and not completed[p]:
                right = ((p // 4 + 1) % 4) * 4
                assert maxprog[p] >= (4 - alive[right:right + 4].sum()) / 4.0 - 1e-12
