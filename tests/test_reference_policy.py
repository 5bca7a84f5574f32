"""Rows a-14 / a-15 of SURVEY.md section 8: the reference's own policy consumes our observation record.

agent_zoo/takeru/policy.py is loaded UNMODIFIED from the reference checkout named by $NMMO_REFERENCE (the two
absent third-party packages are stubbed: pufferlib.models.Policy -> torch.nn.Module,
pufferlib.emulation.unpack_batched_obs -> the record unpacker of nmmo_b200/emulation.py, nmmo's EntityState column names -> include/nmmo_spec.h) and run
on observation records produced by the oracle.  It must find every alive agent's own row, produce one
logit vector per action head with the width of the matching ActionTargets mask, mask exactly the invalid
entries, and its greedy actions must be accepted by the engine step.  Skipped where no reference checkout
is at hand.
"""
import importlib.util
import sys
import types

import numpy as np
import pytest

from nmmo_b200.config import SPEC, ObsLayout
from nmmo_b200.emulation import UnflattenContext, unpack_batched_obs
from util import SMALL, build_world, reference_file

REF = reference_file("agent_zoo", "takeru", "policy.py")
pytestmark = pytest.mark.skipif(REF is None, reason="no reference checkout: set NMMO_REFERENCE")


def _load_reference_policy():
    import torch

    def mod(name):
        m = types.ModuleType(name)
        sys.modules[name] = m
        return m

    saved = {k: sys.modules.get(k) for k in ("pufferlib", "pufferlib.emulation", "pufferlib.models", "nmmo", "nmmo.entity", "nmmo.entity.entity")}
    puf = mod("pufferlib"); emu = mod("pufferlib.emulation"); models = mod("pufferlib.models")
    puf.emulation = emu; puf.models = models
    emu.unpack_batched_obs = unpack_batched_obs

    class Policy(torch.nn.Module):
        def __init__(self, env):
            super().__init__()

    class RecurrentWrapper(torch.nn.Module):
        def __init__(self, env, policy, input_size, hidden_size, num_layers):
            super().__init__()

    models.Policy = Policy; models.RecurrentWrapper = RecurrentWrapper
    nmmo = mod("nmmo"); ent = mod("nmmo.entity"); ee = mod("nmmo.entity.entity"); nmmo.entity = ent; ent.entity = ee
    cols = {k[3:].lower(): v for k, v in SPEC.items() if k.startswith("EA_") and isinstance(v, int) and v < SPEC["EA_N_OBS"] and k != "EA_N_OBS"}
    ee.EntityState = type("EntityState", (), {"State": type("State", (), {"attr_name_to_col": cols})})
    spec = importlib.util.spec_from_file_location("ref_takeru_policy", REF)
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    for k, v in saved.items():
        if v is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = v
    return module


def test_reference_takeru_policy_runs_on_our_records():
    import torch
    from oracle.oracle import OracleEnv
    torch.manual_seed(0)
    module = _load_reference_policy()
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=64, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=2)
    cfg = world[0]
    L = ObsLayout(cfg)
    env = types.SimpleNamespace(unflatten_context=UnflattenContext(cfg))
    policy = module.ReducedModelV2(env, input_size=32, hidden_size=32, task_size=64)
    o = OracleEnv(*world)
    o.reset(4)
    dims = [n for (_, n) in L.masks.values()]
    for t in range(25):
        flat = torch.from_numpy(o.obs.copy())
        alive = torch.from_numpy(o.mask.astype(bool) & ~o.terminated.astype(bool)) if t else torch.ones(o.P, dtype=torch.bool)   # the dead get the zero pad record
        with torch.no_grad():
            hidden, lookup = policy.encode_observations(flat)
            logits, value = policy.decode_actions(hidden, lookup)
        assert value.shape == (o.P, 1) and len(logits) == 12
        out = unpack_batched_obs(flat, env.unflatten_context)
        # every alive agent finds itself among its Entity rows (policy.py:177-182)
        ids = out["Entity"][:, :, SPEC["EA_ID"]]
        me = out["AgentId"][:, 0]
        found = ((ids == me.unsqueeze(1)) & (ids != 0)).any(dim=1)
        assert bool(found[alive].all()) and not bool(found[~alive].any())
        acts = np.zeros((o.P, 12), np.int32)
        for k, ((path, (off, n)), lg) in enumerate(zip(L.masks.items(), logits)):
            assert lg.shape == (o.P, dims[k]), f"{path}: logits {tuple(lg.shape)}"
            a, b = path.split(".")
            mask = out["ActionTargets"][a][b]
            assert bool(((lg == -1e9) == (mask == 0)).all()), f"{path}: masked_fill must hit exactly the zero entries"
            pick = lg.argmax(dim=1)
            ok = mask[torch.arange(o.P), pick] == 1
            assert bool(ok[alive].all()), f"{path}: greedy action of an alive agent is a valid one"
            acts[:, k] = pick.numpy()
        acts[~alive.numpy()] = 0
        o.step(acts)
        if o.episode_done:
            break
    assert t >= 10
