"""nmmo_b200/takeru_policy.py == the reference's agent_zoo/takeru/policy.py (BASELINE.json configs[3] consumer).

The reference module is loaded unmodified (third-party imports stubbed, see test_reference_policy.py), both networks get
the same weights through ``state_dict`` (same parameter names), and logits / values are compared on oracle records --
with and without the per-environment Market de-duplication.  No outputs of the reference module are stored in this
repository, so the test is skipped where no reference checkout ($NMMO_REFERENCE) is at hand."""
import types

import numpy as np
import pytest
import torch

from nmmo_b200.emulation import UnflattenContext
from nmmo_b200.takeru_policy import HEADS, TakeruPolicy
from test_reference_policy import REF, _load_reference_policy
from util import SMALL, build_world


def _records(world, ticks=12, seed=4):
    from oracle.oracle import OracleEnv
    recs = []
    for e in range(3):
        o = OracleEnv(*world); o.reset(seed + e)
        for t in range(ticks):
            o.step(o.sample_actions(7 + e))
        recs.append(o.obs.copy())
    return torch.from_numpy(np.concatenate(recs))


@pytest.mark.skipif(REF is None, reason="no reference checkout: set NMMO_REFERENCE")
@pytest.mark.parametrize("dedup,sparse", [(False, False), (True, False), (True, True)])
def test_same_weights_same_outputs_as_the_reference_module(dedup, sparse):
    torch.manual_seed(0)
    module = _load_reference_policy()
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=64, NC_RES_DEPLETION=1, NC_SPAWN_IMMUNITY=2, NC_WEAPON_DROP_THR=1 << 30)
    cfg = world[0]
    ctx = UnflattenContext(cfg)
    ref = module.ReducedModelV2(types.SimpleNamespace(unflatten_context=ctx), input_size=48, hidden_size=40, task_size=64)
    mine = TakeruPolicy(ctx, input_size=48, hidden_size=40, task_size=64, agents_per_env=16, dedup_market=dedup, sparse_entities=sparse)
    missing = mine.load_state_dict(ref.state_dict(), strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    flat = _records(world)
    assert flat.shape[0] == 48
    with torch.no_grad():
        hidden, lookup = ref.encode_observations(flat)
        ref_logits, ref_value = ref.decode_actions(hidden, lookup)
        my_logits, my_value = mine.logits(flat)
    alive = flat[:, ctx.layout.o_ids:ctx.layout.o_ids + 2].view(torch.int16)[:, 0] != 0
    assert alive.sum() > 8 and len(my_logits) == 12
    for h, a, b in zip(HEADS, ref_logits, my_logits):
        assert a.shape == b.shape, h
        assert torch.allclose(a[alive], b[alive], rtol=1e-5, atol=1e-5), h
    assert torch.allclose(ref_value[alive], my_value[alive], rtol=1e-5, atol=1e-5)
    # sampled actions respect the masks; log-probabilities are those of the sampled entries
    g = torch.Generator().manual_seed(1)
    actions, logprob, value = mine(flat, generator=g)
    assert actions.shape == (48, 12) and actions.dtype == torch.int32
    lp = torch.zeros(48)
    for k, lg in enumerate(my_logits):
        picked = lg[torch.arange(48), actions[:, k].long()]
        assert bool((picked[alive] > -1e8).all()), HEADS[k]
        lp += torch.log_softmax(lg, -1)[torch.arange(48), actions[:, k].long()]
    assert torch.allclose(lp[alive], logprob[alive], atol=1e-4)
    assert torch.allclose(value, my_value.squeeze(-1))
