#!/usr/bin/env python
"""Golden vectors for the rollout storage / sort / GAE path, produced by the REFERENCE's own source lines.

`clean_pufferl.evaluate` and `clean_pufferl.train` cannot be imported here (pufferlib is absent) and the
code in question is inline in those two functions, so this script cuts the exact statements out of
reinforcement_learning/clean_pufferl.py of the reference checkout ($NMMO_REFERENCE) by their first/last lines --
    the masked append   "learner_mask = torch.Tensor(mask * data.policy_pool.mask)" ... "ptr += len(indices)"   (:333-349)
    the sort            "idxs = sorted(range(len(data.sort_keys)), key=data.sort_keys.__getitem__)"            (:413)
    the GAE loop        "advantages = torch.zeros(config.batch_size, device=data.device)" ... end of the loop  (:425-436)
-- and executes them UNMODIFIED (dedented) on torch CPU tensors with a stub `data` / `config`.  Inputs and
outputs are stored in tests/golden/rollout_*.npz; tests/test_rollout.py requires oracle/rollout_oracle.py to
reproduce them bit for bit, and the GPU tests require the CUDA path to equal the oracle bit for bit.

Run with a checkout of the reference baselines repository:  NMMO_REFERENCE=<checkout> python tests/golden/make_golden_rollout.py
"""
from __future__ import annotations

import textwrap
from argparse import Namespace
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
import sys
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))
from rollout_inputs import step_stream  # noqa: E402
from util import reference_file  # noqa: E402
SRC = reference_file("reinforcement_learning", "clean_pufferl.py")


def cut(lines, first, last_pred):
    i0 = next(i for i, l in enumerate(lines) if l.strip().startswith(first))
    i1 = i0
    while not last_pred(lines, i1):
        i1 += 1
    return textwrap.dedent("".join(lines[i0:i1 + 1])), (i0 + 1, i1 + 1)


def reference_blocks():
    lines = SRC.read_text().splitlines(keepends=True)
    store, s_rng = cut(lines, "learner_mask = torch.Tensor(mask * data.policy_pool.mask)", lambda L, i: L[i].strip() == "ptr += len(indices)")
    sort, o_rng = cut(lines, "idxs = sorted(range(len(data.sort_keys))", lambda L, i: True)
    gae, g_rng = cut(lines, "advantages = torch.zeros(config.batch_size, device=data.device)",
                     lambda L, i: L[i].strip() == ")" and "lastgaelam" in L[i - 1])
    return (store, s_rng), (sort, o_rng), (gae, g_rng)


def run_case(name, seed, batch_size, n_slots, stride, p_alive, p_done, p_learner, gamma, lam):
    (store_src, s_rng), (sort_src, o_rng), (gae_src, g_rng) = reference_blocks()
    B = batch_size
    config = Namespace(batch_size=B, gamma=gamma, gae_lambda=lam)
    data = Namespace(device="cpu", sort_keys=[], policy_pool=Namespace(mask=None),
                     obs_ary=np.zeros((B + 1, stride), np.uint8), actions_ary=np.zeros((B + 1, 12), np.int64),
                     logprobs_ary=np.zeros(B + 1, np.float32), rewards_ary=np.zeros(B + 1, np.float32),
                     dones_ary=np.zeros(B + 1, np.float32), values_ary=np.zeros(B + 1, np.float32))
    env_id = np.arange(n_slots)
    ptr, n_steps = 0, 0
    for step, inp in step_stream(seed, n_slots, stride, p_alive, p_done, p_learner):
        if ptr >= B + 1:
            break
        n_steps += 1
        mask, pool_mask = inp["mask"], inp["pool_mask"]
        data.policy_pool.mask = pool_mask
        ns = dict(torch=torch, data=data, config=config, ptr=ptr, step=step, env_id=env_id, mask=mask,
                  o=torch.as_tensor(inp["o"]), value=torch.as_tensor(inp["value"]), actions=inp["actions"],
                  logprob=torch.as_tensor(inp["logprob"]), r=torch.as_tensor(inp["r"]), d=torch.as_tensor(inp["d"]))
        exec(store_src, ns)       # the reference's statements, verbatim
        ptr = ns["ptr"]
    assert ptr == B + 1
    # train(): the arrays are views of torch tensors in the reference (np.asarray(torch.zeros(...)), :191-197)
    data.dones = torch.as_tensor(data.dones_ary); data.values = torch.as_tensor(data.values_ary); data.rewards = torch.as_tensor(data.rewards_ary)
    ns = dict(torch=torch, data=data, config=config)
    exec(sort_src, ns)
    with torch.no_grad():
        exec(gae_src, ns)
    out = HERE / f"{name}.npz"
    np.savez_compressed(out, seed=seed, batch_size=B, n_slots=n_slots, stride=stride, gamma=gamma, gae_lambda=lam, n_steps=n_steps,
                        p_alive=p_alive, p_done=p_done, p_learner=p_learner, src_lines=np.array([s_rng, o_rng, g_rng]),
                        obs=data.obs_ary, actions=data.actions_ary, logprobs=data.logprobs_ary, rewards=data.rewards_ary,
                        dones=data.dones_ary, values=data.values_ary, idxs=np.asarray(ns["idxs"], np.int64),
                        advantages=ns["advantages"].numpy())
    print(f"{name}: {n_steps} steps -> {B + 1} rows, reference lines {s_rng} {o_rng} {g_rng}, {out.stat().st_size} bytes")


def main():
    assert SRC is not None, "set NMMO_REFERENCE to a checkout of the reference baselines repository"
    run_case("rollout_small", 1, batch_size=256, n_slots=96, stride=32, p_alive=0.9, p_done=0.05, p_learner=1.0, gamma=0.99, lam=0.95)
    run_case("rollout_pool", 2, batch_size=700, n_slots=128, stride=48, p_alive=0.8, p_done=0.1, p_learner=0.7, gamma=0.99, lam=0.95)
    run_case("rollout_nodone", 3, batch_size=300, n_slots=64, stride=16, p_alive=0.95, p_done=0.0, p_learner=1.0, gamma=0.97, lam=0.9)


if __name__ == "__main__":
    main()
