"""Device-resident rollout loop: the body of ``clean_pufferl.evaluate`` without host round trips.

Mirrors /root/reference/reinforcement_learning/clean_pufferl.py:279-362 statement by statement
(including the exit test at the top of the loop, :289, so every stored action is also sent):

    o, r, d, t, i, env_id, mask = data.pool.recv()                     :293
    agent_steps_collected += sum(mask); padded_steps_collected += len(mask)   :306-307
    actions, logprob, value, _ = data.policy_pool.forwards(o, lstm)    :317
    indices = where(mask * policy_pool.mask)[: batch_size - ptr + 1]   :333-337
    obs_ary[ptr:end] = o[indices] ... sort_keys.extend(...)            :340-346
    data.pool.send(actions)                                            :357

with ``pool`` = B200VecEnv (CUDA tensors from recv, CUDA actions to send) and the seven fancy-index
stores + ``.cpu()`` copies replaced by one DeviceRollout.store.  The policy is any callable
``policy(flat_obs_uint8[B, obs_sz]) -> (actions int[B, 12], logprob f32[B], value f32[B])`` running on the
same device; the reference's policies qualify once their ``pufferlib.emulation.unpack_batched_obs`` is
nmmo_b200.emulation.unpack_batched_obs (INTEGRATION.md).  Only the step counters come back to the host.
"""
from __future__ import annotations

from types import SimpleNamespace


def evaluate(pool, policy, rollout, learner_mask=None, max_steps: int = 1 << 30):
    """Collect ``rollout.batch_size + 1`` samples (``rollout`` covers all slots of the pool; each batch of an env pool is
    stored at its global slots).  Returns a namespace with the reference's counters:
    agent_steps (sum of mask, :306), global_steps (len(mask), :307), steps, infos (list of dicts)."""
    import torch
    rollout.reset()
    agent_steps = torch.zeros((), dtype=torch.int64, device=rollout.obs.device)
    padded, step, n_recv, infos = 0, 0, 0, []
    cap = rollout.batch_size + 1
    while step < max_steps:
        step += 1
        if rollout.ptr >= cap:        # the one host read per step (the reference's `ptr == batch_size + 1` test, :289)
            break
        o, r, d, t, i, env_id, mask = pool.recv()
        # an env pool (envs_per_batch < num_envs) hands out one batch: its rows are the global slots from slot_base on
        slot_base = pool.batch_env_range[0] * pool.agents_per_env if hasattr(pool, "batch_env_range") else 0
        n_recv += 1
        infos.extend(i)
        agent_steps += mask.sum()
        padded += mask.numel()
        with torch.no_grad():
            actions, logprob, value = policy(o)
        lm = learner_mask
        if lm is not None and lm.numel() != mask.numel():      # a mask over all slots: the batch's part
            lm = lm.reshape(-1)[slot_base:slot_base + mask.numel()]
        rollout.store(o, value, actions, logprob, r, d.float(), mask, step, learner_mask=lm, slot_base=slot_base)
        # the reference always sends the step's actions and only leaves at the top of the next iteration (:289, :357):
        # the stored (action, logprob, value) of the last row are the ones the envs execute, and the next call's
        # first recv() sees fresh outputs
        pool.send(actions)
    return SimpleNamespace(agent_steps=int(agent_steps.item()), global_steps=padded, steps=n_recv, infos=infos)
