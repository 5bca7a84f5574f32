"""GPU: B200VecEnv as an env pool (envs_per_batch < num_envs).  Envs are independent and every draw, the built-in
policy's included, is keyed by (seed, global env, env tick, ...), so stepping the batches on their own streams must give
bit for bit what a lock-step pool gives, round after round, across episode resets."""
from argparse import Namespace
from collections import Counter

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NM_ERR_ARG, NM_ERR_STATE = -1, -4


def _small_env(horizon=60):
    return Namespace(num_agents=16, num_npcs=32, max_episode_length=horizon, maps_path="maps/", map_size=32, num_maps=4,
                     map_force_generation=False, death_fog_tick=None, task_size=64, spawn_immunity=3, resilient_population=0,
                     curriculum_file_path=None)


def _default_env(horizon=60):
    from nmmo_b200.config import default_env_args
    return default_env_args(num_maps=4, max_episode_length=horizon, resilient_population=0)


def _pools(env_ns, E, b, seed=3, collect_infos="async", big=False, monkeypatch=None):
    from nmmo_b200.vecenv import B200VecEnv
    if big:
        monkeypatch.setenv("NMMO_B200_FORCE_BIG", "1")
    try:
        lock = B200VecEnv(env_kwargs={"env": env_ns}, num_envs=E, collect_infos=collect_infos)
        pool = B200VecEnv(env_kwargs={"env": env_ns}, num_envs=E, envs_per_batch=b, env_pool=True, collect_infos=collect_infos)
    finally:
        if big:
            monkeypatch.delenv("NMMO_B200_FORCE_BIG")
    if big:
        assert pool.sim.kernel_names()[1].startswith("nmmo_obs_big"), pool.sim.kernel_names()
    for p in (lock, pool):
        p.sim.set_autosample(11)          # before the reset: the buffer is filled by the reset's observation pass
        p.async_reset(seed)
    return lock, pool


def _entries(pool, infos):
    out = []
    for slot, info in zip(pool.last_info_slots, infos):
        out.append((int(slot), int(info["length"]), float(info["return"]), bool(info.get("episode_done", False))))
    return out


def _lock_tick(lock, log=None):
    i = lock.recv()[4]
    if log is not None:
        log.extend(_entries(lock, i))
    lock.send(lock.sim.actions)


def _pool_round(pool, log=None):
    for _ in range(pool.num_batches):
        i = pool.recv()[4]
        if log is not None:
            log.extend(_entries(pool, i))
        lo, hi = pool.batch_env_range
        pool.send(pool.sim.actions[lo:hi])


def _same_outputs(a, b, tag):
    import torch
    torch.cuda.synchronize()
    for name in ("obs", "rewards", "terminated", "truncated", "mask", "info", "info_valid", "episode_done", "actions"):
        x, y = getattr(a.sim, name), getattr(b.sim, name)
        assert torch.equal(x.view(torch.uint8) if x.dtype == torch.float32 else x,
                           y.view(torch.uint8) if y.dtype == torch.float32 else y), f"{tag}: {name} differ"


def _same_state(a, b, tag):
    for e in range(a.num_envs):
        for x, y in zip(a.sim.snapshot(e), b.sim.snapshot(e)):
            assert np.array_equal(x, y), f"{tag} env {e}: tables differ"


def _run_equal(lock, pool, rounds):
    for r in range(rounds):
        _lock_tick(lock)
        _pool_round(pool)          # no synchronisation inside a round: the batch streams overlap
        _same_outputs(lock, pool, f"round {r}")
        if r % 20 == 19:
            _same_state(lock, pool, f"round {r}")
    episodes = int(pool.sim.stats()[2][2])
    assert episodes >= pool.num_envs, "every env must have reset at least once"
    assert episodes == int(lock.sim.stats()[2][2])


@pytest.mark.parametrize("b", [6, 4, 3])
def test_pool_equals_lock_step_small(b):
    lock, pool = _pools(_small_env(), 12, b)
    _run_equal(lock, pool, 200)
    lock.close(); pool.close()


@pytest.mark.parametrize("b", [4, 2])
def test_pool_equals_lock_step_default_shape(b):
    # 2-env batches leave the 4-env CTA of the step kernel half full
    lock, pool = _pools(_default_env(), 8, b, seed=5)
    assert pool.sim.kernel_names()[0].startswith("nmmo_step4_"), pool.sim.kernel_names()
    _run_equal(lock, pool, 200)
    lock.close(); pool.close()


@pytest.mark.parametrize("b", [6, 3])
def test_pool_equals_lock_step_big_family(monkeypatch, b):
    lock, pool = _pools(_small_env(), 12, b, big=True, monkeypatch=monkeypatch)
    _run_equal(lock, pool, 200)
    lock.close(); pool.close()


@pytest.mark.parametrize("collect_infos", ["async", True])
def test_pool_contract(collect_infos):
    import torch
    E, b = 12, 4
    lock, pool = _pools(_small_env(), E, b, collect_infos=collect_infos)
    P = pool.agents_per_env
    assert pool.num_batches == 3
    got, want = [], []
    for r in range(200):
        _lock_tick(lock, want)
        for k in range(pool.num_batches):
            o, rew, term, trunc, infos, env_id, mask = pool.recv()
            assert pool.batch_env_range == (k * b, (k + 1) * b), "batches rotate in order"
            for x in (o, rew, term, trunc, env_id, mask):
                assert x.shape[0] == b * P
            assert torch.equal(env_id.cpu(), torch.arange(k * b * P, (k + 1) * b * P)), "env_id = the batch's global slots"
            got.extend(_entries(pool, infos))
            if r == 0 and k == 0:
                with pytest.raises(RuntimeError):
                    pool.recv()
            lo, hi = pool.batch_env_range
            pool.send(pool.sim.actions[lo:hi])
    if collect_infos == "async":
        want.extend(_entries(lock, lock.drain_infos()))
        got.extend(_entries(pool, pool.drain_infos()))
    assert len(want) > 2 * E * P, "the run must finish many episodes"
    # the same multiset as the lock-step pool, which hands out every finished agent once: nothing is lost or duplicated
    assert Counter(got) == Counter(want)
    lock.close(); pool.close()


def test_reset_envs_while_a_batch_is_in_flight():
    # pool: batch 0 is stepped (and may still run) when envs 1 (batch 0) and 7 (batch 1) are reset; then batch 1 steps.
    # Lock-step equivalent: reset env 7, one tick, reset env 1.
    E, b, R = 12, 6, 50
    lock, pool = _pools(_small_env(), E, b)
    for _ in range(R):
        _lock_tick(lock)
        _pool_round(pool)
    pool.recv(); pool.send(pool.sim.actions[0:b])
    pool.reset_envs([1, 7], [1001, 1007])
    pool.recv()
    assert pool.batch_env_range == (b, E)
    pool.send(pool.sim.actions[b:E])
    lock.reset_envs([7], [1007])
    _lock_tick(lock)
    lock.reset_envs([1], [1001])
    _same_outputs(lock, pool, "after reset_envs")
    _same_state(lock, pool, "after reset_envs")
    lock.close(); pool.close()


class _Recorder:
    """A DeviceRollout that also keeps host copies of every store() and forwards it to a compact twin."""

    def __init__(self, roll, twin=None, task_id=None):
        self.roll, self.twin, self.task_id, self.calls = roll, twin, task_id, []

    def __getattr__(self, name):
        return getattr(self.roll, name)

    def reset(self):
        self.roll.reset()
        if self.twin is not None:
            self.twin.reset()

    def store(self, o, value, actions, logprob, r, d, mask, step, learner_mask=None, slot_base=0):
        self.calls.append(dict(o=o.cpu().numpy(), value=value.cpu().numpy(), actions=actions.cpu().numpy(),
                               logprob=logprob.cpu().numpy(), r=r.cpu().numpy(), d=d.cpu().numpy(), mask=mask.cpu().numpy(),
                               slot_base=slot_base, step=step))
        self.roll.store(o, value, actions, logprob, r, d, mask, step, learner_mask=learner_mask, slot_base=slot_base)
        if self.twin is not None:
            n = mask.numel()
            self.twin.store(o, value, actions, logprob, r, d, mask, step, learner_mask=learner_mask, slot_base=slot_base,
                            task_id=self.task_id[slot_base:slot_base + n])


def _policy(pool):
    import torch

    def policy(o):
        lo, hi = pool.batch_env_range
        a = pool.sim.actions[lo:hi].reshape(-1, 12).clone()
        x = o[:, :256].to(torch.float32)
        return a, -x[:, :128].mean(1) / 64, x.sum(1) / 4096
    return policy


def _check_against_oracle(rec, B, gamma=0.99, lam=0.95):
    from oracle.rollout_oracle import RolloutOracle
    roll = rec.roll
    o = RolloutOracle(B, roll.obs_stride)
    for c in rec.calls:
        n = len(c["mask"])
        o.store(c["o"], c["value"], c["actions"], c["logprob"], c["r"], c["d"], c["mask"], None,
                np.arange(c["slot_base"], c["slot_base"] + n), c["step"])
    n = o.ptr
    assert roll.ptr == n == B + 1
    assert np.array_equal(roll.obs[:n].cpu().numpy(), o.obs[:n])
    assert np.array_equal(roll.actions[:n].cpu().numpy(), o.actions[:n].astype(np.int32))
    for name in ("logprobs", "rewards", "dones", "values"):
        assert np.array_equal(getattr(roll, name)[:n].cpu().numpy().view(np.uint32), getattr(o, name)[:n].view(np.uint32)), name
    idxs, adv = o.gae(gamma, lam)
    d_idxs, d_adv = roll.gae(gamma, lam)
    d_idxs = d_idxs[:n].cpu().numpy()
    assert np.array_equal(d_idxs, idxs.astype(np.int32)), "sorted (slot, step) order"
    assert np.array_equal(roll.obs[:n].cpu().numpy()[d_idxs], o.obs[idxs]), "rows in sorted order"
    assert np.array_equal(d_adv[:n - 1].cpu().numpy().view(np.uint32), adv.view(np.uint32)), "advantages (bit patterns)"


@pytest.mark.parametrize("b", [6, 12])
def test_evaluate_on_pool_matches_rollout_oracle(b):
    import torch
    from nmmo_b200.evaluate import evaluate
    from nmmo_b200.rollout import DeviceRollout
    from nmmo_b200.vecenv import B200VecEnv
    E, B = 12, 700
    pool = B200VecEnv(env_kwargs={"env": _small_env()}, num_envs=E, envs_per_batch=b, env_pool=True)
    pool.sim.set_autosample(11)
    pool.async_reset(3)
    n_slots = E * pool.agents_per_env
    roll = DeviceRollout(B, n_slots, pool.driver_env.obs_sz)
    comp = DeviceRollout(B, n_slots, pool.driver_env.obs_sz, compact=DeviceRollout.compact_for(pool.sim, max_steps=64))
    rec = _Recorder(roll, comp, pool.sim.task_id)
    res = evaluate(pool, _policy(pool), rec)
    assert res.steps == len(rec.calls) and res.global_steps == res.steps * b * pool.agents_per_env
    if b < E:
        assert {c["slot_base"] for c in rec.calls} == {0, b * pool.agents_per_env}
    _check_against_oracle(rec, B)
    n = roll.ptr
    assert comp.ptr == n
    assert torch.equal(comp.expand(n=n), roll.obs[:n]), "compact rows expand to the plain rows"
    # a compact Market store that is full refuses the next call instead of writing past its end
    full = DeviceRollout(B, n_slots, pool.driver_env.obs_sz, compact=DeviceRollout.compact_for(pool.sim, max_steps=1))
    s0, s1 = 0, b * pool.agents_per_env
    args = (pool.sim.obs[s0:s1], torch.zeros(s1, device="cuda"), pool.sim.actions[0:b], torch.zeros(s1, device="cuda"),
            pool.sim.rewards[s0:s1], torch.zeros(s1, device="cuda"), pool.sim.mask[s0:s1], 1)
    for k in range(E // b):
        full.store(*args, task_id=pool.sim.task_id[s0:s1], slot_base=k * s1)
    with pytest.raises(Exception, match="Market store is full"):
        full.store(*args, task_id=pool.sim.task_id[s0:s1], slot_base=0)
    with pytest.raises(Exception):
        roll.store(*args, slot_base=n_slots - s1 + 1)        # past the last slot
    roll.close(); comp.close(); full.close(); pool.close()


def test_step_envs_refusals():
    import ctypes as C
    import torch
    from nmmo_b200.lib import Simulator
    from util import SMALL, build_world
    world = build_world(task_dim=64, **SMALL, NC_HORIZON=60)
    E = 6
    sim = Simulator(*world[:2], E, *world[2:])
    sim.reset(np.arange(E) + 1)
    buf = torch.zeros(E * sim.P * 12 + 4, dtype=torch.int32, device="cuda")
    st = sim._stream()
    call = lambda lo, hi, ptr: sim.L.nmmo_step_envs(sim.h, lo, hi, C.c_void_p(ptr), st)  # noqa: E731
    for lo, hi in [(0, 0), (3, 3), (4, 2), (-1, 2), (0, E + 1), (E, E + 1)]:
        assert call(lo, hi, buf.data_ptr()) == NM_ERR_ARG, (lo, hi)
    assert call(0, 2, buf.data_ptr() + 4) == NM_ERR_ARG, "misaligned actions"
    assert call(0, 2, 0) == NM_ERR_ARG, "null actions"
    sim.timing(True)
    assert call(0, 2, buf.data_ptr()) == NM_ERR_STATE
    sim.timing(False)
    sim.profile(True)
    assert call(0, 2, buf.data_ptr()) == NM_ERR_STATE
    sim.profile(False)
    assert call(0, 2, buf.data_ptr()) == 0
    with pytest.raises(ValueError):
        sim.step_envs(0, 2, buf[: sim.P * 12].view(1, sim.P, 12))
    torch.cuda.synchronize()
    sim.close()
