"""GPU: saving environments to device blobs and loading them into any slot of any compatible handle (DESIGN.md 2.3).

A loaded env must be byte for byte the env that was saved: its records, outputs, infos, episode flag, tables and task
state right after the load, and everything it produces afterwards under the same actions.  Every engine draw is keyed
by the env's own seed, so this holds in another slot, under another env_base, with three or four envs per CTA and with
the generic kernels in place of the std ones; the CPU oracle checks the other-handle case independently.
"""
import numpy as np
import pytest

from util import SMALL, build_world

pytestmark = pytest.mark.gpu

OUTS = ("obs", "rewards", "terminated", "truncated", "mask", "info", "info_valid")


def _small(agent="takeru", horizon=60, **over):
    return build_world(agent=agent, task_dim=64, **SMALL, NC_HORIZON=horizon, NC_RES_DEPLETION=1, **over)


def _sim(w, E, env_base=0):
    from nmmo_b200.lib import Simulator
    return Simulator(*w[:2], E, *w[2:], env_base=env_base)


def _outputs(sim, envs=None):
    """Device copies of every per-agent output of envs `envs` (default all), the autosample rows and episode_done,
    as uint8 views (byte equality)."""
    import torch
    envs = list(range(sim.E)) if envs is None else list(envs)
    idx = torch.as_tensor(envs, device=sim.obs.device)
    out = {}
    for name in OUTS:
        x = getattr(sim, name).view(sim.E, sim.P, -1)[idx]
        out[name] = x.contiguous().view(torch.uint8).clone()
    out["actions"] = sim.actions[idx].view(torch.uint8).clone()
    out["episode_done"] = sim.episode_done[idx].clone()
    return out


def _state(sim, envs):
    return [(sim.snapshot(e), sim.task_state(e)) for e in envs]


def _assert_outputs(a, b, tag, skip=()):
    import torch
    torch.cuda.synchronize()
    for k in a:
        if k not in skip:
            assert torch.equal(a[k], b[k]), f"{tag}: {k} differ"


def _assert_state(a, b, tag):
    for e, ((sa, ta), (sb, tb)) in enumerate(zip(a, b)):
        for x, y in zip(sa, sb):
            assert np.array_equal(x, y), f"{tag} env #{e}: snapshot tables differ"
        for x, y in zip(ta, tb):
            assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), f"{tag} env #{e}: task state differs"


def _assert_same_blobs(sim, x, y):
    """Blobs of equal small-family states: byte-equal but for the order of the depleted-tile list, which the step kernel
    fills with atomics and keeps unordered (the order changes nothing the env does)."""
    from nmmo_b200.config import SPEC
    a16 = lambda n: (n + 15) & ~15
    off = 128 + 64 + 16 + 16 + a16(SPEC["EA_N"] * (sim.P + sim.N) * 2) + SPEC["IS_N"] * a16(sim.cap * 2) + a16(sim.S * sim.S // 2)
    x, y = x.cpu().numpy(), y.cpu().numpy()
    out = np.ones(x.shape[1], bool)
    out[off:off + 2048] = False
    assert np.array_equal(x[:, out], y[:, out]), "blobs differ outside the depleted-tile list"
    for bx, by in zip(x, y):
        n = int(bx[128:192].view(np.int32)[12])
        assert n == int(by[128:192].view(np.int32)[12])
        dx, dy = bx[off:off + 2048].view(np.uint16), by[off:off + 2048].view(np.uint16)
        assert np.array_equal(np.sort(dx[:max(n, 0)]), np.sort(dy[:max(n, 0)])), "depleted tiles differ"
        assert not dx[max(n, 0):].any() and not dy[max(n, 0):].any()


def _sampled(sim, seed):
    import torch
    buf = torch.zeros_like(sim.actions)
    sim.sample_actions(seed, out=buf)
    return buf


def _round_trip(w, full=False, E=7, seed=5, warm=25, ahead=80):
    import torch
    sim = _sim(w, E)
    sim.set_obs_full(full)
    sim.set_autosample(seed)
    sim.reset(np.arange(E) + 11)
    for _ in range(warm):
        sim.step(sim.actions)
    blobs = sim.save_envs(range(E))
    part = sim.save_envs([5, 1, 3])
    torch.cuda.synchronize()
    assert torch.equal(part, blobs[[5, 1, 3]]), "blobs of equal states differ"
    o0, s0 = _outputs(sim), _state(sim, range(E))
    sums0, counts0, counters0 = sim.stats()
    acts, outs, states = [], [], {}
    for t in range(ahead):
        acts.append(sim.actions.clone())
        sim.step(acts[-1])
        outs.append(_outputs(sim))
        if t % 16 == 15:
            states[t] = _state(sim, range(E))
    sums1, counts1, counters1 = sim.stats()
    assert counters1[2] > counters0[2], "no episode reset between the save and the load"
    sim.load_envs(range(E), blobs)
    _assert_outputs(o0, _outputs(sim), "after load")
    _assert_state(s0, _state(sim, range(E)), "after load")
    assert torch.equal(_sampled(sim, seed), sim.actions), "autosample rows differ from sample_actions"
    sums2, counts2, counters2 = sim.stats()
    assert np.array_equal(counters2[:3], counters1[:3]) and np.array_equal(sums2, sums1) and np.array_equal(counts2, counts1)
    again = sim.save_envs(range(E))
    torch.cuda.synchronize()
    assert torch.equal(again, blobs), "a save right after the load does not return the loaded blobs"
    for t in range(ahead):
        sim.step(acts[t])
        _assert_outputs(outs[t], _outputs(sim), f"replay tick {t}", skip=("actions",))
        if t in states:
            _assert_state(states[t], _state(sim, range(E)), f"replay tick {t}")
    # a permuted subset, saved at the same tick, into the same slots
    sim.load_envs([5, 1, 3], part)
    got = _outputs(sim, [5, 1, 3])
    _assert_outputs(_outputs_sel(o0, [5, 1, 3]), got, "subset load")
    _assert_state([s0[5], s0[1], s0[3]], _state(sim, [5, 1, 3]), "subset load")
    sim.close()


def _outputs_sel(o, envs):
    return {k: v[list(envs)] for k, v in o.items()}


@pytest.mark.parametrize("full", [0, 1])
@pytest.mark.parametrize("agent", ["takeru", "neurips23_start_kit", "yaofeng"])
def test_round_trip_in_place(agent, full):
    _round_trip(_small(agent), full=bool(full))


def test_round_trip_big_family(monkeypatch):
    monkeypatch.setenv("NMMO_B200_FORCE_BIG", "1")
    _round_trip(_small())


def _oracle_check(sim, e, o, tag, state):
    import torch
    torch.cuda.synchronize()
    P = sim.P
    sl = slice(e * P, (e + 1) * P)
    assert np.array_equal(sim.obs[sl].cpu().numpy(), o.obs), f"{tag}: records differ"
    for name, ref in (("mask", o.mask), ("terminated", o.terminated), ("truncated", o.truncated), ("info_valid", o.info_valid)):
        assert np.array_equal(getattr(sim, name)[sl].cpu().numpy(), ref), f"{tag}: {name}"
    assert np.array_equal(sim.rewards[sl].cpu().numpy().view(np.uint32), o.rewards.view(np.uint32)), f"{tag}: rewards"
    assert bool(sim.episode_done[e]) == o.episode_done, f"{tag}: episode_done"
    v = o.info_valid.astype(bool)
    gi, oi = sim.info[sl].cpu().numpy()[v], o.info[v]
    assert ((gi == oi) | (np.isnan(gi) & np.isnan(oi))).all(), f"{tag}: info"
    if state:
        for x, y in zip(sim.snapshot(e)[:3], o.snapshot()):
            assert np.array_equal(x, y), f"{tag}: tables"


def test_other_handle_against_oracle(monkeypatch):
    import torch
    from oracle.oracle import OracleEnv
    w = _small()
    o = OracleEnv(*w)
    a = _sim(w, 1)
    assert a.kernel_names()[0] == "nmmo_step4_kernel"
    o.reset(77); a.reset([77])
    t0 = 30
    for t in range(t0):
        act = o.sample_actions(1000 + t)
        a.actions.copy_(torch.from_numpy(act)[None])
        a.step(a.actions); o.step(act)
    _oracle_check(a, 0, o, "handle A at t0", True)
    blob = a.save_envs([0]).cpu()
    a.close()
    monkeypatch.setenv("NMMO_B200_ENVS_PER_CTA", "3")
    b = _sim(w, 9, env_base=100)
    monkeypatch.delenv("NMMO_B200_ENVS_PER_CTA")
    assert b.kernel_names()[0] == "nmmo_step3_kernel"
    b.set_autosample(3)
    b.reset(np.arange(9) + 500)
    for _ in range(37):
        b.step(b.actions)
    b.load_envs([7], blob)
    done = 0
    for t in range(121):
        _oracle_check(b, 7, o, f"slot 7, {t} ticks after the load", t % 16 == 0)
        done += int(o.episode_done)
        if t == 120:
            break
        act = o.sample_actions(5000 + t)
        acts = b.actions.clone()
        acts[7] = torch.from_numpy(act)
        b.step(acts); o.step(act)
    assert done >= 1, "the loaded env never reached its automatic reset"
    b.close()


def test_branching():
    import torch
    w = _small()
    sim = _sim(w, 6)
    sim.set_autosample(9)
    sim.reset(np.arange(6) + 21)
    for _ in range(20):
        sim.step(sim.actions)
    blob = sim.save_envs([2])
    clones = [0, 1, 3, 4]
    sim.load_envs(clones, blob.repeat(len(clones), 1))
    acts, outs, snaps = [], [], {}
    for t in range(40):
        a = sim.actions.clone()
        if t < 10:                           # identical actions first (the built-in policy's rows differ by slot) ...
            a[clones] = a[0].clone()
        acts.append(a)
        sim.step(a)
        outs.append(_outputs(sim))
        if t < 10:
            for k in clones[1:]:
                for name, v in outs[-1].items():
                    if name != "actions":
                        assert torch.equal(v[k], v[0]), f"tick {t}: clone {k} {name} differs from clone 0 under the same actions"
        if t % 16 == 15:
            snaps[t] = {k: sim.snapshot(k) for k in clones}
    assert any(not torch.equal(outs[-1]["obs"][0], outs[-1]["obs"][k]) for k in clones[1:]), "the clones never diverged"
    # ... then each clone against a replay of the blob with its own actions, in a handle of its own
    for k in clones:
        r = _sim(w, 1)
        r.load_envs([0], blob)
        for t in range(40):
            r.step(acts[t][k][None].contiguous())
            _assert_outputs(_outputs_sel(outs[t], [k]), _outputs(r), f"clone {k} tick {t}", skip=("actions",))
            if t in snaps:
                for x, y in zip(snaps[t][k], r.snapshot(0)):
                    assert np.array_equal(x, y), f"clone {k} tick {t}: tables"
        r.close()
    sim.close()


def test_std_and_generic_share_the_format(monkeypatch):
    import torch
    w = build_world(NC_HORIZON=100)
    a = _sim(w, 5)
    assert a.kernel_names() == ("nmmo_step4_std_kernel", "nmmo_obs_std_kernel")
    monkeypatch.setenv("NMMO_B200_NO_STD_STEP", "1")
    monkeypatch.setenv("NMMO_B200_NO_STD_OBS", "1")
    b = _sim(w, 5)
    assert b.kernel_names() == ("nmmo_step4_kernel", "nmmo_obs_kernel")
    assert a.state_bytes == b.state_bytes
    for s in (a, b):
        s.set_autosample(4)
    a.reset(np.arange(5) + 1); b.reset(np.arange(5) + 40)
    for _ in range(20):
        a.step(a.actions); b.step(b.actions)
    b.load_envs(range(5), a.save_envs(range(5)))
    _assert_outputs(_outputs(a), _outputs(b), "after load")
    for t in range(60):
        act = a.actions.clone()
        a.step(act); b.step(act)
        _assert_outputs(_outputs(a), _outputs(b), f"tick {t}")
    _assert_state(_state(a, range(5)), _state(b, range(5)), "tick 60")
    _assert_same_blobs(a, a.save_envs(range(5)), b.save_envs(range(5)))
    a.close(); b.close()


def test_config5_big_std():
    from bench import world
    from nmmo_b200.config import SPEC
    big_std = ("nmmo_step_big_std_kernel", "nmmo_obs_big_std_kernel")
    cfg, fcfg, maps, tab, emb = world(workload="config5", n_maps=2)
    cfg = cfg.copy()
    cfg[SPEC["NC_HORIZON"]] = 40
    sim = _sim((cfg, fcfg, maps, tab, emb), 2)
    assert sim.kernel_names() == big_std
    sim.set_autosample(1)
    sim.reset([1, 2])
    for _ in range(20):
        sim.step(sim.actions)
    blobs = sim.save_envs([0, 1])
    o0, s0 = _outputs(sim), _state(sim, [0, 1])
    acts, outs = [], []
    for _ in range(30):
        acts.append(sim.actions.clone())
        sim.step(acts[-1])
        outs.append(_outputs(sim))
    sim.load_envs([1, 0], blobs[[1, 0]])
    _assert_outputs(o0, _outputs(sim), "after load")
    _assert_state(s0, _state(sim, [0, 1]), "after load")
    for t in range(30):
        sim.step(acts[t])
        _assert_outputs(outs[t], _outputs(sim), f"replay tick {t}", skip=("actions",))
    assert sim.kernel_names() == big_std
    sim.close()


def test_small_blob_into_big_handle_is_refused(monkeypatch):
    import torch
    from nmmo_b200.lib import NmmoError
    w = _small()
    a = _sim(w, 2)
    a.reset([1, 2])
    blob = a.save_envs([0])
    monkeypatch.setenv("NMMO_B200_FORCE_BIG", "1")
    b = _sim(w, 2)
    assert b.kernel_names()[1].startswith("nmmo_obs_big")
    b.reset([3, 4])
    before = _outputs(b)
    # the families' blobs differ in size (row-major entity table, wider depleted-tile list): the small blob, cut or
    # padded to the big size, keeps its header
    n = min(a.state_bytes, b.state_bytes)
    small = torch.zeros((1, b.state_bytes), dtype=torch.uint8, device=blob.device)
    small[:, :n] = blob[:, :n]
    with pytest.raises(NmmoError, match=r"error -1: .*small-family handle; this handle runs the big family"):
        b.load_envs([0], small)
    with pytest.raises(ValueError, match=f"states must be uint8 \\[1, {b.state_bytes}\\]"):
        b.load_envs([0], blob)
    _assert_outputs(before, _outputs(b), "after the refused load")
    a.close(); b.close()


def test_pool_save_and_load():
    from test_env_pool_gpu import _lock_tick, _pool_round, _pools, _same_outputs, _same_state, _small_env
    import torch
    E, b = 6, 2
    lock, pool = _pools(_small_env(), E, b, collect_infos=True)

    def entries(p, infos):
        return sorted((int(s), int(i["length"]), float(i["return"]), bool(i.get("episode_done", False)))
                      for s, i in zip(p.last_info_slots, infos))

    def lock_round():
        i = lock.recv()[4]
        got = entries(lock, i)
        lock.send(lock.sim.actions)
        return got

    def pool_round():
        got = []
        for _ in range(pool.num_batches):
            i = pool.recv()[4]
            got += entries(pool, i)
            lo, hi = pool.batch_env_range
            pool.send(pool.sim.actions[lo:hi])
        return sorted(got)

    for _ in range(20):
        lock_round(); pool_round()
    # pool: batch 0 (envs 0, 1) is in flight when envs 1 and 4 are saved; lock-step equivalent: env 4 before the tick,
    # env 1 after it
    pool.recv(); pool.send(pool.sim.actions[0:b])
    saved = pool.save_envs([1, 4])
    s4 = lock.save_envs([4])
    _lock_tick(lock)
    s1 = lock.save_envs([1])
    torch.cuda.synchronize()
    assert torch.equal(saved[0], s1[0]) and torch.equal(saved[1], s4[0]), "pool and lock-step saves differ"
    for _ in range(pool.num_batches - 1):
        pool.recv()
        lo, hi = pool.batch_env_range
        pool.send(pool.sim.actions[lo:hi])
    _same_outputs(lock, pool, "after the save")
    n_infos = 0
    for r in range(60):
        if r == 30:
            lock.load_envs([1, 4], saved.cpu()); pool.load_envs([1, 4], saved)
        a, p = lock_round(), pool_round()
        assert a == p, f"round {r}: infos differ"
        n_infos += len(a)
        _same_outputs(lock, pool, f"round {r}")
        if r % 10 == 0:
            _same_state(lock, pool, f"round {r}")
    assert n_infos > 0
    lock.close(); pool.close()


def test_refusals():
    import ctypes as C
    import torch
    from nmmo_b200.lib import NmmoError
    w = _small()
    sim = _sim(w, 4)
    sim.set_autosample(2)
    sim.reset([1, 2, 3, 4])
    for _ in range(10):
        sim.step(sim.actions)
    blob = sim.save_envs([0, 1])
    for _ in range(5):
        sim.step(sim.actions)
    other = _sim(_small(horizon=61), 1)
    other.reset([1])
    foreign = other.save_envs([0])
    assert other.state_bytes == sim.state_bytes
    other.close()
    before, sbefore = _outputs(sim), _state(sim, range(4))
    bad_magic = blob[:1].clone(); bad_magic[0, 0] ^= 1
    bad_version = blob[:1].clone(); bad_version[0, 4] += 1
    cases = [
        (lambda: sim.load_envs([], blob[:0]), "n must be at least 1"),
        (lambda: sim.load_envs([4], blob[:1]), "env id 4 out of range"),
        (lambda: sim.load_envs([-1], blob[:1]), "env id -1 out of range"),
        (lambda: sim.load_envs([2, 2], blob), "appears twice in a load"),
        (lambda: sim.load_envs([1], bad_magic), "bad magic"),
        (lambda: sim.load_envs([1], bad_version), "format version 2"),
        (lambda: sim.load_envs([0, 1], torch.cat([blob[:1], foreign])), "digest mismatch"),
        (lambda: sim.save_envs([4]), "env id 4 out of range"),
        (lambda: sim.save_envs([]), "n must be at least 1"),
    ]
    for fn, msg in cases:
        with pytest.raises(NmmoError, match=f"error -1: .*{msg}"):
            fn()
    # a misaligned device pointer, through the C ABI
    buf = torch.zeros(sim.state_bytes + 16, dtype=torch.uint8, device=blob.device)
    buf[1:1 + sim.state_bytes] = blob[0]
    ids = np.array([1], np.int32)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert sim.L.nmmo_load_envs(sim.h, ids.ctypes.data_as(C.c_void_p), 1, C.c_void_p(buf.data_ptr() + 1), stream) == -1
    assert b"16-byte aligned" in sim.L.nmmo_last_error()
    assert sim.L.nmmo_save_envs(sim.h, ids.ctypes.data_as(C.c_void_p), 1, C.c_void_p(buf.data_ptr() + 1), stream) == -1
    for on, off in ((lambda: sim.timing(True), lambda: sim.timing(False)), (lambda: sim.profile(True), lambda: sim.profile(False))):
        on()
        with pytest.raises(NmmoError, match="error -4: "):
            sim.load_envs([1], blob[:1])
        off()
    _assert_outputs(before, _outputs(sim), "after the refusals")
    _assert_state(sbefore, _state(sim, range(4)), "after the refusals")
    sim.load_envs([3, 0], blob)            # and the handle still loads
    sim.close()
