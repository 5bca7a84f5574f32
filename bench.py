#!/usr/bin/env python
"""bench.py -- throughput of the batched Neural MMO step on B200 (BASELINE.json metric).

One "step" = one lock-step tick of every environment on the GPU: the step kernel (Realm.step +
reward/stat wrapper) and the observation kernel, which also draws the next uniform-random valid
actions from the ActionTargets masks it has just built (BASELINE.json config 2).  Workload at N=1:
configs[1] -- 4096 envs x 128 agents, full NeurIPS23 config with the takeru overrides, from
reset with auto-reset on episode end.  N>1: the same per-GPU workload on every rank (envs
sharded by global index, no collective in the step; one NCCL all-reduce of the episode-stat
vector after the timed region), reported as weak scaling.

  python bench.py --gpus 1 --steps 256 --warmup 16
  python -m torch.distributed.run --nproc-per-node 8 ... bench.py --gpus 8 ...
  python bench.py --impl reference        # the CPU restatement (oracle/) on the host cores

`value` is agent-slot-steps/s (E*128 slots per tick, the reference's `global_step` accounting,
reinforcement_learning/clean_pufferl.py:307); `alive_agent_steps_per_s` is the `sum(mask)`
accounting (:306).  Both are whole-job numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

from nmmo_b200.config import SPEC, ObsLayout, make_config  # noqa: E402
from nmmo_b200.mapgen import generate_maps  # noqa: E402
from nmmo_b200.tasks import default_curriculum, make_task_table  # noqa: E402

METRIC = "agent_steps_per_sec"
UNIT = "agent-slot-steps/s"


NOMINAL_HBM_GBS = 8000.0      # BASELINE.json north_star: "~8 TB/s peak"; reported beside the measured copy peak

WORKLOADS = {
    # BASELINE.json configs[1] (SURVEY.md 8(d) config 2): the configuration the metric is quoted on
    "config2": dict(envs=4096, engine={}, env={},
                    what="configs[1]: {E} lockstep envs x {P} agents per GPU, NeurIPS23 config + takeru overrides, "
                         "synthetic seeded maps, uniform-random valid actions, from reset with auto-reset"),
    # BASELINE.json configs[4] (SURVEY.md 8(d) config 5): 1024 agents per env, NPC_N x8, map centre 512, every agent
    # spawned inside a 32x32 patch, Move chosen with p = 0.9 (collision-heavy); the big kernel family
    "config5": dict(envs=512, engine=dict(NC_SPAWN_PATCH=32, NC_SAMPLE_MOVE_PCT=90),
                    env=dict(num_agents=1024, num_npcs=2048, map_size=512),
                    what="configs[4] stress: {E} lockstep envs x {P} agents per GPU (NPC_N 2048, 544^2 map), clustered "
                         "spawn in a 32x32 patch, Move-biased uniform-random valid actions (p = 0.9), from reset"),
}


def world(agent="takeru", n_maps=None, workload="config2"):
    from nmmo_b200.config import default_env_args, default_wrapper_args
    wl = WORKLOADS[workload]
    env_args = default_env_args(resilient_population=0 if agent in ("takeru", "yaofeng", "hybrid") else 0.2, **wl["env"])
    cfg, fcfg = make_config(env_args, default_wrapper_args(agent), agent, **wl["engine"])
    # "fine" terrain: ponds and groves every ~10 tiles (nmmo_b200/mapgen.py), so that a foraging population can survive
    maps = generate_maps(cfg, 2023, n_maps or (64 if workload == "config2" else 8), terrain="fine")
    tab, emb = make_task_table(default_curriculum(), int(cfg[SPEC["NC_TASK_DIM"]]), seed=3)
    return cfg, fcfg, maps, tab, emb


def committed_traffic(regime_keys):
    """DRAM traffic per launch of the two kernels from the newest committed `ncu --set full` capture whose regime
    matches the timed window (profiles/<tag>_traffic.json, written by tools/summarize_ncu.py).  -> (dict, source)"""
    for tf in sorted((ROOT / "profiles").glob("*_traffic.json"), reverse=True):
        try:
            tj = json.loads(tf.read_text())
        except Exception:  # noqa: BLE001
            continue
        for key in regime_keys:
            found = {k.split(":", 1)[1]: v.get("dram_bytes") for k, v in tj.items() if k.startswith(key + ":")}
            if found:
                return found, f"profiles/{tf.name} capture '{key}' (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)"
    return {}, None


def alg_bytes_per_slot(cfg):
    """Algorithmic bytes of one agent slot-step (DESIGN.md section 4, SURVEY.md 8d):
    dense obs record + actions in + reward/term/trunc/mask out + read and write of the agent's
    own entity row and inventory rows."""
    L = ObsLayout(cfg)
    state = 31 * 2 + 12 * 16 * 2
    return L.alg_bytes + 12 * 4 + (4 + 1 + 1 + 1) + 2 * state, L.alg_bytes


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  NVML is polled in a thread that is already
    running when the region starts (a 33 ms window still gets samples); `nvidia-smi -lms` is the fallback."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:  # noqa: BLE001
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class NvmlSampler(ClockSampler):
    def __init__(self, index: int):
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = "GPU-" + str(torch.cuda.get_device_properties(index).uuid)
            self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
        except Exception:  # noqa: BLE001
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        self.samples = []          # (host time, sm MHz, reasons bitmask, power W)
        self.t0 = self.t1 = None
        self._run = True
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()       # polling starts now, before the warm-up

    def _poll(self):
        nv = self.nv
        while self._run:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.samples.append((time.perf_counter(), sm, rs, pw))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        self.t0 = time.perf_counter()

    def stop(self):
        self.t1 = time.perf_counter()
        time.sleep(0.005)
        self._run = False
        nv = self.nv
        inside = [x for x in self.samples if self.t0 <= x[0] <= self.t1]
        if not inside and self.samples:      # window shorter than one poll: the nearest sample
            inside = [min(self.samples, key=lambda x: abs(x[0] - 0.5 * (self.t0 + self.t1)))]
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(n for n, bit in names.items() if any(x[2] & bit for x in inside))
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception:  # noqa: BLE001
            mx = None
        sm = [x[1] for x in inside]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm),
                "power_w_max": max((x[3] for x in inside), default=None), "source": "NVML polled every ~2 ms, samples inside the timed region"}


def make_clock_sampler(index: int):
    try:
        return NvmlSampler(index)
    except Exception:  # noqa: BLE001
        return ClockSampler(index)


def ref_envs_default(requested: int, P: int, stride: int) -> int:
    """Envs of the CPU arm: the GPU arm's count when the host has the memory for that many oracle envs
    (each holds its own observation records), else as many as fit in a quarter of the free RAM."""
    try:
        import psutil
        free = psutil.virtual_memory().available
    except Exception:  # noqa: BLE001
        free = 16 << 30
    per_env = P * (stride + 4096) + (4 << 20)
    return int(max(16, min(requested, (free // 4) // per_env)))


def cpu_leg(w, n_envs, ticks, warmup=4, seed=1):
    """The CPU restatement (oracle/, OpenMP over envs) on the host cores."""
    from oracle.oracle import OracleBatch
    cores = len(os.sched_getaffinity(0))
    b = OracleBatch(*w, n_envs=n_envs, threads=cores)
    b.reset(np.arange(n_envs) + seed)
    for _ in range(warmup):
        b.sample(seed); b.step()
    alive = 0
    t0 = time.perf_counter()
    for _ in range(ticks):
        b.sample(seed)
        b.step()
        alive += b.alive()
    dt = time.perf_counter() - t0
    P = b.P
    return {"value": n_envs * P * ticks / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_envs} envs x {P} agents x {ticks} ticks from reset (after {warmup} warm-up ticks), "
                      f"C restatement oracle/nmmo_oracle.c, OpenMP {cores} threads",
            "alive_agent_steps_per_s": alive / dt, "seconds": dt}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = world(args.agent, workload=args.workload)
    cores = len(os.sched_getaffinity(0))
    P = int(w[0][SPEC["NC_N_PLAYERS"]])
    gpu_envs = args.envs or WORKLOADS[args.workload]["envs"]
    n_envs = args.ref_envs or ref_envs_default(gpu_envs, P, ObsLayout(w[0]).stride)
    res = cpu_leg(w, n_envs, args.steps, warmup=args.warmup)
    ms = res["seconds"] / args.steps * 1e3
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload]["what"].format(E=n_envs, P=P) + " -- CPU arm: oracle/nmmo_oracle.c (kind: port; the nmmo engine "
                                   "is not installable here), all host cores, one env per OpenMP task",
                       "envs": n_envs, "agents_per_env": P, "same_envs_as_gpu_arm": n_envs == gpu_envs},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "alive_agent_steps_per_s": res["alive_agent_steps_per_s"],
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def dump_outputs(sim, out_dir):
    """Write what a caller of the device-resident step holds after the last timed tick, as float32 .npy files under
    `out_dir` (at most about 45 MB, whatever the size): the per-agent vectors, and the observation records (raw
    bytes), episode infos and next built-in-policy actions, each for a fixed seeded sample of agent slots (all slots
    for the per-agent vectors up to 2^19 of them).  The sampled slots are written beside them as float64 index arrays,
    so that two builds can be compared output for output."""
    import torch
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    n = sim.E * sim.P
    perm = np.random.default_rng(0).permutation(n)
    slots = {"slots": np.sort(perm[:1 << 19]), "wide_slots": np.sort(perm[:1 << 14]), "obs_slots": np.sort(perm[:256])}
    idx = {k: torch.from_numpy(v).to(sim.obs.device) for k, v in slots.items()}
    arrays = {"rewards": sim.rewards[idx["slots"]], "terminated": sim.terminated[idx["slots"]],
              "truncated": sim.truncated[idx["slots"]], "mask": sim.mask[idx["slots"]],
              "info_valid": sim.info_valid[idx["slots"]], "episode_done": sim.episode_done,
              "info": sim.info[idx["wide_slots"]], "actions": sim.actions.view(n, 12)[idx["wide_slots"]],
              "obs": sim.obs[idx["obs_slots"]]}
    # the max-level columns of an episode info are NaN where the key is absent; levels are >= 0, so the dump, whose
    # arrays are all finite, writes -1 there instead
    levels = slice(SPEC["IN_MAXLVL_ARMOR"], SPEC["IN_MAXLVL_CONSUMABLE"] + 1)
    arrays["info"][:, levels] = torch.nan_to_num(arrays["info"][:, levels], nan=-1.0)
    for name, t in arrays.items():
        np.save(out / f"{name}.npy", t.cpu().numpy().astype(np.float32))
    for name, v in slots.items():
        np.save(out / f"{name}.npy", v.astype(np.float64))


def run_native(args):
    import torch
    import torch.distributed as dist
    from nmmo_b200.lib import Simulator, pack_actions_u8

    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    if world_size > 1:
        # NCCL writes its version banner to stdout when the communicator is created; stdout carries exactly one
        # JSON line, so the communicator is created (init + one barrier) with fd 1 pointed at stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    w = world(args.agent, workload=args.workload)
    cfg = w[0]
    E, P = args.envs or WORKLOADS[args.workload]["envs"], int(cfg[SPEC["NC_N_PLAYERS"]])
    clocks = make_clock_sampler(local_rank)      # NVML polling runs from here on, through the warm-up
    sim = Simulator(*w[:2], E, *w[2:], device=local_rank, env_base=rank * E)
    kernel_names = sim.kernel_names()
    seeds = np.arange(E, dtype=np.uint64) + np.uint64(rank * E + args.seed)
    stream = torch.cuda.current_stream()

    # built-in random policy: the observation kernel writes next tick's uniform-random valid
    # actions itself (same draws as the stand-alone sampler kernel, tests/test_parity_gpu.py)
    sim.set_autosample(args.seed, sim.actions)

    def tick(seed):
        sim.step()

    def barrier():
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
            torch.cuda.synchronize()

    n_slots_step = E * P
    # spin-up: a throw-away stretch of ticks so that the first launches of a fresh process (module load, clock ramp) are
    # not inside anything that is timed; the run then restarts from the reset the window is defined from
    sim.reset(seeds)
    for _ in range(48):
        tick(args.seed)
    torch.cuda.synchronize()
    sim.reset(seeds)
    for _ in range(args.warmup):
        tick(args.seed)
    sim.stats(clear=True)
    # ---- device-resident timed region ---------------------------------------------------
    sim.timing(True)
    barrier()
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        tick(args.seed)
    e1.record(stream)
    barrier()
    clk = clocks.stop()
    ms_total = e0.elapsed_time(e1)
    step_ms, obs_ms, n_timed = sim.timing_read()
    sim.timing(False)
    sums, counts, counters = sim.stats(clear=False)
    if args.dump_outputs and rank == 0:          # rank 0's envs only: one dump within the size bound at any world size
        dump_outputs(sim, args.dump_outputs)
    # ---- survival leg (SURVEY.md 8d "run 1024 ticks from reset so the alive-fraction decay is included"): a whole
    # episode under the scripted forager policy (nmmo_forage_actions: walk to water / foliage when hungry), whose
    # population decays like the published trained-policy runs (BASELINE.md 2: alive 0.83 / 0.53 / 0.25 / 0.13 at ticks
    # 32 / 128 / 512 / 1023, time average 0.31) instead of starving by tick ~35 like uniform-random agents do.
    steady = None
    if args.steady_steps > 0:
        horizon = int(cfg[SPEC["NC_HORIZON"]])
        n_ticks = min(args.steady_steps, horizon - 1)
        sim.set_autosample(0, enable=False)
        sim.reset(seeds)
        sim.stats(clear=True)
        marks = {t: None for t in (32, 128, 512, n_ticks - 1) if t < n_ticks}
        sim.timing(True)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(8)]
        g0.record(stream)
        for t in range(n_ticks):
            if t < 8:
                f_ev[t][0].record(stream)
            sim.forage_actions(args.seed)
            if t < 8:
                f_ev[t][1].record(stream)
            sim.step()
            if t in marks:
                marks[t] = sim.mask.sum(dtype=torch.int64)           # stays on the device until the end
        g1.record(stream)
        torch.cuda.synchronize()
        s_step_ms, s_obs_ms, _ = sim.timing_read()
        sim.timing(False)
        _, _, c1 = sim.stats(clear=False)
        ms_s = g0.elapsed_time(g1)
        steady = {"policy": "scripted forager (nmmo_forage_actions), no fighting or trading", "ticks": n_ticks,
                  "ms_per_step": ms_s / n_ticks, "kernels_ms": {"step_kernel": s_step_ms, "obs_kernel": s_obs_ms,
                                                                 "forager_policy_kernel_first_ticks": sum(a.elapsed_time(b) for a, b in f_ev) / len(f_ev)},
                  "value_per_gpu": n_slots_step * n_ticks / (ms_s * 1e-3),
                  "alive_agent_steps_per_s_per_gpu": float(c1[1]) / (ms_s * 1e-3),
                  "alive_fraction": float(c1[1]) / max(1.0, float(c1[0])),
                  "alive_fraction_at_tick": {str(t): float(v.item()) / n_slots_step for t, v in marks.items() if v is not None},
                  "episodes_finished": float(c1[2]),
                  "what": f"one episode from reset, {n_ticks} ticks, every env in lock-step; the policy kernel's time is inside ms_per_step"}
        sim.set_autosample(args.seed, sim.actions)
        sim.reset(seeds)
        sim.stats(clear=True)
    # ---- dense-writer reference point: every byte of every record rewritten each tick ----
    sim.set_obs_full(True)
    for _ in range(2):
        tick(args.seed)
    sim.timing(True)
    for _ in range(8):
        tick(args.seed)
    _, obs_ms_dense, _ = sim.timing_read()
    sim.timing(False)
    sim.set_obs_full(False)
    tick(args.seed)
    # ---- end-to-end through the host-buffer C ABI call ----------------------------------
    # The caller's inputs (actions) start in pinned HOST memory and its results (reward, terminated, truncated,
    # mask) end there, every step, through nmmo_step_host.  To feed it the very actions of the device-resident run,
    # the run is replayed twice from the same reset (it is deterministic): pass A tapes the actions of the last
    # `e2e_steps` ticks of the window into pinned memory (untimed); pass B advances to the same tick on the device
    # and then takes the timed host-buffer steps from the tape.  The built-in policy stays on during pass B (writing
    # to a scratch tensor) so the kernels do the same work as in the device-timed region.
    n = E * P
    e2e_steps = max(4, min(args.steps, 32))
    e2e_warm = 3                                           # untimed host-buffer steps (first-use costs: pinned result buffers)
    pre = max(0, args.warmup + args.steps - e2e_steps - e2e_warm)
    tape = torch.empty((e2e_warm + e2e_steps, E, P, 12), dtype=torch.uint8).pin_memory()      # 12 bytes per agent: nmmo_step_host_u8
    sim.set_autosample(args.seed, sim.actions)
    sim.reset(seeds)
    # (the first ticks after a reset, when nearly every agent is still alive, are timed on the way: this is the
    #  regime a trained policy keeps the simulator in, and the most expensive one per tick)
    early_n = min(24, pre)
    _, _, c0 = sim.stats(clear=False)
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record(stream)
    for _ in range(early_n):
        tick(args.seed)
    h1.record(stream)
    torch.cuda.synchronize()
    _, _, c1 = sim.stats(clear=False)
    ms_early = h0.elapsed_time(h1)
    early = {"ticks": early_n, "ms_per_step": ms_early / max(1, early_n),
             "alive_fraction": float(c1[1] - c0[1]) / max(1.0, float(c1[0] - c0[0])),
             "alive_agent_steps_per_s_per_gpu": float(c1[1] - c0[1]) / max(1e-9, ms_early * 1e-3),
             "what": "the first ticks after reset (nearly all agents alive)"} if early_n > 0 else None
    for _ in range(pre - early_n):
        tick(args.seed)
    for k in range(e2e_warm + e2e_steps):
        tape[k].copy_(pack_actions_u8(sim.actions))      # packed on the device, like a GPU policy would
        tick(args.seed)
    torch.cuda.synchronize()
    sim.reset(seeds)
    for _ in range(pre):
        tick(args.seed)
    scratch = torch.zeros_like(sim.actions)
    torch.cuda.synchronize()
    sim.set_autosample(args.seed, scratch)
    tape_np = tape.numpy()
    for k in range(e2e_warm):
        sim.step_host(tape_np[k])
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(stream)
    for k in range(e2e_warm, e2e_warm + e2e_steps):
        sim.step_host(tape_np[k])                        # H2D actions, step, D2H reward/term/trunc/mask
    f1.record(stream)
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    h2d = n * 12
    d2h = n * (4 + 3)
    # ---- reduce over ranks --------------------------------------------------------------
    t = torch.tensor([ms_total, ms_e2e, step_ms, obs_ms, obs_ms_dense], dtype=torch.float64, device="cuda")
    agg = torch.tensor(np.concatenate([sums, counts, counters.astype(np.float64)]), dtype=torch.float64, device="cuda")
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)       # the only collective: episode stats
    ms_total, ms_e2e, step_ms, obs_ms, obs_ms_dense = t.tolist()
    agg = agg.cpu().numpy()
    IN = SPEC["IN_N"]
    g_sums, g_counts, g_counters = agg[:IN], agg[IN:2 * IN], agg[2 * IN:]
    if rank == 0:
        b_alg, b_obs = alg_bytes_per_slot(cfg)
        total_slots = world_size * n * args.steps
        value = total_slots / (ms_total * 1e-3)
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:  # noqa: BLE001
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        # bytes the observation kernel has to move per launch: the env state it reads plus the record
        # bytes that can differ from the record already in HBM, counted by the kernel itself
        obs_bytes_launch = float(g_counters[4]) / max(1, world_size * args.steps)
        # DRAM traffic of the same kernels from the committed ncu --set full captures (profiles/<tag>_traffic.json,
        # written by tools/summarize_ncu.py from the .ncu-rep of tools/ncu_round.sh); null when none is committed
        alive_frac = float(g_counters[1]) / max(1.0, float(g_counters[0]))
        big = args.workload == "config5"
        k_step, k_obs = kernel_names
        # captures are labelled by regime: "alive" = tick 12 of the driver's window (every agent alive), "tick40" = the
        # mostly-dead regime of long random-action runs, "c5" = config 5; only a capture of the window's regime is quoted
        regime = ["c5"] if big else (["alive"] if alive_frac > 0.8 else ["tick40"])
        tr, traffic_src = committed_traffic(regime)
        traffic = tr.get(k_obs)          # only a capture of the very kernel instantiation that was timed is quoted
        traffic_dense = committed_traffic(["dense"])[0].get(k_obs) if not big else None
        obs_gbs = obs_bytes_launch / (obs_ms * 1e-3) / 1e9
        dense_gbs = n * b_obs / (obs_ms_dense * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload]["what"].format(E=E, P=P),
                       "envs_per_gpu": E, "agents_per_env": P, "npcs_per_env": int(cfg[SPEC["NC_N_NPCS"]]),
                       "obs_record_bytes": int(sim.stride), "sharding": f"env-index x{world_size}",
                       "l2": "inputs larger than L2: the working set per tick (13 GB of obs records, 0.2-0.4 GB of env state) exceeds the 126 MB L2"},
            "alive_agent_steps_per_s": float(g_counters[1]) / (ms_total * 1e-3),
            "alive_fraction": alive_frac,
            "kernels_ms": {"step_kernel": step_ms, "obs_kernel": obs_ms, "launches_timed": n_timed},
            "roofline": None, "roofline_obs_kernel": {"bound": "hbm", "kernel": k_obs, "achieved": obs_gbs, "peak": peak, "unit": "GB/s",
                         "frac": obs_gbs / peak, "peak_nominal": NOMINAL_HBM_GBS, "frac_nominal": obs_gbs / NOMINAL_HBM_GBS,
                         "traffic": traffic, "traffic_source": traffic_src, "traffic_regime": regime[0], "peak_source": peak_src,
                         "alg_bytes_per_launch": obs_bytes_launch,
                         "note": "incremental writer: algorithmic bytes = env state read + record bytes that changed (counted in-kernel)",
                         "dense_mode": {"achieved": dense_gbs, "frac": dense_gbs / peak, "frac_nominal": dense_gbs / NOMINAL_HBM_GBS, "ms": obs_ms_dense,
                                        "alg_bytes_per_launch": n * b_obs, "traffic": traffic_dense,
                                        "what": "same kernel with obs_full=1: all 25 KB of all records rewritten every tick"},
                         "dense_equivalent_gbs": n * b_obs / (obs_ms * 1e-3) / 1e9},
            "e2e": {"value": world_size * n * e2e_steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "path": "nmmo_step_host_u8 (C ABI): one byte per action head from pinned host memory in, reward/term/trunc/mask to pinned host memory out, every "
                            "step; observations stay on the device where the policy reads them; actions = tape of the device-resident run"},
            "survival_episode": steady, "early_window": early,
            "gpu_launches": 2 * args.steps,
            "clocks": clk,
            "episode_stats": {"finished_agents": float(g_counts[SPEC["IN_LENGTH"]]),
                              "mean_length": float(g_sums[SPEC["IN_LENGTH"]] / max(1.0, g_counts[SPEC["IN_LENGTH"]])),
                              "episodes": float(g_counters[2]), "event_ring_overflows": float(g_counters[3])},
        }
        # the step kernel: algorithmic bytes = the env tables in and out (entity table, 4-bit map; the item prefix
        # is a few hundred bytes) + actions in + reward/term/trunc/mask out.  It is latency / instruction-issue
        # bound, not bandwidth bound (DESIGN.md 4.1); the fraction is reported as it is.
        R_ = P + int(cfg[SPEC["NC_N_NPCS"]]); S_ = int(cfg[SPEC["NC_MAP_SIZE"]])
        step_alg = E * (2 * (SPEC["EA_N"] * R_ * 2 + S_ * S_ // 2) + P * 12 * 4 + P * 7)
        step_gbs = step_alg / (step_ms * 1e-3) / 1e9
        traffic_step = tr.get(k_step)
        line["roofline_step_kernel"] = {"bound": "hbm", "kernel": k_step, "achieved": step_gbs, "peak": peak, "unit": "GB/s",
                                        "frac": step_gbs / peak, "peak_nominal": NOMINAL_HBM_GBS, "frac_nominal": step_gbs / NOMINAL_HBM_GBS,
                                        "traffic": traffic_step, "traffic_source": traffic_src, "traffic_regime": regime[0],
                                        "peak_source": peak_src, "alg_bytes_per_launch": step_alg,
                                        "note": "per-env critical path bound by instruction fetch and barrier latency "
                                                "(DESIGN.md 4.1: 2.0 M instruction-line requests per launch), not by bandwidth"}
        dominant = "roofline_step_kernel" if step_ms >= obs_ms else "roofline_obs_kernel"
        other = "roofline_obs_kernel" if dominant == "roofline_step_kernel" else "roofline_step_kernel"
        line["roofline"] = dict(line[dominant], dominant_by="mean launch duration in the timed region",
                                launch_ms={"step_kernel": step_ms, "obs_kernel": obs_ms},
                                other_kernel={"kernel": line[other]["kernel"], "frac": line[other]["frac"], "achieved": line[other]["achieved"],
                                              "see": other})
        if world_size == 1 and not args.no_cpu:
            cores = len(os.sched_getaffinity(0))
            ce = args.ref_envs or (min(1024, ref_envs_default(E, P, sim.stride)) if not big else 32)
            res = cpu_leg(w, n_envs=ce, ticks=min(args.steps, 64), warmup=min(args.warmup, 8))
            line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line))
    sim.close()
    if world_size > 1:
        dist.destroy_process_group()


def run_rollout(args):
    """`--what rollout`: the device rollout append and sort + GAE (SURVEY.md 8(f) rank 1) next to the CPU
    restatement of the reference's Python loop (clean_pufferl.py:329-348, :413-436).  One JSON line."""
    import torch
    from nmmo_b200.rollout import DeviceRollout
    from argparse import Namespace
    a = Namespace(batch=args.rollout_batch, envs=args.envs or 4096, agents=128, stride=25344, alive=0.5, reps=10, cpu_batch=32768)
    n = a.envs * a.agents
    dev = torch.device("cuda")
    g = torch.Generator(device=dev); g.manual_seed(1)
    obs = torch.randint(0, 256, (n, a.stride), dtype=torch.uint8, device=dev, generator=g)
    actions = torch.randint(0, 100, (n, 12), dtype=torch.int32, device=dev, generator=g)
    val = torch.randn(n, device=dev, generator=g); lp = -torch.rand(n, device=dev, generator=g)
    rew = torch.randn(n, device=dev, generator=g); done = (torch.rand(n, device=dev, generator=g) < 0.02).float()
    mask = (torch.rand(n, device=dev, generator=g) < a.alive).to(torch.uint8)
    r = DeviceRollout(a.batch, n, a.stride)
    # ---- append: one recv() fills (part of) the batch
    per_call = min(int(mask.sum().item()), a.batch + 1)
    for _ in range(2):
        r.reset(); r.store(obs, val, actions, lp, rew, done, mask, 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ms = 0.0
    for _ in range(a.reps):
        r.reset()
        e0.record(); r.store(obs, val, actions, lp, rew, done, mask, 1); e1.record()
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1)
    store_ms = ms / a.reps
    store_bytes = per_call * (2 * a.stride + 2 * (12 * 4 + 4 * 4)) + n * 2
    # ---- compact storage: Market once per (step, env), Task as the task id (a row is 8 960 of the 25 344 bytes)
    L = ObsLayout(make_config()[0])
    embed = torch.randn((128, L.task_dim), device=dev, generator=g).half()
    tid = torch.randint(0, 128, (n,), dtype=torch.int32, device=dev, generator=g)
    rc = DeviceRollout(a.batch, n, a.stride, compact=dict(agents_per_env=a.agents, market_off=L.o_market, market_bytes=L.n_mkt * 32,
                                                          task_off=L.o_task, task_bytes=L.task_dim * 2, ids_off=L.o_ids, max_steps=8,
                                                          task_embed_ptr=embed.data_ptr()))
    for _ in range(2):
        rc.reset(); rc.store(obs, val, actions, lp, rew, done, mask, 1, task_id=tid)
    torch.cuda.synchronize()
    ms = 0.0
    for _ in range(a.reps):
        rc.reset()
        e0.record(); rc.store(obs, val, actions, lp, rew, done, mask, 1, task_id=tid); e1.record()
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1)
    cstore_ms = ms / a.reps
    cstore_bytes = per_call * (2 * rc.row_stride + 2 * (12 * 4 + 4 * 4) + 8) + a.envs * 2 * L.n_mkt * 32 + n * 2
    mb = min(16384, per_call)
    pick = torch.randperm(per_call, device=dev, generator=g)[:mb].int()
    out = torch.empty((mb, a.stride), dtype=torch.uint8, device=dev)
    rc.expand(pick, out=out); torch.cuda.synchronize()
    ms = 0.0
    for _ in range(a.reps):
        e0.record(); rc.expand(pick, out=out); e1.record()
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1)
    expand_ms = ms / a.reps
    rc.close()
    # ---- sort + GAE over a full batch collected over several steps
    r.reset()
    step = 0
    while r.ptr < a.batch + 1 and step < 64:
        step += 1
        m = (torch.rand(n, device=dev, generator=g) < 0.2).to(torch.uint8)
        r.store(obs, val, actions, lp, rew, (torch.rand(n, device=dev, generator=g) < 0.02).float(), m, step)
    rows = r.ptr
    r.gae(0.99, 0.95)
    torch.cuda.synchronize()
    ms = 0.0
    for _ in range(a.reps):
        e0.record(); r.gae(0.99, 0.95); e1.record()
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1)
    gae_ms = ms / a.reps
    # ---- CPU restatement of the same loop (Python, like the reference) on a bounded sample
    from oracle.rollout_oracle import RolloutOracle
    cb = min(a.cpu_batch, rows - 1)
    o = RolloutOracle(cb, 16)
    o.rewards[:] = r.rewards[:cb + 1].cpu().numpy(); o.values[:] = r.values[:cb + 1].cpu().numpy(); o.dones[:] = r.dones[:cb + 1].cpu().numpy()
    slot = r.slot[:cb + 1].cpu().numpy(); st = r.step[:cb + 1].cpu().numpy()
    o.sort_keys = list(zip(slot.tolist(), st.tolist())); o.ptr = cb + 1
    t0 = time.perf_counter(); o.gae(0.99, 0.95); cpu_s = time.perf_counter() - t0
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    print(json.dumps({"what": "rollout storage + GAE on the device (clean_pufferl.py:329-348, :413-436)",
                      "n_slots": n, "obs_stride": a.stride, "batch_size": a.batch,
                      "append": {"rows_per_call": per_call, "ms": store_ms, "GB/s": store_bytes / store_ms / 1e6, "peak_GB/s": peak,
                                 "frac": store_bytes / store_ms / 1e6 / peak, "alg_bytes": store_bytes},
                      "append_compact": {"rows_per_call": per_call, "ms": cstore_ms, "row_bytes": a.stride - L.n_mkt * 32 - L.task_dim * 2,
                                         "GB/s": cstore_bytes / cstore_ms / 1e6, "frac": cstore_bytes / cstore_ms / 1e6 / peak, "alg_bytes": cstore_bytes,
                                         "batch_bytes_vs_plain": (per_call * (a.stride - L.n_mkt * 32 - L.task_dim * 2) + a.envs * L.n_mkt * 32) / (per_call * a.stride),
                                         "expand_minibatch": {"rows": mb, "ms": expand_ms, "GB/s": mb * 2 * a.stride / expand_ms / 1e6}},
                      "sort_gae": {"rows": rows, "ms": gae_ms, "samples_per_s": (rows - 1) / gae_ms * 1e3},
                      "cpu_port": {"rows": cb + 1, "seconds": cpu_s, "samples_per_s": cb / cpu_s, "kind": "port (Python loop, like the reference)"}}))
    r.close()



def run_config4(args):
    """`--what config4` (BASELINE.json configs[3]): the rollout loop of clean_pufferl.evaluate
    (/root/reference/reinforcement_learning/clean_pufferl.py:287-357) with the takeru policy, observations and masks
    consumed on the device (no host copy): recv -> policy forward -> rollout store -> send, 4096 envs x 128 agents.
    Reports the reference's own counters (:361-379): SPS (padded slots / elapsed), agent_SPS (sum(mask) / elapsed),
    env_sps (agent steps / env time), inference_sps (padded / inference time).  One JSON line."""
    import torch
    from nmmo_b200.rollout import DeviceRollout
    from nmmo_b200.takeru_policy import TakeruPolicy
    from nmmo_b200.vecenv import B200VecEnv
    torch.backends.cuda.matmul.allow_tf32 = bool(args.tf32)
    torch.backends.cudnn.allow_tf32 = bool(args.tf32)
    E = args.envs or 4096
    pool = B200VecEnv(num_envs=E, agent="takeru", collect_infos=False, curriculum="heldout")
    P = pool.agents_per_env
    n = E * P
    torch.manual_seed(args.seed)
    policy = TakeruPolicy(pool.driver_env.unflatten_context, 256, 256, 2048, agents_per_env=P, envs_per_chunk=args.policy_chunk_envs).cuda().eval()
    batch = min(args.rollout_batch, n)
    roll = DeviceRollout(batch, n, pool.driver_env.obs_sz, compact=DeviceRollout.compact_for(pool.sim, max_steps=4))
    clocks = make_clock_sampler(0)
    pool.async_reset(args.seed)
    gen = torch.Generator(device="cuda"); gen.manual_seed(args.seed)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    marks = []
    agent_steps = torch.zeros((), dtype=torch.int64, device="cuda")
    padded = 0

    def one_step(k, timed):
        nonlocal padded
        e = [ev() for _ in range(4)]
        o, r, d, t, i, env_id, mask = pool.recv()
        e[0].record()
        actions, logprob, value = policy(o, generator=gen)                     # inference (:317-319), on the records in HBM
        e[1].record()
        roll.reset()                                                           # (one recv fills the batch at this env count)
        roll.store(o, value, actions, logprob, r, d.float(), mask, k + 1, task_id=pool.sim.task_id)      # misc: the batch arrays (:333-348), device to device
        e[2].record()
        pool.send(actions)                                                     # env: step + observation kernels (:357, :293)
        e[3].record()
        if timed:
            marks.append(e)
            agent_steps.add_(mask.sum())
            padded += mask.numel()

    for k in range(args.warmup):
        one_step(k, False)
    torch.cuda.synchronize()
    clocks.start()
    t0, t1 = ev(), ev()
    t0.record()
    for k in range(args.steps):
        one_step(args.warmup + k, True)
    t1.record()
    torch.cuda.synchronize()
    clk = clocks.stop()
    total = t0.elapsed_time(t1) * 1e-3
    inf_t = sum(e[0].elapsed_time(e[1]) for e in marks) * 1e-3
    misc_t = sum(e[1].elapsed_time(e[2]) for e in marks) * 1e-3
    env_t = sum(e[2].elapsed_time(e[3]) for e in marks) * 1e-3
    a_steps = int(agent_steps.item())
    rec_bytes = n * pool.driver_env.obs_sz
    line = {"metric": "agent_SPS", "value": a_steps / total, "unit": "agent-steps/s (sum of mask, clean_pufferl.py:306,365)",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int16 env / fp32 policy" + (" (TF32 matmul)" if args.tf32 else ""), "data": "synthetic",
            "config": {"workload": f"configs[3]: clean_pufferl rollout loop with the takeru policy (ReducedModelV2 256/256, random init, no LSTM: "
                                   f"config.yaml:135-136), {E} envs x {P} agents, observations and masks read on the device, held-out task "
                                   f"curriculum with its real 2048-d embeddings, rollout batch {batch} rows stored on the device (compact: Market once per env-step, Task as id)",
                       "envs": E, "agents_per_env": P, "policy_chunk_envs": args.policy_chunk_envs, "obs_record_bytes": pool.driver_env.obs_sz},
            "SPS": padded / total, "agent_SPS": a_steps / total, "alive_fraction": a_steps / max(1, padded),
            "env_sps": a_steps / env_t, "env_sps_padded": padded / env_t, "inference_sps": padded / inf_t,
            "time_share": {"env": env_t / total, "inference": inf_t / total, "misc_rollout_store": misc_t / total},
            "ms": {"env": env_t / args.steps * 1e3, "inference": inf_t / args.steps * 1e3, "rollout_store": misc_t / args.steps * 1e3},
            "host_copies_per_step": 0, "obs_bytes_read_by_policy_per_step": rec_bytes,
            "gpu_launches": 2 * args.steps, "clocks": clk}
    print(json.dumps(line))
    pool.close(); roll.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--envs", type=int, default=0, help="environments per GPU (default: 4096 for config2, 512 for config5)")
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS), help="BASELINE.json configs[1] (default) or configs[4] (1024 agents per env)")
    ap.add_argument("--agent", default="takeru")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--ref-envs", type=int, default=0, help="envs of the CPU sample (default 4 x cores)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--what", default="step", choices=["step", "rollout", "config4"],
                    help="rollout = the device rollout storage / GAE micro-benchmark; config4 = rollout loop with the takeru policy on the device")
    ap.add_argument("--policy-chunk-envs", type=int, default=512, help="config4: environments per policy forward chunk")
    ap.add_argument("--tf32", type=int, default=0, help="config4: allow TF32 in the policy's matmuls / convolutions (the reference runs fp32)")
    ap.add_argument("--rollout-batch", type=int, default=131072)
    ap.add_argument("--steady-steps", type=int, default=1023, help="ticks of the survival leg (one episode under the scripted forager policy; 0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of their last step to DIR/<name>.npy (native step benchmark only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.what != "step" or args.impl != "native"):
        ap.error("--dump-outputs applies to the native step benchmark only")
    if args.what == "rollout":
        run_rollout(args)
    elif args.what == "config4":
        run_config4(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
