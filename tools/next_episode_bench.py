"""What pending next-episode values cost (DESIGN.md 2.5): ms per tick with the feature never enabled, enabled with
nothing pending, and with every automatic reset taking a seed, a map and tasks that torch ops over the flags refill
each tick.

One handle per (workload, mode) built from bench.world, stepped with the built-in random policy (set_autosample, as
bench.py does).  Each measurement resets, warms up `--warmup` ticks and times the next `--steps` ticks with CUDA events
(bench.py's window: --warmup 16 --steps 256); the handles of a workload are taken in turn, `--repeats` times.  In the
"refill" mode every tick first runs, on the current stream and without a host sync,

    free = next_flags == 0;  next_seed / next_map / next_task = where(free, new values, old);  next_flags |= free * 7

so every env's next automatic reset takes all three fields.  Over the window: the environments' resets and the rejected
entries (counters 2 and 5 of stats).  A separate torch.profiler pass over the first min(steps, 64) ticks of the window
gives each kernel's mean device time per tick; "refill_ops_ms" sums the kernels that are not the simulator's.  Prints
one JSON line per measurement; the first line names the GPU and its power limit.

    python tools/next_episode_bench.py [--repeats 3] [--steps 256] [--warmup 16]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import world  # noqa: E402
from nmmo_b200.config import SPEC  # noqa: E402
from nmmo_b200.lib import Simulator  # noqa: E402

SEED = 1
MODES = ("off", "on_nothing_pending", "refill_every_reset")
ALL = SPEC["NM_NEXT_SEED"] | SPEC["NM_NEXT_MAP"] | SPEC["NM_NEXT_TASKS"]


class Refill:
    """Gives every env whose entry was consumed a new seed, map and task, with torch ops on the current stream."""

    def __init__(self, sim):
        self.sim, self.t = sim, 0
        self.ar = torch.arange(sim.E, device=sim.next_flags.device)

    def __call__(self):
        s, ar = self.sim, self.ar
        self.t += 1
        free = s.next_flags == 0
        s.next_seed.copy_(torch.where(free, ar + (1_000_003 * self.t), s.next_seed))
        s.next_map.copy_(torch.where(free, ((ar + self.t) % s.n_maps).to(torch.int32), s.next_map))
        s.next_task.copy_(torch.where(free[:, None], ((ar + 7 * self.t) % s.n_tasks).to(torch.int32)[:, None], s.next_task))
        s.next_flags.bitwise_or_(free.to(torch.uint8) * ALL)


def tick(sim, refill):
    if refill is not None:
        refill()
    sim.step()


def run_window(sim, refill, warmup, steps):
    """Reset, warm up, then `steps` ticks -> (ms per tick, env resets, rejected entries)."""
    sim.reset(np.arange(sim.E, dtype=np.uint64) + 1)
    if sim.next_flags is not None:
        sim.set_next_episodes(True)         # every flag 0
    for _ in range(warmup):
        tick(sim, refill)
    torch.cuda.synchronize()
    sim.stats(clear=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        tick(sim, refill)
    e1.record()
    e1.synchronize()
    counters = sim.stats()[2]
    return e0.elapsed_time(e1) / steps, int(counters[2]), int(counters[5])


def kernel_ms(sim, refill, warmup, steps):
    from torch.profiler import ProfilerActivity, profile
    sim.reset(np.arange(sim.E, dtype=np.uint64) + 1)
    for _ in range(warmup):
        tick(sim, refill)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            tick(sim, refill)
        torch.cuda.synchronize()
    per = {ev.key: ev.device_time_total / 1000.0 / steps for ev in prof.key_averages() if ev.device_time_total > 0}
    ours = {k: round(v, 4) for k, v in per.items() if k.startswith("nmmo_")}
    other = sum(v for k, v in per.items() if not k.startswith("nmmo_") and not k.startswith("Memcpy") and not k.startswith("Memset"))
    return ours, round(other, 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=16)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": gpu[0] if gpu else torch.cuda.get_device_name()}), flush=True)
    for workload, E in (("config2", 4096), ("config5", 512)):
        cfg, fcfg, maps, tab, emb = world(workload=workload)
        sims, refills = {}, {}
        for mode in MODES:
            sims[mode] = Simulator(cfg, fcfg, E, maps, tab, emb)
            sims[mode].set_autosample(SEED)
            if mode != "off":
                sims[mode].set_next_episodes(True)
            refills[mode] = Refill(sims[mode]) if mode == "refill_every_reset" else None
        for rep in range(args.repeats):
            for mode, sim in sims.items():
                ms, resets, rejected = run_window(sim, refills[mode], args.warmup, args.steps)
                print(json.dumps({"workload": workload, "envs": E, "mode": mode, "rep": rep, "warmup": args.warmup,
                                  "steps": args.steps, "ms_per_tick": round(ms, 4), "env_resets": resets,
                                  "rejected_entries": rejected, "kernels": sim.kernel_names()}), flush=True)
        for mode, sim in sims.items():
            k, other = kernel_ms(sim, refills[mode], args.warmup, min(args.steps, 64))
            print(json.dumps({"workload": workload, "envs": E, "mode": mode, "profiler_ms_per_tick": k,
                              "refill_ops_ms": other}), flush=True)
            sim.close()


if __name__ == "__main__":
    main()
