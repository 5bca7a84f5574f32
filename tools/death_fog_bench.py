"""What the death fog costs (DESIGN.md 5): ms per tick with the fog off and on, kernel names and times, alive fraction,
episode lengths.

One handle per (workload, fog) built from bench.world, stepped with the built-in random policy (set_autosample, as
bench.py does).  Fog "off" is the reference's default (death_fog_tick None: the *_std kernels); 0, 128 and 1024 are
death_fog_tick values, which run the generic kernels (the *_std ones fold the fog off).  1024 is the horizon: that fog
never starts, so the handle steps exactly what the fog-off one steps and its row is the cost of the generic kernels
alone.  Each measurement resets, warms up `--warmup` ticks and times the next `--steps` ticks with CUDA events
(bench.py --steps 256 --warmup 16 by default); the handles of a workload are taken in turn, `--repeats` times.  Over
the same window: the alive fraction (mask slots / agent slots), the mean episode length of the agents whose episode
ended in it (info "length"), and the environments' resets.  A separate torch.profiler pass over the first
min(steps, 64) ticks of the window gives each kernel's mean device time per tick.  Prints one JSON line per
measurement; the first line names the GPU and its power limit.

    python tools/death_fog_bench.py [--repeats 3] [--steps 256] [--warmup 16]
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
from nmmo_b200.config import SPEC, death_fog_onset  # noqa: E402
from nmmo_b200.lib import Simulator  # noqa: E402

SEED = 1
FOGS = (None, 0, 128, 1024)


def run_window(sim, warmup, steps):
    """Reset, warm up, then `steps` ticks -> (ms per tick, alive fraction, mean agent episode length, env resets)."""
    sim.reset(np.arange(sim.E, dtype=np.uint64) + 1)
    for _ in range(warmup):
        sim.step()
    torch.cuda.synchronize()
    sim.stats(clear=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sim.step()
    e1.record()
    e1.synchronize()
    sums, counts, counters = sim.stats()
    k = SPEC["IN_LENGTH"]
    length = float(sums[k] / counts[k]) if counts[k] else None
    return e0.elapsed_time(e1) / steps, float(counters[1]) / max(1.0, float(counters[0])), length, int(counters[2])


def kernel_ms(sim, warmup, steps):
    from torch.profiler import ProfilerActivity, profile
    sim.reset(np.arange(sim.E, dtype=np.uint64) + 1)
    for _ in range(warmup):
        sim.step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            sim.step()
        torch.cuda.synchronize()
    return {ev.key: round(ev.device_time_total / 1000.0 / steps, 4) for ev in prof.key_averages() if ev.key.startswith("nmmo_")}


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
        sims = {}
        for fog in FOGS:
            c = cfg.copy()
            c[SPEC["NC_DEATH_FOG"]] = death_fog_onset(fog)
            sims[fog] = Simulator(c, fcfg, E, maps, tab, emb)
            sims[fog].set_autosample(SEED)
        for rep in range(args.repeats):
            for fog, sim in sims.items():
                ms, alive, length, resets = run_window(sim, args.warmup, args.steps)
                print(json.dumps({"workload": workload, "envs": E, "death_fog_tick": fog, "rep": rep,
                                  "warmup": args.warmup, "steps": args.steps, "ms_per_tick": round(ms, 4),
                                  "alive_fraction": round(alive, 4),
                                  "mean_episode_length": None if length is None else round(length, 1),
                                  "env_resets": resets, "kernels": sim.kernel_names()}), flush=True)
        for fog, sim in sims.items():
            k = kernel_ms(sim, args.warmup, min(args.steps, 64))
            print(json.dumps({"workload": workload, "envs": E, "death_fog_tick": fog, "profiler_ms_per_tick": k}), flush=True)
            sim.close()


if __name__ == "__main__":
    main()
