"""What the event log costs (DESIGN.md 2.4): ms per tick with the log off and on, the export kernels' time, rows per tick.

One handle per workload, built from bench.world, stepped with the built-in random policy (set_autosample, as bench.py
does).  "off" steps; "on" steps and exports every env's events with nmmo_events into one device buffer, the way
B200VecEnv(event_log_cap=...) does on the lock-step path.  Both start from the same reset and warm-up, so they cover the
same ticks; they are taken in turn, `--repeats` times.  Windows: "default" = ticks [warmup, warmup + steps) after the
reset (bench.py --steps 256 --warmup 16), "short" = the first ticks, every agent alive (bench.py --steps 20 --warmup 5).
Times are CUDA events around the window.  A separate torch.profiler pass, log on, over the first min(steps, 64) ticks of
the window gives the mean device time of each kernel per tick.  Prints one JSON line per measurement.

    python tools/event_log_bench.py [--repeats 3]
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
from nmmo_b200.lib import Simulator  # noqa: E402

SEED = 1


def run_window(sim, log, warmup, steps, rows, cnt):
    """Log on or off, reset, warm up, then `steps` ticks; -> (ms per tick, mean rows per tick)."""
    sim.set_event_log(log)
    sim.reset(np.arange(sim.E, dtype=np.uint64) + 1)
    total = torch.zeros(1, dtype=torch.int64, device=rows.device)

    def tick():
        sim.step()
        if log:
            sim.events(out=rows, count=cnt)
            total.add_(cnt)
    for _ in range(warmup):
        tick()
    total.zero_()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        tick()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps, float(total.item()) / steps


def kernel_ms(sim, warmup, steps, rows, cnt):
    from torch.profiler import ProfilerActivity, profile
    sim.set_event_log(True)
    sim.reset(np.arange(sim.E, dtype=np.uint64) + 1)
    for _ in range(warmup):
        sim.step(); sim.events(out=rows, count=cnt)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            sim.step(); sim.events(out=rows, count=cnt)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.key.startswith("nmmo_"):
            out[ev.key] = round(ev.device_time_total / 1000.0 / steps, 4)      # ms per tick
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": gpu[0] if gpu else torch.cuda.get_device_name()}), flush=True)
    for workload, E, windows in (("config2", 4096, (("default", 16, 256), ("short", 5, 20))),
                                 ("config5", 512, (("default", 16, 256),))):
        cfg, fcfg, maps, tab, emb = world(workload=workload)
        sim = Simulator(cfg, fcfg, E, maps, tab, emb)
        sim.set_autosample(SEED)
        cap = E * sim.P * 8
        rows = torch.empty((cap, 9), dtype=torch.int32, device="cuda")
        cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
        names = sim.kernel_names()
        for wname, warmup, steps in windows:
            for rep in range(args.repeats):
                for log in (False, True):
                    ms, per_tick = run_window(sim, log, warmup, steps, rows, cnt)
                    print(json.dumps({"workload": workload, "envs": E, "window": wname, "rep": rep, "event_log": log,
                                      "ms_per_tick": round(ms, 4), "rows_per_tick": round(per_tick, 1) if log else None,
                                      "row_bytes_per_tick": round(per_tick * 36) if log else None, "kernels": names}), flush=True)
            k = kernel_ms(sim, warmup, min(steps, 64), rows, cnt)
            print(json.dumps({"workload": workload, "envs": E, "window": wname, "profiler_ms_per_tick": k}), flush=True)
        sim.close()


if __name__ == "__main__":
    main()
