"""Cost of saving and loading environment state (Simulator.save_envs / load_envs, DESIGN.md 2.3).

Cases: 4096 default-shape envs after 64 ticks of the built-in policy (save all, load all, load 64 scattered envs) and
512 config-5 envs after 16 ticks (save all, load all).  Each call is timed with CUDA events around it, after warm-up,
`--repeats` times; a load's time includes its stream synchronise and header read-back.  A torch.profiler pass over
the same calls then splits the device time into the copy kernels and the load's observation pass.  Bytes are what the
copy kernels move: a save reads the live part of each env's buffers and writes whole blobs, a load reads and writes
the live part.  The copy peak is a device-to-device torch copy of 2 GiB in the same process.  Prints one JSON line
per measurement, the first with the card's name and power limit.

    python tools/env_state_bench.py [--repeats 20] [--out DIR]
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

HEADER = 128          # the blob header; the scalars section follows it (nmmo_api.cu state_layout)
SC_N_DANGER, SC_ITEM_HI, SC_N_DEPL = 3, 11, 12


def timed(fn, repeats, warmup=3):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), float(min(ms)), float(max(ms))


def live_bytes(sim, blobs):
    """Bytes of the handle's buffers a save reads (= a load writes) for these blobs: everything but the dead tails of the
    item columns, the depleted-tile list and the danger stack, which the copy kernels skip."""
    sc = blobs[:, HEADER:HEADER + 64].cpu().numpy().view(np.int32)
    big = sim.kernel_names()[0].startswith("nmmo_step_big")
    tile, depl_cap = (4, 4096) if big else (2, 1024)
    ent = (48 if big else SPEC["EA_N"]) * (sim.P + sim.N) * 2
    P = sim.P
    fixed = 64 + 8 + 1 + ent + sim.S * sim.S // 2 + P * (SPEC["ST_N"] * 4 + 3 * 8 + 106 * 4 + 4 + 4 + 4 + SPEC["IN_N"] * 4)
    items = np.clip(sc[:, SC_ITEM_HI], 0, sim.cap) * 2 * SPEC["IS_N"]
    depl = np.clip(sc[:, SC_N_DEPL], 0, depl_cap) * tile
    danger = np.clip(sc[:, SC_N_DANGER], 0, sim.N) * 2
    return int((fixed + items + depl + danger).sum())


def kernel_ms(fn, repeats, names):
    """Mean device time per call of the kernels whose name starts with one of `names`, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(repeats):
            fn()
        torch.cuda.synchronize()
    out = {n: 0.0 for n in names}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            for n in names:
                if ev.name.startswith(n):
                    out[n] += ev.device_time / 1000.0
    return {n: v / repeats for n, v in out.items()}


def case(tag, w, E, ticks, repeats, scattered=0):
    sim = Simulator(*w[:2], E, *w[2:])
    sim.set_autosample(1)
    sim.reset(np.arange(E, dtype=np.uint64) + 1)
    for _ in range(ticks):
        sim.step(sim.actions)
    ids = list(range(E))
    blobs = sim.save_envs(ids)
    torch.cuda.synchronize()
    live = live_bytes(sim, blobs)
    obs_k = sim.kernel_names()[1]
    rows = []
    calls = [("save_all", lambda: sim.save_envs(ids, out=blobs), len(ids), E * sim.state_bytes + live, None),
             ("load_all", lambda: sim.load_envs(ids, blobs), len(ids), 2 * live, (min(ids), max(ids) + 1))]
    if scattered:
        sel = np.sort(np.random.default_rng(0).choice(E, scattered, replace=False))
        sub = blobs[torch.as_tensor(sel, device=blobs.device)].contiguous()
        live_sub = live_bytes(sim, sub)
        calls.append((f"load_{scattered}_scattered", lambda: sim.load_envs(sel, sub), scattered, 2 * live_sub,
                      (int(sel.min()), int(sel.max()) + 1)))
    for name, fn, n, moved, span in calls:
        med, lo, hi = timed(fn, repeats)
        km = kernel_ms(fn, repeats, ["nmmo_state_save_kernel", "nmmo_state_load_kernel", obs_k])
        copy_ms = km["nmmo_state_save_kernel"] + km["nmmo_state_load_kernel"]
        rows.append({"case": tag, "call": name, "envs": n, "state_bytes": sim.state_bytes, "call_ms_median": round(med, 4),
                     "call_ms_min": round(lo, 4), "call_ms_max": round(hi, 4), "copy_kernel_ms": round(copy_ms, 4),
                     "copy_bytes": moved, "copy_GBps": round(moved / copy_ms / 1e6, 1) if copy_ms else None,
                     "obs_pass_ms": round(km[obs_k], 4) if span else None, "obs_pass_envs": (span[1] - span[0]) if span else None,
                     "obs_kernel": obs_k if span else None})
    sim.close()
    return rows


def copy_peak(repeats):
    n = 1 << 31
    a = torch.empty(n, dtype=torch.uint8, device="cuda").fill_(1)
    b = torch.empty_like(a)
    med, lo, hi = timed(lambda: b.copy_(a), repeats)
    del a, b
    torch.cuda.empty_cache()
    return {"call": "copy_peak", "bytes": 2 * n, "ms_median": round(med, 4), "GBps": round(2 * n / lo / 1e6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the lines to DIR/env_state_bench.jsonl")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = [{"gpu": gpu[0] if gpu else torch.cuda.get_device_name()}]
    print(json.dumps(lines[-1]), flush=True)
    lines.append(copy_peak(args.repeats))
    print(json.dumps(lines[-1]), flush=True)
    for row in case("config2_4096", world(n_maps=64), 4096, 64, args.repeats, scattered=64):
        lines.append(row); print(json.dumps(row), flush=True)
    for row in case("config5_512", world(workload="config5", n_maps=8), 512, 16, args.repeats):
        lines.append(row); print(json.dumps(row), flush=True)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        with open(Path(args.out) / "env_state_bench.jsonl", "w") as f:
            for x in lines:
                f.write(json.dumps(x) + "\n")


if __name__ == "__main__":
    main()
