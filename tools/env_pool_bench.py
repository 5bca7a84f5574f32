"""B200VecEnv as an env pool: ms per full round (every env stepped once) on the default shape, by envs_per_batch.

Rows: the built-in random policy with no consumer between recv() and send(); two half-size handles on two streams
(the experiment of DESIGN.md 5.1) for reference; TakeruPolicy on each batch between recv() and send().  Every
measurement starts from the same reset and warm-up, so all of them cover the same ticks of the same episode; the batch
sizes are taken in turn, `--repeats` times.  Times are CUDA events on the current stream, which waits for every batch
stream before the closing event.  Prints one JSON line per measurement.

    python tools/env_pool_bench.py [--envs 4096] [--batches 4096,2048,1024,512] [--rounds 64] [--warmup 16]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from nmmo_b200.vecenv import B200VecEnv  # noqa: E402


def timed(fn, n, join):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    join()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def pool_round(pool, policy=None):
    for _ in range(pool.num_batches):
        o = pool.recv()[0]
        if policy is None:
            lo, hi = pool.batch_env_range
            pool.send(pool.sim.actions[lo:hi])
        else:
            pool.send(policy(o)[0])


def measure_pool(pool, seed, warmup, rounds, policy=None):
    pool.async_reset(seed)
    for _ in range(warmup):
        pool_round(pool, policy)
    join = pool.sim.join_batches if pool.num_batches > 1 else (lambda: None)
    return timed(lambda: pool_round(pool, policy), rounds, join)


def measure_two_handles(sims, streams, seed, warmup, rounds):
    for k, s in enumerate(sims):
        s.reset(np.arange(s.E, dtype=np.uint64) + seed + k * s.E)

    def tick():
        for s, st in zip(sims, streams):
            with torch.cuda.stream(st):
                s.step()

    cur = torch.cuda.current_stream()

    def join():
        for st in streams:
            cur.wait_stream(st)
    for _ in range(warmup):
        tick()
    return timed(tick, rounds, join)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--batches", default="4096,2048,1024,512")
    ap.add_argument("--rounds", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--policy-rounds", type=int, default=4)
    ap.add_argument("--policy-chunk-envs", type=int, default=512)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    E = args.envs
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": gpu[0] if gpu else torch.cuda.get_device_name(), "envs": E}), flush=True)
    batches = [int(b) for b in args.batches.split(",")]
    pools = {}
    for b in batches:
        pools[b] = B200VecEnv(num_envs=E, envs_per_batch=b, agent="takeru", collect_infos=False)
        pools[b].sim.set_autosample(args.seed)
    kernels = pools[batches[0]].sim.kernel_names()
    from nmmo_b200.lib import Simulator
    ref = pools[batches[0]]
    half = [Simulator(ref.cfg, ref.fcfg, E // 2, ref.maps, ref.task_table, ref.task_embed, env_base=k * (E // 2)) for k in range(2)]
    for s in half:
        s.set_autosample(args.seed)
    side = [torch.cuda.Stream() for _ in range(2)]
    from nmmo_b200.takeru_policy import TakeruPolicy
    torch.manual_seed(0)
    policy = TakeruPolicy(ref.driver_env.unflatten_context, agents_per_env=ref.agents_per_env,
                          envs_per_chunk=args.policy_chunk_envs).cuda().eval()
    for rep in range(args.repeats):
        for b in batches:
            ms = measure_pool(pools[b], args.seed, args.warmup, args.rounds)
            print(json.dumps({"row": "random_policy", "rep": rep, "envs_per_batch": b, "ms_per_round": round(ms, 4),
                              "kernels": kernels}), flush=True)
        for name, streams in (("two_handles_two_streams", side), ("two_handles_one_stream", [torch.cuda.current_stream()] * 2)):
            ms = measure_two_handles(half, streams, args.seed, args.warmup, args.rounds)
            print(json.dumps({"row": name, "rep": rep, "envs_per_handle": E // 2, "ms_per_round": round(ms, 4)}), flush=True)
        for b in batches:
            ms = measure_pool(pools[b], args.seed, 2, args.policy_rounds, policy)
            print(json.dumps({"row": "takeru_policy", "rep": rep, "envs_per_batch": b, "ms_per_round": round(ms, 4),
                              "policy_chunk_envs": args.policy_chunk_envs}), flush=True)


if __name__ == "__main__":
    main()
