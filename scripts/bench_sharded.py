"""One bus handle over G GPUs (`Bus(devices=...)`, cpbus_create_sharded) against `LocalShardedBus` driving the same shards
itself, on BASELINE config 3's shape per GPU: 1,048,576 subscribers per GPU, one 1 kHz timer each, 512-event host batches,
throughput mode.  Both publish the same trace from host buffers from ONE thread; at G = 1 the comparison is a plain `Bus`.

    python scripts/bench_sharded.py [--subs-per-gpu N] [--steps K] [--warmup W] [--repeats R] [--shared]

For each G = 1 .. device_count the two arms run alternately, `--repeats` times each, every timed window ending in a device
synchronise (host clock).  One JSON line per G: the GPU's name and power limit, ms per step and deliveries/s of each arm
(median and spread over the repeats), and `parity`: the handle's global digest fold equals the other arm's.  `--shared`
also runs G = 2 and 4 with every shard on device 0 and the same total subscriber count (the one-thread cost of G
fan-outs per step, measurable on a one-GPU box)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from containerpilot_b200 import _native as nat  # noqa: E402
from containerpilot_b200.bus import Bus, EVENT_DTYPE  # noqa: E402
from containerpilot_b200.sharding import LocalShardedBus  # noqa: E402

TICK_NS = 1_000_000   # 1 kHz
DT_NS = 10_000        # virtual time per publish, as bench.py


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return [line.strip() for line in q.stdout.strip().splitlines()]


class HandleArm:
    """one handle over `devices` (sharded=True), or a plain single-GPU Bus"""

    def __init__(self, n_total, devices, batch, sharded=True):
        self.bus = Bus(n_total, ring_cap=1024, batch_cap=batch, timers_per_sub=1, devices=devices if sharded else None,
                       device=devices[0])
        self.bus.subscribe_many(np.full(n_total, nat.MASK_ALL, dtype=np.uint32))
        self.bus.timer_add_many(0, n_total, TICK_NS, source_id0=1_000_000)
        self.n = n_total

    def step(self, ev, now):
        nat.check(self.bus.advance(now), "advance")
        nat.check(self.bus.publish_many(ev), "publish")
        nat.check(self.bus.flush(), "flush")

    def sync(self):
        self.bus.sync()

    def deliveries(self):
        return self.bus.stats()["deliveries"]

    def fold(self):
        return tuple(int(x) for x in self.bus.digest_fold(0, self.n))

    def close(self):
        self.bus.close()


class LocalArm:
    def __init__(self, n_total, devices, batch):
        self.lsb = LocalShardedBus(n_total, devices, batch_cap=batch, timers_per_sub=1)
        self.lsb.subscribe_many(np.full(n_total, nat.MASK_ALL, dtype=np.uint32))
        self.lsb.timer_add_many(TICK_NS, source_id0=1_000_000)

    def step(self, ev, now):
        self.lsb.publish(ev, now)

    def sync(self):
        self.lsb.sync()

    def deliveries(self):
        return sum(bus.stats()["deliveries"] for _, _, bus in self.lsb.shards)

    def fold(self):
        M = (1 << 64) - 1
        c = d = x = n = 0
        for first, count, bus in self.lsb.shards:
            f = bus.digest_fold(first, count)
            c = (c + f[0]) & M; d = (d + f[1]) & M; x ^= f[2]; n += f[3]
        return (c, d, x, n)

    def close(self):
        self.lsb.close()


def run(devices, n_total, args):
    arms = {"handle": HandleArm(n_total, devices, args.batch)}
    if len(devices) > 1:
        arms["local_sharded"] = LocalArm(n_total, devices, args.batch)
    else:
        arms["plain_bus"] = HandleArm(n_total, devices, args.batch, sharded=False)
    rng = np.random.default_rng(0xB200)
    trace = np.zeros((64, args.batch), dtype=EVENT_DTYPE)
    trace["code"] = rng.integers(0, 17, trace.shape); trace["source_id"] = rng.integers(0, 1024, trace.shape)
    state = {name: 0 for name in arms}

    def steps(name, k):
        arm = arms[name]
        for _ in range(k):
            i = state[name]
            arm.step(trace[i % len(trace)], (i + 1) * args.batch * DT_NS)
            state[name] = i + 1

    for name in arms:
        steps(name, args.warmup); arms[name].sync()
    times = {name: [] for name in arms}
    dels = {name: [] for name in arms}
    for _ in range(args.repeats):
        for name, arm in arms.items():
            d0 = arm.deliveries()
            t0 = time.perf_counter()
            steps(name, args.steps)
            arm.sync()
            times[name].append(time.perf_counter() - t0)
            dels[name].append(arm.deliveries() - d0)
    folds = {name: arm.fold() for name, arm in arms.items()}
    for arm in arms.values():
        arm.close()
    out = {}
    for name in arms:
        ms = [1e3 * t / args.steps for t in times[name]]
        rate = [d / t for d, t in zip(dels[name], times[name])]
        out[name] = {"ms_per_step": round(float(np.median(ms)), 4), "ms_per_step_all": [round(v, 4) for v in ms],
                     "deliveries_per_s": float(np.median(rate)), "spread_pct": round(100 * (max(ms) - min(ms)) / np.median(ms), 2)}
    f = list(folds.values())
    return out, f[0] == f[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--subs-per-gpu", type=int, default=1_048_576)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--shared", action="store_true")
    args = ap.parse_args()
    import torch
    ndev = torch.cuda.device_count()
    if ndev == 0:
        sys.exit("no CUDA device: nothing to measure")
    gpus = gpu_info()
    plans = [(list(range(g)), args.subs_per_gpu * g) for g in range(1, ndev + 1)]
    if args.shared:
        plans += [([0] * g, args.subs_per_gpu) for g in (2, 4)]
    for devices, n_total in plans:
        res, parity = run(devices, n_total, args)
        print(json.dumps({"gpus": gpus[:len(set(devices))], "devices": devices, "subscribers_total": n_total,
                          "events_per_step": args.batch, "timers": "1 kHz per subscriber", "steps": args.steps,
                          "repeats": args.repeats, "arms": res, "parity": parity}), flush=True)


if __name__ == "__main__":
    main()
