#!/usr/bin/env python
"""bench.py — events/sec through EventBus.Publish on B200 (BASELINE.json metric).

A "step" is one pass of the hot path over one batch: `batch` published events fanned out to every subscriber mailbox of
every GPU's shard (one fan-out kernel launch per GPU).  Headline unit (BASELINE.md §3): deliveries/s = 32-byte records
landed in mailboxes per second, whole job; publishes/s is reported beside it.

  python bench.py [--gpus N --steps K --warmup W] [--workload default|config2|config3|config5] [--dump-outputs DIR]
  python bench.py --impl reference ...      # the reference's CPU path (restated Go bus) on the host cores

Default: the headline is BASELINE config 3 — the configuration north_star's target is quoted on (1,048,576 subscribers
per GPU, 1 kHz timer per subscriber; at --gpus 8 this IS config 4: 8,388,608 subscribers sharded evenly) — and configs 2
and 5 are measured in the same run and printed under "extra_configs", each with its own roofline / e2e / parity check.
Every configuration is verified after its timed regions (sampled subscribers bit-exact against a 1-subscriber oracle over
the exact trace the bench issued, the shard's total count in closed form, the digest fold across ranks); a mismatch
fails the run (rc != 0).  One JSON line on stdout (rank 0).  Nothing here reads /root/reference.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "events/sec through Bus.Publish (deliveries/s = 32-byte records landed in subscriber mailboxes)"
WORKLOADS = {
    # BASELINE.json configs[1]
    "config2": dict(subs=65_536, events=10_000_000, timers=0, zipf=None, scaling="weak",
                    desc="1xB200: 65,536 subscribers, 10M-event synthetic trace, 32-byte records, all-ones masks"),
    # configs[2] (and configs[3] = the same shard on each of 8 GPUs): the configuration north_star's target is quoted on
    "config3": dict(subs=1_048_576, events=100_000_000, timers=1, zipf=None, scaling="weak",
                    desc="1xB200: 1,048,576 subscribers, 100M events (prefix timed), Timer ticks interleaved at 1 kHz"),
    # configs[4]: Zipf-skewed masks over 16 codes, TOTAL subscriber count fixed as GPUs are added (strong scaling)
    "config5": dict(subs=1_048_576, events=10_000_000, timers=0, zipf=1.0, scaling="strong",
                    desc="filter sweep: 1,048,576 subscribers in total, 16 event codes, Zipf(s=1.0) masks and codes"),
}
DT_NS = 10_000            # virtual time per publish: 1e5 publishes per virtual second
TICK_NS = 1_000_000       # 1 kHz


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=0, help="batches to time (0 = the workload's whole trace, capped)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="cpbus", choices=["cpbus", "reference"])
    ap.add_argument("--workload", default="default", choices=["default"] + sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=512, help="events per step (<= ring/2); 512 measured best: config 2 +1.5 %, config 3 +8 % over 256")
    ap.add_argument("--ring", type=int, default=1024)
    ap.add_argument("--subs", type=int, default=0, help="override subscribers per GPU")
    ap.add_argument("--store", type=int, default=0, help="0 auto, 1 v4, 2 v8, 3 TMA bulk")
    ap.add_argument("--grid", type=int, default=0)
    ap.add_argument("--no-digest", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="default workload: headline only")
    ap.add_argument("--no-verify", action="store_true", help="skip the in-bench oracle check (diagnostics only; the line says so)")
    ap.add_argument("--max-steps", type=int, default=40_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what each configuration's timed fan-out left in the "
                    "mailboxes after its last step to DIR/<config>_<array>.npy (float64, a seeded sample; see dump_outputs)")
    return ap.parse_args()


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (NVML, in-process)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("hw_thermal_slowdown", 0x40),
                              ("sw_thermal_slowdown", 0x20), ("hw_power_brake", 0x80), ("sync_boost", 0x10)):
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        if self.nv is None:
            return
        while not self.stop_flag:
            self.sample()
            time.sleep(0.004)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------- CPU arms ---
def _ref_shape(wl, args, world):
    """Subscribers / events per step of the CPU arm for this workload at `world` GPUs' worth of subscribers."""
    per_gpu = args.subs or (wl["subs"] // world if wl["scaling"] == "strong" else wl["subs"])
    total = per_gpu * world
    # bounded sample: a Go channel of capacity 1000 is 24 KB; 2,097,152 of them are 50 GB of host memory
    return min(total, 2_097_152), total


def cpu_baseline(wl, args, seconds_target: float = 14.0):
    """Restated Go bus (oracle/gobus_baseline.c) on this box's host cores, beside the GPU number (N = 1 only)."""
    import oracle_binding as ob
    cores = os.cpu_count() or 1
    n_subs = min(_ref_shape(wl, args, 1)[0], 262_144)
    probe, _ = ob.gobus_bench_steps2(n_subs, 8, 1, 1, 1000, cores)
    ev = int(max(8, min(args.batch, probe * seconds_target / 4 / n_subs / 3)))
    multi, sec = ob.gobus_bench_steps2(n_subs, ev, 3, 1, 1000, cores)
    ev1 = max(4, ev // max(1, cores // 2))
    single, _ = ob.gobus_bench_steps2(n_subs, ev1, 3, 1, 1000, 1)
    return {"value": multi, "unit": "deliveries/s", "cores": cores, "kind": "port", "single_thread_value": single,
            "sample": f"{n_subs} subscribers x {ev} events x 3 steps sharded over {cores} pinned threads (value), and x {ev1} events "
                      f"x 3 steps on one thread (GOMAXPROCS(1)-faithful); mailbox cap 1000, consumers drain (lossless); "
                      f"restated Go bus — no Go toolchain in this image"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The Go bus cannot be built here (no Go
    toolchain), so this is the oracle port of its cost model with all the host threads it can use, on the same workload
    shape as the cpbus arm: same events per step, subscribers scaled with N (bounded at 2,097,152 = 50 GB of channels)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_binding as ob
    world = max(1, args.gpus)
    name = "config3" if args.workload == "default" else args.workload
    wl = WORKLOADS[name]
    n_subs, n_total = _ref_shape(wl, args, world)
    cores = os.cpu_count() or 1
    steps = args.steps or 8
    warmup = max(0, args.warmup)
    B = args.batch
    probe, _ = ob.gobus_bench_steps2(min(n_subs, 131_072), 8, 1, 1, 1000, cores)
    budget_s = 150.0                                                  # the whole --steps K --warmup W run ends within a few minutes
    ev = int(max(1, min(B, probe * budget_s / n_subs / (steps + warmup))))
    value, sec = ob.gobus_bench_steps2(n_subs, ev, steps, warmup, 1000, cores)
    send_only, _ = ob.gobus_bench_steps2(min(n_subs, 262_144), ev, 3, 1, 1000, cores, send_only=True)
    single, _ = ob.gobus_bench_steps2(min(n_subs, 65_536), max(1, ev // 8), 3, 1, 1000, 1)
    med = float(np.median(sec))
    sample = (f"{steps} steps x {ev} events x {n_subs} subscribers (of the arm's {n_total}"
              f"{'; bounded: 50 GB of channels' if n_subs < n_total else ''}), sharded over {cores} pinned threads, NUMA-local mailboxes, "
              f"consumers drain every step (lossless, the reference's semantics)")
    line = {"impl": "reference", "metric": METRIC, "value": value,
            "unit": "deliveries/s", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * float(sec.sum()) / steps, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": wl["desc"], "subscribers": n_subs, "subscribers_of_arm": n_total, "events_per_step": ev,
                       "events_per_step_of_arm": B, "mailbox_cap": 1000},
            "cpu_baseline": {"value": value, "unit": "deliveries/s", "cores": cores, "kind": "port", "sample": sample},
            "per_step_median_value": n_subs * ev / med if med > 0 else None,
            "single_thread_value": single, "send_only_value": send_only,
            "notes": "single_thread_value = GOMAXPROCS(1)-faithful; send_only_value = no consumer, full mailboxes overwrite "
                     "(what the GPU arm's throughput mode does), all cores",
            "e2e": {"value": value, "unit": "deliveries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- one configuration ---
class Ctx:
    pass


def run_config(cx, name: str, headline: bool):
    import torch
    import trace as tr
    from containerpilot_b200 import _native as nat
    from containerpilot_b200.bus import EVENT_DTYPE
    from containerpilot_b200.sharding import ShardedBus

    args, dist, world, rank, local, dev, stream = cx.args, cx.dist, cx.world, cx.rank, cx.local, cx.dev, cx.stream
    wl = WORKLOADS[name]
    n_subs = args.subs or (wl["subs"] // world if wl["scaling"] == "strong" else wl["subs"])   # per GPU, contiguous shards (SURVEY §8e)
    B, R = args.batch, args.ring
    n_batches_trace = wl["events"] // B
    steps = args.steps or min(n_batches_trace, args.max_steps)
    warmup = max(args.warmup, 3)
    K_timers = 1 if wl["timers"] else 0

    # ---- synthetic trace (rank 0 is the publisher's GPU) ----
    n_trace_batches = min(max(steps + warmup, 2048), 32768)
    n_ev = n_trace_batches * B
    g = torch.Generator(device="cpu"); g.manual_seed(0xC0DEB200 + 2)
    if wl["zipf"]:
        codes = tr.zipf_codes(n_ev, wl["zipf"], 0xC0DEB205).astype(np.uint32)
    else:
        codes = torch.randint(1, 17, (n_ev,), generator=g).numpy().astype(np.uint32)
    srcs = torch.randint(0, 4096, (n_ev,), generator=g).numpy().astype(np.uint32)
    slot_hist = np.stack([np.bincount(codes[i * B:(i + 1) * B], minlength=17) for i in range(n_trace_batches)]) if wl["zipf"] else None

    def make_records(first_seq: int, lo: int = 0, hi: int | None = None) -> np.ndarray:
        hi = n_ev if hi is None else hi
        ev = np.zeros(hi - lo, dtype=EVENT_DTYPE)
        ev["seq"] = first_seq + np.arange(hi - lo, dtype=np.uint64)
        ev["ts_ns"] = (first_seq + 1 + np.arange(hi - lo, dtype=np.uint64)) * DT_NS
        ev["code"], ev["source_id"], ev["target"] = codes[lo:hi], srcs[lo:hi], nat.TARGET_ALL
        return ev

    sb = ShardedBus(0, dist=dist, rank=rank, world=world, device=local, ring_cap=R, batch_cap=B, timers_per_sub=K_timers,
                    digest=not args.no_digest, stream=stream.cuda_stream, store_path=args.store, grid_ctas=args.grid,
                    subs_per_rank=n_subs, stream_slots=64)
    bus = sb.bus
    first = sb.first
    if wl["zipf"]:
        masks = tr.zipf_masks(n_subs, wl["zipf"], 0xC0DEB205 + rank)
    else:
        masks = np.full(n_subs, nat.MASK_ALL, dtype=np.uint32)
    sb.subscribe_many(masks)
    TIMER_SRC0 = 1_000_000
    if K_timers:
        sb.timer_add_many(TICK_NS, source_id0=TIMER_SRC0)

    # ---- the device-resident trace; re-stamped per cycle on the GPU so seq/ts stay monotonic over any number of steps ----
    base = make_records(0)
    use_nccl = bool(os.environ.get("CPBUS_BENCH_NCCL_INGEST"))
    fused = False
    if world > 1 and not use_nccl:
        ptr = sb.attach_trace(n_ev * 32)
        fused = sb.trace_ok
        if not fused and rank == 0:
            print("[bench] peer mapping unavailable: falling back to NCCL broadcast of the event stream", file=sys.stderr)
    if world > 1 and fused:
        if rank == 0:
            class _Raw:                                        # zero-copy torch view of the shared buffer
                __cuda_array_interface__ = {"shape": (n_ev, 32), "typestr": "|u1", "data": (ptr, False), "version": 2}
            trace_dev = torch.as_tensor(_Raw(), device=dev)
            trace_dev.copy_(torch.from_numpy(base.view(np.uint8).reshape(n_ev, 32)))
        else:
            trace_dev = None
    else:
        trace_dev = torch.from_numpy(base.view(np.uint8).reshape(n_ev, 32)).to(dev) if rank == 0 or world == 1 else \
            torch.empty((n_ev, 32), dtype=torch.uint8, device=dev)
        sb.use_local_trace(trace_dev.data_ptr())
    trace_q = trace_dev.view(torch.int64).view(n_ev, 4) if trace_dev is not None else None   # words: seq, ts, code|src, target|flags
    seq0 = torch.arange(n_ev, dtype=torch.int64, device=dev) if rank == 0 else None
    torch.cuda.synchronize()
    sb.barrier()

    def restamp(cycle: int):
        if rank == 0:
            trace_q[:, 0] = seq0 + cycle * n_ev
            trace_q[:, 1] = (seq0 + 1 + cycle * n_ev) * DT_NS

    CHUNK = 64                                                 # batches per NCCL broadcast (512 KiB), fallback ingest only
    state = {"step": 0, "events": 0}
    log = []                                                   # every batch this bus was given: ("dev", slot, seq0, wm) | ("host", slot, seq0, now)
    ingest_mode = sb.ingest if world > 1 and fused else ("nccl-broadcast" if world > 1 else "local")

    def run_steps(k: int):
        """k fan-out steps from the HBM-resident trace."""
        for _ in range(k):
            i = state["step"]
            slot, cycle = i % n_trace_batches, i // n_trace_batches
            if slot == 0 and cycle > 0:
                if world > 1:                                  # nobody may be reading while the publisher re-stamps
                    torch.cuda.synchronize(); dist.barrier()
                restamp(cycle)
                if world > 1:
                    torch.cuda.synchronize(); dist.barrier()
            if world > 1 and not fused and slot % CHUNK == 0:
                hi = min(slot + CHUNK, n_trace_batches)
                dist.broadcast(trace_dev[slot * B: hi * B], src=0)
            wm = (i + 1) * B * DT_NS
            nslot = slot + 2                                   # the batch after next: pulled by THIS launch, hidden under its stores
            nxt = nslot * B * 32 if (fused and nslot < n_trace_batches) else None   # (not across a re-stamp boundary)
            nat.check(sb.fanout_trace(slot * B * 32, B, wm, nxt, B), "fanout_trace")
            log.append(("dev", slot, i * B, wm))
            state["step"] = i + 1
            state["events"] += B

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def jump_to_next_cycle():
        cycle = state["step"] // n_trace_batches + 1
        barrier()
        restamp(cycle)
        barrier()
        state["step"] = cycle * n_trace_batches
        nat.check(bus.advance(state["step"] * B * DT_NS), "cpbus_advance")   # armed timers catch up in bounded windows

    # ---- device-resident timing: `value` ----
    sampler = ClockSampler(local)
    sampler.start()                                            # started early so NVML is warm before the timed region
    run_steps(warmup)
    # settle: a fresh box pages in driver/library code lazily; keep warming (untimed) for 1.2e11 records' worth of
    # all-ones fan-out, about 0.6 s on a B200.  A step count rather than a clock, so that every run (and every build)
    # times the same batches of the same trace and leaves the same mailbox contents behind.
    settle = int(min(20_000, max(10, round(1.2e11 / (n_subs * B)))))
    run_steps(settle)
    torch.cuda.synchronize()
    # if the timed region would straddle the end of the trace, start it at the next cycle instead (re-stamp outside the timing)
    pos = state["step"] % n_trace_batches
    if steps <= n_trace_batches and pos + steps > n_trace_batches:
        jump_to_next_cycle()
    barrier()
    st0 = bus.stats()
    sampler.samples.clear(); sampler.reasons.clear()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    run_steps(steps)
    e1.record(stream)
    sampler.sample()                                           # launches are asynchronous: the GPU is still inside the timed region here
    barrier()
    sampler.stop_flag = True
    ms_local = e0.elapsed_time(e1)
    st1 = bus.stats()
    t = torch.tensor([ms_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    deliv = torch.tensor([st1["deliveries"] - st0["deliveries"], st1["ticks"] - st0["ticks"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(deliv, op=dist.ReduceOp.SUM)
    deliveries, ticks = float(deliv[0].item()), float(deliv[1].item())
    launches = st1["kernel_launches"] - st0["kernel_launches"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, name, bus, first, n_subs, R)
    value = deliveries / (ms * 1e-3)
    publishes_per_s = steps * B / (ms * 1e-3)

    # ---- roofline for the dominant kernel (fan-out): algorithmic bytes per launch / avg launch duration ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    d_local = (st1["deliveries"] - st0["deliveries"]) / steps        # records per launch on this GPU
    # algorithmic bytes per launch (DESIGN.md §4.1): every delivered record is one 32-byte sector; every mailbox's 32-byte
    # control block is read once and written once; an armed timer slot costs its 16-byte hot half read plus, when it fires,
    # the cold half read and both halves written (~64 B); the batch itself is read once from HBM
    per_sub_state = 64 + (64 if K_timers else 0)
    alg_bytes = 32.0 * d_local + n_subs * per_sub_state + B * 32
    kernel_ms = float(ms_local) / steps                              # this rank's launches are back to back on the stream
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = (json.load(open(tp)).get(name) or {}).get(str(B))
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "cpbus_dev::fanout_kernel", "alg_bytes_per_launch": alg_bytes,
                "record_bytes_per_launch": 32.0 * d_local, "state_bytes_per_launch": float(n_subs * per_sub_state + B * 32),
                "kernel_ms": kernel_ms, "peak_source": peak_src}

    # ---- end to end through the public C-ABI with HOST buffers: `e2e` ----
    e2e, launches_e2e = None, 0
    if not args.no_e2e:
        k2 = min(steps, 4000)
        jump_to_next_cycle()                                   # the host leg starts on a fresh trace cycle (clock keeps increasing)
        k2 = min(k2, n_trace_batches - 8)
        host = base                                            # events as a caller holds them (host memory): code + source are read
        nxt = state["step"]
        tickets = []                                           # result reads are pipelined two steps deep
        fold = [None]
        LOOK = 3                                               # N > 1: the publisher's puts run this many batches ahead of the fan-outs
        put_state = {"next": 0}
        stream_events = [0]
        use_stream = world > 1 and sb.stream_ok and not use_nccl
        if world > 1 and not use_stream:
            ingest_buf = torch.empty((B, 32), dtype=torch.uint8, device=dev)
            pinned = torch.from_numpy(np.zeros((B, 32), dtype=np.uint8)).pin_memory() if rank == 0 else None
        total_e2e = k2 + 3

        def e2e_step(j: int):
            i = nxt + j
            now = (i + 1) * B * DT_NS
            lo = (i % n_trace_batches) * B
            if world == 1:
                nat.check(bus.advance(now), "cpbus_advance")
                nat.check(bus.publish_many(host[lo: lo + B]), "cpbus_publish")   # pinned staging + H2D inside
                nat.check(bus.flush(), "cpbus_flush")
            elif use_stream:
                # rank 0: host batch -> the stream ring (pinned staging + H2D + release inside cpbus_stream_put), a few
                # batches ahead; every rank: ONE fan-out launch whose lead CTA pulls the batch over NVLink.  No collective.
                if rank == 0:
                    while put_state["next"] < total_e2e and put_state["next"] <= j + LOOK:
                        q = nxt + put_state["next"]
                        ql = (q % n_trace_batches) * B
                        rc = sb.put(host[ql: ql + B], (q + 1) * B * DT_NS)
                        if rc == nat.EAGAIN:
                            break
                        nat.check(rc, "cpbus_stream_put"); put_state["next"] += 1
                nat.check(sb.fanout(B, now), "cpbus_stream_fanout")
            else:                                              # fallback: H2D on rank 0 + NCCL broadcast + local fan-out, unpipelined
                if rank == 0:
                    rec = make_records(state["events"], lo, lo + B); rec["ts_ns"] = now
                    pinned.copy_(torch.from_numpy(rec.view(np.uint8).reshape(B, 32)))
                    ingest_buf.copy_(pinned, non_blocking=True)
                dist.broadcast(ingest_buf, src=0)
                nat.check(bus.publish_device(ingest_buf.data_ptr(), B, now), "cpbus_publish_device")
            # seq stamped by the bus: cpbus_publish continues the bus's running ordinal; a stream stamps its own put ordinal
            log.append(("host", i % n_trace_batches, stream_events[0] if use_stream else state["events"], now))
            stream_events[0] += B
            state["events"] += B
            tickets.append(bus.step_result_begin())            # 256-byte D2H of the step's result (written by the fan-out kernel)
            if len(tickets) > 2:
                fold[0] = bus.step_result_end(tickets.pop(0))  # ...read two steps later: the GPU never idles

        for j in range(3):
            e2e_step(j)
        while tickets:
            bus.step_result_end(tickets.pop(0))
        barrier()
        s0 = bus.stats()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        f0.record(stream)
        for j in range(3, 3 + k2):
            e2e_step(j)
        while tickets:
            fold[0] = bus.step_result_end(tickets.pop(0))      # every step's result has reached the host
        f1.record(stream)
        barrier()
        wall_ms = (time.perf_counter() - w0) * 1e3
        s1 = bus.stats()
        state["step"] = nxt + 3 + k2
        t2 = torch.tensor([max(f0.elapsed_time(f1), wall_ms)], dtype=torch.float64, device=dev)
        d2 = torch.tensor([s1["deliveries"] - s0["deliveries"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX); dist.all_reduce(d2, op=dist.ReduceOp.SUM)
        api = ("cpbus_advance+cpbus_publish(host events)+cpbus_flush+cpbus_step_result_begin/_end (deliveries + digest checksum of the step, read 2 steps later)"
               if world == 1 else
               ("rank 0: cpbus_stream_put(host events: pinned staging + H2D + release flag, 3 batches ahead); every rank: cpbus_stream_fanout "
                "(lead CTA acquires the flag and pulls the batch over NVLink inside the fan-out launch; no collective) + cpbus_step_result_begin/_end"
                if use_stream else
                "pinned host batch -> H2D on rank 0 -> NCCL broadcast -> cpbus_publish_device + cpbus_step_result_begin/_end"))
        e2e = {"value": float(d2.item()) / (float(t2.item()) * 1e-3), "unit": "deliveries/s",
               "h2d_bytes_per_step": B * 32 + (32 if use_stream else 0), "d2h_bytes_per_step": 256, "steps": k2,
               "ms_per_step": float(t2.item()) / k2, "api": api}
        launches_e2e = s1["kernel_launches"] - s0["kernel_launches"]

    # ---- verification: what the mailboxes hold now must be exactly what the reference bus would have delivered ----
    parity = verify(cx, name, sb, log, base, masks, n_subs, B, K_timers, TIMER_SRC0, slot_hist, make_records) if not args.no_verify else None

    cpu = None
    if headline and rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(wl, args)

    torch.cuda.synchronize()
    sb.close()
    del trace_dev, trace_q
    torch.cuda.empty_cache()
    res = {
        "workload": wl["desc"], "name": name, "steps": steps, "value": value, "unit": "deliveries/s", "ms_per_step": ms / steps,
        "scaling": wl["scaling"], "publishes_per_s": publishes_per_s, "deliveries": deliveries, "ticks": ticks,
        "config": {"workload": wl["desc"], "subscribers_per_gpu": n_subs, "subscribers_total": n_subs * world,
                   "events_per_step": B, "ring_cap": R, "record_bytes": 32, "mode": "overwrite-oldest throughput mode",
                   "digest": not args.no_digest, "timers_per_sub": K_timers, "warmup_settle_steps": settle, "store_path": args.store,
                   "parallelism": f"subscriber shards x{world}" + (f", ingest: {ingest_mode}" if world > 1 else ""),
                   "l2": f"inputs larger than L2: {n_subs * R * 32 / 2**30:.1f} GiB of rings per GPU, "
                         f"{d_local * 32 / 2**20:.0f} MiB written per step vs 126 MB L2",
                   "trace": f"splitmix-seeded {'Zipf' if wl['zipf'] else 'uniform'} codes 1..16, 4096 sources, {n_trace_batches} batches cycled with re-stamped seq/ts"},
        "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu, "gpu_launches": int(launches), "gpu_launches_e2e": int(launches_e2e),
        "clocks": sampler.summary(), "parity_checked": bool(parity and parity["ok"]) if parity is not None else False,
        "parity": parity if parity is not None else {"skipped": "--no-verify"},
    }
    return res


def run_lossless_and_bridge(cx):
    """Two records beside the throughput-mode numbers (N = 1):
    * config 2's shape in LOSSLESS mode — the reference's only semantics (`sub.Rx <- event` blocks on a full channel,
      events/subscriber.go:30-32) — through the host API (cpbus_advance + cpbus_publish + cpbus_flush) with a device-side
      consumer (cpbus_consume_all) that keeps up, so no flush has to be refused;
    * the mailbox -> host bridge (cpbus_drain_many: one gather kernel + two D2H copies into pinned memory), records/s."""
    import torch
    import oracle_binding as ob
    from containerpilot_b200 import _native as nat
    from containerpilot_b200.bus import Bus, EVENT_DTYPE
    args, local, stream = cx.args, cx.local, cx.stream
    n_subs, B, R = 65_536, args.batch, args.ring
    steps = args.steps or 2000
    warmup = max(args.warmup, 3)
    rng = np.random.default_rng(0xC0DEB2A1)
    n_host = 256
    host = np.zeros(n_host * B, dtype=EVENT_DTYPE)
    host["code"] = rng.integers(1, 17, n_host * B); host["source_id"] = rng.integers(0, 4096, n_host * B)
    bus = Bus(n_subs, ring_cap=R, batch_cap=B, lossless=True, digest=True, device=local, stream=stream.cuda_stream)
    bus.subscribe_many(np.full(n_subs, nat.MASK_ALL, dtype=np.uint32))
    orc = ob.Oracle(1, keep_window=8); orc.subscribe()
    step = [0]

    def go(k):
        for _ in range(k):
            i = step[0]
            lo = (i % n_host) * B
            nat.check(bus.advance((i + 1) * B * DT_NS), "cpbus_advance")
            nat.check(bus.publish_many(host[lo:lo + B]), "cpbus_publish")
            nat.check(bus.flush(), "cpbus_flush")                # never EAGAIN: the consumer keeps up
            bus.consume_all()
            step[0] = i + 1
    go(warmup); torch.cuda.synchronize()
    s0 = bus.stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record(stream); go(steps); e1.record(stream)
    torch.cuda.synchronize()
    ms = max(e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3)
    s1 = bus.stats()
    for i in range(step[0]):                                     # the delivered sequence is the same as in throughput mode
        lo = (i % n_host) * B
        orc.advance((i + 1) * B * DT_NS)
        orc.publish_many(host["code"][lo:lo + B], host["source_id"][lo:lo + B])
    dg = bus.digests(0, n_subs)
    ok = bool((dg["count"] == orc.count(0)).all() and (dg["digest"] == orc.digest(0)).all() and s1["overwritten"] == 0)
    deliveries = s1["deliveries"] - s0["deliveries"]
    lossless = {"name": "config2-lossless", "workload": "config 2's shape in lossless mode (reference semantics) with a device consumer that keeps up",
                "value": deliveries / (ms * 1e-3), "unit": "deliveries/s", "steps": steps, "ms_per_step": ms / steps,
                "api": "cpbus_advance + cpbus_publish(host events) + cpbus_flush + cpbus_consume_all per step, host buffers",
                "admit_passes": s1["admit_passes"] - s0["admit_passes"], "admit_skipped": s1["admit_skipped"] - s0["admit_skipped"],
                "parity_checked": ok, "config": {"subscribers_per_gpu": n_subs, "events_per_step": B, "ring_cap": R, "mode": "lossless"}}
    # ---- bridge: what moving mailboxes back to host channels costs (the shim's pump, INTEGRATION.md §4) ----
    n_drain = 8192
    pinned = torch.empty((n_drain * B, 32), dtype=torch.uint8).pin_memory()
    out = pinned.numpy().view(EVENT_DTYPE).reshape(-1)
    times, total = [], 0
    for rep in range(4):
        i = step[0]
        nat.check(bus.advance((i + 1) * B * DT_NS), "cpbus_advance")
        nat.check(bus.publish_many(host[:B]), "cpbus_publish"); nat.check(bus.flush(), "cpbus_flush"); bus.sync()
        step[0] = i + 1
        t0 = time.perf_counter()
        _, offs, cnts = bus.drain_many(0, n_drain, n_drain * B, out=out)
        dt = time.perf_counter() - t0
        if rep:                                                  # first call allocates the device staging
            times.append(dt); total = int(cnts.sum())
        bus.consume_all()
    med = float(np.median(times))
    bridge = {"name": "bridge", "workload": f"cpbus_drain_many: {n_drain} mailboxes x {B} records -> pinned host memory (one gather kernel + two D2H copies)",
              "value": total / med, "unit": "records/s", "gb_per_s": total * 32 / med / 1e9, "ms_per_call": med * 1e3, "records_per_call": total}
    bus.close()
    return lossless, bridge


DUMP_SUBS, DUMP_WINDOWS = 65_536, 64


def _words(a) -> np.ndarray:
    """Unsigned integers as float64, 64-bit ones split into their two 32-bit halves (low first): exact at any value."""
    return np.ascontiguousarray(a).view(np.uint32).astype(np.float64)


def dump_outputs(out_dir, name, bus, first, n_subs, ring_cap):
    """What a caller reads back after the timed fan-out's last step, for this rank's shard: delivered count and digest of
    a seeded sample of subscribers, the mailbox windows (what cpbus_peek_window returns) of a smaller sample, and the
    shard's digest fold.  The sample depends only on the subscriber count; a configuration writes at most 7 MB."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0xC0DEB2D0)
    subs = np.sort(rng.choice(n_subs, min(n_subs, DUMP_SUBS), replace=False))
    dg = bus.digests(first, n_subs)[subs]
    win_subs = np.sort(rng.choice(subs, min(len(subs), DUMP_WINDOWS), replace=False))
    windows = np.full((len(win_subs), ring_cap, 8), -1.0)     # 8 words per record; rows of -1 past a short window
    for k, s in enumerate(win_subs):
        w = _words(bus.peek_window(first + int(s))).reshape(-1, 8)
        windows[k, :len(w)] = w
    arrays = {"subscribers": (first + subs).astype(np.float64), "count": _words(dg["count"]).reshape(-1, 2),
              "digest": _words(dg["digest"]).reshape(-1, 2), "window_subscribers": (first + win_subs).astype(np.float64),
              "windows": windows, "fold": _words(np.array(bus.digest_fold(first, n_subs), dtype=np.uint64)).reshape(4, 2)}
    for key, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}_{key}.npy"), a)


def verify(cx, name, sb, log, base, masks, n_subs, B, K_timers, timer_src0, slot_hist, make_records):
    """After the timed regions: (1) sampled subscribers of this shard — count, order-sensitive digest and the last-1024
    window — against a 1-subscriber oracle placed at that global id and fed the exact batches the bench issued; (2) the
    shard's total delivered count in closed form; (3) the digest fold reduced across ranks.  All ranks must agree."""
    import torch
    import oracle_binding as ob
    from containerpilot_b200.bus import EVENT_DTYPE
    dist, world, rank, dev = cx.dist, cx.world, cx.rank, cx.dev
    bus, first = sb.bus, sb.first
    bus.sync()
    t0 = time.perf_counter()
    rng = np.random.default_rng(1234 + rank)
    sample = sorted({0, n_subs - 1, n_subs // 2, int(rng.integers(0, n_subs))})
    orcs = []
    for s in sample:
        o = ob.Oracle(1, timers_per_sub=K_timers, keep_window=1024, sub_id_base=first + s)
        o.subscribe(int(masks[s]))
        if K_timers:
            o.timer_add(first + s, TICK_NS, timer_src0 + first + s, False)
        orcs.append(o)
    hist_total = np.zeros(17, dtype=np.int64)
    for kind, slot, seq0, t_ in log:
        rec = make_records(seq0, slot * B, (slot + 1) * B)
        if kind == "host":
            rec["ts_ns"] = t_                                  # cpbus_publish / CPBUS_PUT_STAMP: every record of the call carries the clock
        for o in orcs:
            assert o.publish_records(rec, t_) == 0
        if slot_hist is not None:
            hist_total += slot_hist[slot]
    mism = []
    for s, o in zip(sample, orcs):
        d = bus.digests(first + s, 1)
        if int(d["count"][0]) != o.count(first + s) or int(d["digest"][0]) != o.digest(first + s):
            mism.append(f"subscriber {first + s}: count {int(d['count'][0])} vs {o.count(first + s)}, digest {int(d['digest'][0]):#x} vs {o.digest(first + s):#x}")
        w = bus.peek_window(first + s)
        if w.tobytes() != o.mailbox(first + s)[-len(w):].tobytes():
            mism.append(f"subscriber {first + s}: last-{len(w)} window differs")
    # closed form of the shard total
    fold = bus.digest_fold(first, n_subs)
    if slot_hist is None:
        want_total = n_subs * orcs[0].count(first + sample[0])  # all-ones masks, identical timers: every mailbox has the same count
    else:
        bits = ((masks[:, None] >> np.arange(17, dtype=np.uint32)[None, :]) & 1).astype(np.int64)
        want_total = int((bits * hist_total[None, :]).sum())
    if int(fold[0]) != want_total % (1 << 64):
        mism.append(f"shard total count {int(fold[0])} vs closed form {want_total}")
    if slot_hist is None and not K_timers:                      # identical sequences: every digest equals the sampled one
        want_d = (n_subs * orcs[0].digest(first + sample[0])) % (1 << 64)
        if int(fold[1]) != want_d:
            mism.append("sum of digests differs from n_subs x the oracle digest")
    ok = not mism
    gfold = sb.digest_fold_all()
    if world > 1:
        t = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        all_ok = bool(int(t.item()))
    else:
        all_ok = ok
    if mism:
        print(f"[bench] PARITY MISMATCH ({name}, rank {rank}): " + "; ".join(mism[:6]), file=sys.stderr, flush=True)
    return {"ok": all_ok, "sampled_subscribers": [first + s for s in sample], "batches_replayed": len(log),
            "checks": "sampled subscribers: count + digest + last-1024 window vs 1-subscriber oracle over the issued trace; shard total count in closed form; digest fold across ranks",
            "digest_fold": [int(x) for x in gfold], "seconds": round(time.perf_counter() - t0, 2)}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    cx = Ctx()
    cx.args = args
    cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    cx.rank = int(os.environ.get("RANK", "0"))
    cx.local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; cpbus has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(cx.local)
    if cx.world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", cx.local))
    cx.dist = dist
    cx.dev = torch.device("cuda", cx.local)
    cx.stream = torch.cuda.Stream(device=cx.dev)
    torch.cuda.set_stream(cx.stream)

    names = ["config3", "config2", "config5"] if args.workload == "default" else [args.workload]
    if args.no_extras:
        names = names[:1]
    results = [run_config(cx, n, headline=(i == 0)) for i, n in enumerate(names)]
    ok = all(r["parity_checked"] for r in results) or args.no_verify
    side = []
    if cx.world == 1 and args.workload == "default" and not args.no_extras:
        lossless, bridge = run_lossless_and_bridge(cx)
        side = [lossless, bridge]
        ok = ok and lossless["parity_checked"]
    if cx.rank == 0:
        h = results[0]
        line = {
            "metric": METRIC, "value": h["value"], "unit": "deliveries/s", "n_gpus": cx.world,
            "steps": h["steps"], "warmup": max(args.warmup, 3), "ms_per_step": h["ms_per_step"], "higher_is_better": True,
            "scaling": h["scaling"], "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": h["config"],
            "publishes_per_s": h["publishes_per_s"], "deliveries": h["deliveries"], "ticks": h["ticks"],
            "roofline": h["roofline"], "cpu_baseline": h["cpu_baseline"], "e2e": h["e2e"], "gpu_launches": h["gpu_launches"],
            "gpu_launches_e2e": h["gpu_launches_e2e"], "clocks": h["clocks"], "parity_checked": h["parity_checked"], "parity": h["parity"],
            "extra_configs": [{k: r[k] for k in ("name", "workload", "scaling", "steps", "value", "unit", "ms_per_step", "publishes_per_s", "deliveries",
                                                  "ticks", "config", "roofline", "e2e", "gpu_launches", "clocks", "parity_checked", "parity")}
                              for r in results[1:]] + side,
        }
        print(json.dumps(line), flush=True)
    if cx.world > 1:
        dist.destroy_process_group()
    if not ok:
        sys.exit(3)


if __name__ == "__main__":
    main()
