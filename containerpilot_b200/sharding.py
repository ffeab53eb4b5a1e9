"""Multi-GPU bus (SURVEY.md §8e): the subscriber set partitions into contiguous shards, one `Bus` per GPU; rings,
control blocks and timers never move.  The only thing every shard must see is the publisher's batch sequence, and that
exchange is fused into the fan-out kernel (libcpbus `cpbus_stream_*`: a flagged ring in the publisher GPU's HBM that the
other GPUs' lead CTAs pull over NVLink) — there is no collective on the data path.  Because records carry GLOBAL
subscriber ids (`cpbus_config.sub_id_base`), a subscriber's sequence and digest do not depend on the shard count.

Two drivers over the same C-ABI:

* `ShardedBus`      — one process per GPU (`torch.distributed.run`); torch.distributed (NCCL or gloo) is used ONLY for the
                      construction handshake (the 64-byte CUDA-IPC handle) and for reducing statistics.
* `LocalShardedBus` — one process driving G buses (what a cgo shim inside the single ContainerPilot process does):
                      `cpbus_stream_attach`, peer access instead of IPC; also runs with all shards on ONE GPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat
from .bus import Bus, EVENT_DTYPE


def shard_range(n_total: int, world: int, rank: int) -> tuple[int, int]:
    """Contiguous, near-even partition: returns (first_global_id, count) of `rank`'s shard (libcpbus `cpbus_shard_range`, the
    partition `cpbus_create_sharded` uses)."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    first, count = C.c_uint32(), C.c_uint32()
    nat.check(nat.load().cpbus_shard_range(n_total, world, rank, C.byref(first), C.byref(count)), "cpbus_shard_range")
    return first.value, count.value


def owner_of(sub_id: int, n_total: int, world: int) -> int:
    """Rank that holds global subscriber `sub_id` (inverse of shard_range)."""
    base, extra = divmod(n_total, world)
    cut = extra * (base + 1)
    return sub_id // (base + 1) if sub_id < cut else extra + (sub_id - cut) // max(base, 1)


def stamp_trace(codes: np.ndarray, sources: np.ndarray, dt_ns: int, first_seq: int = 0) -> np.ndarray:
    """Complete 32-byte records for a device-resident trace: seq = publish ordinal, ts = (seq+1)*dt."""
    n = len(codes)
    ev = np.zeros(n, dtype=EVENT_DTYPE)
    ev["seq"] = first_seq + np.arange(n, dtype=np.uint64)
    ev["ts_ns"] = (first_seq + 1 + np.arange(n, dtype=np.uint64)) * np.uint64(dt_ns)
    ev["code"], ev["source_id"], ev["target"] = codes, sources, 0xFFFFFFFF
    return ev


def broadcast_events(dist, events_u8, src: int = 0):
    """Fallback ingest when no peer mapping can be made (no NVLink/IPC): broadcast a batch (uint8 tensor [n, 32] on the
    backend's device) from `src` with the collective backend — NCCL on GPUs, gloo in the CPU tests."""
    dist.broadcast(events_u8, src=src)
    return events_u8


class _ShardOps:
    """What both drivers share: a shard is a `Bus` plus its end of the publisher's stream."""

    bus: Bus
    first: int
    count: int

    # -- membership / timers on this shard (global ids) --------------------
    def subscribe_many(self, masks) -> int:
        return self.bus.subscribe_many(masks)

    def timer_add_many(self, period_ns: int, source_id0: int = 0, source_ids=None, oneshot: bool = False):
        self.bus.timer_add_many(self.first, self.count, period_ns, source_ids=source_ids,
                                source_id0=source_id0 + (0 if source_ids is not None else self.first), oneshot=oneshot)

    def digests(self):
        return self.bus.digests(self.first, self.count)


class ShardedBus(_ShardOps):
    """One rank's shard; constructed collectively by every rank of `dist` (torch.distributed, already initialised).

    Data path per step (SPMD: every rank knows n and now_ns of each batch):
        rank 0       : put(events, now_ns)            host batch -> the stream ring (H2D + release), may run ahead
        every rank   : fanout(n, now_ns)              one fan-out launch; the batch is pulled inside the kernel
    Device-resident traces (the publisher's events already in its HBM): attach_trace / fanout_trace.
    """

    def __init__(self, n_subs_total: int, dist=None, rank: int = 0, world: int = 1, device: int = -1, ring_cap: int = 1024,
                 batch_cap: int = 512, timers_per_sub: int = 0, digest: bool = True, stream_slots: int = 64,
                 stream=None, store_path: int = nat.STORE_AUTO, grid_ctas: int = 0, subs_per_rank: int | None = None,
                 bus_factory=Bus):
        self.dist, self.rank, self.world = dist, rank, world
        if subs_per_rank is not None:               # weak scaling: fixed shard size
            self.first, self.count = rank * subs_per_rank, subs_per_rank
        else:
            self.first, self.count = shard_range(n_subs_total, world, rank)
        self.bus = bus_factory(max(self.count, 1), ring_cap=ring_cap, batch_cap=batch_cap, timers_per_sub=timers_per_sub, digest=digest,
                       device=device, sub_id_base=self.first, store_path=store_path, stream=stream, grid_ctas=grid_ctas)
        self.batch_cap = batch_cap
        self._st = None
        self._peer_trace = None      # (mapped pointer, owner?) of the attached device trace
        self._trace_ptr = None
        self._trace_local = False
        self.ingest = "local"
        self._open_stream(stream_slots)

    # -- construction handshake -------------------------------------------
    def _all_ok(self, ok: bool) -> bool:
        if self.world == 1:
            return ok
        import torch
        dev = "cuda" if self.dist.get_backend() == "nccl" else "cpu"
        t = torch.tensor([1 if ok else 0], device=dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(int(t.item()))

    def _open_stream(self, slots: int):
        ok, handle = True, None
        if self.rank == 0:
            try:
                self._st, handle = self.bus.stream_create(slots, self.world)
            except nat.CpbusError as ex:                    # pragma: no cover - depends on the box
                self._err = ex
                ok, handle = False, None
        if self.world > 1:
            box = [handle]
            self.dist.broadcast_object_list(box, src=0)
            if self.rank != 0:
                if box[0] is None:
                    ok = False
                else:
                    try:
                        self._st = self.bus.stream_open(box[0], self.rank)
                    except nat.CpbusError as ex:            # pragma: no cover
                        self._err = ex
                        ok = False
        self.stream_ok = self._all_ok(ok)
        if self.stream_ok:
            self.ingest = "nvlink-stream (flagged ring, pulled inside the fan-out kernel)" if self.world > 1 else "local stream"

    # -- host batches ------------------------------------------------------
    def put(self, events: np.ndarray, now_ns: int, raw: bool = False) -> int:
        """Publisher rank only (no-op elsewhere).  EAGAIN: the consumers are a whole ring behind."""
        if self.rank != 0:
            return nat.OK
        return self.bus.stream_put(self._st, events, now_ns, raw)

    def fanout(self, n: int, now_ns: int) -> int:
        return self.bus.stream_fanout(self._st, n, now_ns)

    def publish(self, events: np.ndarray, now_ns: int) -> int:
        """put + fanout for callers that do not pipeline."""
        rc = self.put(events, now_ns)
        return rc if rc else self.fanout(len(events), now_ns)

    # -- device-resident trace (publisher's events already in its HBM) ----
    def attach_trace(self, nbytes: int):
        """Rank 0 allocates a shareable buffer of `nbytes` and returns its device pointer (fill it, then call
        `trace_ready()`); the other ranks map it over NVLink.  Returns the local pointer on rank 0, None elsewhere."""
        ok, handle, ptr = True, None, None
        if self.rank == 0:
            try:
                ptr, handle = self.bus.shared_alloc(nbytes)
            except nat.CpbusError as ex:                    # pragma: no cover
                self._err = ex
                ok = False
        if self.world > 1:
            box = [handle]
            self.dist.broadcast_object_list(box, src=0)
            if self.rank != 0:
                if box[0] is None:
                    ok = False
                else:
                    try:
                        self._peer_trace = self.bus.shared_open(box[0])
                    except nat.CpbusError as ex:            # pragma: no cover
                        self._err = ex
                        ok = False
        self.trace_ok = self._all_ok(ok)
        self._trace_ptr = ptr if self.rank == 0 else self._peer_trace
        if self.trace_ok and self.world > 1:
            self.ingest = "nvlink-peer-pull (fused into the fan-out kernel)"
        return ptr

    def use_local_trace(self, ptr: int):
        """The trace already sits in THIS GPU's memory at `ptr` (single GPU, or a replicated / NCCL-broadcast copy)."""
        self._trace_ptr, self._trace_local = ptr, True

    def fanout_trace(self, offset_bytes: int, n: int, watermark_ns: int, next_offset_bytes: int | None = None, next_n: int = 0) -> int:
        """Fan out records [offset, offset + 32 n) of the attached trace; `next_offset_bytes` names a LATER batch (best: the
        one after next) that this launch pulls across the link while its stores are in flight."""
        base = self._trace_ptr
        if self.world == 1 or self._trace_local:
            return self.bus.publish_device(base + offset_bytes, n, watermark_ns)
        nxt = base + next_offset_bytes if next_offset_bytes is not None else 0
        return self.bus.publish_device_staged(base + offset_bytes, n, watermark_ns, nxt, next_n if nxt else 0)

    def fanout_broadcast(self, batch_u8, n: int, watermark_ns: int) -> int:
        """Fallback (no peer mapping): `batch_u8` is a [n, 32] uint8 CUDA tensor, valid on rank 0; NCCL broadcast, then a
        local fan-out.  One collective per call — the caller batches several steps per call to amortise it."""
        if self.world > 1:
            broadcast_events(self.dist, batch_u8, src=0)
        return self.bus.publish_device(batch_u8.data_ptr(), n, watermark_ns)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    # -- reductions (verification, statistics) -----------------------------
    def digest_fold_all(self):
        """(sum count, sum digest, xor H(digest, count, id), n) over EVERY shard — equal for any shard count."""
        f = self.bus.digest_fold(self.first, self.count)
        if self.world == 1:
            return f
        gathered = [None] * self.world
        self.dist.all_gather_object(gathered, tuple(int(x) for x in f))
        M = (1 << 64) - 1
        c = d = x = n = 0
        for g in gathered:
            c = (c + g[0]) & M; d = (d + g[1]) & M; x ^= g[2]; n += g[3]
        return (c, d, x, n)

    def close(self):
        if self._peer_trace is not None:
            try:
                self.bus.shared_close(self._peer_trace)
            except nat.CpbusError:                          # pragma: no cover - teardown only
                pass
            self._peer_trace = None
        if self.world > 1 and self.rank != 0 and self._st is not None:
            self.bus.stream_close(self._st); self._st = None   # importers unmap before the owner frees
        if self.world > 1:
            self.dist.barrier()
        if self._st is not None:
            self.bus.stream_close(self._st); self._st = None
        self.bus.close()


class LocalShardedBus:
    """G shards driven by ONE process (shard g on `devices[g]`; all on one GPU is allowed): what a cgo shim inside the
    single ContainerPilot process does.  Same stream protocol as `ShardedBus`, attached in-process."""

    def __init__(self, n_subs_total: int, devices, ring_cap: int = 1024, batch_cap: int = 512, timers_per_sub: int = 0,
                 digest: bool = True, stream_slots: int = 64):
        self.world = len(devices)
        self.shards = []
        for g, dev in enumerate(devices):
            first, count = shard_range(n_subs_total, self.world, g)
            self.shards.append((first, count, Bus(max(count, 1), ring_cap=ring_cap, batch_cap=batch_cap, timers_per_sub=timers_per_sub,
                                                  digest=digest, device=dev, sub_id_base=first)))
        pub = self.shards[0][2]
        st0, _ = pub.stream_create(stream_slots, self.world)
        self._st = [st0] + [self.shards[g][2].stream_attach(st0, g) for g in range(1, self.world)]

    def bus_of(self, sub_id: int) -> Bus:
        for first, count, bus in self.shards:
            if first <= sub_id < first + count:
                return bus
        raise KeyError(sub_id)

    def subscribe_many(self, masks):
        """global masks array, split by shard"""
        masks = np.asarray(masks, dtype=np.uint32)
        for first, count, bus in self.shards:
            if count:
                bus.subscribe_many(masks[first:first + count])

    def timer_add_many(self, period_ns: int, source_id0: int = 0):
        for first, count, bus in self.shards:
            if count:
                bus.timer_add_many(first, count, period_ns, source_id0=source_id0 + first)

    def publish(self, events: np.ndarray, now_ns: int, raw: bool = False):
        """One batch to every shard: put once, fan out on each GPU (never ahead of its own fan-outs, so it may wait)."""
        nat.check(self.shards[0][2].stream_put(self._st[0], events, now_ns, raw), "cpbus_stream_put")
        self.fanout(len(events), now_ns)

    def put(self, events: np.ndarray, now_ns: int, raw: bool = False) -> int:
        """Run ahead of the fan-outs.  One thread drives publisher and consumers here, so this never waits: EAGAIN means
        "fan out (or sync) first" — the slot's previous batch has not been pulled by every shard yet."""
        return self.shards[0][2].stream_put(self._st[0], events, now_ns, raw, nowait=True)

    def fanout(self, n: int, now_ns: int):
        for g, (_, _, bus) in enumerate(self.shards):
            nat.check(bus.stream_fanout(self._st[g], n, now_ns), "cpbus_stream_fanout")

    def sync(self):
        for _, _, bus in self.shards:
            bus.sync()

    def digests(self):
        """(count, digest) of every subscriber, in global id order"""
        parts = [bus.digests(first, count) for first, count, bus in self.shards if count]
        return np.concatenate(parts)

    def close(self):
        for g in range(self.world - 1, -1, -1):
            self.shards[g][2].stream_close(self._st[g])
        for _, _, bus in self.shards:
            bus.close()
