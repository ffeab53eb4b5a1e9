"""`Bus`: a thin numpy-friendly wrapper over the libcpbus C-ABI (include/cpbus.h).

One `Bus` = one GPU's shard of subscriber mailboxes.  Every method maps 1:1 to a
`cpbus_*` entry point; no event ever takes a Python/CPU data path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat

EVENT_DTYPE = np.dtype([("seq", "<u8"), ("ts_ns", "<u8"), ("code", "<u4"), ("source_id", "<u4"),
                        ("target", "<u4"), ("flags", "<u4")])
assert EVENT_DTYPE.itemsize == 32


class Bus:
    def __init__(self, n_max_subs: int, ring_cap: int = 1024, batch_cap: int = 256, timers_per_sub: int = 0,
                 lossless: bool = False, digest: bool = True, device: int = -1, sub_id_base: int = 0,
                 store_path: int = nat.STORE_AUTO, stream: int | None = None, grid_ctas: int = 0, devices=None):
        """`devices`: a list of CUDA ordinals makes this ONE handle over len(devices) shards (`cpbus_create_sharded`):
        shard k on devices[k], the same ids, records and digests as one bus with the same arguments; `device` is then
        ignored."""
        self._lib = nat.load()
        cfg = nat.Config()
        cfg.n_max_subs, cfg.ring_cap, cfg.batch_cap, cfg.timers_per_sub = n_max_subs, ring_cap, batch_cap, timers_per_sub
        cfg.flags = (nat.CFG_LOSSLESS if lossless else 0) | (nat.CFG_DIGEST if digest else 0)
        cfg.device, cfg.sub_id_base, cfg.store_path, cfg.grid_ctas = device, sub_id_base, store_path, grid_ctas
        cfg.stream = C.c_void_p(stream) if stream else None
        self._h = C.c_void_p()
        if devices is None:
            nat.check(self._lib.cpbus_create(C.byref(cfg), C.byref(self._h)), "cpbus_create")
        else:
            devs = (C.c_int32 * max(1, len(devices)))(*devices)
            nat.check(self._lib.cpbus_create_sharded(C.byref(cfg), devs, len(devices), C.byref(self._h)), "cpbus_create_sharded")
        self.ring_cap, self.batch_cap, self.sub_id_base = ring_cap, batch_cap, sub_id_base

    # -- lifecycle ---------------------------------------------------------
    def close(self):
        if self._h:
            self._lib.cpbus_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- intern ------------------------------------------------------------
    def intern(self, s: str) -> int:
        raw = s.encode()
        out = C.c_uint32()
        nat.check(self._lib.cpbus_intern(self._h, raw, len(raw), C.byref(out)), "cpbus_intern")
        return out.value

    def intern_ephemeral(self, s: str) -> int:
        """payload strings (Metric "key|value"): ids from the bounded, recycled region"""
        raw = s.encode()
        out = C.c_uint32()
        nat.check(self._lib.cpbus_intern_ephemeral(self._h, raw, len(raw), C.byref(out)), "cpbus_intern_ephemeral")
        return out.value

    def source(self, source_id: int) -> str:
        n = C.c_size_t()
        nat.check(self._lib.cpbus_source(self._h, source_id, None, 0, C.byref(n)), "cpbus_source")
        buf = C.create_string_buffer(max(1, n.value))
        nat.check(self._lib.cpbus_source(self._h, source_id, buf, n.value, C.byref(n)), "cpbus_source")
        return buf.raw[: n.value].decode()

    # -- membership --------------------------------------------------------
    def subscribe(self, mask: int = nat.MASK_ALL) -> int:
        out = C.c_uint32()
        nat.check(self._lib.cpbus_subscribe(self._h, mask, C.byref(out)), "cpbus_subscribe")
        return out.value

    def subscribe_many(self, masks) -> int:
        m = np.ascontiguousarray(masks, dtype=np.uint32)
        out = C.c_uint32()
        nat.check(self._lib.cpbus_subscribe_many(self._h, m.ctypes.data, m.size, C.byref(out)), "cpbus_subscribe_many")
        return out.value

    def subscribe_pairs(self, mask: int, pairs) -> int:
        """second-level filter: `pairs` = exact (code, source_id) cases delivered on top of the code mask"""
        pr = np.ascontiguousarray([(int(c), int(s)) for c, s in pairs], dtype=np.uint32).reshape(-1, 2)
        out = C.c_uint32()
        nat.check(self._lib.cpbus_subscribe_pairs(self._h, mask, pr.ctypes.data if len(pr) else None, len(pr), C.byref(out)),
                  "cpbus_subscribe_pairs")
        return out.value

    def subscribe_pairs_many(self, masks, pairs_per_sub) -> int:
        """a whole fleet in one call: masks[i] and pairs_per_sub[i] = list of (code, source_id), at most 16 each"""
        m = np.ascontiguousarray(masks, dtype=np.uint32)
        n = m.size
        rows = np.full((n, 16, 2), 0xFFFFFFFF, dtype=np.uint32)
        cnt = np.zeros(n, dtype=np.uint32)
        for i, pr in enumerate(pairs_per_sub):
            if len(pr) > 16:
                raise nat.CpbusError(nat.EINVAL, "cpbus_subscribe_pairs_many")
            cnt[i] = len(pr)
            if len(pr):
                rows[i, :len(pr)] = np.asarray(pr, dtype=np.uint32).reshape(-1, 2)
        out = C.c_uint32()
        nat.check(self._lib.cpbus_subscribe_pairs_many(self._h, m.ctypes.data, rows.ctypes.data, cnt.ctypes.data, n, C.byref(out)),
                  "cpbus_subscribe_pairs_many")
        return out.value

    def set_mask(self, sub_id: int, mask: int):
        nat.check(self._lib.cpbus_set_mask(self._h, sub_id, mask), "cpbus_set_mask")

    def unsubscribe(self, sub_id: int):
        nat.check(self._lib.cpbus_unsubscribe(self._h, sub_id), "cpbus_unsubscribe")

    # -- timers ------------------------------------------------------------
    def timer_add(self, sub_id: int, period_ns: int, source_id: int, oneshot: bool = False) -> int:
        out = C.c_uint32()
        nat.check(self._lib.cpbus_timer_add(self._h, sub_id, period_ns, source_id, int(oneshot), C.byref(out)), "cpbus_timer_add")
        return out.value

    def timer_add_many(self, first_sub: int, n: int, period_ns: int, source_ids=None, source_id0: int = 0, oneshot: bool = False):
        ptr = None
        if source_ids is not None:
            arr = np.ascontiguousarray(source_ids, dtype=np.uint32)
            ptr = arr.ctypes.data
        nat.check(self._lib.cpbus_timer_add_many(self._h, first_sub, n, period_ns, ptr, source_id0, int(oneshot)), "cpbus_timer_add_many")

    def timer_cancel(self, timer_id: int):
        nat.check(self._lib.cpbus_timer_cancel(self._h, timer_id), "cpbus_timer_cancel")

    # -- hot path ----------------------------------------------------------
    def publish(self, code: int, source_id: int = 0) -> int:
        ev = nat.Event(0, 0, code, source_id, 0, 0)
        return self._lib.cpbus_publish(self._h, C.byref(ev), 1)

    def publish_many(self, events: np.ndarray) -> int:
        """events: EVENT_DTYPE array (only code/source_id are read)."""
        ev = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
        return self._lib.cpbus_publish(self._h, ev.ctypes.data, ev.size)

    def send(self, sub_id: int, code: int, source_id: int = 0) -> int:
        ev = nat.Event(0, 0, code, source_id, 0, 0)
        return self._lib.cpbus_send(self._h, sub_id, C.byref(ev))

    def advance(self, now_ns: int) -> int:
        return self._lib.cpbus_advance(self._h, now_ns)

    def flush(self) -> int:
        return self._lib.cpbus_flush(self._h)

    def sync(self):
        nat.check(self._lib.cpbus_sync(self._h), "cpbus_sync")

    def publish_device(self, dev_ptr: int, n: int, watermark_ns: int) -> int:
        return self._lib.cpbus_publish_device(self._h, C.c_void_p(dev_ptr), n, watermark_ns)

    def publish_device_staged(self, dev_ptr: int, n: int, watermark_ns: int, next_ptr: int = 0, next_n: int = 0) -> int:
        """dev_ptr / next_ptr may be peer-mapped pointers into another GPU's HBM (fused NVLink ingest)."""
        return self._lib.cpbus_publish_device_staged(self._h, C.c_void_p(dev_ptr), n, watermark_ns,
                                                     C.c_void_p(next_ptr) if next_ptr else None, next_n)

    # -- the publisher's stream across GPUs (one process per GPU) ------------
    def stream_create(self, n_slots: int, n_consumers: int):
        """publisher rank: (stream handle, 64-byte IPC handle for the other ranks)"""
        st, handle = C.c_void_p(), C.create_string_buffer(64)
        nat.check(self._lib.cpbus_stream_create(self._h, n_slots, n_consumers, C.byref(st), handle), "cpbus_stream_create")
        return st, handle.raw

    def stream_open(self, handle: bytes, consumer_index: int):
        st = C.c_void_p()
        nat.check(self._lib.cpbus_stream_open(self._h, handle, consumer_index, C.byref(st)), "cpbus_stream_open")
        return st

    def stream_attach(self, owner_stream, consumer_index: int):
        """same-process consumer of a stream created by another Bus of this process (peer access instead of IPC)"""
        st = C.c_void_p()
        nat.check(self._lib.cpbus_stream_attach(self._h, owner_stream, consumer_index, C.byref(st)), "cpbus_stream_attach")
        return st

    def stream_put(self, st, events: np.ndarray, now_ns: int, raw: bool = False, nowait: bool = False) -> int:
        ev = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
        flags = (nat.PUT_RAW if raw else nat.PUT_STAMP) | (nat.PUT_NOWAIT if nowait else 0)
        return self._lib.cpbus_stream_put(st, ev.ctypes.data if ev.size else None, ev.size, now_ns, flags)

    def stream_fanout(self, st, n: int, now_ns: int) -> int:
        return self._lib.cpbus_stream_fanout(st, n, now_ns)

    def stream_poll(self, st):
        """(n, now_ns) of the next batch if the publisher has released it, else None — for consumers that are not told"""
        ready, n, now = C.c_int(), C.c_size_t(), C.c_uint64()
        nat.check(self._lib.cpbus_stream_poll(st, C.byref(ready), C.byref(n), C.byref(now)), "cpbus_stream_poll")
        return (n.value, now.value) if ready.value else None

    def stream_status(self, st) -> int:
        return self._lib.cpbus_stream_status(st)

    def stream_set_timeout(self, st, microseconds: int):
        nat.check(self._lib.cpbus_stream_set_timeout(st, microseconds), "cpbus_stream_set_timeout")

    def stream_close(self, st):
        nat.check(self._lib.cpbus_stream_close(st), "cpbus_stream_close")

    def shared_alloc(self, nbytes: int):
        """(device pointer, 64-byte IPC handle) of a new buffer on this bus's GPU, mappable by the other GPUs."""
        ptr, handle = C.c_void_p(), C.create_string_buffer(64)
        nat.check(self._lib.cpbus_shared_alloc(self._h, nbytes, C.byref(ptr), handle), "cpbus_shared_alloc")
        return ptr.value, handle.raw

    def shared_open(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        nat.check(self._lib.cpbus_shared_open(self._h, handle, C.byref(ptr)), "cpbus_shared_open")
        return ptr.value

    def shared_close(self, ptr: int):
        nat.check(self._lib.cpbus_shared_close(self._h, C.c_void_p(ptr)), "cpbus_shared_close")

    # -- consumer side -----------------------------------------------------
    def drain(self, sub_id: int, cap: int | None = None):
        cap = cap or self.ring_cap
        out = np.zeros(cap, dtype=EVENT_DTYPE)
        n, lost = C.c_size_t(), C.c_uint64()
        nat.check(self._lib.cpbus_drain(self._h, sub_id, out.ctypes.data, cap, C.byref(n), C.byref(lost)), "cpbus_drain")
        return out[: n.value]

    def consume_all(self):
        """device-side consumer: every mailbox read to the end, records discarded"""
        nat.check(self._lib.cpbus_consume_all(self._h), "cpbus_consume_all")

    def drain_many(self, first_sub: int, n: int, cap: int, out=None):
        """Bulk drain: returns (records, offsets, counts); mailbox i's FIFO run is records[offsets[i]:offsets[i]+counts[i]].
        `out`: a preallocated EVENT_DTYPE array of at least `cap` records (pinned memory makes the D2H a straight DMA)."""
        if out is None:
            out = np.zeros(cap, dtype=EVENT_DTYPE)
        offs, cnts = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint32)
        total = C.c_size_t()
        nat.check(self._lib.cpbus_drain_many(self._h, first_sub, n, out.ctypes.data, cap, offs.ctypes.data, cnts.ctypes.data,
                                             C.byref(total)), "cpbus_drain_many")
        return out, offs, cnts

    def peek_window(self, sub_id: int, cap: int | None = None) -> np.ndarray:
        cap = cap or self.ring_cap
        out = np.zeros(cap, dtype=EVENT_DTYPE)
        n = C.c_size_t()
        nat.check(self._lib.cpbus_peek_window(self._h, sub_id, out.ctypes.data, cap, C.byref(n)), "cpbus_peek_window")
        return out[: n.value]

    def digests(self, first_sub: int, n: int):
        out = np.zeros(n, dtype=[("count", "<u8"), ("digest", "<u8")])
        nat.check(self._lib.cpbus_digest(self._h, first_sub, n, out.ctypes.data), "cpbus_digest")
        return out

    def digest_fold(self, first_sub: int, n: int):
        out = (C.c_uint64 * 4)()
        nat.check(self._lib.cpbus_digest_fold(self._h, first_sub, n, C.byref(out)), "cpbus_digest_fold")
        return tuple(out)

    def digest_fold_begin(self, first_sub: int, n: int) -> int:
        t = C.c_uint32()
        nat.check(self._lib.cpbus_digest_fold_begin(self._h, first_sub, n, C.byref(t)), "cpbus_digest_fold_begin")
        return t.value

    def digest_fold_end(self, ticket: int):
        out = (C.c_uint64 * 4)()
        nat.check(self._lib.cpbus_digest_fold_end(self._h, ticket, C.byref(out)), "cpbus_digest_fold_end")
        return tuple(out)

    def step_result_begin(self) -> int:
        t = C.c_uint32()
        nat.check(self._lib.cpbus_step_result_begin(self._h, C.byref(t)), "cpbus_step_result_begin")
        return t.value

    def step_result_end(self, ticket: int):
        out = (C.c_uint64 * 4)()
        nat.check(self._lib.cpbus_step_result_end(self._h, ticket, C.byref(out)), "cpbus_step_result_end")
        return tuple(out)

    def debug_events(self):
        out = np.zeros(10, dtype=EVENT_DTYPE)
        n = C.c_size_t()
        nat.check(self._lib.cpbus_debug_events(self._h, out.ctypes.data, 10, C.byref(n)), "cpbus_debug_events")
        return out[: n.value]

    def stats(self) -> dict:
        st = nat.Stats()
        nat.check(self._lib.cpbus_stats(self._h, C.byref(st)), "cpbus_stats")
        d = {k: getattr(st, k) for k, _ in nat.Stats._fields_ if k != "published_by_code"}
        d["published_by_code"] = list(st.published_by_code)
        return d

    def publish_counts(self) -> dict:
        """{(code, source_id): count} — the reference's containerpilot_events{code, source} counter (Metric excluded)"""
        n = C.c_size_t()
        nat.check(self._lib.cpbus_publish_counts(self._h, None, 0, C.byref(n)), "cpbus_publish_counts")
        buf = (nat.PairCount * max(1, n.value))()
        nat.check(self._lib.cpbus_publish_counts(self._h, buf, n.value, C.byref(n)), "cpbus_publish_counts")
        return {(buf[i].code, buf[i].source_id): buf[i].count for i in range(n.value)}

    def device_ptrs(self) -> dict:
        ring, ctl = C.c_void_p(), C.c_void_p()
        nat.check(self._lib.cpbus_device_ptrs(self._h, C.byref(ring), C.byref(ctl)), "cpbus_device_ptrs")
        return {"ring": ring.value, "ctl": ctl.value}
