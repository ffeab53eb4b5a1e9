"""One bus handle over several shards (cpbus_create_sharded): every value a caller reads back equals what one bus created
with the same configuration returns.  Shards sit on devices i % device_count, so a one-GPU box runs everything with the
shards sharing device 0; the cases that need distinct GPUs skip there."""
import os
import subprocess

import numpy as np
import pytest

import oracle_binding as ob
from containerpilot_b200 import _native as nat
from containerpilot_b200 import events
from containerpilot_b200.bus import Bus, EVENT_DTYPE

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ndev():
    import torch
    return torch.cuda.device_count()


def _devices(g, distinct=False):
    n = _ndev()
    if distinct and n < g:
        pytest.skip(f"needs {g} GPUs, {n} visible")
    return [i % n for i in range(g)]


RC_METHODS = {"publish_many", "send", "advance", "flush", "publish_device"}   # Bus methods that return the status


def _call(fn, *a, **kw):
    """(status, value) of a Bus call, whether the method returns its status or raises it"""
    try:
        r = fn(*a, **kw)
    except nat.CpbusError as e:
        return e.status, None
    if getattr(fn, "__name__", "") in RC_METHODS:
        return r, None
    return nat.OK, r


def _view(x):
    if isinstance(x, np.ndarray):
        return x.tobytes()
    if isinstance(x, tuple):
        return tuple(_view(v) for v in x)
    if isinstance(x, dict):
        return {k: _view(v) for k, v in x.items()}
    return x


def _readback(bus, n_max, log):
    """everything a caller can read without consuming"""
    st = bus.stats()
    st.pop("batches"); st.pop("kernel_launches")
    log.append(("stats", st))
    log.append(("debug", _view(bus.debug_events())))
    log.append(("counts", bus.publish_counts()))
    n = st["n_subs"]
    log.append(("digests_all", _view(_call(lambda: bus.digests(bus.sub_id_base, n_max)))))
    ok, d = _call(lambda: bus.digest_fold(bus.sub_id_base, max(1, n)))
    log.append(("fold", ok, d))
    t = bus.step_result_begin()
    log.append(("step", bus.step_result_end(t)))


def _mixed_trace(bus, seed, n_max, log):
    """The same random sequence of calls on any Bus; every status and readback goes to `log`."""
    rng = np.random.default_rng(seed)
    base = bus.sub_id_base
    B, R = bus.batch_cap, bus.ring_cap
    src = [bus.intern(f"src-{i}") for i in range(8)]
    log.append(("intern", src, bus.intern_ephemeral("k|1"), bus.source(src[3])))
    timers, now = [], 0
    for step in range(160):
        op = rng.integers(0, 16)
        if op == 0:
            k = int(rng.integers(1, 9))
            masks = np.where(rng.random(k) < 0.5, nat.MASK_ALL, rng.integers(0, 1 << 17, k)).astype(np.uint32)
            log.append(("sub_many", _call(bus.subscribe_many, masks)))
        elif op == 1:
            log.append(("sub", _call(bus.subscribe, int(rng.integers(0, 1 << 17)))))
        elif op == 2:
            k = int(rng.integers(1, 6))
            pairs = [[(int(rng.integers(0, 17)), src[int(rng.integers(0, 8))]) for _ in range(int(rng.integers(0, 4)))] for _ in range(k)]
            masks = rng.integers(0, 1 << 17, k).astype(np.uint32) & np.uint32(0x1FF0)
            log.append(("sub_pairs_many", _call(bus.subscribe_pairs_many, masks, pairs)))
        elif op == 3:
            log.append(("sub_pairs", _call(bus.subscribe_pairs, 1 << 3, [(5, src[1]), (7, src[2])])))
        elif op == 4:
            log.append(("unsub", _call(bus.unsubscribe, base + int(rng.integers(0, n_max + 2)))))
        elif op == 5:
            log.append(("mask", _call(bus.set_mask, base + int(rng.integers(0, n_max + 2)), int(rng.integers(0, 1 << 17)))))
        elif op == 6:
            r = _call(bus.timer_add, base + int(rng.integers(0, n_max)), int(rng.choice([20_000, 50_000])), src[0],
                      oneshot=bool(rng.integers(0, 2)))
            log.append(("timer", r))
            if r[0] == nat.OK:
                timers.append(r[1])
        elif op == 7 and timers:
            log.append(("cancel", _call(bus.timer_cancel, timers[int(rng.integers(0, len(timers)))])))
        elif op == 8:
            f = int(rng.integers(0, n_max)); k = int(rng.integers(1, 12))
            log.append(("timer_many", _call(bus.timer_add_many, base + f, k, 50_000, source_id0=src[4])))
        elif op in (9, 10):
            n = int(rng.integers(1, int(2.5 * B)))
            ev = np.zeros(n, dtype=EVENT_DTYPE)
            ev["code"] = rng.integers(0, 17, n); ev["source_id"] = np.array(src)[rng.integers(0, 8, n)]
            log.append(("publish", _call(bus.publish_many, ev)))
        elif op == 11:
            for _ in range(int(rng.integers(1, 6))):
                log.append(("send", _call(bus.send, base + int(rng.integers(0, n_max + 1)), int(rng.integers(0, 17)), src[5])))
        elif op == 12:
            now += int(rng.choice([1_000, 30_000, 3_000_000]))   # 3 ms: wider than the 20 us timers' window
            log.append(("advance", _call(bus.advance, now)))
        elif op == 13:
            log.append(("flush", _call(bus.flush)))
        elif op == 14:
            s = base + int(rng.integers(0, n_max + 1))
            log.append(("drain", _view(_call(bus.drain, s, cap=int(rng.integers(1, R + 1))))))
            log.append(("peek", _view(_call(bus.peek_window, s, cap=int(rng.integers(1, R + 1))))))
        elif op == 15:
            f = int(rng.integers(0, n_max)); k = int(rng.integers(1, n_max - f + 1))
            # enough cap for every mailbox: which runs a short cap admits depends on the order the mailboxes claim space, on
            # one bus as on a handle (test_drain_many_with_a_short_cap covers that contract)
            st, r = _call(bus.drain_many, base + f, k, k * R)
            runs = None
            if st == nat.OK:
                out, offs, cnts = r
                runs = [out[o:o + c].tobytes() for o, c in zip(offs, cnts)]   # per-mailbox runs: their placement may differ
            log.append(("drain_many", st, runs))
        if step % 20 == 19:
            _readback(bus, n_max, log)
    log.append(("final_flush", _call(bus.flush)))
    bus.sync()
    _readback(bus, n_max, log)
    for s in range(n_max):
        log.append(("peek_end", s, _view(_call(bus.peek_window, base + s))))


def _compare(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x == y, (i, x, y)


@pytest.mark.parametrize("lossless", [False, True])
@pytest.mark.parametrize("g", [2, 3, 4])
def test_mixed_trace_equals_one_bus(g, lossless):
    n_max = 24
    kw = dict(ring_cap=128, batch_cap=32, timers_per_sub=2, lossless=lossless, sub_id_base=1000)
    for seed in (11, 12):
        logs = []
        for devices in (None, _devices(g)):
            log = []
            with Bus(n_max, devices=devices, **kw) as bus:
                _mixed_trace(bus, seed * 10 + g, n_max, log)
            logs.append(log)
        _compare(logs[0], logs[1])


@pytest.mark.parametrize("g", [2, 4, 8])
def test_mixed_trace_on_distinct_gpus(g):
    devices = _devices(g, distinct=True)
    n_max = 40
    kw = dict(ring_cap=128, batch_cap=32, timers_per_sub=2, lossless=False)
    logs = []
    for devs in (None, devices):
        log = []
        with Bus(n_max, devices=devs, **kw) as bus:
            _mixed_trace(bus, 77, n_max, log)
        logs.append(log)
    _compare(logs[0], logs[1])


@pytest.mark.parametrize("g", [2, 3])
def test_fleet_matches_the_oracle(g):
    """A full fleet with one timer each, unicast sends to every shard, publish bursts and clock jumps: every subscriber's
    (count, digest) and mailbox window equal the oracle's."""
    N, R, B = 48, 256, 64
    rng = np.random.default_rng(5 + g)
    masks = np.where(rng.random(N) < 0.5, nat.MASK_ALL, rng.integers(0, 1 << 17, N)).astype(np.uint32)
    orc = ob.Oracle(N, timers_per_sub=1, keep_window=R)
    for m in masks:
        orc.subscribe(int(m))
    with Bus(N, ring_cap=R, batch_cap=B, timers_per_sub=1, devices=_devices(g)) as bus:
        bus.subscribe_many(masks)
        bus.timer_add_many(0, N, 40_000, source_id0=100)
        for s in range(N):
            orc.timer_add(s, 40_000, 100 + s, False)
        now = 0
        for step in range(40):
            now += int(rng.choice([7_000, 90_000, 2_000_000]))
            nat.check(bus.advance(now), "advance"); orc.advance(now)
            n = int(rng.integers(1, 3 * B))
            ev = np.zeros(n, dtype=EVENT_DTYPE)
            ev["code"] = rng.integers(0, 17, n); ev["source_id"] = rng.integers(0, 30, n)
            nat.check(bus.publish_many(ev), "publish"); orc.publish_many(ev["code"], ev["source_id"])
            for _ in range(3):
                s, c = int(rng.integers(0, N)), int(rng.integers(0, 17))
                nat.check(bus.send(s, c, 9), "send"); orc.receive(s, c, 9)
        nat.check(bus.flush(), "flush")
        bus.sync()
        got = bus.digests(0, N)
        for s in range(N):
            assert (int(got["count"][s]), int(got["digest"][s])) == (orc.count(s), orc.digest(s)), s
            assert bus.peek_window(s).tobytes() == orc.mailbox(s).tobytes(), s
        st = bus.stats()
        assert st["deliveries"] == orc.total_deliveries() and st["ticks"] == orc.total_ticks()
        _drain_many_with_a_short_cap(bus, orc, N, R)


def _drain_many_with_a_short_cap(bus, orc, N, R):
    """drain_many with a cap that cuts inside a shard, repeated until nothing is left: every returned run is a whole
    mailbox in FIFO order, a mailbox left out has counts[i] = 0, and over the calls nothing is lost or duplicated."""
    runs = [None] * N
    for _ in range(4 * N):
        out, offs, cnts = bus.drain_many(0, N, R + 7)
        if not cnts.any():
            break
        for i in np.nonzero(cnts)[0]:
            assert runs[i] is None, i                             # taken once
            runs[i] = out[offs[i]:offs[i] + cnts[i]].tobytes()
    for s in range(N):
        assert runs[s] == orc.mailbox(s).tobytes(), s


@pytest.mark.parametrize("stalled", ["first", "middle", "last"])
def test_lossless_stall_on_one_shard(stalled):
    """Every mailbox is drained after each flush except one (on the first, a middle or the last of 4 shards).  The flush
    stops with EAGAIN after exactly the prefix one bus delivers; the mailboxes equal the oracle's with the same capacity;
    after that one is drained too, the flush resumes."""
    R, B, N, G = 128, 64, 16, 4
    P = 48                                                        # events per flush: the victim's room runs out mid-batch
    victim = {"first": 1, "middle": 9, "last": 14}[stalled]
    rng = np.random.default_rng(31)
    orc = ob.Oracle(N, keep_window=0, mailbox_cap=R)
    for _ in range(N):
        orc.subscribe(nat.MASK_ALL)
    buses = [Bus(N, ring_cap=R, batch_cap=B, lossless=True), Bus(N, ring_cap=R, batch_cap=B, lossless=True, devices=_devices(G))]
    try:
        for b in buses:
            b.subscribe_many(np.full(N, nat.MASK_ALL, dtype=np.uint32))
        stalls = 0
        i_orc = 0
        events_all = []
        for step in range(12):
            ev = np.zeros(P, dtype=EVENT_DTYPE)
            ev["code"] = rng.integers(1, 17, P); ev["source_id"] = step * P + np.arange(P)
            events_all.extend(zip(ev["code"], ev["source_id"]))
            for b in buses:
                nat.check(b.publish_many(ev), "publish")
            while True:
                rcs = [b.flush() for b in buses]
                assert rcs[0] == rcs[1], rcs
                while i_orc < len(events_all):
                    r = orc.publish(int(events_all[i_orc][0]), int(events_all[i_orc][1]))
                    if r == ob.EAGAIN:
                        break
                    i_orc += 1
                counts = [b.digests(0, N)["count"].tolist() for b in buses]
                assert counts[0] == counts[1] == [orc.count(s) for s in range(N)]
                for s in range(N):
                    if s != victim or rcs[0] == nat.EAGAIN and stalls >= 2:
                        got = [b.drain(s, cap=R).tobytes() for b in buses]
                        assert got[0] == got[1] == orc.consume(s, R).tobytes()
                if rcs[0] == nat.OK:
                    break
                assert rcs[0] == nat.EAGAIN
                stalls += 1
        st = [b.stats() for b in buses]
        assert stalls > 0
        assert st[1]["admit_passes"] > 0 and st[1]["admit_partial"] > 0
        for k in ("admit_passes", "admit_skipped", "admit_partial", "deliveries", "publishes"):
            assert st[0][k] == st[1][k], k
    finally:
        for b in buses:
            b.close()


def test_device_batches_split_like_one_bus():
    """An oversize device batch (more than batch_cap records, a watermark step wider than the timer window) with timers, in
    throughput mode: the same digests, step result and statistics as one bus.  Lossless mode refuses it (EINVAL)."""
    import torch
    N, B = 40, 64
    rng = np.random.default_rng(3)
    n = 5 * B + 7
    ev = np.zeros(n, dtype=EVENT_DTYPE)
    ev["seq"] = np.arange(n); ev["ts_ns"] = 1_000 * (1 + np.arange(n)); ev["code"] = rng.integers(0, 17, n)
    ev["source_id"] = rng.integers(0, 20, n); ev["target"] = 0xFFFFFFFF
    ev["target"][::9] = rng.integers(0, N, len(ev[::9])); ev["flags"][::9] = nat.F_UNICAST
    d = torch.from_numpy(ev.view(np.uint8).reshape(n, 32).copy()).cuda(0)
    res = []
    for devs in (None, _devices(3)):
        with Bus(N, ring_cap=512, batch_cap=B, timers_per_sub=1, devices=devs, device=0) as bus:
            bus.subscribe_many(np.full(N, nat.MASK_ALL, dtype=np.uint32))
            bus.timer_add_many(0, N, 3_000, source_id0=50)
            nat.check(bus.publish_device(d.data_ptr(), n, int(ev["ts_ns"][-1]) + 500), "publish_device")
            bus.sync()
            st = bus.stats(); st.pop("batches"); st.pop("kernel_launches")
            res.append((bus.digests(0, N).tobytes(), bus.step_result_end(bus.step_result_begin()), st,
                        bus.debug_events().tobytes(), bus.publish_counts()))
            assert st["device_splits"] > 1
    assert res[0] == res[1]
    with Bus(N, ring_cap=512, batch_cap=B, lossless=True, devices=_devices(2)) as bus:
        bus.subscribe_many(np.full(N, nat.MASK_ALL, dtype=np.uint32))
        assert bus.publish_device(d.data_ptr(), B, int(ev["ts_ns"][B - 1])) == nat.EINVAL


def test_refused_calls():
    with Bus(9, ring_cap=128, batch_cap=32, devices=_devices(3), sub_id_base=100) as bus:
        lib, h = bus._lib, bus._h
        import ctypes as C
        assert lib.cpbus_publish_device_staged(h, None, 0, 0, None, 0) == nat.EINVAL
        st, handle = C.c_void_p(), C.create_string_buffer(64)
        assert lib.cpbus_stream_create(h, 8, 2, C.byref(st), handle) == nat.EINVAL
        assert lib.cpbus_stream_open(h, handle, 1, C.byref(st)) == nat.EINVAL
        p = C.c_void_p()
        assert lib.cpbus_shared_alloc(h, 64, C.byref(p), handle) == nat.EINVAL
        assert lib.cpbus_shared_open(h, handle, C.byref(p)) == nat.EINVAL
        assert lib.cpbus_shared_close(h, C.c_void_p(64)) == nat.EINVAL
        assert lib.cpbus_device_ptrs(h, C.byref(p), C.byref(p)) == nat.EINVAL
        with Bus(4, ring_cap=128, batch_cap=32, device=0) as other:
            ost, _ = other.stream_create(8, 2)
            assert lib.cpbus_stream_attach(h, ost, 1, C.byref(st)) == nat.EINVAL
            other.stream_close(ost)
        assert bus.subscribe_many(np.full(9, nat.MASK_ALL, dtype=np.uint32)) == 100
        with pytest.raises(nat.CpbusError) as e:
            bus.subscribe()
        assert e.value.status == nat.ENOSPC
        for call in (lambda: bus.drain(109), lambda: bus.peek_window(109), lambda: bus.unsubscribe(109),
                     lambda: bus.digests(105, 5), lambda: bus.drain_many(108, 2, 64), lambda: bus.unsubscribe(99)):
            with pytest.raises(nat.CpbusError) as e:
                call()
            assert e.value.status == nat.ENOENT
        assert bus.send(109, 1) == nat.ENOENT
        assert bus.send(108, 1) == nat.OK


def test_go_shaped_scenarios_on_three_shards():
    """events_test.go:64-113 sequences, a timer on a watch's private channel, Unsubscribe ordering and DebugEvents through
    events.EventBus(devices=[0, 0, 0], n_max_subs=6): two subscribers per shard, so the third lands on shard 1."""
    from containerpilot_b200.events import Event
    bus = events.EventBus(n_max_subs=6, devices=_devices(3))
    pub = events.Publisher(); pub.Register(bus)
    subs = [events.Subscriber(events.Chan(100)) for _ in range(3)]
    for s in subs:
        s.Subscribe(bus)
    pub.Publish(Event(events.Startup, "serviceA"))
    for sig in ("SIGHUP", "SIGUSR2"):
        bus.PublishSignal(sig)
    want = [Event(events.Startup, "serviceA"), Event(events.Signal, "SIGHUP"), Event(events.Signal, "SIGUSR2")]
    assert [s.Received() for s in subs] == [want] * 3
    subs[1].Unsubscribe()                                 # ordered with publishes: sees nothing after this
    bus.Publish(Event(events.StatusHealthy, "serviceA"))
    assert subs[1].Received() == []
    assert subs[2].Received() == [Event(events.StatusHealthy, "serviceA")]
    rx = events.Chan(100)                                 # a watch's private channel (watches.go:37,71): an implicit subscriber
    ctx, cancel = events.WithCancel()
    events.NewEventTimer(ctx, rx, 1_000, "w.poll")
    bus.Advance(3_500)
    bus.Publish(Event(events.StatusChanged, "w"))
    tick = Event(events.TimerExpired, "w.poll")
    assert rx.recv_all() == [tick, tick, tick]
    assert subs[0].Received() == [Event(events.StatusHealthy, "serviceA"), Event(events.StatusChanged, "w")]
    cancel()
    bus.Advance(10_000)
    bus.Publish(events.GlobalShutdown)
    assert rx.recv_all() == []
    assert bus.DebugEvents() == want + [Event(events.StatusHealthy, "serviceA"), Event(events.StatusChanged, "w"),
                                        events.GlobalShutdown]
    pub.Unregister()
    bus.close()


def test_cpp_mirror_runs_on_a_sharded_handle():
    exe = os.path.join(ROOT, "containerpilot_b200", "csrc", "host", "events_sharded_test")
    assert os.path.exists(exe), "built by __graft_entry__.build()"
    r = subprocess.run([exe, *map(str, _devices(3))], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
