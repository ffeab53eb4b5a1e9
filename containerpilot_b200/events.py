"""Host-side mirror of ContainerPilot's `events` package over the GPU bus.

Same names, argument meaning and error behaviour as the Go API
(/root/reference/events/), so that parity tests read like the reference's own:

    EventCode / Event / FromString / Global*           events/events.go
    EventBus: Register Unregister Subscribe Unsubscribe
              Publish PublishSignal SetReloadFlag
              Shutdown Wait DebugEvents                events/bus.go
    Publisher / Subscriber (+ Rx)                      events/publisher.go, subscriber.go
    NewEventTimer / NewEventTimeout                    events/timer.go

`NewEventTimer` / `NewEventTimeout` take any `Chan`, exactly as the Go functions take any `chan Event`
(events/timer.go:12-16,40-45): when the channel is not the Rx of a subscribed Subscriber (a Watch's private channel,
watches/watches.go:37,71) the bus gives it a mailbox of its own — an implicit subscriber with an empty code mask that
receives only the ticks and direct sends — on the bus most recently created in this process (the reference has exactly
one live bus per App run, core/app.go:142).

Differences, all forced by running under a virtual clock in tests:
  * `Rx` is a `Chan` whose receive side drains the subscriber's HBM mailbox
    (`cpbus_drain`) — in the Go shim a drain goroutine pumps a real `chan Event`;
  * time only moves when `EventBus.Advance(ns)` is called (the Go shim calls
    cpbus_advance with the monotonic clock);
  * Go panics become Python exceptions (`BusPanic`).
Every delivery goes through libcpbus (CUDA).  There is no CPU data path here.
"""
from __future__ import annotations

import weakref
from collections import deque
from dataclasses import dataclass

import numpy as np

from . import _native as nat
from .bus import Bus, EVENT_DTYPE

# EventCode enum — events/events.go:21-39
(None_, ExitSuccess, ExitFailed, Stopping, Stopped, StatusHealthy, StatusUnhealthy, StatusChanged, TimerExpired,
 EnterMaintenance, ExitMaintenance, Error, Quit, Metric, Startup, Shutdown, Signal) = range(17)


class BusPanic(RuntimeError):
    """A condition on which the Go bus panics (closed mailbox, double Unsubscribe, bad type)."""


def CodeString(code: int) -> str:
    """EventCode.String — events/eventcode_string.go:9-15"""
    name = nat.load().cpbus_code_name(code)
    return name.decode() if name is not None else f"EventCode({code})"


def FromString(name: str):
    """FromString — events/events.go:52-86. Returns (code, err)."""
    code = nat.load().cpbus_code_from_string(name.encode())
    if code < 0:
        return None_, ValueError(f"{name} is not a valid event code")
    return code, None


@dataclass(frozen=True)
class Event:
    """Event — events/events.go:10-13 (comparable by value, usable as a dict key)."""
    Code: int = None_
    Source: str = ""

    def __repr__(self):
        return f"{{{CodeString(self.Code)} {self.Source}}}"


# global events — events/events.go:42-49
GlobalStartup = Event(Startup, "global")
GlobalShutdown = Event(Shutdown, "global")
NonEvent = Event(None_, "")
GlobalEnterMaintenance = Event(EnterMaintenance, "global")
GlobalExitMaintenance = Event(ExitMaintenance, "global")
QuitByTest = Event(Quit, "closed")


class Chan:
    """Stand-in for `chan Event` with capacity `cap` (make(chan Event, n))."""

    def __init__(self, cap: int = 1000):
        self.cap = cap
        self.closed = False
        self._local = deque()       # sends made while no subscriber is attached
        self._sub = None            # owning Subscriber once subscribed

    def close(self):
        """close(rx).  A timer goroutine that then sends into it panics, recovers and exits (events/timer.go:26-30,
        50-54): the implicit mailbox behind a timer-only channel is released, and with it its timers."""
        self.closed = True
        sub = self._sub
        if sub is not None and getattr(sub, "_implicit", False) and sub.Bus is not None and sub._id is not None:
            sub.Bus._release_implicit(sub)

    def send(self, event: Event):
        """`rx <- event`: direct mailbox write (jobs/jobs.go:262)."""
        if self.closed:
            raise BusPanic("send on closed channel")
        sub = self._sub
        if sub is not None and sub.Bus is not None and sub._id is not None:
            sub.Bus._send(sub, event)
        else:
            self._local.append(event)

    def recv_all(self):
        """Drain everything currently in the mailbox, FIFO."""
        out = list(self._local)
        self._local.clear()
        sub = self._sub
        if sub is not None and sub.Bus is not None and sub._id is not None:
            out.extend(sub.Bus._drain(sub))
        return out


class EventBus:
    """EventBus — events/bus.go:12-22.  NewEventBus() == EventBus().

    `EventBus(devices=[0, 1, ...])` puts the subscribers on several GPUs behind one handle (`Bus(devices=...)`); nothing
    else about the API changes."""

    def __init__(self, n_max_subs: int = 64, ring_cap: int = 1024, batch_cap: int = 256, timers_per_sub: int = 4,
                 lossless: bool = True, **kw):
        self._bus = Bus(n_max_subs, ring_cap=ring_cap, batch_cap=batch_cap, timers_per_sub=timers_per_sub,
                        lossless=lossless, digest=True, **kw)
        self.reload = False
        self._done = 0              # sync.WaitGroup counter (bus.go:16)
        self._subs = {}             # Subscriber -> sub_id  (registry, bus.go:13)
        self._implicit = {}         # Chan -> implicit Subscriber (timer-only channels; NOT in the registry or the WaitGroup)
        _live_buses.append(weakref.ref(self))

    # ---- lifecycle accounting ----
    def Register(self, publisher):          # bus.go:91-95
        self._done += 1

    def Unregister(self, publisher):        # bus.go:98-102
        self._done -= 1
        if self._done < 0:
            raise BusPanic("sync: negative WaitGroup counter")

    def Subscribe(self, subscriber, mask: int = nat.MASK_ALL, cases=None):   # bus.go:105-111
        """`cases`: exact Event values of the consumer's switch (jobs/jobs.go:197-231) delivered on top of `mask`"""
        if not isinstance(subscriber, Subscriber):
            raise BusPanic("interface conversion: EventSubscriber is not *Subscriber")
        imp = self._implicit.pop(subscriber.Rx, None) if subscriber.Rx is not None else None
        if imp is not None and not cases:
            # the channel already carries timer ticks (NewEventTimer came first): keep that mailbox and its timers, open the mask
            self._bus.set_mask(imp._id, mask)
            subscriber._id, subscriber._tail = imp._id, imp._tail
        elif cases:
            subscriber._id = self._bus.subscribe_pairs(mask, [(e.Code, self._bus.intern(e.Source)) for e in cases])
        else:
            subscriber._id = self._bus.subscribe(mask)
        if subscriber.Rx is not None:
            subscriber.Rx._sub = subscriber
        self._subs[subscriber] = subscriber._id
        self._done += 1

    def Unsubscribe(self, subscriber):      # bus.go:114-122
        if not isinstance(subscriber, Subscriber):
            raise BusPanic("interface conversion: EventSubscriber is not *Subscriber")
        if subscriber in self._subs:
            subscriber._tail = self._drain(subscriber)       # keep what was delivered before the unsubscribe
            self._bus.unsubscribe(self._subs.pop(subscriber))
            subscriber._id = None
        self._done -= 1
        if self._done < 0:
            raise BusPanic("sync: negative WaitGroup counter")

    def SetReloadFlag(self):                # bus.go:150-154
        self.reload = True

    def Wait(self) -> bool:                 # bus.go:164-169 (non-blocking mirror)
        if self._done > 0:
            raise BlockingIOError("EventBus.Wait would block: %d registrations outstanding" % self._done)
        return self.reload

    # ---- hot path ----
    def Publish(self, event: Event):        # bus.go:125-140
        for sub in self._subs:
            if sub.Rx is not None and sub.Rx.closed:
                raise BusPanic("send on closed channel")     # bus.go:135-137
        rc = self._bus.publish(event.Code, self._intern(event))
        if rc == nat.EAGAIN:
            raise BlockingIOError("Publish would block: a subscriber mailbox is full")
        nat.check(rc, "cpbus_publish")

    def PublishMany(self, events):
        """A burst of Publish calls as one batch (one `cpbus_publish` call, one staging pass): what a fan-in caller such as
        the /v3/metric handler (control/endpoints.go:125-128) hands over.  Same per-event semantics as Publish."""
        for sub in self._subs:
            if sub.Rx is not None and sub.Rx.closed:
                raise BusPanic("send on closed channel")     # bus.go:135-137
        batch = np.zeros(len(events), dtype=EVENT_DTYPE)
        batch["code"] = [e.Code for e in events]
        batch["source_id"] = [self._intern(e) for e in events]
        rc = self._bus.publish_many(batch)
        if rc == nat.EAGAIN:
            raise BlockingIOError("Publish would block: a subscriber mailbox is full")
        nat.check(rc, "cpbus_publish")

    def _intern(self, event: Event) -> int:
        """Source -> id.  A Metric event's Source is a payload ("key|value", control/endpoints.go:125-126), not a name:
        it goes to the bounded ephemeral region so the intern table cannot grow with every posted value."""
        return self._bus.intern_ephemeral(event.Source) if event.Code == Metric else self._bus.intern(event.Source)

    def PublishSignal(self, sig: str):      # bus.go:144-146
        self.Publish(Event(Signal, sig))

    def Shutdown(self):                     # bus.go:158-160
        self.Publish(GlobalShutdown)

    def DebugEvents(self):                  # bus.go:34-54
        return [Event(int(r["code"]), self._bus.source(int(r["source_id"]))) for r in self._bus.debug_events()]

    # ---- virtual clock (test-only control; the Go shim feeds the monotonic clock) ----
    def Advance(self, now_ns: int):
        nat.check(self._bus.advance(now_ns), "cpbus_advance")

    def Flush(self):
        rc = self._bus.flush()
        if rc == nat.EAGAIN:
            raise BlockingIOError("flush would block: a subscriber mailbox is full")
        nat.check(rc, "cpbus_flush")

    # ---- used by Chan / Subscriber ----
    def _send(self, sub, event: Event):
        rc = self._bus.send(sub._id, event.Code, self._intern(event))
        if rc == nat.EAGAIN:
            raise BlockingIOError("send would block: mailbox full")
        nat.check(rc, "cpbus_send")

    def _drain(self, sub):
        self.Flush()
        recs = self._bus.drain(sub._id)
        return [Event(int(r["code"]), self._bus.source(int(r["source_id"]))) for r in recs]

    # ---- timer-only channels ----
    def _implicit_for(self, rx: "Chan"):
        sub = self._implicit.get(rx)
        if sub is None:
            sub = Subscriber(rx)
            sub.Bus, sub._implicit = self, True
            sub._id = self._bus.subscribe(0)          # empty mask: broadcasts never land here, ticks and direct sends do
            self._implicit[rx] = sub
        return sub

    def _release_implicit(self, sub):
        self._implicit.pop(sub.Rx, None)
        try:
            self._bus.unsubscribe(sub._id)            # disarms its timers too
        except nat.CpbusError:
            pass
        sub._id = None

    def close(self):
        self._bus.close()
        _live_buses[:] = [r for r in _live_buses if r() is not None and r() is not self]


_live_buses: list = []


def _current_bus() -> EventBus:
    """The bus a bus-less call (`NewEventTimer(ctx, rx, ...)` on an unsubscribed channel) refers to: the most recently
    created live one.  ContainerPilot has exactly one per App run (core/app.go:142)."""
    for r in reversed(_live_buses):
        b = r()
        if b is not None and b._bus._h:
            return b
    raise BusPanic("NewEventTimer: no EventBus exists in this process")


NewEventBus = EventBus


class Publisher:
    """Publisher — events/publisher.go:13-36"""

    def __init__(self):
        self.Bus = None

    def Publish(self, event: Event):
        self.Bus.Publish(event)

    def Register(self, bus: EventBus):
        self.Bus = bus
        bus.Register(self)

    def Unregister(self):
        self.Bus.Unregister(self)

    def Wait(self):
        return self.Bus.Wait()


class Subscriber:
    """Subscriber — events/subscriber.go:13-37"""

    def __init__(self, rx: Chan | None = None):
        self.Rx = rx
        self.Bus = None
        self._id = None
        self._tail = []
        self._implicit = False      # True: the bus made this mailbox for a timer-only channel (NewEventTimer on an unsubscribed rx)
        if rx is not None:
            rx._sub = self

    def __hash__(self):
        return id(self)

    def __eq__(self, other):
        return self is other

    def Subscribe(self, bus: EventBus, mask: int = nat.MASK_ALL, cases=None):
        self.Bus = bus
        if self.Rx is not None:
            self.Rx._sub = self
        bus.Subscribe(self, mask, cases)

    def Unsubscribe(self):
        self.Bus.Unsubscribe(self)

    def Receive(self, event: Event):        # subscriber.go:30-32
        self.Rx.send(event)

    def Wait(self):
        return self.Bus.Wait()

    def Received(self):
        """Everything delivered so far, FIFO (test observation point: `<-sub.Rx` until empty)."""
        out, self._tail = self._tail, []
        out.extend(self.Rx.recv_all() if self.Rx is not None else [])
        return out


class Context:
    """context.WithCancel stand-in: cancel() disarms every timer started under it."""

    def __init__(self):
        self._timers = []
        self.done = False

    def cancel(self):
        self.done = True
        for bus, tid in self._timers:
            try:
                bus._bus.timer_cancel(tid)
            except nat.CpbusError as e:      # one-shot already fired
                if e.status != nat.ENOENT:
                    raise
        self._timers.clear()


def WithCancel():
    ctx = Context()
    return ctx, ctx.cancel


def _new_timer(ctx: Context, rx: Chan, tick_ns: int, name: str, oneshot: bool):
    sub = rx._sub
    if sub is None or sub.Bus is None or sub._id is None:
        # any `chan Event` will do (events/timer.go:40-46 takes only ctx, rx, tick, name): a Watch passes a private
        # channel that is not a bus subscriber (watches/watches.go:37,71)
        if rx.closed:
            return                              # the goroutine's first send would panic and be recovered: no tick ever arrives
        sub = _current_bus()._implicit_for(rx)
    bus = sub.Bus
    tid = bus._bus.timer_add(sub._id, tick_ns, bus._bus.intern(name), oneshot)
    ctx._timers.append((bus, tid))


def NewEventTimeout(ctx: Context, rx: Chan, tick_ns: int, name: str):
    """NewEventTimeout — events/timer.go:12-37: one {TimerExpired, name} after `tick`."""
    _new_timer(ctx, rx, tick_ns, name, True)


def NewEventTimer(ctx: Context, rx: Chan, tick_ns: int, name: str):
    """NewEventTimer — events/timer.go:40-71: {TimerExpired, name} every `tick` until cancelled."""
    _new_timer(ctx, rx, tick_ns, name, False)
