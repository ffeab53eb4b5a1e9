// events.hpp — C++ mirror of ContainerPilot's Go package `events`, on top of the libcpbus C-ABI.
//
// Same names, argument meaning and error behaviour as /root/reference/events/:
//   EventCode, Event, FromString, Global*            events/events.go
//   EventBus  (Register Unregister Subscribe Unsubscribe Publish PublishSignal
//              SetReloadFlag Shutdown Wait DebugEvents)   events/bus.go
//   EventPublisher / Publisher, EventSubscriber / Subscriber (with a real bounded Rx channel)
//                                                    events/publisher.go, events/subscriber.go
//   NewEventTimer / NewEventTimeout(ctx, rx, tick, name)   events/timer.go — `rx` is ANY channel, as in Go: the Rx of a
//       subscribed Subscriber (jobs/jobs.go:147-158) or a private channel nobody subscribed (watches/watches.go:37,71);
//       the latter gets an implicit mailbox with an empty code mask on the current bus (ticks + direct sends only)
// This is the host side a cgo shim would be (INTEGRATION.md shows the Go version); Go is not
// installed in this image, so the compiled-language mirror is C++17.  Go panics are `events::Panic`.
// Every delivery goes through libcpbus (CUDA): mailboxes live in HBM and a pump moves them into `Rx`.
#pragma once
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../../include/cpbus.h"

namespace events {

struct Panic : std::runtime_error { using std::runtime_error::runtime_error; };

// EventCode — events/events.go:18-39
enum EventCode : int {
  None = 0, ExitSuccess, ExitFailed, Stopping, Stopped, StatusHealthy, StatusUnhealthy, StatusChanged, TimerExpired,
  EnterMaintenance, ExitMaintenance, Error, Quit, Metric, Startup, Shutdown, Signal
};

inline std::string String(EventCode c) {   // events/eventcode_string.go:9-15
  const char* n = cpbus_code_name((int)c);
  return n ? std::string(n) : "EventCode(" + std::to_string((int)c) + ")";
}

// FromString — events/events.go:52-86: (code, "") or (None, "<name> is not a valid event code")
inline std::pair<EventCode, std::string> FromString(const std::string& name) {
  int c = cpbus_code_from_string(name.c_str());
  if (c < 0) return {None, name + " is not a valid event code"};
  return {(EventCode)c, ""};
}

struct Event {   // events/events.go:10-13
  EventCode Code = None;
  std::string Source;
  bool operator==(const Event& o) const { return Code == o.Code && Source == o.Source; }
  bool operator!=(const Event& o) const { return !(*this == o); }
  bool operator<(const Event& o) const { return Code != o.Code ? Code < o.Code : Source < o.Source; }
};

// global events — events/events.go:42-49
inline const Event GlobalStartup{Startup, "global"}, GlobalShutdown{Shutdown, "global"}, NonEvent{None, ""},
    GlobalEnterMaintenance{EnterMaintenance, "global"}, GlobalExitMaintenance{ExitMaintenance, "global"},
    QuitByTest{Quit, "closed"};

// `chan Event` with a capacity: make(chan Event, n)
class Chan {
 public:
  explicit Chan(size_t cap) : cap_(cap) {}
  // `rx <- e`: blocks while full; panics when closed
  void Send(const Event& e) {
    std::unique_lock<std::mutex> l(m_);
    not_full_.wait(l, [&] { return closed_ || q_.size() < cap_; });
    if (closed_) throw Panic("send on closed channel");
    q_.push_back(e);
    not_empty_.notify_one();
  }
  bool TrySend(const Event& e) {
    std::lock_guard<std::mutex> l(m_);
    if (closed_) throw Panic("send on closed channel");
    if (q_.size() >= cap_) return false;
    q_.push_back(e);
    not_empty_.notify_one();
    return true;
  }
  // `e, ok := <-rx` with a timeout standing in for `select { case <-ctx.Done() }`
  bool Recv(Event* out, std::chrono::milliseconds wait = std::chrono::milliseconds(0)) {
    std::unique_lock<std::mutex> l(m_);
    if (!not_empty_.wait_for(l, wait, [&] { return closed_ || !q_.empty(); })) return false;
    if (q_.empty()) return false;
    *out = q_.front();
    q_.pop_front();
    not_full_.notify_one();
    return true;
  }
  void Close() {
    std::lock_guard<std::mutex> l(m_);
    closed_ = true;
    not_full_.notify_all();
    not_empty_.notify_all();
  }
  bool Closed() const { std::lock_guard<std::mutex> l(m_); return closed_; }
  size_t Len() const { std::lock_guard<std::mutex> l(m_); return q_.size(); }

 private:
  mutable std::mutex m_;
  std::condition_variable not_full_, not_empty_;
  std::deque<Event> q_;
  size_t cap_;
  bool closed_ = false;
};
using ChanPtr = std::shared_ptr<Chan>;
inline ChanPtr MakeChan(size_t cap) { return std::make_shared<Chan>(cap); }

class EventBus;

struct EventPublisher {   // events/publisher.go:5-9
  virtual void Publish(const Event&) = 0;
  virtual void Register(EventBus*) = 0;
  virtual void Unregister() = 0;
  virtual ~EventPublisher() = default;
};
struct EventSubscriber {   // events/subscriber.go:5-9
  virtual void Subscribe(EventBus*) = 0;
  virtual void Unsubscribe() = 0;
  virtual void Receive(const Event&) = 0;
  virtual ~EventSubscriber() = default;
};

class Subscriber : public EventSubscriber {   // events/subscriber.go:13-37
 public:
  ChanPtr Rx;
  EventBus* Bus = nullptr;
  void Subscribe(EventBus* bus) override;
  void Subscribe(EventBus* bus, uint32_t mask, const std::vector<Event>& cases);   // filtered (masks + exact cases)
  void Unsubscribe() override;
  void Receive(const Event& e) override;
  void Wait();

 private:
  friend class EventBus;
  friend void NewEventTimeout(class Context&, const ChanPtr&, std::chrono::nanoseconds, const std::string&);
  friend void NewEventTimer(class Context&, const ChanPtr&, std::chrono::nanoseconds, const std::string&);
  uint32_t id_ = UINT32_MAX;
  bool implicit_ = false;       // made by the bus for a timer-only channel: not in the WaitGroup, released when Rx is closed
  std::deque<Event> pending_;   // drained from HBM but Rx was full
};

class Publisher : public EventPublisher {   // events/publisher.go:13-36
 public:
  EventBus* Bus = nullptr;
  void Publish(const Event& e) override;
  void Register(EventBus* bus) override;
  void Unregister() override;
  void Wait();
};

// context.WithCancel stand-in: Cancel() runs every registered hook once (ctx.Done())
class Context {
 public:
  void Cancel() {
    std::vector<std::function<void()>> h;
    { std::lock_guard<std::mutex> l(m_); if (done_) return; done_ = true; h.swap(hooks_); }
    for (auto& f : h) f();
  }
  bool Done() const { return done_; }
  void OnDone(std::function<void()> f) {
    { std::lock_guard<std::mutex> l(m_); if (!done_) { hooks_.push_back(std::move(f)); return; } }
    f();
  }

 private:
  std::mutex m_;
  std::atomic<bool> done_{false};
  std::vector<std::function<void()>> hooks_;
};

namespace detail {
// which Subscriber (of which bus) owns a channel: kept by Subscribe / Unsubscribe, looked up by the timer functions
// (Go needs no such table because the timer goroutine writes the channel itself)
struct RxOwner { EventBus* bus; Subscriber* sub; };
inline std::map<Chan*, RxOwner>& RxRegistry() { static std::map<Chan*, RxOwner> r; return r; }
}  // namespace detail

class EventBus {   // events/bus.go:12-22
 public:
  enum class Clock { Virtual, Monotonic };
  // NewEventBus() — events/bus.go:72-88.  Clock::Virtual: time moves only through Advance() (tests);
  // Clock::Monotonic: a pump thread feeds std::chrono::steady_clock every millisecond.
  // `devices` non-empty: the subscribers are sharded over these GPUs behind one handle (cpbus_create_sharded); nothing
  // else about the bus changes.
  explicit EventBus(Clock clock = Clock::Monotonic, uint32_t n_max_subs = 256, uint32_t mailbox_cap = 1024,
                    std::vector<int> devices = {}) : clock_(clock) {
    cpbus_config cfg{};
    cfg.n_max_subs = n_max_subs; cfg.ring_cap = mailbox_cap; cfg.batch_cap = mailbox_cap >= 512 ? 256 : mailbox_cap / 2;
    cfg.timers_per_sub = 4; cfg.flags = CPBUS_CFG_LOSSLESS | CPBUS_CFG_DIGEST; cfg.device = -1;
    batch_cap_ = cfg.batch_cap;
    const std::vector<int32_t> devs(devices.begin(), devices.end());
    int rc = devs.empty() ? cpbus_create(&cfg, &h_) : cpbus_create_sharded(&cfg, devs.data(), (uint32_t)devs.size(), &h_);
    if (rc) throw std::runtime_error(std::string(devs.empty() ? "cpbus_create: " : "cpbus_create_sharded: ") + cpbus_strerror(rc) +
                                     " " + cpbus_last_cuda_error());
    start_ = std::chrono::steady_clock::now();
    life_->h = h_;
    { std::lock_guard<std::mutex> g(CurrentMutex()); CurrentSlot() = this; }
    if (clock_ == Clock::Monotonic) pump_ = std::thread([this] { PumpLoop(); });
  }
  ~EventBus() {
    stop_ = true;
    if (pump_.joinable()) pump_.join();
    { std::lock_guard<std::mutex> g(CurrentMutex()); if (CurrentSlot() == this) CurrentSlot() = nullptr; }
    {
      std::lock_guard<std::recursive_mutex> l(lock_);
      life_->alive = false;                       // ctx.OnDone hooks that fire later find a dead bus and do nothing
      for (auto& kv : registry_) detail::RxRegistry().erase(kv.first->Rx.get());
    }
    cpbus_destroy(h_);
  }
  // The bus a bus-less call refers to (NewEventTimer on a channel nobody subscribed): the most recently created live one.
  // ContainerPilot has exactly one per App run (core/app.go:142).
  static EventBus* Current() { std::lock_guard<std::mutex> g(CurrentMutex()); return CurrentSlot(); }

  // NewEventTimer / NewEventTimeout (events/timer.go:12-71) for any channel
  static void StartTimer(Context& ctx, const ChanPtr& rx, std::chrono::nanoseconds tick, const std::string& name, int oneshot);
  EventBus(const EventBus&) = delete;

  void Register(EventPublisher*) { std::lock_guard<std::recursive_mutex> l(lock_); done_.Add(1); }   // bus.go:91-95
  void Unregister(EventPublisher*) { std::lock_guard<std::recursive_mutex> l(lock_); done_.Done(); }  // bus.go:98-102

  void Subscribe(EventSubscriber* subscriber) { Subscribe(subscriber, CPBUS_MASK_ALL, {}); }   // bus.go:105-111
  // The consumer's switch pushed down: `mask` = codes taken whatever the source, `cases` = the exact Event values of its
  // `switch event { case events.Event{Code, Source}: ... }` (jobs/jobs.go:197-231), at most CPBUS_MAX_PAIRS.
  void Subscribe(EventSubscriber* subscriber, uint32_t mask, const std::vector<Event>& cases) {
    std::lock_guard<std::recursive_mutex> l(lock_);
    auto* sub = dynamic_cast<Subscriber*>(subscriber);
    if (!sub) throw Panic("interface conversion: EventSubscriber is not *Subscriber");   // bus.go:108
    uint32_t id = 0;
    std::vector<cpbus_pair> pairs;
    for (const Event& e : cases) pairs.push_back(cpbus_pair{(uint32_t)e.Code, Intern(e.Source)});
    auto imp = sub->Rx ? implicit_.find(sub->Rx.get()) : implicit_.end();
    if (imp != implicit_.end() && pairs.empty()) {
      // the channel already carries timer ticks (NewEventTimer came first): keep that mailbox and its timers, open the mask
      Subscriber* old = imp->second.get();
      id = old->id_;
      Retry([&] { return cpbus_set_mask(h_, id, mask); }, "cpbus_set_mask");
      sub->pending_ = std::move(old->pending_);
      registry_.erase(old);
      implicit_.erase(imp);
    } else {
      Retry([&] { return cpbus_subscribe_pairs(h_, mask, pairs.data(), (uint32_t)pairs.size(), &id); }, "cpbus_subscribe_pairs");
    }
    sub->id_ = id;
    registry_[sub] = id;
    if (sub->Rx) detail::RxRegistry()[sub->Rx.get()] = {this, sub};
    done_.Add(1);
  }

  void Unsubscribe(EventSubscriber* subscriber) {   // bus.go:114-122
    std::lock_guard<std::recursive_mutex> l(lock_);
    auto* sub = dynamic_cast<Subscriber*>(subscriber);
    if (!sub) throw Panic("interface conversion: EventSubscriber is not *Subscriber");
    auto it = registry_.find(sub);
    if (it != registry_.end()) {
      FlushLocked();
      DrainOne(sub, /*blocking=*/false);   // what was published before the unsubscribe still reaches Rx
      Retry([&] { return cpbus_unsubscribe(h_, it->second); }, "cpbus_unsubscribe");
      registry_.erase(it);
      if (sub->Rx) detail::RxRegistry().erase(sub->Rx.get());
      sub->id_ = UINT32_MAX;
    }
    done_.Done();   // negative counter => panic, as sync.WaitGroup does (bus.go:121)
  }

  void Publish(const Event& event) {   // bus.go:125-140
    std::lock_guard<std::recursive_mutex> l(lock_);
    for (auto& kv : registry_)
      if (kv.first->Rx && kv.first->Rx->Closed()) throw Panic("send on closed channel");   // bus.go:135-137
    if (String(event.Code) != "Metric") counter_[{String(event.Code), event.Source}]++;     // bus.go:130-132
    cpbus_event ev{};
    ev.code = (uint32_t)event.Code; ev.source_id = Intern(event);
    for (;;) {
      int rc = cpbus_publish(h_, &ev, 1);
      if (rc == CPBUS_EAGAIN) { DrainAll(/*blocking=*/true); continue; }   // the Go publisher would block in chansend
      Check(rc, "cpbus_publish");
      break;
    }
    if (clock_ == Clock::Virtual) { FlushLocked(); DrainAll(false); }
  }
  // A burst of Publish calls handed over as batches (one cpbus_publish call and one fan-out per batch_cap events): what a
  // fan-in caller such as the /v3/metric handler produces (control/endpoints.go:125-128).  Same per-event semantics as
  // Publish; a full mailbox blocks the batch until the consumers have drained, like a blocked chansend.
  void PublishMany(const std::vector<Event>& events) {
    std::lock_guard<std::recursive_mutex> l(lock_);
    for (auto& kv : registry_)
      if (kv.first->Rx && kv.first->Rx->Closed()) throw Panic("send on closed channel");   // bus.go:135-137
    FlushLocked();   // staging buffer empty from here on: a chunk of <= batch_cap_ events never triggers a flush of its own
    std::vector<cpbus_event> evs;
    for (size_t i = 0; i < events.size(); i += batch_cap_) {
      const size_t n = std::min<size_t>(batch_cap_, events.size() - i);
      evs.assign(n, cpbus_event{});
      for (size_t j = 0; j < n; j++) {
        const Event& e = events[i + j];
        if (String(e.Code) != "Metric") counter_[{String(e.Code), e.Source}]++;            // bus.go:130-132
        evs[j].code = (uint32_t)e.Code; evs[j].source_id = Intern(e);
      }
      Check(cpbus_publish(h_, evs.data(), n), "cpbus_publish");
      FlushLocked();
    }
    if (clock_ == Clock::Virtual) DrainAll(false);
  }
  void PublishSignal(const std::string& sig) { Publish(Event{Signal, sig}); }   // bus.go:144-146
  void SetReloadFlag() { std::lock_guard<std::recursive_mutex> l(lock_); reload_ = true; }   // bus.go:150-154
  void Shutdown() { Publish(GlobalShutdown); }   // bus.go:158-160
  bool Wait() { done_.Wait(); std::lock_guard<std::recursive_mutex> l(lock_); return reload_; }   // bus.go:164-169

  std::vector<Event> DebugEvents() {   // bus.go:34-54
    std::this_thread::sleep_for(std::chrono::milliseconds(clock_ == Clock::Virtual ? 0 : 100));
    std::lock_guard<std::recursive_mutex> l(lock_);
    cpbus_event buf[10]; size_t n = 0;
    Check(cpbus_debug_events(h_, buf, 10, &n), "cpbus_debug_events");
    std::vector<Event> out;
    for (size_t i = 0; i < n && i < 10; i++) out.push_back(Event{(EventCode)buf[i].code, Source(buf[i].source_id)});
    return out;
  }

  // virtual clock (Clock::Virtual only): the runtime clock reaching `now_ns`
  void Advance(uint64_t now_ns) {
    std::lock_guard<std::recursive_mutex> l(lock_);
    Check(cpbus_advance(h_, now_ns), "cpbus_advance");
    FlushLocked();
    DrainAll(false);
  }
  uint64_t CounterValue(const std::string& code, const std::string& source) {
    std::lock_guard<std::recursive_mutex> l(lock_);
    auto it = counter_.find({code, source});
    return it == counter_.end() ? 0 : it->second;
  }
  cpbus_t* handle() { return h_; }

 private:
  friend class Subscriber;
  friend void NewEventTimeout(Context&, const ChanPtr&, std::chrono::nanoseconds, const std::string&);
  friend void NewEventTimer(Context&, const ChanPtr&, std::chrono::nanoseconds, const std::string&);

  struct WaitGroup {   // sync.WaitGroup
    void Add(long n) { std::lock_guard<std::mutex> l(m); c += n; if (c < 0) throw Panic("sync: negative WaitGroup counter"); if (c == 0) cv.notify_all(); }
    void Done() { Add(-1); }
    void Wait() { std::unique_lock<std::mutex> l(m); cv.wait(l, [&] { return c == 0; }); }
    std::mutex m; std::condition_variable cv; long c = 0;
  };

  // state a ctx.OnDone hook may still hold after the bus is gone
  struct Life { std::recursive_mutex m; bool alive = true; cpbus_t* h = nullptr; };
  static std::mutex& CurrentMutex() { static std::mutex m; return m; }
  static EventBus*& CurrentSlot() { static EventBus* b = nullptr; return b; }

  // libcpbus flushes staged events inside membership / timer calls; in lossless mode a full mailbox makes them return
  // CPBUS_EAGAIN: let the consumers run (drain into Rx) and try again, like a blocked chansend would
  template <class F>
  void Retry(F&& call, const char* where) {
    for (;;) {
      const int rc = call();
      if (rc == CPBUS_EAGAIN) { DrainAll(/*blocking=*/true); continue; }
      Check(rc, where);
      return;
    }
  }
  // the mailbox behind a channel nobody subscribed (watches/watches.go:37,71): empty code mask, so only ticks and
  // direct sends land in it; pumped into `rx` like any other; not part of the WaitGroup
  Subscriber* ImplicitFor(const ChanPtr& rx) {
    auto it = implicit_.find(rx.get());
    if (it != implicit_.end()) return it->second.get();
    auto sub = std::make_unique<Subscriber>();
    sub->Rx = rx; sub->Bus = this; sub->implicit_ = true;
    uint32_t id = 0;
    Retry([&] { return cpbus_subscribe(h_, 0u, &id); }, "cpbus_subscribe");
    sub->id_ = id;
    registry_[sub.get()] = id;
    detail::RxRegistry()[rx.get()] = {this, sub.get()};
    Subscriber* raw = sub.get();
    implicit_[rx.get()] = std::move(sub);
    return raw;
  }
  // close(rx) on a timer-only channel: the Go timer goroutine panics on its next send, recovers and exits
  // (events/timer.go:26-30,50-54) — release the mailbox and with it the timers
  void ReleaseImplicit(Subscriber* sub) {
    cpbus_unsubscribe(h_, sub->id_);
    registry_.erase(sub);
    detail::RxRegistry().erase(sub->Rx.get());
    implicit_.erase(sub->Rx.get());
  }

  static void Check(int rc, const char* where) {
    if (rc == CPBUS_ECLOSED) throw Panic("sync: negative WaitGroup counter");
    if (rc) throw std::runtime_error(std::string(where) + ": " + cpbus_strerror(rc) + " " + cpbus_last_cuda_error());
  }
  uint32_t Intern(const std::string& s) { uint32_t id = 0; Check(cpbus_intern(h_, s.data(), s.size(), &id), "cpbus_intern"); return id; }
  // A Metric event's Source is a payload ("key|value", control/endpoints.go:125-126), not a name: bounded ephemeral region
  uint32_t Intern(const Event& e) {
    if (e.Code != Metric) return Intern(e.Source);
    uint32_t id = 0; Check(cpbus_intern_ephemeral(h_, e.Source.data(), e.Source.size(), &id), "cpbus_intern_ephemeral"); return id;
  }
  std::string Source(uint32_t id) {
    size_t n = 0; cpbus_source(h_, id, nullptr, 0, &n);
    std::string s(n, '\0'); if (n) cpbus_source(h_, id, &s[0], n, &n);
    return s;
  }
  void FlushLocked() {
    for (;;) {
      int rc = cpbus_flush(h_);
      if (rc == CPBUS_EAGAIN) { DrainAll(true); continue; }
      Check(rc, "cpbus_flush");
      return;
    }
  }
  // HBM mailbox -> the subscriber's real Rx channel (`chan Event`), FIFO, lossless
  void DrainOne(Subscriber* sub, bool blocking) {
    if (sub->id_ == UINT32_MAX) return;
    cpbus_event buf[256];
    for (;;) {
      size_t n = 0; uint64_t lost = 0;
      Check(cpbus_drain(h_, sub->id_, buf, 256, &n, &lost), "cpbus_drain");
      for (size_t i = 0; i < n; i++) sub->pending_.push_back(Event{(EventCode)buf[i].code, Source(buf[i].source_id)});
      if (n < 256) break;
    }
    while (!sub->pending_.empty() && sub->Rx) {
      if (blocking) sub->Rx->Send(sub->pending_.front());
      else if (!sub->Rx->TrySend(sub->pending_.front())) break;
      sub->pending_.pop_front();
    }
  }
  // All mailboxes at once: one gather kernel + two D2H copies (cpbus_drain_many) instead of a round trip per subscriber.
  void DrainAll(bool blocking) {
    if (registry_.empty()) return;
    uint32_t lo = UINT32_MAX, hi = 0;
    for (auto& kv : registry_) { lo = std::min(lo, kv.second); hi = std::max(hi, kv.second); }
    const uint32_t n = hi - lo + 1;
    if (drain_buf_.size() < kDrainCap) drain_buf_.resize(kDrainCap);
    drain_off_.resize(n); drain_cnt_.resize(n);
    std::vector<Subscriber*> by_id(n, nullptr);
    for (auto& kv : registry_) by_id[kv.second - lo] = kv.first;
    for (;;) {
      size_t total = 0;
      Check(cpbus_drain_many(h_, lo, n, drain_buf_.data(), kDrainCap, drain_off_.data(), drain_cnt_.data(), &total), "cpbus_drain_many");
      if (!total) break;
      for (uint32_t i = 0; i < n; i++) {
        if (!drain_cnt_[i] || !by_id[i]) continue;
        const cpbus_event* r = drain_buf_.data() + drain_off_[i];
        for (uint32_t j = 0; j < drain_cnt_[i]; j++) by_id[i]->pending_.push_back(Event{(EventCode)r[j].code, Source(r[j].source_id)});
      }
    }
    std::vector<Subscriber*> dead;
    for (auto& kv : registry_) {
      Subscriber* sub = kv.first;
      try {
        while (!sub->pending_.empty() && sub->Rx) {
          if (blocking) sub->Rx->Send(sub->pending_.front());
          else if (!sub->Rx->TrySend(sub->pending_.front())) break;
          sub->pending_.pop_front();
        }
      } catch (const Panic&) {
        if (!sub->implicit_) throw;          // bus.go:135-137: publishing into a closed subscriber channel is a panic
        dead.push_back(sub);                 // timer.go:50-54: the timer goroutine recovers and exits
      }
    }
    for (Subscriber* sub : dead) ReleaseImplicit(sub);
  }
  void PumpLoop() {
    while (!stop_) {
      std::this_thread::sleep_for(std::chrono::milliseconds(1));
      std::lock_guard<std::recursive_mutex> l(lock_);
      uint64_t now = (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - start_).count();
      cpbus_advance(h_, now);
      int rc = cpbus_flush(h_);
      if (rc != CPBUS_OK && rc != CPBUS_EAGAIN) continue;
      try { DrainAll(false); } catch (const Panic&) { /* closed Rx: the timer goroutine recovers (timer.go:26-30,50-54) */ }
    }
  }

  static constexpr size_t kDrainCap = 1 << 16;
  std::vector<cpbus_event> drain_buf_;
  std::vector<uint32_t> drain_off_, drain_cnt_;
  cpbus_t* h_ = nullptr;
  std::shared_ptr<Life> life_ = std::make_shared<Life>();
  std::recursive_mutex& lock_ = life_->m;   // bus.lock (bus.go:14): serialises publishers and membership changes
  std::map<Chan*, std::unique_ptr<Subscriber>> implicit_;   // timer-only channels
  bool reload_ = false;
  WaitGroup done_;
  std::map<Subscriber*, uint32_t> registry_;   // bus.go:13
  uint32_t batch_cap_ = 32;                    // events per cpbus_publish batch (PublishMany)
  std::map<std::pair<std::string, std::string>, uint64_t> counter_;   // containerpilot_events{code,source}
  Clock clock_;
  std::chrono::steady_clock::time_point start_;
  std::thread pump_;
  std::atomic<bool> stop_{false};
};

inline void Subscriber::Subscribe(EventBus* bus) { Bus = bus; bus->Subscribe(this); }   // subscriber.go:19-22
inline void Subscriber::Subscribe(EventBus* bus, uint32_t mask, const std::vector<Event>& cases) { Bus = bus; bus->Subscribe(this, mask, cases); }
inline void Subscriber::Unsubscribe() { Bus->Unsubscribe(this); }                       // subscriber.go:25-27
inline void Subscriber::Wait() { Bus->Wait(); }                                         // subscriber.go:35-37
inline void Subscriber::Receive(const Event& e) {                                       // subscriber.go:30-32: `sub.Rx <- event`
  if (Rx && Rx->Closed()) throw Panic("send on closed channel");
  if (Bus && id_ != UINT32_MAX) {   // direct mailbox write, ordered with publishes, bypasses the filter
    std::lock_guard<std::recursive_mutex> l(Bus->lock_);
    cpbus_event ev{};
    ev.code = (uint32_t)e.Code; ev.source_id = Bus->Intern(e);
    for (;;) {
      int rc = cpbus_send(Bus->h_, id_, &ev);
      if (rc == CPBUS_EAGAIN) { Bus->DrainAll(true); continue; }
      EventBus::Check(rc, "cpbus_send");
      break;
    }
    if (Bus->clock_ == EventBus::Clock::Virtual) { Bus->FlushLocked(); Bus->DrainAll(false); }
  } else if (Rx) Rx->Send(e);
}
inline void Publisher::Publish(const Event& e) { Bus->Publish(e); }                     // publisher.go:18-20
inline void Publisher::Register(EventBus* bus) { Bus = bus; bus->Register(this); }      // publisher.go:23-26
inline void Publisher::Unregister() { Bus->Unregister(this); }                          // publisher.go:29-31
inline void Publisher::Wait() { Bus->Wait(); }                                          // publisher.go:34-36

namespace detail {
struct TimerTarget { EventBus* bus; Subscriber* sub; };
// `rx` is the Rx of a subscribed Subscriber, or any other channel: then the current bus makes it a mailbox of its own
inline TimerTarget TargetOf(const ChanPtr& rx) {
  auto& reg = RxRegistry();
  auto it = reg.find(rx.get());
  if (it != reg.end() && it->second.sub->Bus) return {it->second.bus, it->second.sub};
  EventBus* bus = EventBus::Current();
  if (!bus) throw Panic("NewEventTimer: no EventBus exists in this process");
  return {bus, nullptr};
}
}  // namespace detail

inline void EventBus::StartTimer(Context& ctx, const ChanPtr& rx, std::chrono::nanoseconds tick, const std::string& name, int oneshot) {
  if (rx->Closed()) return;   // the goroutine's first send would panic and be recovered: no tick ever arrives
  detail::TimerTarget t = detail::TargetOf(rx);
  EventBus* bus = t.bus;
  std::lock_guard<std::recursive_mutex> l(bus->lock_);
  Subscriber* sub = t.sub ? t.sub : bus->ImplicitFor(rx);
  uint32_t tid = 0;
  const uint32_t src = bus->Intern(name);
  bus->Retry([&] { return cpbus_timer_add(bus->h_, sub->id_, (uint64_t)tick.count(), src, oneshot, &tid); }, "cpbus_timer_add");
  // ctx.Done() (timer.go:20-22,57-58).  The hook may outlive the bus: it holds the bus's Life, not the bus.  Timer ids
  // carry a generation, so a late cancel can never disarm a slot that has been re-armed since.
  std::shared_ptr<Life> life = bus->life_;
  ctx.OnDone([life, bus, tid] {
    std::lock_guard<std::recursive_mutex> g(life->m);
    if (!life->alive) return;
    for (;;) {
      const int rc = cpbus_timer_cancel(life->h, tid);
      if (rc != CPBUS_EAGAIN) break;          // ENOENT: already fired / gone
      bus->DrainAll(/*blocking=*/true);       // a full mailbox held back the flush in front of the cancel: let consumers run
    }
  });
}
namespace detail {
inline void StartTimer(Context& ctx, const ChanPtr& rx, std::chrono::nanoseconds tick, const std::string& name, int oneshot) {
  EventBus::StartTimer(ctx, rx, tick, name, oneshot);
}
}  // namespace detail

// Callers pass `rx` exactly as in Go (jobs/jobs.go:147-158, watches/watches.go:71): any `chan Event`.
inline void NewEventTimeout(Context& ctx, const ChanPtr& rx, std::chrono::nanoseconds tick, const std::string& name) {   // timer.go:12-37
  detail::StartTimer(ctx, rx, tick, name, 1);
}
inline void NewEventTimer(Context& ctx, const ChanPtr& rx, std::chrono::nanoseconds tick, const std::string& name) {     // timer.go:40-71
  detail::StartTimer(ctx, rx, tick, name, 0);
}

}  // namespace events
