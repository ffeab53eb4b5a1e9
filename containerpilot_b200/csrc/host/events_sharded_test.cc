// events_sharded_test.cc — the C++ mirror (events.hpp) on a bus sharded over three shards behind one handle
// (EventBus(..., devices)), with the real pump thread.  The three devices come from the command line (default 0 0 0).
// Six subscribers, two per shard: the third subscriber lands on shard 1.  Exit code 0 = all passed.  Needs a GPU.
#include <cstdio>
#include <cstdlib>
#include <thread>

#include "events.hpp"

using namespace events;

static int failures = 0;
#define EXPECT(cond)                                                           \
  do {                                                                         \
    if (!(cond)) { std::printf("  FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); failures++; } \
  } while (0)

static std::vector<Event> RecvAll(Chan* rx, size_t want) {   // the pump delivers asynchronously: wait (bounded) for `want`
  std::vector<Event> got;
  Event e;
  for (int spin = 0; spin < 2000 && got.size() < want; spin++)
    if (rx->Recv(&e, std::chrono::milliseconds(1))) got.push_back(e);
  while (rx->Recv(&e)) got.push_back(e);
  return got;
}

// events/events_test.go:64-113 on three shards: publish, signals, Unsubscribe ordering, DebugEvents
static void TestPubSubOnShards(const std::vector<int>& devices) {
  std::printf("TestPubSubOnShards\n");
  EventBus bus(EventBus::Clock::Monotonic, 6, 1024, devices);
  Publisher pub;
  pub.Register(&bus);
  Subscriber subs[3];
  for (auto& s : subs) { s.Rx = MakeChan(100); s.Subscribe(&bus); }
  pub.Publish(Event{Startup, "serviceA"});
  bus.PublishSignal("SIGHUP");
  bus.PublishSignal("SIGUSR2");
  const std::vector<Event> want{Event{Startup, "serviceA"}, Event{Signal, "SIGHUP"}, Event{Signal, "SIGUSR2"}};
  for (auto& s : subs) EXPECT(RecvAll(s.Rx.get(), want.size()) == want);
  subs[1].Unsubscribe();                         // ordered with publishes: sees nothing published after this
  pub.Publish(Event{StatusHealthy, "serviceA"});
  EXPECT((RecvAll(subs[2].Rx.get(), 1) == std::vector<Event>{Event{StatusHealthy, "serviceA"}}));
  EXPECT((RecvAll(subs[0].Rx.get(), 1) == std::vector<Event>{Event{StatusHealthy, "serviceA"}}));
  EXPECT(RecvAll(subs[1].Rx.get(), 0).empty());
  std::vector<Event> debug = want;
  debug.push_back(Event{StatusHealthy, "serviceA"});
  EXPECT(bus.DebugEvents() == debug);
  subs[0].Unsubscribe(); subs[2].Unsubscribe();
  pub.Unregister();
  EXPECT(bus.Wait() == false);
}

int main(int argc, char** argv) {
  std::vector<int> devices{0, 0, 0};
  for (int i = 1; i < argc && i <= 3; i++) devices[i - 1] = std::atoi(argv[i]);
  TestPubSubOnShards(devices);
  std::printf(failures ? "FAILED (%d)\n" : "PASS\n", failures);
  return failures ? 1 : 0;
}
