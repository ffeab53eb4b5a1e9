// cpbus.cu — libcpbus: C-ABI (include/cpbus.h) over the sm_100a kernels.
//
// Host-side bookkeeping that the reference keeps in Go (events/bus.go): the
// registry, the 10-slot debug ring, per-code publish counts, the Source intern
// table, the virtual clock, staging of published events into pinned batches.
// There is NO CPU data path: without a CUDA device cpbus_create fails with
// CPBUS_ENODEV, and nothing here touches oracle/.
#include "cpbus_kernels.cuh"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

using namespace cpbus_dev;

namespace {

thread_local char g_cuda_err[256] = "";

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      snprintf(g_cuda_err, sizeof(g_cuda_err), "%s:%d %s: %s", __FILE__, __LINE__, #call,          \
               cudaGetErrorString(e_));                                                            \
      return CPBUS_ECUDA;                                                                          \
    }                                                                                              \
  } while (0)

// debug ring entry awaiting enqueue: a concrete event, or "the broadcast events of device launch `launch`"
struct DbgItem { bool marker; unsigned long long launch; cpbus_event ev; };

// publish counts by (code << 32 | source_id): the label set of `containerpilot_events` (events/bus.go:131).  Flat
// open-addressing table (key + 1 stored, 0 = empty): an increment is one probe in the common case, and a burst of n
// events is counted in two passes (slots prefetched, then incremented) so that cache misses of a high-cardinality
// source set overlap instead of adding up (a std::unordered_map here cost ~40 ns per published event).
struct PairCounter {
  std::vector<uint64_t> keys, cnts;
  size_t used = 0;
  static uint64_t mix(uint64_t k) { k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; return k; }
  void grow() {
    std::vector<uint64_t> ok, oc;
    ok.swap(keys); oc.swap(cnts);
    const size_t cap = ok.empty() ? 1024 : ok.size() * 2;
    keys.assign(cap, 0); cnts.assign(cap, 0); used = 0;
    for (size_t i = 0; i < ok.size(); i++) if (ok[i]) add(ok[i] - 1, oc[i]);
  }
  void add(uint64_t key, uint64_t by) {
    if ((used + 1) * 2 > keys.size()) grow();
    const size_t mask = keys.size() - 1;
    for (size_t i = mix(key) & mask;; i = (i + 1) & mask) {
      if (keys[i] == key + 1) { cnts[i] += by; return; }
      if (!keys[i]) { keys[i] = key + 1; cnts[i] = by; used++; return; }
    }
  }
  void prefetch(uint64_t key) const { if (!keys.empty()) { const size_t i = mix(key) & (keys.size() - 1); __builtin_prefetch(&keys[i]); __builtin_prefetch(&cnts[i]); } }
};

struct HostTimer { bool active = false, oneshot = false; uint8_t gen = 0; uint64_t period = 0, next_due = 0; uint32_t source_id = 0; };
// timer id = slot index (subscriber * K + k) | generation << 26: a late cancel from an old context cannot disarm a re-armed slot
constexpr uint32_t kTimerSlotBits = 26, kTimerSlotMask = (1u << kTimerSlotBits) - 1u;

}  // namespace

struct cpbus_stream;

struct cpbus {
  cpbus_config cfg{};
  int device = 0, sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  uint32_t N = 0, R = 0, B = 0, K = 0;
  int store = CPBUS_STORE_V8;
  bool lossless = false, use_digest = false;

  // HBM-resident state (SoA, one entry per subscriber of this shard)
  cpbus_event* d_ring = nullptr;          // N * R records: each mailbox is one contiguous 32*R-byte ring
  SubCtl* d_ctl = nullptr;                // N control blocks: {tail, head, digest, mask}, one sector each
  DevTimer* d_timers = nullptr;           // N * K
  DevStats* d_stats = nullptr;
  uint64_t* d_pow = nullptr;              // P^0..: digest multiplier powers, TMA-loaded by every CTA
  unsigned char* d_desc = nullptr;        // per-launch batch descriptor (CTA 0 writes, the others read)
  unsigned long long* d_desc_ready = nullptr;
  unsigned long long launch_seq = 0;
  cpbus_event* d_batch_local = nullptr;    // staged ingest: CTA 0's local copy of a peer batch
  static constexpr int kPrefetch = 3;      // fused ingest: later batches pulled over NVLink by earlier launches
  cpbus_event* d_prefetch[kPrefetch] = {};
  const void* pf_ptr[kPrefetch] = {};      // which peer batch sits in d_prefetch[i] ...
  size_t pf_n[kPrefetch] = {};
  unsigned long long pf_seq[kPrefetch] = {};   // ... and which launch wrote it
  int pf_next = 0;
  std::vector<void*> shared_owned, shared_mapped;   // cpbus_shared_alloc / cpbus_shared_open
  // stream mode (cpbus_stream_*): device-managed prefetch of later stream batches + sticky error word
  unsigned long long* d_pf_state = nullptr;   // [kStreamPrefetch]: which stream batch sits in d_prefetch[i]
  cpbus_event* d_pf_buf = nullptr;            // kStreamPrefetch x batch_cap records (one allocation)
  unsigned int* h_err = nullptr;              // pinned + mapped: kErr* bits written by the fan-out kernel
  unsigned int* d_err = nullptr;              // device alias of h_err
  uint32_t stream_spin_us = 0;                // bound of the in-kernel wait for a stream batch (0 = 2 s)
  // accounting of device-published batches (cpbus_publish_device*, cpbus_stream_fanout): done by the kernel's lead CTA
  DevPubAcct* d_acct = nullptr;
  DevPubAcct* h_acct = nullptr;               // pinned staging for cpbus_stats / cpbus_debug_events / cpbus_publish_counts
  std::deque<DbgItem> dbg_pending;            // debug-ring entries not yet enqueued (events, or markers of device batches)
  PairCounter pub_pairs;                              // host publishes by (code << 32 | source_id), Metric excluded (bus.go:130-132)
  cpbus_event* d_drain = nullptr; size_t drain_cap = 0;        // cpbus_drain_many staging
  uint2* d_drain_idx = nullptr; size_t drain_idx_cap = 0;
  uint32_t subs_per_warp = 0;             // 0 = auto
  uint32_t order_block = 0;               // mask order is built per block of this many consecutive subscribers (0 = one global order)
  bool order_heavy_first = true;          // within a block: masks with more codes first (CPBUS_ORDER_HEAVY=0: plain mask order)
  bool pdl = true;                        // programmatic dependent launch of consecutive fan-outs
  int h2d_spin_us = 30;                   // how long cpbus_flush waits on the host for the batch's H2D before inserting a stream wait
  bool zero_copy = false;                 // fan-out pulls host-staged batches straight from pinned memory (experiment: CPBUS_ZERO_COPY=1)
  cudaEvent_t launched = nullptr;         // recorded after the latest fan-out (step results are read on the copy stream)
  int hints = -1;                         // -1 auto; bit0: control blocks / timer slots evict_last in L2
  static constexpr int kFoldSlots = 8;
  unsigned long long* d_fold = nullptr;   // kFoldSlots x 4 words
  cudaEvent_t fold_done[kFoldSlots] = {};
  uint32_t fold_next = 0;
  static constexpr int kStage = 8;         // staging ring: the host may run several flushes ahead of the GPU
  static constexpr int kEpoch = 4;         // a `consumed` event is recorded only after every kEpoch-th buffer, so that most
                                           // consecutive fan-outs are adjacent in the stream (programmatic dependent launch)
  static constexpr int kDevSlots = 64, kDevEpoch = 16;
  cpbus_event* d_stage = nullptr;          // kDevSlots x batch_cap records: device side of the staging ring
  cudaEvent_t epoch_done[kDevSlots / kDevEpoch] = {};   // on the bus stream, after the last fan-out of each epoch of slots
  uint32_t dev_slot = 0;
  cpbus_event* h_batch[kStage] = {};       // pinned staging
  cudaEvent_t h2d_done[kStage] = {};       // on copy_stream: batch c has reached HBM
  cudaEvent_t consumed[kStage] = {};       // on the bus stream: the fan-out that read d_batch[c] has finished
  cudaStream_t copy_stream = nullptr;      // H2D of batch i+1 overlaps the fan-out of batch i
  cudaStream_t result_stream = nullptr;    // D2H of step results: must not queue in front of the next batch's H2D
  // per-launch results written by the fan-out kernel itself (no extra kernel to read a step's result)
  DevResultSlot* d_result = nullptr;       // kResultRing x kResultSub slots
  DevResultSlot* h_result = nullptr;       // pinned, kFoldSlots tickets x kResultSub
  cudaEvent_t result_done[8] = {};
  uint32_t result_next = 0;
  DevStats* h_stats = nullptr;            // pinned
  unsigned long long* h_fold = nullptr;   // pinned
  int cur = 0;
  size_t n_staged = 0;

  // registry mirror (events/bus.go:13 `registry map[*Subscriber]bool`)
  std::vector<uint32_t> h_mask;
  std::vector<uint8_t> h_active;
  std::vector<uint8_t> h_npairs;          // second-level filter: exact {code, source} cases per subscriber (empty until first use)
  uint2* d_pairs = nullptr;               // N x CPBUS_MAX_PAIRS, allocated by the first cpbus_subscribe_pairs
  uint32_t n_paired = 0;                  // active subscribers with a pair table
  uint32_t* d_order = nullptr;            // active subscribers sorted by code mask (ORDERED fan-out)
  uint32_t n_order = 0, n_filtered = 0;   // n_filtered: active subscribers whose mask is not CPBUS_MASK_ALL
  bool order_dirty = true;
  int use_order = 1;                      // CPBUS_ORDER: 0 never, 1 when some subscriber is filtered (default), 2 also for all-ones masks (experiment)
  std::vector<size_t> oneshot_idx;        // armed one-shot timers (index into h_timers)
  std::vector<HostTimer> h_timers;        // N*K, allocated on first timer
  uint32_t n_next = 0, n_active = 0, n_timers = 0;
  uint64_t min_period = UINT64_MAX;       // conservative lower bound over armed periodic timers

  // clock and ordinals
  uint64_t now = 0, last_watermark = 0, seq = 0;
  // lossless mode: a lower bound of the free slots of the FULLEST mailbox.  While a batch provably fits (bound >= what it
  // can append to one mailbox) the admission pass and its host sync are skipped; the bound is refreshed exactly whenever
  // the admission kernel does run, and reset by cpbus_consume_all.
  uint64_t room_lb = 0;

  // DebugEvents ring (events/bus.go:18-21, 24-54)
  int dbg_head = -1, dbg_tail = 0;
  cpbus_event dbg[10]{};

  // intern table (Event.Source string <-> u32)
  std::unordered_map<std::string, uint32_t> intern;
  std::vector<std::string> sources;
  size_t intern_bytes = 0;
  // bounded region for payload strings (Metric "key|value"): recycled oldest-first
  struct EphSlot { std::string s; uint32_t gen = 0; bool live = false; };
  std::vector<EphSlot> eph;
  std::unordered_map<std::string, uint32_t> eph_map;
  uint32_t eph_next = 0;
  uint64_t eph_live = 0, eph_recycled = 0;
  std::vector<cpbus_stream*> streams;     // open streams (closed by cpbus_destroy if the caller did not)

  cpbus_stats_t st{};
  std::mutex mu;   // drain/stats from a second thread

  // Sharded handle (cpbus_create_sharded): G shard buses behind this one.  The handle keeps what the kernels never see
  // (intern table, clock, publish ordinal, debug ring, host publish counts, lossless room bound) and stages events into
  // h_batch[0]; a flush puts the staged records into the stream owned by shard 0 and fans them out on every shard.
  std::vector<cpbus*> shards;             // empty: an ordinary bus
  std::vector<uint32_t> shard_first;      // shard k holds local ids [shard_first[k], shard_first[k+1]) (global = sub_id_base + local)
  std::vector<cpbus_stream*> shard_st;    // shard k's end of the handle's stream (shard 0 owns it)
  cpbus_event* d_batch_host = nullptr;    // device alias of the pinned, portable staging buffer (admission reads it in place)
  bool any_timer = false;                 // a timer has been armed on some shard (cpbus_timer_cancel's "no timer table yet")
  std::vector<std::pair<uint32_t, uint32_t>> fold_parts[kFoldSlots];   // handle ticket -> (shard, shard ticket)
  std::vector<uint32_t> result_parts[8];
  bool sharded() const { return !shards.empty(); }
};

namespace {

// counting sort of the active subscribers by their 17-bit code mask (stable: ids ascending inside a mask)
int rebuild_order(cpbus* b);

int dev_guard(cpbus* b) {
  CK(cudaSetDevice(b->device));
  return CPBUS_OK;
}

uint32_t mask_word(const cpbus* b, uint32_t local) {
  uint32_t hint = 0;
  if (b->K && !b->h_timers.empty())
    for (uint32_t k = 0; k < b->K; k++)
      if (b->h_timers[(size_t)local * b->K + k].active) hint = k + 1;
  if (!b->h_active[local]) return 0;
  const uint32_t pair_bit = (!b->h_npairs.empty() && b->h_npairs[local]) ? kPairBit : 0u;
  return (b->h_mask[local] & CPBUS_MASK_ALL) | (hint << kTimerHintShift) | pair_bit | kActiveBit;
}

void dbg_ring_put(cpbus* b, const cpbus_event& e) {   // events/bus.go:24-31
  b->dbg[(b->dbg_head + 1) % 10] = e;
  int old = b->dbg_head;
  b->dbg_head = (b->dbg_head + 1) % 10;
  if (old != -1 && b->dbg_head == b->dbg_tail) b->dbg_tail = (b->dbg_tail + 1) % 10;
}

// While the broadcast events of a device-published batch are still unknown to the host (a marker is pending), later
// enqueues queue up behind it so that the ring keeps the global publish order; cpbus_debug_events resolves them.
void dbg_enqueue(cpbus* b, const cpbus_event& e) {
  if (b->dbg_pending.empty()) { dbg_ring_put(b, e); return; }
  b->dbg_pending.push_back(DbgItem{false, 0ull, e});
  if (b->dbg_pending.size() > (size_t)kAcctDbgRing) b->dbg_pending.pop_front();
}

void dbg_mark_device_batch(cpbus* b, unsigned long long launch) {
  b->dbg_pending.push_back(DbgItem{true, launch, cpbus_event{}});
  if (b->dbg_pending.size() > (size_t)kAcctDbgRing) b->dbg_pending.pop_front();
}

// The mask order of the ORDERED build, host-only (exported as cpbus_mask_order so that it can be tested without a GPU).
// Equal masks become neighbours, so a warp's consecutive mailboxes share one filter pass.
//  * Blocks.  A GLOBAL order scatters the mailboxes that are written at the same time over the whole ring area (1,048,576
//    rings = 32 GiB = 16,384 2-MiB pages, all live at once); ordering block by block of consecutive subscribers keeps the
//    concurrently written rings within a few hundred pages, at the price of shorter runs.  Same box, Zipf masks, us per launch
//    (profiles/r02_ab_kernel_variants.md table 8): 1,048,576 subscribers (32 GiB of rings) global order 1347.5, blocks of
//    524,288 subscribers 1292, of 262,144 or 131,072 1279.5 (-5.0 %), of 4,096 1287; 524,288 subscribers (16 GiB): global
//    635.4, blocks of 262,144 643.7 (shorter runs cost 1.3 %).  Policy (block == 0): one global order up to 16 GiB of rings,
//    blocks of 8 GiB beyond.
//  * Heavy first.  Within a block a second, stable pass by the number of codes in the mask, most first: CTAs are dispatched
//    in block order, so the mailboxes that take the most records start first and the launch's last wave is made of the light
//    ones (shorter tail before the next launch may start); equal masks stay neighbours.  Table 9: 131,072 subscribers
//    167.2 -> 162.0 us per launch, 262,144 319.5 -> 309.2, 1,048,576 1279.4 -> 1274.6.
static void mask_order(const uint32_t* masks, const uint8_t* active, uint32_t n, uint32_t ring_cap, uint32_t block, bool heavy_first,
                       std::vector<uint32_t>& order) {
  order.clear();
  order.reserve(n);
  const uint64_t ring_bytes = (uint64_t)ring_cap * sizeof(cpbus_event);
  uint32_t blk = block;
  if (!blk) blk = (uint64_t)n * ring_bytes <= (16ull << 30) ? std::max(1u, n) : (uint32_t)std::max<uint64_t>(4096, (8ull << 30) / ring_bytes);
  if (block == 0xFFFFFFFFu) blk = std::max(1u, n);   // one global order (A/B)
  std::vector<uint32_t> count((size_t)CPBUS_MASK_ALL + 2), tmp;
  for (uint32_t lo = 0; lo < n; lo += blk) {
    const uint32_t hi = (uint32_t)std::min<uint64_t>((uint64_t)lo + blk, n);
    std::fill(count.begin(), count.end(), 0u);
    for (uint32_t i = lo; i < hi; i++) if (!active || active[i]) count[(masks[i] & CPBUS_MASK_ALL) + 1]++;
    for (size_t k = 1; k < count.size(); k++) count[k] += count[k - 1];
    const size_t base = order.size();
    order.resize(base + count.back());
    for (uint32_t i = lo; i < hi; i++) if (!active || active[i]) order[base + count[masks[i] & CPBUS_MASK_ALL]++] = i;
    if (heavy_first) {
      const size_t nb = order.size() - base;
      uint32_t pc_count[34] = {};
      for (size_t k = 0; k < nb; k++) pc_count[32 - __builtin_popcount(masks[order[base + k]] & CPBUS_MASK_ALL) + 1]++;
      for (int k = 1; k < 34; k++) pc_count[k] += pc_count[k - 1];
      tmp.resize(nb);
      for (size_t k = 0; k < nb; k++) tmp[pc_count[32 - __builtin_popcount(masks[order[base + k]] & CPBUS_MASK_ALL)]++] = order[base + k];
      std::copy(tmp.begin(), tmp.end(), order.begin() + base);
    }
  }
}

int rebuild_order(cpbus* b) {
  std::vector<uint32_t> order;
  static_assert(sizeof(b->h_active[0]) == 1, "h_active is a byte vector");
  mask_order(b->h_mask.data(), reinterpret_cast<const uint8_t*>(b->h_active.data()), b->n_next, b->R, b->order_block, b->order_heavy_first, order);
  b->n_order = (uint32_t)order.size();
  if (b->n_order) {
    CK(cudaMemcpyAsync(b->d_order, order.data(), (size_t)b->n_order * 4, cudaMemcpyHostToDevice, b->stream));
    CK(cudaStreamSynchronize(b->stream));
  }
  b->order_dirty = false;
  return CPBUS_OK;
}

template <int STORE, bool TIMERS, bool DIGEST, bool ORDERED, bool PAIRS = false>
int launch_fanout_t(cpbus* b, const FanoutParams& p, uint32_t grid, size_t smem) {
  static bool attr_done[64] = {};   // per instantiation AND per device: function attributes are per-device state
  const int dev = b->device & 63;
  if (!attr_done[dev]) {
    CK(cudaFuncSetAttribute(fanout_kernel<STORE, TIMERS, DIGEST, ORDERED, PAIRS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_done[dev] = true;
  }
  if (!grid) {
    // Several waves of short-lived CTAs rather than one persistent wave: the hardware CTA scheduler
    // balances the two dies / SM speed spread for free (pure-store microbenchmark, scripts/write_ceiling.cu:
    // 6.0 TB/s with one resident wave, 6.9 TB/s with >= 32 CTAs per SM).  Per-CTA setup here is a descriptor
    // copy + TMA wait (~2 us), so the sweet spot measured on the real kernel is 2-16 mailboxes per warp
    // (65,536 subscribers: 2-4 per warp -> 97 % of the copy peak, 1 per warp 89 %, persistent 83 %;
    //  1,048,576 subscribers with timers: 8-16 per warp -> 94 %, 4 or 32 per warp 85 %).
    const uint32_t need = (p.n_subs + kWarpsPerCta - 1) / kWarpsPerCta;
    uint32_t spw = b->subs_per_warp;
    if (!spw) {
      // ~constant bytes per warp: the counts above were measured at 256-event batches; a 512-event batch halves them
      const uint32_t scale = std::max(1u, (p.n_ev + 128u) / 256u);
      const uint32_t cap = std::max(1u, 16u / scale);
      spw = std::max(1u, std::min(cap, (need + (uint32_t)b->sm_count * 7 * scale) / ((uint32_t)b->sm_count * 14 * scale)));
    }
    grid = std::max(1u, std::min((need + spw - 1) / spw, need));
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = b->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // PDL: the next fan-out's prologue overlaps this one's tail
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = b->pdl ? 1 : 0;
  CK(cudaLaunchKernelEx(&cfg, fanout_kernel<STORE, TIMERS, DIGEST, ORDERED, PAIRS>, p));
  CK(cudaGetLastError());
  return CPBUS_OK;
}

// fan out `n` records at d_src with watermark w (all checks done by the caller)
struct StreamArgs {   // stream mode (cpbus_stream_fanout): where this batch's header / ack words live
  const StreamHdr* hdr = nullptr; unsigned long long* ack = nullptr; unsigned long long seq = 0;
  const StreamHdr* next_hdr = nullptr;
};

int launch_fanout(cpbus* b, const cpbus_event* d_src, uint32_t n, uint64_t w, int staged = 0,
                  const cpbus_event* prefetch_src = nullptr, cpbus_event* prefetch_dst = nullptr, uint32_t prefetch_n = 0,
                  bool batch_dep = false, bool account = false, const StreamArgs* sa = nullptr) {
  if (b->n_next == 0 && !sa) return CPBUS_OK;
  if (n == 0 && b->n_timers == 0 && !sa) return CPBUS_OK;   // (a stream batch is always consumed: its slot must be acknowledged)
  FanoutParams p{};
  p.batch = d_src; p.ring = b->d_ring; p.ctl = b->d_ctl; p.timers = b->d_timers; p.stats = b->d_stats; p.pow_table = b->d_pow; p.launch_seq = ++b->launch_seq;
  p.desc = b->d_desc + (p.launch_seq & 1) * ((fanout_desc_bytes(2048) + 255) & ~(size_t)255);   // two descriptor buffers: launch i+1 may write while launch i reads
  p.desc_ready = b->d_desc_ready + (p.launch_seq & 1) * 16; p.w_now = w;
  p.result = b->d_result + (size_t)(p.launch_seq % kResultRing) * kResultSub;
  p.result_next = b->d_result + (size_t)((p.launch_seq + 1) % kResultRing) * kResultSub;
  p.batch_local = b->d_batch_local; p.staged = (uint32_t)staged;
  p.err_word = b->d_err; p.acct = account ? b->d_acct : nullptr;
  p.pf_state = b->d_pf_state; p.pf_buf = b->d_pf_buf; p.pf_stride = b->B; p.spin_us = b->stream_spin_us;
  if (sa) { p.stream_hdr = sa->hdr; p.stream_ack = sa->ack; p.stream_seq = sa->seq; p.stream_next_hdr = sa->next_hdr; }
  p.prefetch_src = prefetch_src; p.prefetch_dst = prefetch_dst; p.prefetch_n = prefetch_n;
  p.batch_dep = batch_dep ? 1u : 0u; p.n_ev = n;
  p.n_subs = b->n_next; p.ring_cap = b->R; p.K = b->K; p.sub_base = b->cfg.sub_id_base;
  p.use_digest = b->use_digest; p.lossless = b->lossless; p.timers_on = b->n_timers > 0 && b->K > 0;
  p.smem_cap = (n + 31u) & ~31u;
  // evict_last on control blocks / timer slots: they are re-read and re-written by every launch while the ring stream passes
  // through L2 once.  Round 2, same box (gpurun_out/r2k_ab.txt): with the hint at 1,048,576 subscribers config 5 (32 MiB of
  // control blocks, scattered by the mask order) 1424 -> 1355 us per launch (-4.9 %), config 3 (64 MiB with timer slots)
  // 2671 -> 2662 (-0.4 %); round 1's kernel had lost 8 % there.  Kept while the hot state is at most half of the 126 MB L2.
  const size_t hot_bytes = (size_t)b->n_next * (sizeof(SubCtl) + (p.timers_on ? b->K * sizeof(DevTimer) : 0));
  p.hints = b->hints >= 0 ? (uint32_t)b->hints : (hot_bytes <= (64u << 20) ? 1u : 0u);
  const uint32_t need = (b->n_next + kWarpsPerCta - 1) / kWarpsPerCta;
  uint32_t grid = b->cfg.grid_ctas ? std::max(1u, std::min(b->cfg.grid_ctas, need)) : 0u;   // 0: sized from occupancy
  int rc;
  // ORDERED build (no timers armed, at least one filtered subscriber): walk the mailboxes in code-mask order so that
  // equal masks are neighbours and share one filter pass (cost ~ deliveries + distinct masks, not subscribers x events)
  // PAIRS build (some subscriber has exact {code, source} cases): the timers build with the second-level test in its
  // general path; subscribers without a pair table take the same paths as before
  const bool pairs_on = b->n_paired > 0 && b->d_pairs;
  p.pairs = pairs_on ? b->d_pairs : nullptr;
  const size_t smem = fanout_smem_bytes(p.smem_cap) + (pairs_on ? kPairFilterBytes : 0);   // + the batch's {code, source} presence filter
  if (!pairs_on && !p.timers_on && (b->use_order == 2 || (b->use_order == 1 && b->n_filtered > 0))) {
    if (b->order_dirty) { const int rc_order = rebuild_order(b); if (rc_order) return rc_order; }
    if (b->n_order) {
      const uint32_t scale = std::max(1u, (p.n_ev + 128u) / 256u);
      // measured at 512-event batches: 8 mailboxes per warp from 524,288 subscribers up, 6 at 262,144 (-0.7 %), 4 at 131,072
      // (-2.8 %: short launches want more, shorter CTAs) — gpurun_out/r2y_ab.txt
      uint32_t spw = b->subs_per_warp ? std::min(32u, b->subs_per_warp)
                                      : std::max(4u, std::min(16u / scale, b->n_order / (20480u * scale)));
      p.order = b->d_order; p.n_order = b->n_order; p.spw = spw;
      const uint32_t warps = (b->n_order + spw - 1) / spw;
      grid = std::max(1u, (warps + kWarpsPerCta - 1) / kWarpsPerCta);
    }
  }
  if (pairs_on && !b->cfg.grid_ctas) {   // PAIRS build: lane-parallel triage over blocks of 32 mailboxes per warp turn
    const uint32_t blocks = (b->n_next + 31u) / 32u;
    grid = std::max(1u, std::min((blocks + kWarpsPerCta - 1) / kWarpsPerCta, (uint32_t)b->sm_count * 16u));
  }
  const int variant = pairs_on ? (p.use_digest ? 7 : 6) : (p.timers_on ? 2 : 0) | (p.use_digest ? 1 : 0) | (p.order ? 4 : 0);
#define CPBUS_DISPATCH(ST)                                                                \
  switch (variant) {                                                                     \
    case 0: rc = launch_fanout_t<ST, false, false, false>(b, p, grid, smem); break;      \
    case 1: rc = launch_fanout_t<ST, false, true, false>(b, p, grid, smem); break;       \
    case 2: rc = launch_fanout_t<ST, true, false, false>(b, p, grid, smem); break;       \
    case 3: rc = launch_fanout_t<ST, true, true, false>(b, p, grid, smem); break;        \
    case 4: rc = launch_fanout_t<ST, false, false, true>(b, p, grid, smem); break;       \
    case 5: rc = launch_fanout_t<ST, false, true, true>(b, p, grid, smem); break;        \
    case 6: rc = launch_fanout_t<ST, true, false, false, true>(b, p, grid, smem); break; \
    default: rc = launch_fanout_t<ST, true, true, false, true>(b, p, grid, smem); break; \
  }
  switch (b->store) {
    case CPBUS_STORE_V4: CPBUS_DISPATCH(CPBUS_STORE_V4); break;
    case CPBUS_STORE_BULK: CPBUS_DISPATCH(CPBUS_STORE_BULK); break;
    default: CPBUS_DISPATCH(CPBUS_STORE_V8); break;
  }
#undef CPBUS_DISPATCH
  if (rc) return rc;
  b->st.batches++; b->st.kernel_launches++;
  b->last_watermark = w;
  if (account && n) dbg_mark_device_batch(b, p.launch_seq);
  return CPBUS_OK;
}

// the most a launch of n events up to watermark w can append to ONE mailbox: every event + every firing of its timer slots
uint64_t admit_need(uint32_t n, uint32_t K, bool timers, uint64_t min_period, uint64_t last_watermark, uint64_t w) {
  uint64_t need = n;
  if (timers && K) {
    const uint64_t per_slot = (min_period != UINT64_MAX && w > last_watermark) ? (w - last_watermark) / min_period + 2 : 2;
    need += (uint64_t)K * per_slot;
  }
  return need;
}

// enqueue the admission kernel and the D2H of its result words into h_stats (the caller synchronises b->stream)
int admit_launch(cpbus* b, const cpbus_event* d_src, uint32_t n, uint64_t w) {
  CK(cudaMemsetAsync(&b->d_stats->admit_overflow, 0, 4 * sizeof(unsigned long long), b->stream));   // overflow, overwritten, max_used, deficit
  const uint32_t threads = 256, grid = (b->n_next + threads - 1) / threads;
  admit_kernel<<<grid, threads, 0, b->stream>>>(d_src, n, w, b->d_ctl, b->d_timers, b->n_next, b->R, b->K,
                                                b->cfg.sub_id_base, b->n_timers > 0 && b->K > 0, b->d_stats,
                                                b->n_paired > 0 ? b->d_pairs : nullptr);
  CK(cudaGetLastError());
  b->st.kernel_launches++;
  CK(cudaMemcpyAsync(&b->h_stats->admit_overflow, &b->d_stats->admit_overflow, 4 * sizeof(unsigned long long),
                     cudaMemcpyDeviceToHost, b->stream));
  return CPBUS_OK;
}

// lossless admission (reference: the sender blocks on a full channel, events/subscriber.go:30-32)
int admit(cpbus* b, const cpbus_event* d_src, uint32_t n, uint64_t w, bool* ok, uint32_t* prefix = nullptr) {
  *ok = true;
  if (prefix) *prefix = n;
  if (!b->lossless || b->n_next == 0) return CPBUS_OK;
  const uint64_t need = admit_need(n, b->K, b->n_timers > 0, b->min_period, b->last_watermark, w);
  if (b->room_lb >= need) { b->room_lb -= need; b->st.admit_skipped++; return CPBUS_OK; }   // provably fits: no kernel, no sync
  int rc = admit_launch(b, d_src, n, w); if (rc) return rc;
  b->st.admit_passes++;
  CK(cudaStreamSynchronize(b->stream));
  *ok = b->h_stats->admit_overflow == 0;
  if (!*ok && prefix) *prefix = n - (uint32_t)std::min<unsigned long long>(n, b->h_stats->admit_deficit);   // events every mailbox can still take
  const uint64_t used = b->h_stats->admit_max_used;            // fullest mailbox, this batch included
  // admitted: the batch is in; refused: nothing was appended, so the fullest mailbox holds at most `used` minus its share (>= 0):
  // keep the conservative figure either way
  b->room_lb = used >= b->R ? 0 : b->R - used;
  return CPBUS_OK;
}

// host mirror of one-shot timers that have fired on the device (events/timer.go:19-33):
// a one-shot whose due time is <= the last launched watermark has disarmed itself.
void retire_oneshots(cpbus* b, uint64_t w) {
  size_t keep = 0;
  for (size_t i = 0; i < b->oneshot_idx.size(); i++) {
    HostTimer& t = b->h_timers[b->oneshot_idx[i]];
    if (t.active && t.oneshot && t.next_due <= w) { t.active = false; b->n_timers--; continue; }
    if (t.active && t.oneshot) b->oneshot_idx[keep++] = b->oneshot_idx[i];
  }
  b->oneshot_idx.resize(keep);
  if (b->n_timers == 0) b->min_period = UINT64_MAX;
}

int flush_sharded(cpbus* h, uint64_t w);

int flush_staged(cpbus* b, uint64_t w) {
  if (b->sharded()) return flush_sharded(b, w);
  const uint32_t n = (uint32_t)b->n_staged;
  if (n == 0 && b->n_timers == 0) { b->last_watermark = std::max(b->last_watermark, w); return CPBUS_OK; }   // nothing armed: the watermark follows the clock
  if (n == 0 && w == b->last_watermark) return CPBUS_OK;
  const int c = b->cur;
  int rc;
  if (b->zero_copy && !b->lossless) {
    // Zero-copy ingest: the pinned staging buffer is mapped into the device address space; CTA 0 of the fan-out pulls the
    // batch over PCIe in its prologue (the staged path) — no H2D op, no stream waits, consecutive fan-outs stay adjacent.
    rc = launch_fanout(b, b->h_batch[c], n, w, /*staged=*/1);
    if (rc) return rc;
    if ((c & (cpbus::kEpoch - 1)) == cpbus::kEpoch - 1) CK(cudaEventRecord(b->consumed[c], b->stream));
    b->n_staged = 0;
    b->cur = (b->cur + 1) % cpbus::kStage;
    CK(cudaEventSynchronize(b->consumed[b->cur | (cpbus::kEpoch - 1)]));   // the launch that read the buffer we are about to overwrite has finished
    return CPBUS_OK;
  }
  // Device staging is a long ring (kDevSlots batches): a slot is reused only kDevSlots flushes later, far beyond how far the
  // host can run ahead, so the H2D never has to wait for an old fan-out and lands within microseconds.  Reuse safety is a
  // host-side check once per epoch of kDevEpoch slots (almost always already satisfied).
  const uint32_t slot = b->dev_slot;
  cpbus_event* d_dst = b->d_stage + (size_t)slot * b->B;
  if (slot % cpbus::kDevEpoch == 0) CK(cudaEventSynchronize(b->epoch_done[slot / cpbus::kDevEpoch]));   // last round's users of this epoch are done
  if (n) {
    CK(cudaMemcpyAsync(d_dst, b->h_batch[c], (size_t)n * sizeof(cpbus_event), cudaMemcpyHostToDevice, b->copy_stream));
    CK(cudaEventRecord(b->h2d_done[c], b->copy_stream));
    // Give the 8-16 KiB copy a few microseconds to land.  If it has, the bus stream needs no wait node, consecutive fan-outs
    // stay adjacent in the stream and the next launch's prologue overlaps this one's tail (programmatic dependent launch).
    bool landed = false;
    const auto t_spin = std::chrono::steady_clock::now();
    do {
      const cudaError_t q = cudaEventQuery(b->h2d_done[c]);
      if (q == cudaSuccess) { landed = true; break; }
      if (q != cudaErrorNotReady) { CK(q); }
    } while (std::chrono::steady_clock::now() - t_spin < std::chrono::microseconds(b->h2d_spin_us));
    if (!landed) CK(cudaStreamWaitEvent(b->stream, b->h2d_done[c], 0));
  }
  bool ok = true;
  uint32_t m = n;
  rc = admit(b, d_dst, n, w, &ok, &m);
  if (rc) return rc;
  if (!ok) {
    // Some mailbox lacks the room.  Like the Go bus, which blocks at the first event a full channel cannot take
    // (events/subscriber.go:30-32), deliver the longest prefix EVERY mailbox can take — with the ticks due by its last
    // event — keep the rest staged and report the stall; the caller lets the consumers run and flushes again.
    if (m == 0) return CPBUS_EAGAIN;
    const uint64_t w_part = b->h_batch[c][m - 1].ts_ns;
    rc = launch_fanout(b, d_dst, m, w_part);
    if (rc) return rc;
    if (slot % cpbus::kDevEpoch == cpbus::kDevEpoch - 1) CK(cudaEventRecord(b->epoch_done[slot / cpbus::kDevEpoch], b->stream));
    b->dev_slot = (slot + 1) % cpbus::kDevSlots;
    memmove(b->h_batch[c], b->h_batch[c] + m, (size_t)(n - m) * sizeof(cpbus_event));   // (the H2D of this buffer completed before the admission pass)
    b->n_staged = n - m;
    b->room_lb = 0;
    b->st.admit_partial++;
    return CPBUS_EAGAIN;
  }
  rc = launch_fanout(b, d_dst, n, w);
  if (rc) return rc;
  if (slot % cpbus::kDevEpoch == cpbus::kDevEpoch - 1) CK(cudaEventRecord(b->epoch_done[slot / cpbus::kDevEpoch], b->stream));
  b->dev_slot = (slot + 1) % cpbus::kDevSlots;
  b->n_staged = 0;
  b->cur = (b->cur + 1) % cpbus::kStage;
  CK(cudaEventSynchronize(b->h2d_done[b->cur]));   // the pinned buffer we are about to overwrite has left the host
  return CPBUS_OK;
}

// armed timers; on a sharded handle the sum over its shards
uint32_t timers_armed(const cpbus* b) {
  uint32_t n = b->n_timers;
  for (const cpbus* s : b->shards) n += s->n_timers;
  return n;
}

// (a sharded handle keeps min_period the way one bus would; each shard's own bound is never below it, so every shard
// accepts the handle's step)
uint64_t max_window(const cpbus* b) {
  if (!b->K || timers_armed(b) == 0 || b->min_period == UINT64_MAX) return UINT64_MAX;
  const uint64_t J = 32u / b->K;
  return b->min_period > UINT64_MAX / J ? UINT64_MAX : b->min_period * J;
}

int stage_one(cpbus* b, uint32_t code, uint32_t source_id, uint32_t target, uint32_t flags) {
  if (b->n_staged == b->B) { int rc = flush_staged(b, b->now); if (rc) return rc; }
  cpbus_event& e = b->h_batch[b->cur][b->n_staged++];
  e.seq = b->seq++; e.ts_ns = b->now; e.code = code; e.source_id = source_id; e.target = target; e.flags = flags;
  return CPBUS_OK;
}

bool is_pow2(uint32_t x) { return x && !(x & (x - 1)); }

// ---- sharded handle (cpbus_create_sharded): the entry points below route here; definitions at the end of the file ----
int sh_subscribe_many(cpbus* h, const uint32_t* masks, uint32_t n, uint32_t* first_sub_id);
int sh_subscribe_pairs(cpbus* h, uint32_t mask, const cpbus_pair* pairs, uint32_t n_pairs, uint32_t* sub_id);
int sh_subscribe_pairs_many(cpbus* h, const uint32_t* masks, const cpbus_pair* pairs, const uint32_t* n_pairs, uint32_t n, uint32_t* first_sub_id);
int sh_unsubscribe(cpbus* h, uint32_t sub_id);
int sh_set_mask(cpbus* h, uint32_t sub_id, uint32_t mask);
int sh_timer_add(cpbus* h, uint32_t sub_id, uint64_t period_ns, uint32_t source_id, int oneshot, uint32_t* timer_id);
int sh_timer_add_many(cpbus* h, uint32_t first_sub, uint32_t n, uint64_t period_ns, const uint32_t* source_ids, uint32_t source_id0, int oneshot);
int sh_timer_cancel(cpbus* h, uint32_t timer_id);
int sh_send(cpbus* h, uint32_t sub_id, const cpbus_event* ev);
int sh_publish_device(cpbus* h, const void* d_events, size_t n, uint64_t watermark_ns);
int sh_drain_many(cpbus* h, uint32_t first_sub, uint32_t n, cpbus_event* out, size_t cap, uint32_t* offsets, uint32_t* counts, size_t* total);
int sh_digest(cpbus* h, uint32_t first_sub, uint32_t n, cpbus_digest_t* out);
int sh_digest_fold_begin(cpbus* h, uint32_t first_sub, uint32_t n, uint32_t* ticket);
int sh_digest_fold_end(cpbus* h, uint32_t ticket, uint64_t out[4]);
int sh_step_result_begin(cpbus* h, uint32_t* ticket);
int sh_step_result_end(cpbus* h, uint32_t ticket, uint64_t out[4]);
int sh_stats(cpbus* h, cpbus_stats_t* out);
// the shard that holds the subscriber with global id sub_id, or nullptr (CPBUS_ENOENT) if the handle has not handed it out
cpbus* sh_owner(const cpbus* h, uint32_t sub_id);

}  // namespace

extern "C" {
// Nothing may unwind through the C boundary (cgo, ctypes): every status-returning entry point is a function-try-block.
#define CPBUS_CATCH                                                                                   \
  catch (const std::bad_alloc&) { return CPBUS_ENOMEM; }                                              \
  catch (...) { snprintf(g_cuda_err, sizeof(g_cuda_err), "unexpected C++ exception"); return CPBUS_ECUDA; }

uint32_t cpbus_abi_version(void) { return 2; }
static int split_plan(const uint64_t* ts, size_t n, uint32_t batch_cap, uint64_t now, uint64_t watermark, uint64_t window,
                      std::vector<size_t>& end, std::vector<uint64_t>& wm);
int cpbus_split_plan(const uint64_t* ts, size_t n, uint32_t batch_cap, uint64_t now_ns, uint64_t watermark_ns, uint64_t window_ns,
                     size_t* ends, uint64_t* watermarks, size_t cap, size_t* n_slices) try {
  if ((!ts && n) || !n_slices || (cap && (!ends || !watermarks))) return CPBUS_EINVAL;
  std::vector<size_t> end; std::vector<uint64_t> wm;
  const int rc = split_plan(ts, n, batch_cap, now_ns, watermark_ns, window_ns, end, wm);
  if (rc) return rc;
  *n_slices = end.size();
  for (size_t k = 0; k < end.size() && k < cap; k++) { ends[k] = end[k]; watermarks[k] = wm[k]; }
  return CPBUS_OK;
} CPBUS_CATCH
size_t cpbus_mask_order(const uint32_t* masks, const uint8_t* active, uint32_t n, uint32_t ring_cap, uint32_t block, int heavy_first, uint32_t* out) {
  if (!masks || !out || !ring_cap) return 0;
  try {
    std::vector<uint32_t> order;
    mask_order(masks, active, n, ring_cap, block, heavy_first != 0, order);
    std::copy(order.begin(), order.end(), out);
    return order.size();
  } catch (const std::bad_alloc&) { return 0; }
}

const char* cpbus_last_cuda_error(void) { return g_cuda_err; }

const char* cpbus_strerror(int s) {
  switch (s) {
    case CPBUS_OK: return "ok";
    case CPBUS_EINVAL: return "invalid argument";
    case CPBUS_ENOMEM: return "out of memory";
    case CPBUS_ECUDA: return "CUDA error";
    case CPBUS_EAGAIN: return "mailbox full (lossless mode): drain and retry";
    case CPBUS_ENOSPC: return "capacity exhausted";
    case CPBUS_ENOENT: return "no such subscriber or timer";
    case CPBUS_ECLOSED: return "subscriber already unsubscribed";
    case CPBUS_ENODEV: return "no CUDA device (libcpbus has no CPU fallback)";
    case CPBUS_EORDER: return "clock moved backwards, batch unsorted or timer window exceeded";
    case CPBUS_ETIMEDOUT: return "stream batch never arrived (publisher stalled or consumer a whole ring behind)";
    default: return "unknown status";
  }
}

// EventCode.String — events/eventcode_string.go:5-15
const char* cpbus_code_name(int code) {
  static const char* const names[CPBUS_N_CODES] = {
      "None", "ExitSuccess", "ExitFailed", "Stopping", "Stopped", "StatusHealthy", "StatusUnhealthy", "StatusChanged",
      "TimerExpired", "EnterMaintenance", "ExitMaintenance", "Error", "Quit", "Metric", "Startup", "Shutdown", "Signal"};
  return (code < 0 || code >= CPBUS_N_CODES) ? nullptr : names[code];
}

// FromString — events/events.go:52-86
int cpbus_code_from_string(const char* name) try {
  if (!name) return -1;
  static const std::unordered_map<std::string, int> table = {
      {"exitSuccess", CPBUS_EXIT_SUCCESS}, {"exitFailed", CPBUS_EXIT_FAILED}, {"stopping", CPBUS_STOPPING},
      {"stopped", CPBUS_STOPPED}, {"healthy", CPBUS_STATUS_HEALTHY}, {"unhealthy", CPBUS_STATUS_UNHEALTHY},
      {"changed", CPBUS_STATUS_CHANGED}, {"timerExpired", CPBUS_TIMER_EXPIRED},
      {"enterMaintenance", CPBUS_ENTER_MAINTENANCE}, {"exitMaintenance", CPBUS_EXIT_MAINTENANCE},
      {"error", CPBUS_ERROR}, {"quit", CPBUS_QUIT}, {"startup", CPBUS_STARTUP}, {"shutdown", CPBUS_SHUTDOWN},
      {"SIGHUP", CPBUS_SIGNAL}, {"SIGUSR2", CPBUS_SIGNAL}};
  auto it = table.find(name);
  return it == table.end() ? -1 : it->second;
} CPBUS_CATCH

uint64_t cpbus_record_hash(const cpbus_event* e) {
  return record_hash_words(e->seq, e->ts_ns, (uint64_t)e->code | ((uint64_t)e->source_id << 32),
                           (uint64_t)e->target | ((uint64_t)e->flags << 32));
}
uint64_t cpbus_digest_multiplier(void) { return kDigestP; }

static bool config_ok(const cpbus_config* cfg) {
  const uint32_t R = cfg->ring_cap ? cfg->ring_cap : 1024;
  const uint32_t B = cfg->batch_cap ? cfg->batch_cap : std::min(256u, R / 2);
  const uint32_t K = cfg->timers_per_sub;
  if (!cfg->n_max_subs || !is_pow2(R) || R < 64 || B == 0 || B > R / 2 || (B % 32) != 0 || B > 1024) return false;   // 1024: the kernel keeps one match word per 32-event chunk in a lane
  if (!(K == 0 || K == 1 || K == 2 || K == 4 || K == 8)) return false;
  if ((uint64_t)cfg->n_max_subs * std::max(K, 1u) > kTimerSlotMask) return false;   // timer ids keep 6 generation bits
  return cfg->store_path <= CPBUS_STORE_BULK;
}

int cpbus_create(const cpbus_config* cfg, cpbus_t** out) try {
  if (!cfg || !out) return CPBUS_EINVAL;
  *out = nullptr;
  if (!config_ok(cfg)) return CPBUS_EINVAL;
  const uint32_t R = cfg->ring_cap ? cfg->ring_cap : 1024;
  const uint32_t B = cfg->batch_cap ? cfg->batch_cap : std::min(256u, R / 2);
  const uint32_t K = cfg->timers_per_sub;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "no CUDA device visible");
    return CPBUS_ENODEV;
  }
  cpbus* b = new (std::nothrow) cpbus();
  if (!b) return CPBUS_ENOMEM;
  b->cfg = *cfg; b->cfg.ring_cap = R; b->cfg.batch_cap = B;
  b->N = cfg->n_max_subs; b->R = R; b->B = B; b->K = K;
  b->lossless = cfg->flags & CPBUS_CFG_LOSSLESS; b->use_digest = cfg->flags & CPBUS_CFG_DIGEST;
  b->room_lb = R;
  b->store = cfg->store_path == CPBUS_STORE_AUTO ? CPBUS_STORE_V8 : (int)cfg->store_path;
  if (const char* e = getenv("CPBUS_H2D_SPIN_US")) b->h2d_spin_us = atoi(e);
  if (const char* e = getenv("CPBUS_ORDER")) b->use_order = atoi(e);
  if (const char* e = getenv("CPBUS_PDL")) b->pdl = atoi(e) != 0;
  if (const char* e = getenv("CPBUS_ZERO_COPY")) b->zero_copy = atoi(e) != 0;
  if (const char* e = getenv("CPBUS_HINTS")) b->hints = atoi(e);
  if (const char* e = getenv("CPBUS_SUBS_PER_WARP")) b->subs_per_warp = (uint32_t)atoi(e);   // tuning knob for experiments
  if (const char* e = getenv("CPBUS_ORDER_BLOCK")) b->order_block = (uint32_t)atoll(e);
  if (const char* e = getenv("CPBUS_ORDER_HEAVY")) b->order_heavy_first = atoi(e) != 0;
  int rc = CPBUS_OK;
  auto fail = [&](int code) { cpbus_destroy(b); return code; };
  if (cfg->device >= 0) b->device = cfg->device;
  else if (cudaGetDevice(&b->device) != cudaSuccess) return fail(CPBUS_ECUDA);
  if (b->device >= ndev) return fail(CPBUS_EINVAL);
  if ((rc = dev_guard(b))) return fail(rc);
  cudaDeviceProp prop{};
  if (cudaGetDeviceProperties(&prop, b->device) == cudaSuccess) b->sm_count = prop.multiProcessorCount;
  if (cfg->stream) b->stream = (cudaStream_t)cfg->stream;
  else {
    if (cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess) return fail(CPBUS_ECUDA);
    b->own_stream = true;
  }
  const size_t N = b->N;
#define ALLOC(ptr, bytes)                                                                     \
  if (cudaMalloc((void**)&(ptr), (bytes)) != cudaSuccess) {                                   \
    snprintf(g_cuda_err, sizeof(g_cuda_err), "cudaMalloc(%zu) failed", (size_t)(bytes));     \
    return fail(CPBUS_ENOMEM);                                                                \
  }
  ALLOC(b->d_ring, N * R * sizeof(cpbus_event));
  ALLOC(b->d_ctl, N * sizeof(SubCtl)); ALLOC(b->d_order, N * 4);
  if (K) ALLOC(b->d_timers, N * K * sizeof(DevTimer));
  ALLOC(b->d_stats, sizeof(DevStats)); ALLOC(b->d_fold, 32 * cpbus::kFoldSlots); ALLOC(b->d_pow, kPowTableLen * 8);
  ALLOC(b->d_desc, 2 * ((fanout_desc_bytes(2048) + 255) & ~(size_t)255)); ALLOC(b->d_desc_ready, 256);
  if (cudaMemsetAsync(b->d_desc_ready, 0, 256, b->stream) != cudaSuccess) return fail(CPBUS_ECUDA);
  if (cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(CPBUS_ECUDA);
  if (cudaStreamCreateWithFlags(&b->result_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(CPBUS_ECUDA);
  if (cudaEventCreateWithFlags(&b->launched, cudaEventDisableTiming) != cudaSuccess) return fail(CPBUS_ECUDA);
  ALLOC(b->d_stage, (size_t)cpbus::kDevSlots * B * sizeof(cpbus_event));
  for (int i = 0; i < cpbus::kDevSlots / cpbus::kDevEpoch; i++)
    if (cudaEventCreateWithFlags(&b->epoch_done[i], cudaEventDisableTiming) != cudaSuccess) return fail(CPBUS_ECUDA);
  for (int i = 0; i < cpbus::kStage; i++) {
    if (cudaMallocHost((void**)&b->h_batch[i], (size_t)B * sizeof(cpbus_event)) != cudaSuccess) return fail(CPBUS_ENOMEM);
    if (cudaEventCreateWithFlags(&b->h2d_done[i], cudaEventDisableTiming) != cudaSuccess) return fail(CPBUS_ECUDA);
    if (cudaEventCreateWithFlags(&b->consumed[i], cudaEventDisableTiming) != cudaSuccess) return fail(CPBUS_ECUDA);
  }
  ALLOC(b->d_batch_local, (size_t)B * sizeof(cpbus_event));
  ALLOC(b->d_pf_buf, (size_t)kStreamPrefetch * B * sizeof(cpbus_event)); ALLOC(b->d_pf_state, 64);
  ALLOC(b->d_acct, sizeof(DevPubAcct));
  if (cudaMemsetAsync(b->d_pf_state, 0, 64, b->stream) != cudaSuccess ||
      cudaMemsetAsync(b->d_acct, 0, sizeof(DevPubAcct), b->stream) != cudaSuccess) return fail(CPBUS_ECUDA);
  if (cudaHostAlloc((void**)&b->h_err, 64, cudaHostAllocMapped) != cudaSuccess) return fail(CPBUS_ENOMEM);
  memset(b->h_err, 0, 64);
  if (cudaHostGetDevicePointer((void**)&b->d_err, b->h_err, 0) != cudaSuccess) return fail(CPBUS_ECUDA);
  if (cudaMallocHost((void**)&b->h_acct, offsetof(DevPubAcct, pair_key)) != cudaSuccess) return fail(CPBUS_ENOMEM);
  for (int i = 0; i < cpbus::kPrefetch; i++) ALLOC(b->d_prefetch[i], (size_t)B * sizeof(cpbus_event));
  ALLOC(b->d_result, sizeof(DevResultSlot) * kResultRing * kResultSub);
  if (cudaMemsetAsync(b->d_result, 0, sizeof(DevResultSlot) * kResultRing * kResultSub, b->stream) != cudaSuccess) return fail(CPBUS_ECUDA);
  if (cudaMallocHost((void**)&b->h_result, sizeof(DevResultSlot) * 8 * kResultSub) != cudaSuccess) return fail(CPBUS_ENOMEM);
  for (int i = 0; i < 8; i++)
    if (cudaEventCreateWithFlags(&b->result_done[i], cudaEventDisableTiming) != cudaSuccess) return fail(CPBUS_ECUDA);
#undef ALLOC
  if (cudaMallocHost((void**)&b->h_stats, sizeof(DevStats)) != cudaSuccess) return fail(CPBUS_ENOMEM);
  if (cudaMallocHost((void**)&b->h_fold, 32 * cpbus::kFoldSlots) != cudaSuccess) return fail(CPBUS_ENOMEM);
  for (int i = 0; i < cpbus::kFoldSlots; i++)
    if (cudaEventCreateWithFlags(&b->fold_done[i], cudaEventDisableTiming) != cudaSuccess) return fail(CPBUS_ECUDA);
  // rings are NOT cleared: a slot is only ever read after it has been written (head/tail bound every read)
  bool ok = cudaMemsetAsync(b->d_ctl, 0, N * sizeof(SubCtl), b->stream) == cudaSuccess &&
            cudaMemsetAsync(b->d_stats, 0, sizeof(DevStats), b->stream) == cudaSuccess &&
            (!K || cudaMemsetAsync(b->d_timers, 0xFF, N * K * sizeof(DevTimer), b->stream) == cudaSuccess) &&   // every slot idle
            cudaStreamSynchronize(b->stream) == cudaSuccess;
  if (!ok) return fail(CPBUS_ECUDA);
  {
    std::vector<uint64_t> pw(kPowTableLen);
    uint64_t x = 1;
    for (uint32_t i = 0; i < kPowTableLen; i++) { pw[i] = x; x *= kDigestP; }
    if (cudaMemcpyAsync(b->d_pow, pw.data(), kPowTableLen * 8, cudaMemcpyHostToDevice, b->stream) != cudaSuccess ||
        cudaStreamSynchronize(b->stream) != cudaSuccess) return fail(CPBUS_ECUDA);
  }
  b->h_mask.assign(N, 0);
  b->h_active.assign(N, 0);
  b->intern.emplace(std::string(), 0u);   // "" -> 0 so that NonEvent == {None, 0} (events/events.go:45)
  b->sources.emplace_back();
  *out = b;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_destroy(cpbus_t* b) try {
  if (!b) return CPBUS_EINVAL;
  if (b->sharded()) {
    for (size_t k = b->shard_st.size(); k-- > 0;) cpbus_stream_close(b->shard_st[k]);   // attached ends before the owner
    for (size_t k = b->shards.size(); k-- > 0;) cpbus_destroy(b->shards[k]);
    if (b->h_batch[0]) cudaFreeHost(b->h_batch[0]);
    delete b;
    return CPBUS_OK;
  }
  cudaSetDevice(b->device);
  if (b->stream) cudaStreamSynchronize(b->stream);
  while (!b->streams.empty()) cpbus_stream_close(b->streams.back());
  cudaFree(b->d_ring); cudaFree(b->d_ctl); cudaFree(b->d_order); cudaFree(b->d_pairs);
  cudaFree(b->d_timers); cudaFree(b->d_stats); cudaFree(b->d_fold); cudaFree(b->d_pow); cudaFree(b->d_desc); cudaFree(b->d_desc_ready);
  if (b->copy_stream) cudaStreamSynchronize(b->copy_stream);
  if (b->result_stream) { cudaStreamSynchronize(b->result_stream); cudaStreamDestroy(b->result_stream); }
  for (int i = 0; i < cpbus::kStage; i++) {
    if (b->h_batch[i]) cudaFreeHost(b->h_batch[i]);
    if (b->h2d_done[i]) cudaEventDestroy(b->h2d_done[i]);
    if (b->consumed[i]) cudaEventDestroy(b->consumed[i]);
  }
  cudaFree(b->d_stage);
  for (int i = 0; i < cpbus::kDevSlots / cpbus::kDevEpoch; i++) if (b->epoch_done[i]) cudaEventDestroy(b->epoch_done[i]);
  if (b->copy_stream) cudaStreamDestroy(b->copy_stream);
  if (b->launched) cudaEventDestroy(b->launched);
  cudaFree(b->d_drain); cudaFree(b->d_drain_idx);
  cudaFree(b->d_result); cudaFree(b->d_batch_local); cudaFree(b->d_pf_buf); cudaFree(b->d_pf_state); cudaFree(b->d_acct);
  if (b->h_err) cudaFreeHost(b->h_err);
  if (b->h_acct) cudaFreeHost(b->h_acct);
  for (int i = 0; i < cpbus::kPrefetch; i++) cudaFree(b->d_prefetch[i]);
  for (void* p : b->shared_mapped) cudaIpcCloseMemHandle(p);
  for (void* p : b->shared_owned) cudaFree(p);
  if (b->h_result) cudaFreeHost(b->h_result);
  for (int i = 0; i < 8; i++) if (b->result_done[i]) cudaEventDestroy(b->result_done[i]);
  if (b->h_stats) cudaFreeHost(b->h_stats);
  if (b->h_fold) cudaFreeHost(b->h_fold);
  for (int i = 0; i < cpbus::kFoldSlots; i++) if (b->fold_done[i]) cudaEventDestroy(b->fold_done[i]);
  if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
  delete b;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_intern(cpbus_t* b, const char* s, size_t len, uint32_t* source_id) try {
  if (!b || (!s && len) || !source_id) return CPBUS_EINVAL;
  std::string key(s ? s : "", len);
  auto it = b->intern.find(key);
  if (it != b->intern.end()) { *source_id = it->second; return CPBUS_OK; }
  if (b->sources.size() >= 0xFFFFFFF0u) return CPBUS_ENOSPC;
  if (b->sources.size() >= CPBUS_EPHEMERAL_BIT) return CPBUS_ENOSPC;   // permanent ids never carry the ephemeral bit
  const uint32_t id = (uint32_t)b->sources.size();
  b->sources.push_back(key);
  b->intern_bytes += key.size();
  b->intern.emplace(std::move(key), id);
  *source_id = id;
  return CPBUS_OK;
} CPBUS_CATCH

// Bounded region for payload strings (control/endpoints.go:125-126: Source = "key|value" of every posted metric).
// id = EPHEMERAL_BIT | generation(15) << 16 | slot(16); the slot's previous string is dropped when it is reused.
int cpbus_intern_ephemeral(cpbus_t* b, const char* s, size_t len, uint32_t* source_id) try {
  if (!b || (!s && len) || !source_id) return CPBUS_EINVAL;
  std::string key(s ? s : "", len);
  auto perm = b->intern.find(key);
  if (perm != b->intern.end()) { *source_id = perm->second; return CPBUS_OK; }   // already a name: keep one id per string
  auto it = b->eph_map.find(key);
  if (it != b->eph_map.end()) {
    const cpbus::EphSlot& e = b->eph[it->second];
    *source_id = CPBUS_EPHEMERAL_BIT | ((e.gen & 0x7FFFu) << 16) | it->second;
    return CPBUS_OK;
  }
  if (b->eph.empty()) b->eph.resize(CPBUS_EPHEMERAL_SLOTS);
  const uint32_t slot = b->eph_next;
  b->eph_next = (slot + 1) % CPBUS_EPHEMERAL_SLOTS;
  cpbus::EphSlot& e = b->eph[slot];
  if (e.live) { b->eph_map.erase(e.s); b->eph_recycled++; } else b->eph_live++;
  e.gen++; e.live = true; e.s = key;
  b->eph_map.emplace(std::move(key), slot);
  *source_id = CPBUS_EPHEMERAL_BIT | ((e.gen & 0x7FFFu) << 16) | slot;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_source(cpbus_t* b, uint32_t id, char* out, size_t cap, size_t* len) try {
  if (!b) return CPBUS_EINVAL;
  if (id & CPBUS_EPHEMERAL_BIT) {
    const uint32_t slot = id & 0xFFFFu, gen = (id >> 16) & 0x7FFFu;
    if (slot >= b->eph.size() || !b->eph[slot].live || (b->eph[slot].gen & 0x7FFFu) != gen) return CPBUS_ENOENT;   // recycled
    const std::string& s = b->eph[slot].s;
    if (len) *len = s.size();
    if (out && cap) memcpy(out, s.data(), std::min(cap, s.size()));
    return CPBUS_OK;
  }
  if (id >= b->sources.size()) return CPBUS_ENOENT;
  const std::string& s = b->sources[id];
  if (len) *len = s.size();
  if (out && cap) memcpy(out, s.data(), std::min(cap, s.size()));
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_subscribe_many(cpbus_t* b, const uint32_t* masks, uint32_t n, uint32_t* first_sub_id) try {
  if (!b || !n) return CPBUS_EINVAL;
  if ((uint64_t)b->n_next + n > b->N) return CPBUS_ENOSPC;
  if (b->sharded()) return sh_subscribe_many(b, masks, n, first_sub_id);
  int rc = dev_guard(b); if (rc) return rc;
  if ((rc = flush_staged(b, b->now))) return rc;   // ordered with publishes (events/bus.go:105-107 takes the same lock)
  const uint32_t first = b->n_next;
  std::vector<SubCtl> blocks(n);
  memset(blocks.data(), 0, (size_t)n * sizeof(SubCtl));
  for (uint32_t i = 0; i < n; i++) {
    b->h_mask[first + i] = (masks ? masks[i] : CPBUS_MASK_ALL) & CPBUS_MASK_ALL;
    blocks[i].mask = b->h_mask[first + i] | kActiveBit;
    b->h_active[first + i] = 1;
    if (b->h_mask[first + i] != CPBUS_MASK_ALL) b->n_filtered++;
  }
  CK(cudaMemcpyAsync(b->d_ctl + first, blocks.data(), (size_t)n * sizeof(SubCtl), cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  b->n_next += n; b->n_active += n; b->order_dirty = true;
  if (first_sub_id) *first_sub_id = b->cfg.sub_id_base + first;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_subscribe(cpbus_t* b, uint32_t mask, uint32_t* sub_id) { return cpbus_subscribe_many(b, &mask, 1, sub_id); }

static int push_mask_words(cpbus* b, uint32_t first, uint32_t n);

int cpbus_subscribe_pairs(cpbus_t* b, uint32_t mask, const cpbus_pair* pairs, uint32_t n_pairs, uint32_t* sub_id) try {
  if (!b || n_pairs > CPBUS_MAX_PAIRS || (n_pairs && !pairs)) return CPBUS_EINVAL;
  for (uint32_t j = 0; j < n_pairs; j++) if (pairs[j].code >= CPBUS_N_CODES) return CPBUS_EINVAL;
  if (b->sharded()) return sh_subscribe_pairs(b, mask, pairs, n_pairs, sub_id);
  // a pair whose code is already in the mask adds nothing; what is left decides whether a table is needed at all
  uint2 row[CPBUS_MAX_PAIRS];
  uint32_t used = 0;
  for (uint32_t j = 0; j < n_pairs; j++)
    if (!((mask >> pairs[j].code) & 1u)) row[used++] = make_uint2(pairs[j].code, pairs[j].source_id);
  if (used == 0) return cpbus_subscribe_many(b, &mask, 1, sub_id);
  int rc = dev_guard(b); if (rc) return rc;
  if (!b->d_pairs) {
    if (cudaMalloc((void**)&b->d_pairs, (size_t)b->N * CPBUS_MAX_PAIRS * sizeof(uint2)) != cudaSuccess) {
      snprintf(g_cuda_err, sizeof(g_cuda_err), "cudaMalloc(pair tables) failed");
      return CPBUS_ENOMEM;
    }
    CK(cudaMemsetAsync(b->d_pairs, 0xFF, (size_t)b->N * CPBUS_MAX_PAIRS * sizeof(uint2), b->stream));   // every slot unused
    b->h_npairs.assign(b->N, 0);
  }
  uint32_t id = 0;
  if ((rc = cpbus_subscribe_many(b, &mask, 1, &id))) return rc;
  const uint32_t l = id - b->cfg.sub_id_base;
  for (uint32_t j = used; j < CPBUS_MAX_PAIRS; j++) row[j] = make_uint2(kPairNone, kPairNone);
  CK(cudaMemcpyAsync(b->d_pairs + (size_t)l * CPBUS_MAX_PAIRS, row, sizeof(row), cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));   // `row` is on the stack
  b->h_npairs[l] = (uint8_t)used; b->n_paired++;
  if ((rc = push_mask_words(b, l, 1))) return rc;
  if (sub_id) *sub_id = id;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_subscribe_pairs_many(cpbus_t* b, const uint32_t* masks, const cpbus_pair* pairs, const uint32_t* n_pairs,
                               uint32_t n, uint32_t* first_sub_id) try {
  if (!b || !n || !masks || !pairs || !n_pairs) return CPBUS_EINVAL;
  for (uint32_t i = 0; i < n; i++) {
    if (n_pairs[i] > CPBUS_MAX_PAIRS) return CPBUS_EINVAL;
    for (uint32_t j = 0; j < n_pairs[i]; j++) if (pairs[(size_t)i * CPBUS_MAX_PAIRS + j].code >= CPBUS_N_CODES) return CPBUS_EINVAL;
  }
  if ((uint64_t)b->n_next + n > b->N) return CPBUS_ENOSPC;
  if (b->sharded()) return sh_subscribe_pairs_many(b, masks, pairs, n_pairs, n, first_sub_id);
  int rc = dev_guard(b); if (rc) return rc;
  if (!b->d_pairs) {
    if (cudaMalloc((void**)&b->d_pairs, (size_t)b->N * CPBUS_MAX_PAIRS * sizeof(uint2)) != cudaSuccess) {
      snprintf(g_cuda_err, sizeof(g_cuda_err), "cudaMalloc(pair tables) failed");
      return CPBUS_ENOMEM;
    }
    CK(cudaMemsetAsync(b->d_pairs, 0xFF, (size_t)b->N * CPBUS_MAX_PAIRS * sizeof(uint2), b->stream));   // every slot unused
    b->h_npairs.assign(b->N, 0);
  }
  uint32_t first = 0;
  if ((rc = cpbus_subscribe_many(b, masks, n, &first))) return rc;
  const uint32_t l0 = first - b->cfg.sub_id_base;
  std::vector<uint2> rows((size_t)n * CPBUS_MAX_PAIRS, make_uint2(kPairNone, kPairNone));
  uint32_t paired = 0;
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t m = masks[i] & CPBUS_MASK_ALL;
    uint32_t used = 0;
    for (uint32_t j = 0; j < n_pairs[i]; j++) {
      const cpbus_pair& pr = pairs[(size_t)i * CPBUS_MAX_PAIRS + j];
      if (!((m >> pr.code) & 1u)) rows[(size_t)i * CPBUS_MAX_PAIRS + used++] = make_uint2(pr.code, pr.source_id);
    }
    b->h_npairs[l0 + i] = (uint8_t)used;
    if (used) paired++;
  }
  CK(cudaMemcpyAsync(b->d_pairs + (size_t)l0 * CPBUS_MAX_PAIRS, rows.data(), rows.size() * sizeof(uint2), cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  b->n_paired += paired;
  if (paired && (rc = push_mask_words(b, l0, n))) return rc;
  if (first_sub_id) *first_sub_id = first;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_unsubscribe(cpbus_t* b, uint32_t sub_id) try {
  if (!b) return CPBUS_EINVAL;
  if (b->sharded()) return sh_unsubscribe(b, sub_id);
  const uint32_t l = sub_id - b->cfg.sub_id_base;
  if (sub_id < b->cfg.sub_id_base || l >= b->n_next) return CPBUS_ENOENT;
  int rc = dev_guard(b); if (rc) return rc;
  if ((rc = flush_staged(b, b->now))) return rc;
  // second Unsubscribe drives the WaitGroup negative in Go (events/bus.go:121) => panic
  if (!b->h_active[l]) return CPBUS_ECLOSED;
  b->h_active[l] = 0;
  if (b->h_mask[l] != CPBUS_MASK_ALL) b->n_filtered--;
  if (!b->h_npairs.empty() && b->h_npairs[l]) { b->h_npairs[l] = 0; b->n_paired--; }
  b->order_dirty = true;
  const uint32_t word = 0;
  CK(cudaMemcpyAsync(&b->d_ctl[l].mask, &word, 4, cudaMemcpyHostToDevice, b->stream));
  if (b->K && !b->h_timers.empty()) {
    for (uint32_t k = 0; k < b->K; k++) {
      HostTimer& t = b->h_timers[(size_t)l * b->K + k];
      if (t.active) { t.active = false; b->n_timers--; }
    }
    CK(cudaMemsetAsync(b->d_timers + (size_t)l * b->K, 0xFF, b->K * sizeof(DevTimer), b->stream));
  }
  CK(cudaStreamSynchronize(b->stream));
  b->n_active--;
  return CPBUS_OK;
} CPBUS_CATCH

// Change a subscriber's code mask in place (ordered with publishes like Subscribe): the subscriber keeps its mailbox,
// its timers and its exact cases.  Used when a mailbox that so far only received timer ticks / direct sends (mask 0:
// NewEventTimer on a channel that was not subscribed, watches/watches.go:37,71) is subscribed to the bus after all.
int cpbus_set_mask(cpbus_t* b, uint32_t sub_id, uint32_t mask) try {
  if (!b) return CPBUS_EINVAL;
  if (b->sharded()) return sh_set_mask(b, sub_id, mask);
  const uint32_t l = sub_id - b->cfg.sub_id_base;
  if (sub_id < b->cfg.sub_id_base || l >= b->n_next) return CPBUS_ENOENT;
  if (!b->h_active[l]) return CPBUS_ECLOSED;
  int rc = dev_guard(b); if (rc) return rc;
  if ((rc = flush_staged(b, b->now))) return rc;
  mask &= CPBUS_MASK_ALL;
  if (b->h_mask[l] != CPBUS_MASK_ALL) b->n_filtered--;
  if (mask != CPBUS_MASK_ALL) b->n_filtered++;
  b->h_mask[l] = mask; b->order_dirty = true;
  return push_mask_words(b, l, 1);
} CPBUS_CATCH

static int push_mask_words(cpbus* b, uint32_t first, uint32_t n) {
  std::vector<uint32_t> words(n);
  for (uint32_t i = 0; i < n; i++) words[i] = mask_word(b, first + i);
  CK(cudaMemcpy2DAsync(&b->d_ctl[first].mask, sizeof(SubCtl), words.data(), 4, 4, n, cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return CPBUS_OK;
}

int cpbus_timer_add(cpbus_t* b, uint32_t sub_id, uint64_t period_ns, uint32_t source_id, int oneshot, uint32_t* timer_id) try {
  if (!b || !period_ns) return CPBUS_EINVAL;
  if (!b->K) return CPBUS_ENOSPC;
  if (b->sharded()) return sh_timer_add(b, sub_id, period_ns, source_id, oneshot, timer_id);
  const uint32_t l = sub_id - b->cfg.sub_id_base;
  if (sub_id < b->cfg.sub_id_base || l >= b->n_next) return CPBUS_ENOENT;
  int rc = dev_guard(b); if (rc) return rc;
  if ((rc = flush_staged(b, b->now))) return rc;
  if (b->h_timers.empty()) b->h_timers.resize((size_t)b->N * b->K);
  retire_oneshots(b, b->last_watermark);
  if (!b->h_active[l]) return CPBUS_ECLOSED;
  for (uint32_t k = 0; k < b->K; k++) {
    HostTimer& t = b->h_timers[(size_t)l * b->K + k];
    if (t.active) continue;
    t.active = true; t.oneshot = oneshot != 0; t.period = period_ns; t.next_due = b->now + period_ns; t.source_id = source_id;
    DevTimer d{}; d.next_due = t.next_due; d.period = oneshot ? 0 : period_ns; d.source_id = source_id; d.fired = 0;
    CK(cudaMemcpyAsync(b->d_timers + (size_t)l * b->K + k, &d, sizeof(d), cudaMemcpyHostToDevice, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    b->n_timers++;
    if (!oneshot) b->min_period = std::min(b->min_period, period_ns);
    else b->oneshot_idx.push_back((size_t)l * b->K + k);
    t.gen = (uint8_t)((t.gen + 1) & 0x3F);
    if (timer_id) *timer_id = (l * b->K + k) | ((uint32_t)t.gen << kTimerSlotBits);
    return push_mask_words(b, l, 1);
  }
  return CPBUS_ENOSPC;
} CPBUS_CATCH

int cpbus_timer_add_many(cpbus_t* b, uint32_t first_sub, uint32_t n, uint64_t period_ns, const uint32_t* source_ids,
                         uint32_t source_id0, int oneshot) try {
  if (!b || !period_ns || !n) return CPBUS_EINVAL;
  if (!b->K) return CPBUS_ENOSPC;
  if (b->sharded()) return sh_timer_add_many(b, first_sub, n, period_ns, source_ids, source_id0, oneshot);
  const uint32_t l0 = first_sub - b->cfg.sub_id_base;
  if (first_sub < b->cfg.sub_id_base || (uint64_t)l0 + n > b->n_next) return CPBUS_ENOENT;
  int rc = dev_guard(b); if (rc) return rc;
  if ((rc = flush_staged(b, b->now))) return rc;
  if (b->h_timers.empty()) b->h_timers.resize((size_t)b->N * b->K);
  // bulk arm: uses slot 0 of each subscriber (must be free)
  retire_oneshots(b, b->last_watermark);
  for (uint32_t i = 0; i < n; i++) {
    if (!b->h_active[l0 + i]) return CPBUS_ECLOSED;
    if (b->h_timers[(size_t)(l0 + i) * b->K].active) return CPBUS_ENOSPC;
  }
  std::vector<DevTimer> dev((size_t)n * b->K);
  memset(dev.data(), 0, dev.size() * sizeof(DevTimer));
  CK(cudaMemcpyAsync(dev.data(), b->d_timers + (size_t)l0 * b->K, dev.size() * sizeof(DevTimer), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  for (uint32_t i = 0; i < n; i++) {
    HostTimer& t = b->h_timers[(size_t)(l0 + i) * b->K];
    t.active = true; t.oneshot = oneshot != 0; t.period = period_ns; t.next_due = b->now + period_ns;
    t.source_id = source_ids ? source_ids[i] : source_id0 + i;
    DevTimer& d = dev[(size_t)i * b->K];
    d.next_due = t.next_due; d.period = oneshot ? 0 : period_ns; d.source_id = t.source_id; d.fired = 0; d.pad[0] = d.pad[1] = 0;
    if (oneshot) b->oneshot_idx.push_back((size_t)(l0 + i) * b->K);
  }
  CK(cudaMemcpyAsync(b->d_timers + (size_t)l0 * b->K, dev.data(), dev.size() * sizeof(DevTimer), cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  b->n_timers += n;
  if (!oneshot) b->min_period = std::min(b->min_period, period_ns);
  return push_mask_words(b, l0, n);
} CPBUS_CATCH

int cpbus_timer_cancel(cpbus_t* b, uint32_t timer_id) try {
  if (!b) return CPBUS_EINVAL;
  if (b->sharded()) return sh_timer_cancel(b, timer_id);
  if (!b->K || b->h_timers.empty()) return CPBUS_ENOENT;
  const uint32_t slot_index = timer_id & kTimerSlotMask, gen = timer_id >> kTimerSlotBits;
  const uint32_t l = slot_index / b->K, k = slot_index % b->K;
  if (l >= b->n_next) return CPBUS_ENOENT;
  int rc = dev_guard(b); if (rc) return rc;
  if ((rc = flush_staged(b, b->now))) return rc;   // firings due before the cancel still happen
  retire_oneshots(b, b->last_watermark);
  HostTimer& t = b->h_timers[(size_t)l * b->K + k];
  if (!t.active || t.gen != gen) return CPBUS_ENOENT;   // already fired / cancelled, or the slot has been re-armed since
  t.active = false; b->n_timers--;
  CK(cudaMemsetAsync(b->d_timers + (size_t)l * b->K + k, 0xFF, sizeof(DevTimer), b->stream));
  CK(cudaStreamSynchronize(b->stream));
  if (b->n_timers == 0) b->min_period = UINT64_MAX;
  return push_mask_words(b, l, 1);
} CPBUS_CATCH

int cpbus_publish(cpbus_t* b, const cpbus_event* ev, size_t n) try {
  if (!b || (!ev && n)) return CPBUS_EINVAL;
  int rc = dev_guard(b); if (rc) return rc;
  for (size_t i = 0; i < n; i++) {   // counter slots of the whole burst: requested up front, touched in the loop below
    if (ev[i].code < CPBUS_N_CODES && ev[i].code != CPBUS_METRIC) b->pub_pairs.prefetch(((uint64_t)ev[i].code << 32) | ev[i].source_id);
  }
  // The debug ring holds 10 entries (events/bus.go:24-31): of a burst only the last 10 published can ever be seen, so only
  // those are enqueued — including when the call stops early (CPBUS_EAGAIN from an automatic flush in lossless mode).
  auto dbg_tail = [&](size_t published) {
    for (size_t j = published > 10 ? published - 10 : 0; j < published; j++) {
      cpbus_event e{};
      e.seq = b->seq - (published - j); e.ts_ns = b->now; e.code = ev[j].code; e.source_id = ev[j].source_id; e.target = CPBUS_TARGET_ALL;
      dbg_enqueue(b, e);
    }
  };
  for (size_t i = 0; i < n; i++) if (ev[i].code >= CPBUS_N_CODES) return CPBUS_EINVAL;   // nothing of an invalid burst is published
  for (size_t i = 0; i < n; i++) {
    const uint32_t code = ev[i].code;
    if ((rc = stage_one(b, code, ev[i].source_id, CPBUS_TARGET_ALL, 0))) { dbg_tail(i); return rc; }
    if (code != CPBUS_METRIC) {                                  // events/bus.go:130-132
      b->st.published_by_code[code]++;
      b->pub_pairs.add(((uint64_t)code << 32) | ev[i].source_id, 1);
    }
    b->st.publishes++;
  }
  dbg_tail(n);                                                   // events/bus.go:139
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_send(cpbus_t* b, uint32_t sub_id, const cpbus_event* ev) try {
  if (!b || !ev || ev->code >= CPBUS_N_CODES) return CPBUS_EINVAL;
  if (b->sharded()) return sh_send(b, sub_id, ev);
  const uint32_t l = sub_id - b->cfg.sub_id_base;
  if (sub_id < b->cfg.sub_id_base || l >= b->n_next) return CPBUS_ENOENT;
  if (!b->h_active[l]) return CPBUS_ECLOSED;   // the mailbox is gone (Go: send on a closed channel panics)
  int rc = dev_guard(b); if (rc) return rc;
  if ((rc = stage_one(b, ev->code, ev->source_id, sub_id, CPBUS_F_UNICAST))) return rc;
  b->st.publishes++;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_advance(cpbus_t* b, uint64_t now_ns) try {
  if (!b) return CPBUS_EINVAL;
  if (now_ns < b->now) return CPBUS_EORDER;
  if (now_ns == b->now) return CPBUS_OK;
  int rc = dev_guard(b); if (rc) return rc;
  // the kernel looks at <= 32/K candidate firings per timer slot per launch: keep every
  // flush window within that many periods of the fastest periodic timer
  const uint64_t win = max_window(b);
  while (win != UINT64_MAX && now_ns - b->last_watermark > win) {
    b->now = b->last_watermark + win;
    if ((rc = flush_staged(b, b->now))) return rc;
  }
  b->now = now_ns;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_flush(cpbus_t* b) try {
  if (!b) return CPBUS_EINVAL;
  int rc = dev_guard(b); if (rc) return rc;
  return flush_staged(b, b->now);
} CPBUS_CATCH

int cpbus_sync(cpbus_t* b) try {
  if (!b) return CPBUS_EINVAL;
  for (cpbus* s : b->shards) { const int rc = cpbus_sync(s); if (rc) return rc; }
  if (b->sharded()) return CPBUS_OK;
  int rc = dev_guard(b); if (rc) return rc;
  CK(cudaStreamSynchronize(b->stream));
  return CPBUS_OK;
} CPBUS_CATCH

static int publish_device_impl(cpbus_t* b, const void* d_events, size_t n, uint64_t watermark_ns, bool staged,
                               const void* d_next, size_t n_next);

// A device batch that one launch cannot take — more than batch_cap records, or a watermark further from the last one than the
// 32/K firings per timer slot a launch examines — is cut into slices that can (round 1 answered CPBUS_EINVAL / CPBUS_EORDER).
// The cut needs the records' timestamps: one strided D2H of 8 bytes per record, on this slow path only.  A slice ends at
// batch_cap records or at the window's edge, whichever comes first, and its watermark is its last record's timestamp (cut by
// size) or the edge (cut by time): ticks due by then are merged exactly where the unsplit launch would have put them, because
// a tick is ordered in front of every event with ts >= its due time and such events are either in this slice behind it or
// in a later one.  The host path does the same at cpbus_advance.  (events/timer.go:40-71 has no such limit: a Go timer
// that fell behind fires late, never "not at all".)
// The cut itself, host-only (exported as cpbus_split_plan so that it can be tested without a GPU): slice k = records
// [end[k-1], end[k]) launched with watermark wm[k].  `now` = the bus clock (= the last launched watermark once staged events
// are flushed), `window` = the widest watermark step one launch may take (UINT64_MAX: no timer armed).
static int split_plan(const uint64_t* ts, size_t n, uint32_t batch_cap, uint64_t now, uint64_t watermark, uint64_t window,
                      std::vector<size_t>& end, std::vector<uint64_t>& wm) {
  for (size_t i = 1; i < n; i++) if (ts[i] < ts[i - 1]) return CPBUS_EORDER;
  if (!batch_cap || !window) return CPBUS_EINVAL;
  if (watermark < now || (n && ts[n - 1] > watermark)) return CPBUS_EORDER;
  size_t i = 0;
  uint64_t lw = now;
  for (;;) {
    const uint64_t edge = (window == UINT64_MAX || watermark - lw <= window) ? watermark : lw + window;
    size_t j = std::upper_bound(ts + i, ts + n, edge) - ts;
    uint64_t w = edge;
    if (j - i > batch_cap) { j = i + batch_cap; w = std::max(ts[j - 1], lw); }   // (records older than the clock ride with it)
    end.push_back(j); wm.push_back(w);
    i = j; lw = w;
    if (j == n && w == watermark) return CPBUS_OK;
  }
}

static int publish_device_split(cpbus_t* b, const cpbus_event* d_events, size_t n, uint64_t watermark_ns, bool staged,
                                const void* d_next, size_t n_next) {
  std::vector<uint64_t> ts, wm;
  std::vector<size_t> end;
  ts.resize(n);
  if (n) {
    CK(cudaMemcpy2DAsync(ts.data(), 8, reinterpret_cast<const unsigned char*>(d_events) + offsetof(cpbus_event, ts_ns), sizeof(cpbus_event),
                         8, n, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
  }
  int rc = split_plan(ts.data(), n, b->B, b->now, watermark_ns, max_window(b), end, wm);   // (a one-shot retiring mid-way can only widen the window)
  if (rc) return rc;
  size_t i = 0;
  for (size_t k = 0; k < end.size(); k++) {
    const bool last = k + 1 == end.size();
    rc = publish_device_impl(b, d_events + i, end[k] - i, wm[k], staged, last ? d_next : nullptr, last ? n_next : 0);
    if (rc) return rc;
    b->st.device_splits++;
    i = end[k];
  }
  return CPBUS_OK;
}

static int publish_device_impl(cpbus_t* b, const void* d_events, size_t n, uint64_t watermark_ns, bool staged,
                               const void* d_next, size_t n_next) {
  if (!b || (!d_events && n) || ((uintptr_t)d_events & 31u) || n_next > b->B || ((uintptr_t)d_next & 31u)) return CPBUS_EINVAL;
  int rc = dev_guard(b); if (rc) return rc;
  if ((rc = flush_staged(b, b->now))) return rc;
  if (watermark_ns < b->now) return CPBUS_EORDER;
  if (staged && b->lossless) return CPBUS_EINVAL;   // admission would have to read the peer batch: not supported
  if (n > b->B || watermark_ns - b->last_watermark > max_window(b)) {
    // lossless mode stays all-or-nothing per call (the caller owns the batch and could not tell how far a refused call got)
    if (b->lossless) return n > b->B ? CPBUS_EINVAL : CPBUS_EORDER;
    return publish_device_split(b, (const cpbus_event*)d_events, n, watermark_ns, staged, d_next, n_next);
  }
  bool ok = true;
  if ((rc = admit(b, (const cpbus_event*)d_events, (uint32_t)n, watermark_ns, &ok))) return rc;
  if (!ok) return CPBUS_EAGAIN;
  b->now = watermark_ns;
  const cpbus_event* src = (const cpbus_event*)d_events;
  bool dep = false;
  // Prefetch cache: a peer batch an earlier launch already pulled into d_prefetch[i].  An entry is good for ONE use, only
  // while it is recent (the caller may re-stamp or reuse the peer buffer later), and the newest match wins.
  for (int i = 0; i < cpbus::kPrefetch; i++)
    if (b->pf_ptr[i] && b->launch_seq - b->pf_seq[i] > (unsigned long long)cpbus::kPrefetch) b->pf_ptr[i] = nullptr;
  if (staged && n) {
    int hit = -1;
    for (int i = 0; i < cpbus::kPrefetch; i++)
      if (b->pf_ptr[i] == d_events && b->pf_n[i] == n && (hit < 0 || b->pf_seq[i] > b->pf_seq[hit])) hit = i;
    if (hit >= 0) {
      src = b->d_prefetch[hit];          // plain local launch
      staged = false;
      dep = b->pf_seq[hit] == b->launch_seq;   // written by the IMMEDIATELY preceding launch: its prologue must not run ahead
      for (int i = 0; i < cpbus::kPrefetch; i++) if (b->pf_ptr[i] == d_events) b->pf_ptr[i] = nullptr;   // consumed (and any older copy dropped)
    }
  }
  const cpbus_event* pf_src = nullptr; cpbus_event* pf_dst = nullptr;
  int slot = -1;
  if (d_next && n_next) {
    slot = b->pf_next;
    if (b->d_prefetch[slot] == src) slot = (slot + 1) % cpbus::kPrefetch;   // never overwrite the buffer this launch reads
    pf_src = (const cpbus_event*)d_next; pf_dst = b->d_prefetch[slot];
    for (int i = 0; i < cpbus::kPrefetch; i++) if (b->pf_ptr[i] == d_next) b->pf_ptr[i] = nullptr;   // superseded
  }
  if ((rc = launch_fanout(b, src, (uint32_t)n, watermark_ns, staged ? 1 : 0, pf_src, pf_dst, (uint32_t)n_next, dep, /*account=*/true))) return rc;
  if (slot >= 0) { b->pf_ptr[slot] = d_next; b->pf_n[slot] = n_next; b->pf_seq[slot] = b->launch_seq; b->pf_next = (slot + 1) % cpbus::kPrefetch; }
  b->st.publishes += n; b->seq += n;
  return CPBUS_OK;
}

int cpbus_publish_device(cpbus_t* b, const void* d_events, size_t n, uint64_t watermark_ns) try {
  if (b && b->sharded()) return sh_publish_device(b, d_events, n, watermark_ns);
  return publish_device_impl(b, d_events, n, watermark_ns, false, nullptr, 0);
} CPBUS_CATCH

// Multi-GPU ingest fused into the fan-out kernel: d_events (and d_next) may point into ANOTHER GPU's HBM (the
// publisher's event stream, peer-mapped over NVLink).  One CTA pulls the batch across the link, stages it in local
// HBM and publishes it with the batch descriptor; if the caller names the NEXT batch, that one is pulled by the
// same launch while its stores are in flight, so the following call starts from local memory.  No collective.
int cpbus_publish_device_staged(cpbus_t* b, const void* d_events, size_t n, uint64_t watermark_ns, const void* d_next, size_t n_next) try {
  if (b && b->sharded()) return CPBUS_EINVAL;   // the handle already feeds its shards; a peer batch is meant for one shard bus
  return publish_device_impl(b, d_events, n, watermark_ns, true, d_next, n_next);
} CPBUS_CATCH

// ---- buffers shared between the GPUs of one box (CUDA IPC; NVLink peer mapping on the importing side) ----
int cpbus_shared_alloc(cpbus_t* b, size_t bytes, void** dptr, unsigned char handle[64]) try {
  if (!b || !dptr || !handle || !bytes || b->sharded()) return CPBUS_EINVAL;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  int rc = dev_guard(b); if (rc) return rc;
  void* p = nullptr;
  if (cudaMalloc(&p, bytes) != cudaSuccess) { snprintf(g_cuda_err, sizeof(g_cuda_err), "cudaMalloc(%zu) failed", bytes); return CPBUS_ENOMEM; }
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); snprintf(g_cuda_err, sizeof(g_cuda_err), "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); return CPBUS_ECUDA; }
  memcpy(handle, &h, 64);
  b->shared_owned.push_back(p);
  *dptr = p;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_shared_open(cpbus_t* b, const unsigned char handle[64], void** dptr) try {
  if (!b || !dptr || !handle || b->sharded()) return CPBUS_EINVAL;
  int rc = dev_guard(b); if (rc) return rc;      // the IMPORTING device must be current: the mapping is made for it
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  void* p = nullptr;
  CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  b->shared_mapped.push_back(p);
  *dptr = p;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_shared_close(cpbus_t* b, void* dptr) try {
  if (!b || !dptr || b->sharded()) return CPBUS_EINVAL;
  int rc = dev_guard(b); if (rc) return rc;
  CK(cudaStreamSynchronize(b->stream));
  for (int i = 0; i < cpbus::kPrefetch; i++) b->pf_ptr[i] = nullptr;   // prefetched copies of anything in that buffer are void
  for (size_t i = 0; i < b->shared_owned.size(); i++)
    if (b->shared_owned[i] == dptr) { cudaFree(dptr); b->shared_owned.erase(b->shared_owned.begin() + i); return CPBUS_OK; }
  for (size_t i = 0; i < b->shared_mapped.size(); i++)
    if (b->shared_mapped[i] == dptr) { cudaIpcCloseMemHandle(dptr); b->shared_mapped.erase(b->shared_mapped.begin() + i); return CPBUS_OK; }
  return CPBUS_ENOENT;
} CPBUS_CATCH

// ---- the publisher's event stream across the GPUs of one box (include/cpbus.h: cpbus_stream_*) ----
struct cpbus_stream {
  cpbus* bus = nullptr;
  bool owner = false, attached = false;      // attached: same-process consumer sharing the owner's pointer (peer access, no IPC)
  uint32_t n_slots = 0, n_consumers = 0, consumer = 0, B = 0;
  unsigned char* base = nullptr;             // the ring: local memory on the publisher, NVLink peer mapping elsewhere
  StreamHdr* hdr = nullptr;
  unsigned long long* ack = nullptr;         // consumer c's word is ack[4 * c] (one sector each)
  cpbus_event* payload = nullptr;
  unsigned long long put_seq = 0, get_seq = 0;   // batches released / fanned out so far (ordinals are 1-based)
  unsigned long long pub_seq = 0;            // publisher: publish ordinal stamped into the next record (CPBUS_PUT_STAMP)
  unsigned long long min_ack = 0;            // publisher: cached min over the consumers' acks
  // publisher staging: pinned payload + header buffers, copies on their own stream
  static constexpr int kStage = 8;
  cpbus_event* h_stage[kStage] = {};
  StreamHdr* h_hdr = nullptr;                // kStage headers
  unsigned long long* h_ack = nullptr;       // kStreamMaxConsumers x 4 words
  cudaEvent_t staged_done[kStage] = {};
  cudaStream_t put_stream = nullptr;
};

static int stream_bind(cpbus_stream* st) {
  st->hdr = reinterpret_cast<StreamHdr*>(st->base + stream_hdr_off());
  st->ack = reinterpret_cast<unsigned long long*>(st->base + stream_ack_off(st->n_slots));
  st->payload = reinterpret_cast<cpbus_event*>(st->base + stream_payload_off(st->n_slots));
  return CPBUS_OK;
}

// (a sharded handle uses the stream in lossless mode too: it runs the admission of every shard itself before each put)
static int stream_create_impl(cpbus* b, uint32_t n_slots, uint32_t n_consumers, cpbus_stream** out, unsigned char handle[64]);

int cpbus_stream_create(cpbus_t* b, uint32_t n_slots, uint32_t n_consumers, cpbus_stream_t** out, unsigned char handle[64]) try {
  if (!b || !out || !handle || n_slots < 4 || n_consumers == 0 || n_consumers > kStreamMaxConsumers) return CPBUS_EINVAL;
  if (b->lossless || b->sharded()) return CPBUS_EINVAL;   // admission would have to see every shard: throughput mode only
  return stream_create_impl(b, n_slots, n_consumers, out, handle);
} CPBUS_CATCH

static int stream_create_impl(cpbus* b, uint32_t n_slots, uint32_t n_consumers, cpbus_stream** out, unsigned char handle[64]) {
  *out = nullptr;
  int rc = dev_guard(b); if (rc) return rc;
  cpbus_stream* st = new (std::nothrow) cpbus_stream();
  if (!st) return CPBUS_ENOMEM;
  st->bus = b; st->owner = true; st->n_slots = n_slots; st->n_consumers = n_consumers; st->consumer = 0; st->B = b->B;
  st->pub_seq = b->seq;
  const size_t bytes = stream_bytes(n_slots, b->B);
  auto fail = [&](int code) { cpbus_stream_close(st); return code; };
  b->streams.push_back(st);
  if (cudaMalloc((void**)&st->base, bytes) != cudaSuccess) { snprintf(g_cuda_err, sizeof(g_cuda_err), "cudaMalloc(%zu) failed", bytes); return fail(CPBUS_ENOMEM); }
  if (cudaMemset(st->base, 0, stream_payload_off(n_slots)) != cudaSuccess) return fail(CPBUS_ECUDA);
  StreamMeta meta{}; meta.magic = kStreamMagic; meta.n_slots = n_slots; meta.batch_cap = b->B; meta.n_consumers = n_consumers;
  if (cudaMemcpy(st->base, &meta, sizeof(meta), cudaMemcpyHostToDevice) != cudaSuccess) return fail(CPBUS_ECUDA);
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, st->base) != cudaSuccess) { snprintf(g_cuda_err, sizeof(g_cuda_err), "cudaIpcGetMemHandle failed"); return fail(CPBUS_ECUDA); }
  memcpy(handle, &h, 64);
  stream_bind(st);
  if (cudaStreamCreateWithFlags(&st->put_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(CPBUS_ECUDA);
  for (int i = 0; i < cpbus_stream::kStage; i++) {
    if (cudaMallocHost((void**)&st->h_stage[i], (size_t)b->B * sizeof(cpbus_event)) != cudaSuccess) return fail(CPBUS_ENOMEM);
    if (cudaEventCreateWithFlags(&st->staged_done[i], cudaEventDisableTiming) != cudaSuccess) return fail(CPBUS_ECUDA);
  }
  if (cudaMallocHost((void**)&st->h_hdr, sizeof(StreamHdr) * cpbus_stream::kStage) != cudaSuccess) return fail(CPBUS_ENOMEM);
  if (cudaMallocHost((void**)&st->h_ack, (size_t)kStreamMaxConsumers * 32) != cudaSuccess) return fail(CPBUS_ENOMEM);
  *out = st;
  return CPBUS_OK;
}

int cpbus_stream_open(cpbus_t* b, const unsigned char handle[64], uint32_t consumer_index, cpbus_stream_t** out) try {
  if (!b || !out || !handle || consumer_index == 0 || consumer_index >= kStreamMaxConsumers) return CPBUS_EINVAL;
  if (b->lossless || b->sharded()) return CPBUS_EINVAL;
  *out = nullptr;
  int rc = dev_guard(b); if (rc) return rc;      // the IMPORTING device must be current: the mapping is made for it
  cpbus_stream* st = new (std::nothrow) cpbus_stream();
  if (!st) return CPBUS_ENOMEM;
  st->bus = b; st->owner = false; st->consumer = consumer_index;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  cudaError_t e = cudaIpcOpenMemHandle((void**)&st->base, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) { snprintf(g_cuda_err, sizeof(g_cuda_err), "cudaIpcOpenMemHandle: %s", cudaGetErrorString(e)); delete st; return CPBUS_ECUDA; }
  StreamMeta meta{};
  e = cudaMemcpy(&meta, st->base, sizeof(meta), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess || meta.magic != kStreamMagic || meta.batch_cap != b->B || consumer_index >= meta.n_consumers) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "stream meta mismatch (magic %x, batch_cap %u vs %u, consumers %u)", meta.magic, meta.batch_cap, b->B, meta.n_consumers);
    cudaIpcCloseMemHandle(st->base); delete st;
    return e != cudaSuccess ? CPBUS_ECUDA : CPBUS_EINVAL;
  }
  st->n_slots = meta.n_slots; st->n_consumers = meta.n_consumers; st->B = meta.batch_cap;
  stream_bind(st);
  b->streams.push_back(st);
  *out = st;
  return CPBUS_OK;
} CPBUS_CATCH

// Same-process consumer (one host process driving several GPUs, as a cgo shim would): no IPC handle — the owner's
// pointer is used directly, with peer access enabled when the consumer's bus lives on another GPU.
static int stream_attach_impl(cpbus* b, cpbus_stream* owner, uint32_t consumer_index, cpbus_stream** out);

int cpbus_stream_attach(cpbus_t* b, cpbus_stream_t* owner, uint32_t consumer_index, cpbus_stream_t** out) try {
  if (!b || !owner || !owner->owner || !out || consumer_index == 0 || consumer_index >= owner->n_consumers) return CPBUS_EINVAL;
  if (b->lossless || b->sharded() || b->B != owner->B) return CPBUS_EINVAL;
  return stream_attach_impl(b, owner, consumer_index, out);
} CPBUS_CATCH

static int stream_attach_impl(cpbus* b, cpbus_stream* owner, uint32_t consumer_index, cpbus_stream** out) {
  *out = nullptr;
  int rc = dev_guard(b); if (rc) return rc;
  if (b->device != owner->bus->device) {
    int can = 0;
    CK(cudaDeviceCanAccessPeer(&can, b->device, owner->bus->device));
    if (!can) { snprintf(g_cuda_err, sizeof(g_cuda_err), "device %d cannot access device %d", b->device, owner->bus->device); return CPBUS_ECUDA; }
    const cudaError_t e = cudaDeviceEnablePeerAccess(owner->bus->device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { CK(e); }
    cudaGetLastError();   // clear "already enabled"
  }
  cpbus_stream* st = new (std::nothrow) cpbus_stream();
  if (!st) return CPBUS_ENOMEM;
  st->bus = b; st->attached = true; st->consumer = consumer_index;
  st->n_slots = owner->n_slots; st->n_consumers = owner->n_consumers; st->B = owner->B; st->base = owner->base;
  stream_bind(st);
  b->streams.push_back(st);
  *out = st;
  return CPBUS_OK;
}

int cpbus_stream_close(cpbus_stream_t* st) try {
  if (!st) return CPBUS_EINVAL;
  cpbus* b = st->bus;
  cudaSetDevice(b->device);
  cudaStreamSynchronize(b->stream);
  if (st->put_stream) { cudaStreamSynchronize(st->put_stream); cudaStreamDestroy(st->put_stream); }
  for (int i = 0; i < cpbus_stream::kStage; i++) {
    if (st->h_stage[i]) cudaFreeHost(st->h_stage[i]);
    if (st->staged_done[i]) cudaEventDestroy(st->staged_done[i]);
  }
  if (st->h_hdr) cudaFreeHost(st->h_hdr);
  if (st->h_ack) cudaFreeHost(st->h_ack);
  if (st->base) { if (st->owner) cudaFree(st->base); else if (!st->attached) cudaIpcCloseMemHandle(st->base); }
  b->streams.erase(std::remove(b->streams.begin(), b->streams.end(), st), b->streams.end());
  delete st;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_stream_set_timeout(cpbus_stream_t* st, uint32_t microseconds) try {
  if (!st) return CPBUS_EINVAL;
  st->bus->stream_spin_us = microseconds;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_stream_status(cpbus_stream_t* st) try {
  if (!st) return CPBUS_EINVAL;
  return (*(volatile unsigned int*)st->bus->h_err) ? CPBUS_ETIMEDOUT : CPBUS_OK;
} CPBUS_CATCH

// Publisher: copy the batch into the next slot, then release it (header after payload, same stream).
int cpbus_stream_put(cpbus_stream_t* st, const cpbus_event* ev, size_t n, uint64_t now_ns, uint32_t flags) try {
  if (!st || !st->owner || (!ev && n) || n > st->B) return CPBUS_EINVAL;
  cpbus* b = st->bus;
  int rc = dev_guard(b); if (rc) return rc;
  const unsigned long long q = st->put_seq + 1;
  if (q > st->n_slots && st->min_ack + st->n_slots < q) {
    // The slot still holds batch q - n_slots: every consumer must have pulled it.  Acks are device words written by the
    // consumers' kernels; refresh the cached minimum, and — unless the caller asked not to wait — give consumers that
    // are merely behind (their launches are queued, the GPUs are busy) up to the stream timeout to get there.
    const auto t0 = std::chrono::steady_clock::now();
    const auto budget = std::chrono::microseconds(b->stream_spin_us ? b->stream_spin_us : 2000000u);
    for (;;) {
      CK(cudaMemcpyAsync(st->h_ack, st->ack, (size_t)st->n_consumers * 32, cudaMemcpyDeviceToHost, st->put_stream));
      CK(cudaStreamSynchronize(st->put_stream));
      unsigned long long m = ~0ull;
      for (uint32_t c = 0; c < st->n_consumers; c++) m = std::min(m, st->h_ack[4 * c]);
      st->min_ack = m;
      if (st->min_ack + st->n_slots >= q) break;
      if ((flags & CPBUS_PUT_NOWAIT) || std::chrono::steady_clock::now() - t0 > budget || *(volatile unsigned int*)b->h_err) return CPBUS_EAGAIN;
      std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
  }
  const int s = (int)(q % cpbus_stream::kStage);
  CK(cudaEventSynchronize(st->staged_done[s]));   // the pinned buffers of batch q - kStage have left the host
  cpbus_event* dst = st->h_stage[s];
  if (flags & CPBUS_PUT_RAW) { if (n) memcpy(dst, ev, n * sizeof(cpbus_event)); }
  else {
    for (size_t i = 0; i < n; i++) {
      const uint32_t code = ev[i].code;
      if (code >= CPBUS_N_CODES) return CPBUS_EINVAL;
      dst[i].seq = st->pub_seq + i; dst[i].ts_ns = now_ns; dst[i].code = code; dst[i].source_id = ev[i].source_id;
      dst[i].target = CPBUS_TARGET_ALL; dst[i].flags = 0;
    }
  }
  const uint32_t slot = (uint32_t)(q % st->n_slots);
  if (n) CK(cudaMemcpyAsync(st->payload + (size_t)slot * st->B, dst, n * sizeof(cpbus_event), cudaMemcpyHostToDevice, st->put_stream));
  StreamHdr* hh = &st->h_hdr[s];
  memset(hh, 0, sizeof(*hh));
  hh->seq = q; hh->watermark = now_ns; hh->n = (uint32_t)n;
  if (!(flags & CPBUS_PUT_RAW)) st->pub_seq += n;
  CK(cudaMemcpyAsync(&st->hdr[slot], hh, sizeof(StreamHdr), cudaMemcpyHostToDevice, st->put_stream));   // the release: after the payload
  CK(cudaEventRecord(st->staged_done[s], st->put_stream));
  st->put_seq = q;
  return CPBUS_OK;
} CPBUS_CATCH

// Consumers that are NOT told n / now_ns by their driver: look at the next slot's header (one 32-byte copy across the link).
// *ready = 0: the publisher has not released that batch yet.
int cpbus_stream_poll(cpbus_stream_t* st, int* ready, size_t* n, uint64_t* now_ns) try {
  if (!st || !ready) return CPBUS_EINVAL;
  cpbus* b = st->bus;
  int rc = dev_guard(b); if (rc) return rc;
  if (*(volatile unsigned int*)b->h_err) return CPBUS_ETIMEDOUT;
  const unsigned long long q = st->get_seq + 1;
  StreamHdr h{};
  CK(cudaMemcpyAsync(&h, &st->hdr[q % st->n_slots], sizeof(h), cudaMemcpyDeviceToHost, b->result_stream));
  CK(cudaStreamSynchronize(b->result_stream));
  *ready = h.seq == q ? 1 : 0;
  if (*ready) { if (n) *n = h.n; if (now_ns) *now_ns = h.watermark; }
  return CPBUS_OK;
} CPBUS_CATCH

// One fan-out launch for the next batch of the stream (checks done by the caller).  account = false: the batch's events
// were already counted where they were published (a sharded handle's cpbus_publish).
static int stream_launch(cpbus_stream* st, size_t n, uint64_t w, bool account) {
  cpbus* b = st->bus;
  const unsigned long long q = st->get_seq + 1;
  StreamArgs sa;
  const uint32_t slot = (uint32_t)(q % st->n_slots), slot2 = (uint32_t)((q + 2) % st->n_slots);
  sa.hdr = &st->hdr[slot]; sa.ack = &st->ack[4 * st->consumer]; sa.seq = q; sa.next_hdr = &st->hdr[slot2];
  const int rc = launch_fanout(b, st->payload + (size_t)slot * st->B, (uint32_t)n, w, /*staged=*/2,
                               st->payload + (size_t)slot2 * st->B, b->d_pf_buf + (size_t)((q + 2) % kStreamPrefetch) * b->B, 0,
                               /*batch_dep=*/false, account, &sa);
  if (rc) return rc;
  st->get_seq = q;
  return CPBUS_OK;
}

// Every rank (the publisher's included): fan out the next batch of the stream to this GPU's shard.
int cpbus_stream_fanout(cpbus_stream_t* st, size_t n, uint64_t now_ns) try {
  if (!st || n > st->B) return CPBUS_EINVAL;
  cpbus* b = st->bus;
  int rc = dev_guard(b); if (rc) return rc;
  if (*(volatile unsigned int*)b->h_err) return CPBUS_ETIMEDOUT;
  if ((rc = flush_staged(b, b->now))) return rc;
  if (now_ns < b->now) return CPBUS_EORDER;
  if (now_ns - b->last_watermark > max_window(b)) return CPBUS_EORDER;
  b->now = now_ns;
  if ((rc = stream_launch(st, n, now_ns, /*account=*/true))) return rc;
  b->st.publishes += n; b->seq += n;
  return CPBUS_OK;
} CPBUS_CATCH

static int read_cursors(cpbus* b, uint32_t l, uint64_t* tail, uint64_t* head, uint64_t* lost = nullptr) {
  SubCtl c{};
  CK(cudaMemcpyAsync(&c, b->d_ctl + l, sizeof(SubCtl), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  *tail = c.tail;
  // overwrite-oldest: the consumer's cursor can never be older than the oldest record still in the ring
  *head = (!b->lossless && c.tail > b->R && c.tail - b->R > c.head) ? c.tail - b->R : c.head;
  if (lost) *lost = *head - c.head;   // records overwritten since the consumer's stored cursor
  return CPBUS_OK;
}

static int copy_slots(cpbus* b, uint32_t l, uint64_t from, size_t n, cpbus_event* out) {
  const cpbus_event* ring = b->d_ring + (size_t)l * b->R;
  const uint32_t s0 = (uint32_t)(from & (b->R - 1));
  const size_t first = std::min<size_t>(n, b->R - s0);
  if (first) CK(cudaMemcpyAsync(out, ring + s0, first * sizeof(cpbus_event), cudaMemcpyDeviceToHost, b->stream));
  if (n > first) CK(cudaMemcpyAsync(out + first, ring, (n - first) * sizeof(cpbus_event), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return CPBUS_OK;
}

int cpbus_drain(cpbus_t* b, uint32_t sub_id, cpbus_event* out, size_t cap, size_t* n, uint64_t* lost) try {
  if (!b || !n || (!out && cap)) return CPBUS_EINVAL;
  if (b->sharded()) { cpbus* s = sh_owner(b, sub_id); return s ? cpbus_drain(s, sub_id, out, cap, n, lost) : CPBUS_ENOENT; }
  const uint32_t l = sub_id - b->cfg.sub_id_base;
  if (sub_id < b->cfg.sub_id_base || l >= b->n_next) return CPBUS_ENOENT;
  std::lock_guard<std::mutex> g(b->mu);
  int rc = dev_guard(b); if (rc) return rc;
  uint64_t tail = 0, head = 0;
  uint64_t gone = 0;
  if ((rc = read_cursors(b, l, &tail, &head, &gone))) return rc;
  if (lost) *lost = gone;
  const size_t take = (size_t)std::min<uint64_t>(tail - head, cap);
  if (take && (rc = copy_slots(b, l, head, take, out))) return rc;
  head += take;
  CK(cudaMemcpyAsync(&b->d_ctl[l].head, &head, 8, cudaMemcpyHostToDevice, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  *n = take;
  return CPBUS_OK;
} CPBUS_CATCH

// Bulk drain: everything undrained in mailboxes [first_sub, first_sub+n) in ONE kernel + two D2H copies.
// out receives the records (each mailbox's run contiguous and FIFO), offsets[i]/counts[i] say where mailbox i's run is.
int cpbus_drain_many(cpbus_t* b, uint32_t first_sub, uint32_t n, cpbus_event* out, size_t cap, uint32_t* offsets,
                     uint32_t* counts, size_t* total) try {
  if (!b || !n || !out || !cap || !offsets || !counts || !total || cap > 0xFFFFFFFFull) return CPBUS_EINVAL;
  if (b->sharded()) return sh_drain_many(b, first_sub, n, out, cap, offsets, counts, total);
  const uint32_t l = first_sub - b->cfg.sub_id_base;
  if (first_sub < b->cfg.sub_id_base || (uint64_t)l + n > b->n_next) return CPBUS_ENOENT;
  std::lock_guard<std::mutex> g(b->mu);
  int rc = dev_guard(b); if (rc) return rc;
  if (b->drain_cap < cap || b->drain_idx_cap < n) {   // device staging grows on demand and is kept
    if (b->drain_cap < cap) { cudaFree(b->d_drain); b->d_drain = nullptr; CK(cudaMalloc((void**)&b->d_drain, cap * sizeof(cpbus_event))); b->drain_cap = cap; }
    if (b->drain_idx_cap < n) { cudaFree(b->d_drain_idx); b->d_drain_idx = nullptr; CK(cudaMalloc((void**)&b->d_drain_idx, (size_t)n * sizeof(uint2) + 16)); b->drain_idx_cap = n; }
  }
  unsigned int* cursor = reinterpret_cast<unsigned int*>(b->d_drain_idx + n);
  CK(cudaMemsetAsync(cursor, 0, sizeof(unsigned int), b->stream));
  const uint32_t threads = 256, grid = std::min<uint32_t>((n + 7) / 8, (uint32_t)b->sm_count * 8);
  drain_many_kernel<<<grid, threads, 0, b->stream>>>(b->d_ctl, b->d_ring, l, n, b->R, b->lossless ? 1u : 0u, b->d_drain,
                                                     (uint32_t)cap, b->d_drain_idx, cursor);
  CK(cudaGetLastError());
  b->st.kernel_launches++;
  std::vector<uint2> idx(n);
  CK(cudaMemcpyAsync(idx.data(), b->d_drain_idx, (size_t)n * sizeof(uint2), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  size_t tot = 0, hi = 0;
  for (uint32_t i = 0; i < n; i++) {
    offsets[i] = idx[i].x; counts[i] = idx[i].y; tot += idx[i].y;
    hi = std::max<size_t>(hi, (size_t)idx[i].x + idx[i].y);
  }
  if (hi) CK(cudaMemcpyAsync(out, b->d_drain, hi * sizeof(cpbus_event), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  *total = tot;
  return CPBUS_OK;
} CPBUS_CATCH

// Device-side consumer: every mailbox of this shard is read to the end and its records are discarded.
int cpbus_consume_all(cpbus_t* b) try {
  if (!b) return CPBUS_EINVAL;
  if (b->sharded()) {
    for (cpbus* s : b->shards) { const int rc = cpbus_consume_all(s); if (rc) return rc; }
    b->room_lb = b->R;
    return CPBUS_OK;
  }
  std::lock_guard<std::mutex> g(b->mu);
  int rc = dev_guard(b); if (rc) return rc;
  if (b->n_next) {
    const uint32_t threads = 256, grid = std::min<uint32_t>((b->n_next + threads - 1) / threads, (uint32_t)b->sm_count * 8);
    consume_all_kernel<<<grid, threads, 0, b->stream>>>(b->d_ctl, b->n_next);
    CK(cudaGetLastError());
    b->st.kernel_launches++;
  }
  b->room_lb = b->R;   // stream-ordered behind every earlier fan-out: from here on every mailbox is empty
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_peek_window(cpbus_t* b, uint32_t sub_id, cpbus_event* out, size_t cap, size_t* n) try {
  if (!b || !n || (!out && cap)) return CPBUS_EINVAL;
  if (b->sharded()) { cpbus* s = sh_owner(b, sub_id); return s ? cpbus_peek_window(s, sub_id, out, cap, n) : CPBUS_ENOENT; }
  const uint32_t l = sub_id - b->cfg.sub_id_base;
  if (sub_id < b->cfg.sub_id_base || l >= b->n_next) return CPBUS_ENOENT;
  std::lock_guard<std::mutex> g(b->mu);
  int rc = dev_guard(b); if (rc) return rc;
  uint64_t tail = 0, head = 0;
  if ((rc = read_cursors(b, l, &tail, &head))) return rc;
  const size_t take = (size_t)std::min<uint64_t>(std::min<uint64_t>(tail, b->R), cap);
  if (take && (rc = copy_slots(b, l, tail - take, take, out))) return rc;
  *n = take;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_digest(cpbus_t* b, uint32_t first_sub, uint32_t n, cpbus_digest_t* out) try {
  if (!b || !out || !n) return CPBUS_EINVAL;
  if (b->sharded()) return sh_digest(b, first_sub, n, out);
  const uint32_t l = first_sub - b->cfg.sub_id_base;
  if (first_sub < b->cfg.sub_id_base || (uint64_t)l + n > b->n_next) return CPBUS_ENOENT;
  std::lock_guard<std::mutex> g(b->mu);
  int rc = dev_guard(b); if (rc) return rc;
  std::vector<SubCtl> c(n);
  CK(cudaMemcpyAsync(c.data(), b->d_ctl + l, (size_t)n * sizeof(SubCtl), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  for (uint32_t i = 0; i < n; i++) { out[i].count = c[i].tail; out[i].digest = c[i].digest; }
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_digest_fold_begin(cpbus_t* b, uint32_t first_sub, uint32_t n, uint32_t* ticket) try {
  if (!b || !ticket || !n) return CPBUS_EINVAL;
  if (b->sharded()) return sh_digest_fold_begin(b, first_sub, n, ticket);
  const uint32_t l = first_sub - b->cfg.sub_id_base;
  if (first_sub < b->cfg.sub_id_base || (uint64_t)l + n > b->n_next) return CPBUS_ENOENT;
  std::lock_guard<std::mutex> g(b->mu);
  int rc = dev_guard(b); if (rc) return rc;
  const uint32_t slot = b->fold_next++ % cpbus::kFoldSlots;
  unsigned long long* d = b->d_fold + 4 * slot;
  CK(cudaMemsetAsync(d, 0, 32, b->stream));
  const uint32_t threads = 256, grid = std::min<uint32_t>((n + threads - 1) / threads, (uint32_t)b->sm_count * 4);
  digest_fold_kernel<<<grid, threads, 0, b->stream>>>(b->d_ctl, l, n, b->cfg.sub_id_base, d);
  CK(cudaGetLastError());
  b->st.kernel_launches++;
  CK(cudaMemcpyAsync(b->h_fold + 4 * slot, d, 32, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaEventRecord(b->fold_done[slot], b->stream));
  *ticket = slot;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_digest_fold_end(cpbus_t* b, uint32_t ticket, uint64_t out[4]) try {
  if (!b || !out || ticket >= (uint32_t)cpbus::kFoldSlots) return CPBUS_EINVAL;
  if (b->sharded()) return sh_digest_fold_end(b, ticket, out);
  int rc = dev_guard(b); if (rc) return rc;
  CK(cudaEventSynchronize(b->fold_done[ticket]));
  for (int i = 0; i < 4; i++) out[i] = b->h_fold[4 * ticket + i];
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_digest_fold(cpbus_t* b, uint32_t first_sub, uint32_t n, uint64_t out[4]) try {
  uint32_t ticket = 0;
  int rc = cpbus_digest_fold_begin(b, first_sub, n, &ticket);
  return rc ? rc : cpbus_digest_fold_end(b, ticket, out);
} CPBUS_CATCH

// The fan-out kernel leaves {deliveries, ticks, sum of the new digests} of each launch in a small ring;
// reading a step's result therefore costs one 256-byte D2H and no extra kernel.
int cpbus_step_result_begin(cpbus_t* b, uint32_t* ticket) try {
  if (!b || !ticket) return CPBUS_EINVAL;
  if (b->sharded()) return sh_step_result_begin(b, ticket);
  std::lock_guard<std::mutex> g(b->mu);
  int rc = dev_guard(b); if (rc) return rc;
  const uint32_t t = b->result_next++ % 8;
  const DevResultSlot* src = b->d_result + (size_t)(b->launch_seq % kResultRing) * kResultSub;
  // read it on a side stream, behind an event recorded after the launch: neither the next fan-out nor the next batch's
  // H2D queues behind this D2H
  CK(cudaEventRecord(b->launched, b->stream));
  CK(cudaStreamWaitEvent(b->result_stream, b->launched, 0));
  CK(cudaMemcpyAsync(b->h_result + (size_t)t * kResultSub, src, sizeof(DevResultSlot) * kResultSub, cudaMemcpyDeviceToHost, b->result_stream));
  CK(cudaEventRecord(b->result_done[t], b->result_stream));
  *ticket = t;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_step_result_end(cpbus_t* b, uint32_t ticket, uint64_t out[4]) try {
  if (!b || !out || ticket >= 8) return CPBUS_EINVAL;
  if (b->sharded()) return sh_step_result_end(b, ticket, out);
  int rc = dev_guard(b); if (rc) return rc;
  CK(cudaEventSynchronize(b->result_done[ticket]));
  out[0] = out[1] = out[2] = out[3] = 0;
  for (int i = 0; i < kResultSub; i++) {
    const DevResultSlot& r = b->h_result[(size_t)ticket * kResultSub + i];
    out[0] += r.deliveries; out[1] += r.ticks; out[2] += r.digest_sum; out[3] += r.launch_seq;
  }
  return CPBUS_OK;
} CPBUS_CATCH

// DebugEvents — events/bus.go:34-54
// Broadcast events of device-published batches join the debug ring here, in publish order (the kernel's lead CTA kept
// the last 10 of each such batch; launches older than kAcctDbgRing are no longer resolvable and are skipped).
static int dbg_resolve(cpbus* b) {
  if (b->dbg_pending.empty()) return CPBUS_OK;
  bool any_marker = false;
  for (const DbgItem& it : b->dbg_pending) any_marker |= it.marker;
  cpbus* a = b->sharded() ? b->shards[0] : b;   // the bus whose kernel accounted the device batches
  if (any_marker) {
    int rc = dev_guard(a); if (rc) return rc;
    CK(cudaMemcpyAsync(a->h_acct->tail, a->d_acct->tail, sizeof(a->h_acct->tail), cudaMemcpyDeviceToHost, a->stream));
    CK(cudaStreamSynchronize(a->stream));
  }
  for (const DbgItem& it : b->dbg_pending) {
    if (!it.marker) { dbg_ring_put(b, it.ev); continue; }
    const DevDbgTail& t = a->h_acct->tail[it.launch % kAcctDbgRing];
    if (t.launch_seq != it.launch) continue;
    for (uint32_t j = 0; j < t.n_kept && j < (uint32_t)kAcctDbgKeep; j++) dbg_ring_put(b, t.ev[j]);
  }
  b->dbg_pending.clear();
  return CPBUS_OK;
}

int cpbus_debug_events(cpbus_t* b, cpbus_event* out, size_t cap, size_t* n) try {
  if (!b || !n || (!out && cap)) return CPBUS_EINVAL;
  { const int rc = dbg_resolve(b); if (rc) return rc; }
  size_t k = 0;
  for (;;) {
    if (b->dbg_head == -1) break;
    const cpbus_event e = b->dbg[b->dbg_tail % 10];
    if (b->dbg_tail == b->dbg_head) { b->dbg_head = -1; b->dbg_tail = 0; }
    else b->dbg_tail = (b->dbg_tail + 1) % 10;
    if (e.code == CPBUS_NONE && e.source_id == 0) break;   // == NonEvent
    if (k < cap) out[k] = e;
    k++;
  }
  *n = k;
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_stats(cpbus_t* b, cpbus_stats_t* out) try {
  if (!b || !out) return CPBUS_EINVAL;
  if (b->sharded()) return sh_stats(b, out);
  std::lock_guard<std::mutex> g(b->mu);
  int rc = dev_guard(b); if (rc) return rc;
  CK(cudaMemsetAsync(&b->d_stats->overwritten, 0, sizeof(unsigned long long), b->stream));
  if (!b->lossless && b->n_next) {
    const uint32_t threads = 256, grid = std::min<uint32_t>((b->n_next + threads - 1) / threads, (uint32_t)b->sm_count * 4);
    overwritten_kernel<<<grid, threads, 0, b->stream>>>(b->d_ctl, b->n_next, b->R, &b->d_stats->overwritten);
    CK(cudaGetLastError());
  }
  CK(cudaMemcpyAsync(b->h_stats, b->d_stats, sizeof(DevStats), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaMemcpyAsync(b->h_acct->by_code, b->d_acct->by_code, sizeof(b->h_acct->by_code), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  retire_oneshots(b, b->last_watermark);
  b->st.deliveries = b->st.ticks = 0;
  b->st.overwritten = b->h_stats->overwritten;
  for (int i = 0; i < kStatSlots; i++) { b->st.deliveries += b->h_stats->slot[i].deliveries; b->st.ticks += b->h_stats->slot[i].ticks; }
  b->st.n_subs = b->n_active; b->st.n_timers = b->n_timers; b->st.now_ns = b->now;
  b->st.intern_entries = b->sources.size(); b->st.intern_bytes = b->intern_bytes;
  b->st.ephemeral_live = b->eph_live; b->st.ephemeral_recycled = b->eph_recycled;
  *out = b->st;
  for (int c = 0; c < CPBUS_N_CODES; c++) out->published_by_code[c] += b->h_acct->by_code[c];   // device-published batches (kernel-counted)
  return CPBUS_OK;
} CPBUS_CATCH

// containerpilot_events{code, source} (events/bus.go:60-68,130-132): host publishes are counted in cpbus_publish, batches
// that arrive in device memory by the fan-out kernel's lead CTA (DevPubAcct).
int cpbus_publish_counts(cpbus_t* b, cpbus_pair_count* out, size_t cap, size_t* n) try {
  if (!b || !n || (!out && cap)) return CPBUS_EINVAL;
  std::lock_guard<std::mutex> g(b->mu);
  cpbus* a = b->sharded() ? b->shards[0] : b;   // the bus whose kernel accounted the device batches
  int rc = dev_guard(a); if (rc) return rc;
  std::unordered_map<uint64_t, uint64_t> merged;
  for (size_t i = 0; i < b->pub_pairs.keys.size(); i++) if (b->pub_pairs.keys[i]) merged[b->pub_pairs.keys[i] - 1] += b->pub_pairs.cnts[i];
  if (a->launch_seq) {
    std::vector<unsigned long long> keys(kAcctPairSlots), cnts(kAcctPairSlots);
    CK(cudaMemcpyAsync(keys.data(), a->d_acct->pair_key, sizeof(unsigned long long) * kAcctPairSlots, cudaMemcpyDeviceToHost, a->stream));
    CK(cudaMemcpyAsync(cnts.data(), a->d_acct->pair_cnt, sizeof(unsigned long long) * kAcctPairSlots, cudaMemcpyDeviceToHost, a->stream));
    CK(cudaStreamSynchronize(a->stream));
    for (uint32_t i = 0; i < kAcctPairSlots; i++) if (keys[i]) merged[keys[i] - 1] += cnts[i];
  }
  std::vector<std::pair<uint64_t, uint64_t>> v(merged.begin(), merged.end());
  std::sort(v.begin(), v.end());
  for (size_t i = 0; i < v.size() && i < cap; i++) out[i] = cpbus_pair_count{(uint32_t)(v[i].first >> 32), (uint32_t)v[i].first, v[i].second};
  *n = v.size();
  return CPBUS_OK;
} CPBUS_CATCH

int cpbus_device_ptrs(cpbus_t* b, void** ring, void** ctl) try {
  if (!b || b->sharded()) return CPBUS_EINVAL;   // the layout is per shard
  if (ring) *ring = b->d_ring;
  if (ctl) *ctl = b->d_ctl;
  return CPBUS_OK;
} CPBUS_CATCH


// ---- one handle over several GPUs (include/cpbus.h: cpbus_create_sharded) ----
int cpbus_shard_range(uint32_t n_max_subs, uint32_t n_shards, uint32_t shard, uint32_t* first, uint32_t* count) {
  if (!n_shards || shard >= n_shards || !first || !count) return CPBUS_EINVAL;
  const uint32_t base = n_max_subs / n_shards, extra = n_max_subs % n_shards;
  *first = shard * base + std::min(shard, extra);
  *count = base + (shard < extra ? 1u : 0u);
  return CPBUS_OK;
}

int cpbus_create_sharded(const cpbus_config* cfg, const int32_t* devices, uint32_t n_shards, cpbus_t** out) try {
  if (!cfg || !out) return CPBUS_EINVAL;
  *out = nullptr;
  if (!devices || !n_shards || n_shards > kStreamMaxConsumers || cfg->stream || !config_ok(cfg) || cfg->n_max_subs < n_shards)
    return CPBUS_EINVAL;
  cpbus_config c = *cfg;
  if (n_shards == 1) { c.device = devices[0]; return cpbus_create(&c, out); }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "no CUDA device visible");
    return CPBUS_ENODEV;
  }
  for (uint32_t k = 0; k < n_shards; k++) if (devices[k] < 0 || devices[k] >= ndev) return CPBUS_EINVAL;
  cpbus* h = new (std::nothrow) cpbus();
  if (!h) return CPBUS_ENOMEM;
  auto fail = [&](int code) { cpbus_destroy(h); return code; };
  h->R = cfg->ring_cap ? cfg->ring_cap : 1024;
  h->B = cfg->batch_cap ? cfg->batch_cap : std::min(256u, h->R / 2);
  h->cfg = *cfg; h->cfg.ring_cap = h->R; h->cfg.batch_cap = h->B; h->cfg.device = devices[0];
  h->N = cfg->n_max_subs; h->K = cfg->timers_per_sub; h->device = devices[0];
  h->lossless = cfg->flags & CPBUS_CFG_LOSSLESS; h->use_digest = cfg->flags & CPBUS_CFG_DIGEST;
  h->room_lb = h->R;
  for (uint32_t k = 0; k < n_shards; k++) {
    uint32_t first = 0, count = 0;
    cpbus_shard_range(cfg->n_max_subs, n_shards, k, &first, &count);
    c = *cfg; c.n_max_subs = count; c.sub_id_base = cfg->sub_id_base + first; c.device = devices[k];
    cpbus* s = nullptr;
    const int rc = cpbus_create(&c, &s);
    if (rc) return fail(rc);
    h->shards.push_back(s); h->shard_first.push_back(first);
  }
  // the handle's stream: shard 0 owns it, the others attach in-process (peer access when they live on another GPU).  16 slots
  // let the host run that many flushes ahead of the slowest shard before cpbus_stream_put waits for it.
  unsigned char ipc[64];
  cpbus_stream* st0 = nullptr;
  int rc = stream_create_impl(h->shards[0], 16, n_shards, &st0, ipc);
  if (rc) return fail(rc);
  h->shard_st.push_back(st0);
  for (uint32_t k = 1; k < n_shards; k++) {
    cpbus_stream* st = nullptr;
    if ((rc = stream_attach_impl(h->shards[k], st0, k, &st))) return fail(rc);
    h->shard_st.push_back(st);
  }
  // staging: pinned, portable and mapped, so that the admission kernel of every shard can read it in place
  if ((rc = dev_guard(h))) return fail(rc);
  if (cudaHostAlloc((void**)&h->h_batch[0], (size_t)h->B * sizeof(cpbus_event), cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess)
    return fail(CPBUS_ENOMEM);
  if (cudaHostGetDevicePointer((void**)&h->d_batch_host, h->h_batch[0], 0) != cudaSuccess) return fail(CPBUS_ECUDA);
  h->intern.emplace(std::string(), 0u);
  h->sources.emplace_back();
  *out = h;
  return CPBUS_OK;
} CPBUS_CATCH

}  // extern "C"

namespace {

uint32_t sh_index(const cpbus* h, uint32_t l) {   // shard holding local id l < N
  return (uint32_t)(std::upper_bound(h->shard_first.begin(), h->shard_first.end(), l) - h->shard_first.begin()) - 1u;
}
uint32_t sh_end(const cpbus* h, uint32_t k) { return k + 1 < h->shards.size() ? h->shard_first[k + 1] : h->N; }

cpbus* sh_owner(const cpbus* h, uint32_t sub_id) {
  const uint32_t l = sub_id - h->cfg.sub_id_base;
  if (sub_id < h->cfg.sub_id_base || l >= h->n_next) return nullptr;
  return h->shards[sh_index(h, l)];
}

// f(shard index, first local id, count) for each shard's piece of local ids [l, l + n), in id order; stops at an error
template <class F>
int sh_pieces(const cpbus* h, uint32_t l, uint32_t n, F f) {
  const uint64_t hi = (uint64_t)l + n;
  for (uint32_t lo = l; lo < hi;) {
    const uint32_t k = sh_index(h, lo), e = (uint32_t)std::min<uint64_t>(hi, sh_end(h, k));
    const int rc = f(k, lo, e - lo);
    if (rc) return rc;
    lo = e;
  }
  return CPBUS_OK;
}

bool sh_in_range(const cpbus* h, uint32_t first_sub, uint32_t n) {
  return first_sub >= h->cfg.sub_id_base && (uint64_t)(first_sub - h->cfg.sub_id_base) + n <= h->n_next;
}

// The shards follow the handle's clock: a shard's timers are armed relative to its `now`, and its own flush (which every
// membership / timer call runs first) then finds nothing to do.
void sh_sync_clocks(cpbus* h) {
  for (cpbus* s : h->shards) { s->now = h->now; s->last_watermark = h->last_watermark; }
}

void sh_retire_oneshots(cpbus* h) {   // where one bus would retire its fired one-shots: on every shard at once
  for (cpbus* s : h->shards) retire_oneshots(s, s->last_watermark);
  if (timers_armed(h) == 0) h->min_period = UINT64_MAX;
}

// Lossless admission over every shard: the handle keeps one room bound like a single bus; when it is used up, the admission
// kernel runs on every shard (each reads the pinned staging buffer in place) and the results merge as if one kernel had seen
// every mailbox: any overflow refuses, the shortest prefix wins, the fullest mailbox sets the new bound.
int sh_admit(cpbus* h, uint32_t n, uint64_t w, bool* ok, uint32_t* prefix) {
  *ok = true; *prefix = n;
  if (h->n_next == 0) return CPBUS_OK;
  const uint64_t need = admit_need(n, h->K, timers_armed(h) > 0, h->min_period, h->last_watermark, w);
  if (h->room_lb >= need) { h->room_lb -= need; h->st.admit_skipped++; return CPBUS_OK; }
  int rc;
  for (cpbus* s : h->shards)
    if (s->n_next && ((rc = dev_guard(s)) || (rc = admit_launch(s, h->d_batch_host, n, w)))) return rc;
  unsigned long long overflow = 0, deficit = 0, used = 0;
  for (cpbus* s : h->shards) {
    if (!s->n_next) continue;
    if ((rc = dev_guard(s))) return rc;
    CK(cudaStreamSynchronize(s->stream));
    overflow += s->h_stats->admit_overflow;
    deficit = std::max(deficit, s->h_stats->admit_deficit);
    used = std::max(used, s->h_stats->admit_max_used);
  }
  h->st.admit_passes++;
  *ok = overflow == 0;
  if (!*ok) *prefix = n - (uint32_t)std::min<unsigned long long>(n, deficit);
  h->room_lb = used >= h->R ? 0 : h->R - used;
  return CPBUS_OK;
}

// One flush of a handle = one put of the staged records into the stream + one stream fan-out per shard (flush_staged's rules).
int flush_sharded(cpbus* h, uint64_t w) {
  const uint32_t n = (uint32_t)h->n_staged;
  const uint32_t timers = timers_armed(h);
  if ((n == 0 && timers == 0) || (n == 0 && w == h->last_watermark)) {
    if (n == 0 && timers == 0) h->last_watermark = std::max(h->last_watermark, w);
    sh_sync_clocks(h);
    return CPBUS_OK;
  }
  if (h->n_next == 0) {   // no mailbox yet: one bus launches nothing and drops the batch, so does the handle
    h->n_staged = 0;
    sh_sync_clocks(h);
    return CPBUS_OK;
  }
  bool ok = true;
  uint32_t m = n;
  int rc;
  if (h->lossless && (rc = sh_admit(h, n, w, &ok, &m))) return rc;
  if (!ok) {
    if (m == 0) return CPBUS_EAGAIN;
    w = h->h_batch[0][m - 1].ts_ns;   // the prefix every mailbox of every shard can take, with the ticks due by its last event
  }
  for (cpbus* s : h->shards) if (*(volatile unsigned int*)s->h_err) return CPBUS_ETIMEDOUT;
  // the default put waits (bounded) for the slot's previous batch: its fan-outs are already queued behind earlier puts
  if ((rc = cpbus_stream_put(h->shard_st[0], h->h_batch[0], m, w, CPBUS_PUT_RAW))) return rc;
  for (size_t k = 0; k < h->shards.size(); k++) {
    if ((rc = dev_guard(h->shards[k]))) return rc;
    if ((rc = stream_launch(h->shard_st[k], m, w, /*account=*/false))) return rc;
  }
  h->last_watermark = w;
  sh_sync_clocks(h);
  if (!ok) {
    memmove(h->h_batch[0], h->h_batch[0] + m, (size_t)(n - m) * sizeof(cpbus_event));   // (the put copied the prefix out)
    h->n_staged = n - m;
    h->room_lb = 0;
    h->st.admit_partial++;
    return CPBUS_EAGAIN;
  }
  h->n_staged = 0;
  return CPBUS_OK;
}

// flush the handle (membership and timer calls are ordered with publishes, events/bus.go:105-122), then work on the shards
int sh_prepare(cpbus* h) {
  int rc = dev_guard(h); if (rc) return rc;
  return flush_staged(h, h->now);
}

int sh_subscribe_many(cpbus* h, const uint32_t* masks, uint32_t n, uint32_t* first_sub_id) {
  int rc = sh_prepare(h); if (rc) return rc;
  const uint32_t first = h->n_next;
  rc = sh_pieces(h, first, n, [&](uint32_t k, uint32_t lo, uint32_t cnt) {
    const int r = cpbus_subscribe_many(h->shards[k], masks ? masks + (lo - first) : nullptr, cnt, nullptr);
    if (!r) h->n_next += cnt;
    return r;
  });
  if (rc) return rc;
  if (first_sub_id) *first_sub_id = h->cfg.sub_id_base + first;
  return CPBUS_OK;
}

int sh_subscribe_pairs(cpbus* h, uint32_t mask, const cpbus_pair* pairs, uint32_t n_pairs, uint32_t* sub_id) {
  if (h->n_next >= h->N) return CPBUS_ENOSPC;
  int rc = sh_prepare(h); if (rc) return rc;
  if ((rc = cpbus_subscribe_pairs(h->shards[sh_index(h, h->n_next)], mask, pairs, n_pairs, sub_id))) return rc;
  h->n_next++;
  return CPBUS_OK;
}

int sh_subscribe_pairs_many(cpbus* h, const uint32_t* masks, const cpbus_pair* pairs, const uint32_t* n_pairs, uint32_t n,
                            uint32_t* first_sub_id) {
  int rc = sh_prepare(h); if (rc) return rc;
  const uint32_t first = h->n_next;
  rc = sh_pieces(h, first, n, [&](uint32_t k, uint32_t lo, uint32_t cnt) {
    const size_t i = lo - first;
    const int r = cpbus_subscribe_pairs_many(h->shards[k], masks + i, pairs + i * CPBUS_MAX_PAIRS, n_pairs + i, cnt, nullptr);
    if (!r) h->n_next += cnt;
    return r;
  });
  if (rc) return rc;
  if (first_sub_id) *first_sub_id = h->cfg.sub_id_base + first;
  return CPBUS_OK;
}

int sh_unsubscribe(cpbus* h, uint32_t sub_id) {
  cpbus* s = sh_owner(h, sub_id);
  if (!s) return CPBUS_ENOENT;
  int rc = sh_prepare(h); if (rc) return rc;
  return cpbus_unsubscribe(s, sub_id);
}

int sh_set_mask(cpbus* h, uint32_t sub_id, uint32_t mask) {
  cpbus* s = sh_owner(h, sub_id);
  if (!s) return CPBUS_ENOENT;
  if (!s->h_active[sub_id - s->cfg.sub_id_base]) return CPBUS_ECLOSED;
  int rc = sh_prepare(h); if (rc) return rc;
  return cpbus_set_mask(s, sub_id, mask);
}

// timer ids of a handle are global slots: (id - sub_id_base) * K + k, with the shard's generation bits
int sh_timer_add(cpbus* h, uint32_t sub_id, uint64_t period_ns, uint32_t source_id, int oneshot, uint32_t* timer_id) {
  cpbus* s = sh_owner(h, sub_id);
  if (!s) return CPBUS_ENOENT;
  int rc = sh_prepare(h); if (rc) return rc;
  sh_retire_oneshots(h);
  h->any_timer = true;
  uint32_t local = 0;
  if ((rc = cpbus_timer_add(s, sub_id, period_ns, source_id, oneshot, &local))) return rc;
  if (!oneshot) h->min_period = std::min(h->min_period, period_ns);
  const uint32_t shift = (s->cfg.sub_id_base - h->cfg.sub_id_base) * h->K;
  if (timer_id) *timer_id = ((local & kTimerSlotMask) + shift) | (local & ~kTimerSlotMask);
  return CPBUS_OK;
}

int sh_timer_add_many(cpbus* h, uint32_t first_sub, uint32_t n, uint64_t period_ns, const uint32_t* source_ids, uint32_t source_id0,
                      int oneshot) {
  if (!sh_in_range(h, first_sub, n)) return CPBUS_ENOENT;
  int rc = sh_prepare(h); if (rc) return rc;
  sh_retire_oneshots(h);
  h->any_timer = true;
  const uint32_t l0 = first_sub - h->cfg.sub_id_base;
  // all or nothing, as on one bus: check every piece before arming any
  rc = sh_pieces(h, l0, n, [&](uint32_t k, uint32_t lo, uint32_t cnt) {
    const cpbus* s = h->shards[k];
    for (uint32_t i = lo - h->shard_first[k], e = i + cnt; i < e; i++) {
      if (!s->h_active[i]) return (int)CPBUS_ECLOSED;
      if (!s->h_timers.empty() && s->h_timers[(size_t)i * s->K].active) return (int)CPBUS_ENOSPC;
    }
    return (int)CPBUS_OK;
  });
  if (rc) return rc;
  if ((rc = sh_pieces(h, l0, n, [&](uint32_t k, uint32_t lo, uint32_t cnt) {
        const uint32_t i = lo - l0;
        return cpbus_timer_add_many(h->shards[k], h->cfg.sub_id_base + lo, cnt, period_ns, source_ids ? source_ids + i : nullptr,
                                    source_id0 + i, oneshot);
      })))
    return rc;
  if (!oneshot) h->min_period = std::min(h->min_period, period_ns);
  return CPBUS_OK;
}

int sh_timer_cancel(cpbus* h, uint32_t timer_id) {
  if (!h->K || !h->any_timer) return CPBUS_ENOENT;
  const uint32_t slot = timer_id & kTimerSlotMask, l = slot / h->K;
  if (l >= h->n_next) return CPBUS_ENOENT;
  int rc = sh_prepare(h); if (rc) return rc;
  sh_retire_oneshots(h);
  const uint32_t k = sh_index(h, l);
  rc = cpbus_timer_cancel(h->shards[k], (slot - h->shard_first[k] * h->K) | (timer_id & ~kTimerSlotMask));
  if (timers_armed(h) == 0) h->min_period = UINT64_MAX;
  return rc;
}

int sh_send(cpbus* h, uint32_t sub_id, const cpbus_event* ev) {
  cpbus* s = sh_owner(h, sub_id);
  if (!s) return CPBUS_ENOENT;
  if (!s->h_active[sub_id - s->cfg.sub_id_base]) return CPBUS_ECLOSED;
  int rc = dev_guard(h); if (rc) return rc;
  if ((rc = stage_one(h, ev->code, ev->source_id, sub_id, CPBUS_F_UNICAST))) return rc;   // global target: the owner's kernel takes it
  h->st.publishes++;
  return CPBUS_OK;
}

// one slice that every shard's launch can take: shard 0 reads the batch locally, the others pull it from shard 0's GPU
int sh_device_slice(cpbus* h, const cpbus_event* d_events, size_t n, uint64_t w) {
  for (size_t k = 0; k < h->shards.size(); k++) {
    const int rc = publish_device_impl(h->shards[k], d_events, n, w, /*staged=*/k > 0, nullptr, 0);
    if (rc) return rc;
  }
  cpbus* s0 = h->shards[0];
  for (const DbgItem& it : s0->dbg_pending) {   // shard 0's kernel accounted the batch: its debug-ring markers move to the handle
    h->dbg_pending.push_back(it);
    if (h->dbg_pending.size() > (size_t)kAcctDbgRing) h->dbg_pending.pop_front();
  }
  for (cpbus* s : h->shards) s->dbg_pending.clear();
  h->now = h->last_watermark = w;
  h->st.publishes += n; h->seq += n;
  sh_sync_clocks(h);
  return CPBUS_OK;
}

int sh_publish_device(cpbus* h, const void* d_events, size_t n, uint64_t watermark_ns) {
  if ((!d_events && n) || ((uintptr_t)d_events & 31u)) return CPBUS_EINVAL;
  if (h->lossless) return CPBUS_EINVAL;   // admission would have to read the batch from every shard: not supported
  int rc = dev_guard(h); if (rc) return rc;
  if ((rc = flush_staged(h, h->now))) return rc;
  if (watermark_ns < h->now) return CPBUS_EORDER;
  const cpbus_event* ev = (const cpbus_event*)d_events;
  const uint64_t window = max_window(h);
  if (n <= h->B && watermark_ns - h->last_watermark <= window) return sh_device_slice(h, ev, n, watermark_ns);
  // the same cut as publish_device_split, planned once for all shards
  std::vector<uint64_t> ts(n), wm;
  std::vector<size_t> end;
  cpbus* s0 = h->shards[0];
  if (n) {
    CK(cudaMemcpy2DAsync(ts.data(), 8, reinterpret_cast<const unsigned char*>(ev) + offsetof(cpbus_event, ts_ns), sizeof(cpbus_event),
                         8, n, cudaMemcpyDeviceToHost, s0->stream));
    CK(cudaStreamSynchronize(s0->stream));
  }
  if ((rc = split_plan(ts.data(), n, h->B, h->now, watermark_ns, window, end, wm))) return rc;
  size_t i = 0;
  for (size_t k = 0; k < end.size(); k++) {
    if ((rc = sh_device_slice(h, ev + i, end[k] - i, wm[k]))) return rc;
    h->st.device_splits++;
    i = end[k];
  }
  return CPBUS_OK;
}

int sh_drain_many(cpbus* h, uint32_t first_sub, uint32_t n, cpbus_event* out, size_t cap, uint32_t* offsets, uint32_t* counts,
                  size_t* total) {
  if (!sh_in_range(h, first_sub, n)) return CPBUS_ENOENT;
  const uint32_t l0 = first_sub - h->cfg.sub_id_base;
  size_t used = 0, tot = 0;
  const int rc = sh_pieces(h, l0, n, [&](uint32_t k, uint32_t lo, uint32_t cnt) {
    uint32_t* offs = offsets + (lo - l0);
    uint32_t* cnts = counts + (lo - l0);
    if (used >= cap) {   // no room left: these mailboxes stay untouched for the next call
      memset(offs, 0, cnt * sizeof(uint32_t)); memset(cnts, 0, cnt * sizeof(uint32_t));
      return (int)CPBUS_OK;
    }
    size_t t = 0, hi = 0;
    const int r = cpbus_drain_many(h->shards[k], h->cfg.sub_id_base + lo, cnt, out + used, cap - used, offs, cnts, &t);
    if (r) return r;
    for (uint32_t i = 0; i < cnt; i++)
      if (cnts[i]) { hi = std::max<size_t>(hi, (size_t)offs[i] + cnts[i]); offs[i] += (uint32_t)used; }
    used += hi; tot += t;
    return (int)CPBUS_OK;
  });
  if (rc) return rc;
  *total = tot;
  return CPBUS_OK;
}

int sh_digest(cpbus* h, uint32_t first_sub, uint32_t n, cpbus_digest_t* out) {
  if (!sh_in_range(h, first_sub, n)) return CPBUS_ENOENT;
  const uint32_t l0 = first_sub - h->cfg.sub_id_base;
  return sh_pieces(h, l0, n, [&](uint32_t k, uint32_t lo, uint32_t cnt) {
    return cpbus_digest(h->shards[k], h->cfg.sub_id_base + lo, cnt, out + (lo - l0));
  });
}

int sh_digest_fold_begin(cpbus* h, uint32_t first_sub, uint32_t n, uint32_t* ticket) {
  if (!sh_in_range(h, first_sub, n)) return CPBUS_ENOENT;
  const uint32_t slot = h->fold_next++ % cpbus::kFoldSlots;
  auto& parts = h->fold_parts[slot];
  parts.clear();
  const int rc = sh_pieces(h, first_sub - h->cfg.sub_id_base, n, [&](uint32_t k, uint32_t lo, uint32_t cnt) {
    uint32_t t = 0;
    const int r = cpbus_digest_fold_begin(h->shards[k], h->cfg.sub_id_base + lo, cnt, &t);
    if (!r) parts.emplace_back(k, t);
    return r;
  });
  if (rc) return rc;
  *ticket = slot;
  return CPBUS_OK;
}

int sh_digest_fold_end(cpbus* h, uint32_t ticket, uint64_t out[4]) {
  out[0] = out[1] = out[2] = out[3] = 0;
  for (const auto& p : h->fold_parts[ticket]) {   // the fold's own combination: sums, XOR, sum of n
    uint64_t o[4];
    const int rc = cpbus_digest_fold_end(h->shards[p.first], p.second, o);
    if (rc) return rc;
    out[0] += o[0]; out[1] += o[1]; out[2] ^= o[2]; out[3] += o[3];
  }
  return CPBUS_OK;
}

int sh_step_result_begin(cpbus* h, uint32_t* ticket) {
  const uint32_t t = h->result_next++ % 8;
  auto& parts = h->result_parts[t];
  parts.clear();
  for (cpbus* s : h->shards) {
    uint32_t st = 0;
    const int rc = cpbus_step_result_begin(s, &st);
    if (rc) return rc;
    parts.push_back(st);
  }
  *ticket = t;
  return CPBUS_OK;
}

// deliveries, ticks and digest sums add up over the shards; the launch ordinal is the same on every shard (shard 0's)
int sh_step_result_end(cpbus* h, uint32_t ticket, uint64_t out[4]) {
  out[0] = out[1] = out[2] = out[3] = 0;
  const auto& parts = h->result_parts[ticket];
  for (size_t k = 0; k < parts.size(); k++) {
    uint64_t o[4];
    const int rc = cpbus_step_result_end(h->shards[k], parts[k], o);
    if (rc) return rc;
    out[0] += o[0]; out[1] += o[1]; out[2] += o[2];
    if (k == 0) out[3] = o[3];
  }
  return CPBUS_OK;
}

int sh_stats(cpbus* h, cpbus_stats_t* out) {
  *out = h->st;
  out->deliveries = out->ticks = out->batches = out->kernel_launches = out->overwritten = 0;
  out->n_subs = out->n_timers = 0;
  for (size_t k = 0; k < h->shards.size(); k++) {
    cpbus_stats_t s{};
    const int rc = cpbus_stats(h->shards[k], &s);
    if (rc) return rc;
    out->deliveries += s.deliveries; out->ticks += s.ticks; out->batches += s.batches; out->kernel_launches += s.kernel_launches;
    out->overwritten += s.overwritten; out->n_subs += s.n_subs; out->n_timers += s.n_timers;
    if (k == 0) for (int c = 0; c < CPBUS_N_CODES; c++) out->published_by_code[c] += s.published_by_code[c];   // device batches (shard 0's kernel)
  }
  if (timers_armed(h) == 0) h->min_period = UINT64_MAX;   // (the shards' statistics retired their fired one-shots)
  out->now_ns = h->now;
  out->intern_entries = h->sources.size(); out->intern_bytes = h->intern_bytes;
  out->ephemeral_live = h->eph_live; out->ephemeral_recycled = h->eph_recycled;
  return CPBUS_OK;
}

}  // namespace
