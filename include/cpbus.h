/*
 * cpbus.h — C-ABI of libcpbus, the B200-native event bus that sits behind
 * ContainerPilot's `events` package (reference: /root/reference/events/).
 *
 * This header is the drop-in boundary (SURVEY.md §8b).  It is what a cgo shim
 * for package `events` binds (see INTEGRATION.md for the Go side).  Everything
 * is plain C: pointers + sizes, `int` status returns (0 = OK, negative =
 * CPBUS_E*), no exceptions, no torch types.  The library never keeps a caller
 * pointer past the call (cgo pointer rule).  One publisher thread at a time
 * per bus (the shim keeps `bus.lock`, reference events/bus.go:126); drain and
 * stats may be called from another thread between flushes.
 *
 * Record format (frozen): one 32-byte, 32-byte-aligned record = exactly one
 * HBM/L2 sector.  Go's `Event{Code EventCode; Source string}`
 * (events/events.go:10-13) maps to {code, source_id} through the host-side
 * intern table (cpbus_intern); seq/ts/target/flags are bus bookkeeping.
 */
#ifndef CPBUS_H
#define CPBUS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- event codes: events/events.go:21-39 (iota order is the wire value) ---- */
enum {
  CPBUS_NONE = 0, CPBUS_EXIT_SUCCESS, CPBUS_EXIT_FAILED, CPBUS_STOPPING,
  CPBUS_STOPPED, CPBUS_STATUS_HEALTHY, CPBUS_STATUS_UNHEALTHY,
  CPBUS_STATUS_CHANGED, CPBUS_TIMER_EXPIRED, CPBUS_ENTER_MAINTENANCE,
  CPBUS_EXIT_MAINTENANCE, CPBUS_ERROR, CPBUS_QUIT, CPBUS_METRIC,
  CPBUS_STARTUP, CPBUS_SHUTDOWN, CPBUS_SIGNAL,
  CPBUS_N_CODES /* 17 */
};

/* subscription mask: bit i set <=> subscriber wants EventCode i.
 * CPBUS_MASK_ALL reproduces the reference exactly (the reference bus has no
 * filter: events/bus.go:134-138 delivers every event to every subscriber). */
#define CPBUS_MASK_ALL 0x0001FFFFu

/* one exact case of a consumer's event switch: events.Event{Code, Source} (jobs/jobs.go:197-231) */
typedef struct cpbus_pair { uint32_t code, source_id; } cpbus_pair;
#define CPBUS_MAX_PAIRS 16

#define CPBUS_TARGET_ALL 0xFFFFFFFFu /* broadcast (EventBus.Publish)            */
#define CPBUS_F_TICK     0x1u        /* record produced by a timer (events/timer.go) */
#define CPBUS_F_UNICAST  0x2u        /* direct mailbox send (`sub.Rx <- ev`, jobs/jobs.go:262) */

typedef struct cpbus_event {
  uint64_t seq;       /* publish: global publish ordinal (0-based, bus lifetime).
                         tick: firing ordinal of that timer (0-based).          */
  uint64_t ts_ns;     /* virtual clock when published / due time of the tick    */
  uint32_t code;      /* EventCode                                              */
  uint32_t source_id; /* interned Event.Source                                  */
  uint32_t target;    /* CPBUS_TARGET_ALL, or the global subscriber id          */
  uint32_t flags;     /* CPBUS_F_*                                              */
} cpbus_event;        /* sizeof == 32 */

/* ---- status codes ---- */
enum {
  CPBUS_OK = 0,
  CPBUS_EINVAL = -1,   /* bad argument                                           */
  CPBUS_ENOMEM = -2,   /* host or device allocation failed                       */
  CPBUS_ECUDA = -3,    /* CUDA runtime error (cpbus_last_cuda_error has detail)  */
  CPBUS_EAGAIN = -4,   /* lossless mode: a targeted mailbox is full; drain+retry */
  CPBUS_ENOSPC = -5,   /* subscriber / timer / intern table capacity exhausted   */
  CPBUS_ENOENT = -6,   /* unknown subscriber / timer id                          */
  CPBUS_ECLOSED = -7,  /* subscriber already unsubscribed (Go: panic, bus.go:121)*/
  CPBUS_ENODEV = -8,   /* no CUDA device: there is NO CPU fallback               */
  CPBUS_EORDER = -9,   /* device batch not sorted by ts / clock moved backwards  */
  CPBUS_ETIMEDOUT = -10 /* stream mode: a batch never arrived (publisher stalled or the consumer fell a whole ring
                           behind); sticky: the bus reports it from every later stream call */
};

/* cpbus_config.flags */
#define CPBUS_CFG_LOSSLESS 0x1u /* reference semantics: never drop; a full mailbox
                                   stalls the publisher (events/subscriber.go:30-32).
                                   The library keeps a lower bound of the free room of
                                   the fullest mailbox: while a batch provably fits it
                                   goes straight to the fan-out; the admission kernel
                                   (and its host sync) runs only when the bound is used
                                   up, and refreshes it exactly.
                                   Without it the bus runs in overwrite-oldest
                                   throughput mode (no consumer needed).          */
#define CPBUS_CFG_DIGEST   0x2u /* maintain the per-subscriber order-sensitive
                                   64-bit digest in-kernel                       */

/* cpbus_config.store_path: how records reach the rings (all are bit-identical) */
enum {
  CPBUS_STORE_AUTO = 0, /* library default = best measured (see DESIGN.md)       */
  CPBUS_STORE_V4   = 1, /* st.global.v4.b32: lane pair per record, 16 B / lane   */
  CPBUS_STORE_V8   = 2, /* st.global.v8.b32: one lane per record, 32 B / lane    */
  CPBUS_STORE_BULK = 3  /* cp.async.bulk smem->global (TMA) for dense segments   */
};

typedef struct cpbus_config {
  uint32_t n_max_subs;     /* capacity of this shard's subscriber table           */
  uint32_t ring_cap;       /* records per mailbox; power of two, >= 64 (1024 = default; reference channel cap is 1000, jobs/jobs.go:23) */
  uint32_t batch_cap;      /* max events per flush; <= min(ring_cap/2, 1024), multiple of 32 */
  uint32_t timers_per_sub; /* timer slots per subscriber: 0,1,2,4,8               */
  uint32_t flags;          /* CPBUS_CFG_*                                         */
  int32_t  device;         /* CUDA device ordinal; -1 = current device            */
  uint32_t sub_id_base;    /* global id of this shard's subscriber 0 (multi-GPU:
                              contiguous shards, SURVEY.md §8e)                   */
  uint32_t store_path;     /* CPBUS_STORE_*                                       */
  void*    stream;         /* cudaStream_t to run on; NULL = library-owned stream */
  uint32_t grid_ctas;      /* 0 = auto (multiple of the SM count)                 */
  uint32_t reserved[5];
} cpbus_config;

typedef struct cpbus_digest_t {
  uint64_t count;  /* records ever delivered to this mailbox (broadcast + unicast + ticks) */
  uint64_t digest; /* rolling h = h*P + H(record) over the delivered sequence (mod 2^64)  */
} cpbus_digest_t;

typedef struct cpbus_stats_t {
  uint64_t publishes;      /* events that entered Publish/Send                    */
  uint64_t deliveries;     /* 32-B records landed in mailboxes (incl. ticks)      */
  uint64_t ticks;          /* timer records among the deliveries                  */
  uint64_t batches;        /* fan-out launches                                    */
  uint64_t kernel_launches;/* all kernels this bus launched                       */
  uint64_t overwritten;    /* undrained records currently lost to overwrite-oldest:
                              sum over mailboxes of max(0, tail - ring_cap - head) */
  uint64_t published_by_code[CPBUS_N_CODES]; /* reconciliation of the Prometheus
                              `containerpilot_events` counter (events/bus.go:130-132) */
  uint32_t n_subs;         /* currently subscribed                                */
  uint32_t n_timers;       /* currently armed                                     */
  uint64_t now_ns;         /* virtual clock                                       */
  /* ABI v2 */
  uint64_t intern_entries; /* permanent Source strings held by the intern table  */
  uint64_t intern_bytes;   /* ... and their total length                          */
  uint64_t ephemeral_live; /* payload strings currently held by the bounded ephemeral region (cpbus_intern_ephemeral) */
  uint64_t ephemeral_recycled; /* ephemeral ids that have been recycled so far   */
  uint64_t admit_passes;   /* lossless mode: flushes that needed the admission kernel (+ one host sync) ... */
  uint64_t admit_skipped;  /* ... and flushes that provably fitted and went straight to the fan-out        */
  uint64_t admit_partial;  /* flushes that delivered only the prefix every mailbox could take (then EAGAIN)  */
  uint64_t device_splits;  /* slices launched for device batches one launch could not take (see cpbus_publish_device) */
} cpbus_stats_t;

typedef struct cpbus cpbus_t;

/* ---- lifecycle: NewEventBus (events/bus.go:72-88); reload = destroy+create (core/app.go:142) ---- */
int cpbus_create(const cpbus_config* cfg, cpbus_t** out);
int cpbus_destroy(cpbus_t* bus);

/* ---- one handle over several GPUs ----------------------------------------------------------------------------------------
 * G shard buses behind ONE handle: every other cpbus_* entry point takes it unchanged, and every value a caller reads back
 * equals what one bus created with the same cfg returns (status codes, records, lost, digests, folds, step results, debug
 * events, publish counts, source ids, statistics) — except cpbus_stats.batches and .kernel_launches, which are sums over
 * the shards.  cfg means what it means for cpbus_create (total capacity, ring, batch, timers, flags, store path, grid);
 * cfg->device is ignored: shard k lives on devices[k] (a device may repeat).  n_shards == 1 is exactly cpbus_create on
 * devices[0].  CPBUS_EINVAL (before any device is touched): what cpbus_create rejects, devices == NULL, n_shards == 0 or
 * > 64, n_max_subs < n_shards, cfg->stream != NULL.  If a shard cannot be created, what was made is destroyed.
 *   Ids.  Shard k owns the contiguous global ids sub_id_base + cpbus_shard_range(n_max_subs, n_shards, k); ids are handed
 *   out in order from sub_id_base as on one bus, so a fleet that fills the handle spreads evenly and a few subscribers all
 *   sit on shard 0.  Timer ids are global slots ((id - sub_id_base) * K + k, with the generation bits).
 *   Routing.  Intern/source: one table at the handle.  Ranges (subscribe_many, subscribe_pairs_many, timer_add_many, digest,
 *   digest_fold*, drain_many) are cut at the shard boundaries; drain_many keeps its contract when cap is short (every run is
 *   complete and FIFO, a mailbox left out has counts[i] = 0).  Single-subscriber calls go to the owner shard after the
 *   staged events are flushed.  cpbus_step_result_end: deliveries, ticks and digest sums added over the shards, the launch
 *   ordinal of shard 0.
 *   Data path.  The handle stages events like one bus (seq = publish ordinal, ts = its clock).  A flush puts the staged
 *   records into a stream owned by shard 0 and launches one stream fan-out per shard (cpbus_stream_*: each shard's lead CTA
 *   pulls the batch); cpbus_advance cuts clock steps at the narrowest timer window over the shards.  Lossless mode: a flush
 *   delivers, on every shard, the longest prefix every mailbox of every shard can take (the admission pass runs on each shard
 *   when the handle's room bound is used up) and returns CPBUS_EAGAIN for the rest, as one bus does.
 *   cpbus_publish_device: throughput mode only (shard 0 reads the batch locally, the others pull it from shard 0's GPU;
 *   oversize batches are cut once for all shards; shard 0's kernel accounts them); CPBUS_EINVAL in lossless mode.
 *   CPBUS_EINVAL on a handle: cpbus_publish_device_staged, cpbus_stream_create/open/attach, cpbus_shared_*, cpbus_device_ptrs. */
int cpbus_create_sharded(const cpbus_config* cfg, const int32_t* devices, uint32_t n_shards, cpbus_t** out);
/* The id partition of cpbus_create_sharded, host-only (no device): shard `shard` of n_shards holds local ids
 * [*first, *first + *count) of n_max_subs; the first n_max_subs % n_shards shards hold one more.  CPBUS_EINVAL: n_shards == 0,
 * shard >= n_shards, or a NULL output. */
int cpbus_shard_range(uint32_t n_max_subs, uint32_t n_shards, uint32_t shard, uint32_t* first, uint32_t* count);

/* ---- Event.Source interning (events/events.go:12; SURVEY F7) ---- */
int cpbus_intern(cpbus_t* bus, const char* s, size_t len, uint32_t* source_id);
/* copies at most cap bytes; *len receives the full length.  CPBUS_ENOENT: unknown id, or an ephemeral id whose
 * slot has been recycled since. */
int cpbus_source(cpbus_t* bus, uint32_t source_id, char* out, size_t cap, size_t* len);
/* Payload strings that are NOT names: every POST /v3/metric publishes Event{Metric, "key|value"}
 * (control/endpoints.go:125-126) and each distinct value would otherwise live in the intern table for the bus's
 * lifetime (the reference keeps Metric out of its per-source counter for the same cardinality reason, events/bus.go:130).
 * Ephemeral ids come from a bounded region of CPBUS_EPHEMERAL_SLOTS strings that is recycled oldest-first: an id
 * (bit 31 set) stays resolvable until CPBUS_EPHEMERAL_SLOTS newer distinct payloads have been interned — far beyond the
 * lifetime of a record in a 1024-slot mailbox.  Equal strings that are both still live get the same id. */
#define CPBUS_EPHEMERAL_SLOTS 65536u
#define CPBUS_EPHEMERAL_BIT   0x80000000u
int cpbus_intern_ephemeral(cpbus_t* bus, const char* s, size_t len, uint32_t* source_id);

/* ---- membership: Subscribe/Unsubscribe (events/bus.go:105-122).  Ordered with
 *      publishes: any staged events are flushed first. ---- */
int cpbus_subscribe(cpbus_t* bus, uint32_t code_mask, uint32_t* sub_id);
int cpbus_subscribe_many(cpbus_t* bus, const uint32_t* code_masks, uint32_t n, uint32_t* first_sub_id);
/* Second-level filter (SURVEY.md §8f N3).  A consumer's `switch event { case events.Event{Code, Source}: ... }`
 * (jobs/jobs.go:188-231) compares whole Event values, so each case is an exact {code, source} pair.  The subscriber
 * receives a broadcast event when its code is in code_mask (any source) OR {code, source_id} equals one of the
 * n_pairs <= CPBUS_MAX_PAIRS pairs.  Unicast records and timer ticks bypass both levels, like a direct channel send.
 * CPBUS_EINVAL: n_pairs > CPBUS_MAX_PAIRS, a pair's code >= CPBUS_N_CODES, or pairs == NULL with n_pairs > 0. */
int cpbus_subscribe_pairs(cpbus_t* bus, uint32_t code_mask, const cpbus_pair* pairs, uint32_t n_pairs, uint32_t* sub_id);
/* bulk form for a whole fleet: subscriber i gets code_masks[i] and the first n_pairs[i] (<= CPBUS_MAX_PAIRS) entries of
 * row i of `pairs` (n rows of CPBUS_MAX_PAIRS entries; the rest of a row is ignored).  One upload instead of n calls. */
int cpbus_subscribe_pairs_many(cpbus_t* bus, const uint32_t* code_masks, const cpbus_pair* pairs, const uint32_t* n_pairs,
                               uint32_t n, uint32_t* first_sub_id);
int cpbus_unsubscribe(cpbus_t* bus, uint32_t sub_id);
/* Change a subscriber's code mask in place (ordered with publishes).  Mailbox, timers and exact cases are kept.  The
 * shims use it when a channel that only carried timer ticks (implicit mask-0 subscriber, see NewEventTimer in
 * INTEGRATION.md) is subscribed to the bus afterwards. */
int cpbus_set_mask(cpbus_t* bus, uint32_t sub_id, uint32_t code_mask);

/* ---- timers: NewEventTimer / NewEventTimeout (events/timer.go:40-71 / 12-37).
 *      The first firing is due at now + period_ns; a periodic timer then fires
 *      every period_ns, a one-shot exactly once.  cancel = ctx.Done().  A timer id carries a generation: cancelling an
 *      id whose slot has fired (one-shot) or been re-armed since returns CPBUS_ENOENT and touches nothing. ---- */
int cpbus_timer_add(cpbus_t* bus, uint32_t sub_id, uint64_t period_ns, uint32_t source_id, int oneshot, uint32_t* timer_id);
/* one periodic timer per subscriber [first_sub, first_sub+n); source_ids[i] (or source_id0+i if NULL) */
int cpbus_timer_add_many(cpbus_t* bus, uint32_t first_sub, uint32_t n, uint64_t period_ns, const uint32_t* source_ids, uint32_t source_id0, int oneshot);
int cpbus_timer_cancel(cpbus_t* bus, uint32_t timer_id);

/* ---- the hot path: EventBus.Publish (events/bus.go:125-140) ---- */
/* Stages n events; only code/source_id are read from ev (seq, ts, target, flags
 * are stamped by the bus).  Flushes automatically whenever batch_cap is reached.
 * Lossless mode: if an automatic flush hits a full mailbox the call stops and returns
 * CPBUS_EAGAIN; events before the one that triggered the flush are staged, that one and
 * the rest are not (cpbus_stats.publishes tells how many were taken).  Publishing one
 * event per call, as the Go bus does, makes the retry point unambiguous.  cpbus_flush in
 * lossless mode blocks PER EVENT like the Go bus: when some mailbox lacks the room, the longest
 * prefix of the staged events that every targeted mailbox can take is delivered (with the timer
 * ticks due by its last event), the rest stays staged and the call returns CPBUS_EAGAIN; after the
 * consumers have drained, the next flush continues with the first undelivered event.
 * (Batches handed over in device memory, cpbus_publish_device, stay all-or-nothing: the caller owns them.) */
int cpbus_publish(cpbus_t* bus, const cpbus_event* ev, size_t n);
/* Direct mailbox write, bypassing the filter (`job.Rx <- ev`, jobs/jobs.go:262;
 * Subscriber.Receive, events/subscriber.go:30).  Ordered with publishes. */
int cpbus_send(cpbus_t* bus, uint32_t sub_id, const cpbus_event* ev);
/* Move the virtual clock; timers whose due time <= now_ns fire at the next flush,
 * ordered before any event published after this call. */
int cpbus_advance(cpbus_t* bus, uint64_t now_ns);
/* Launch the fan-out for everything staged (async on the bus stream). */
int cpbus_flush(cpbus_t* bus);
int cpbus_sync(cpbus_t* bus);
/* Fan out a batch that is already resident in HBM (multi-GPU: the NCCL-broadcast
 * stream, SURVEY.md §8e; bench: device-resident trace).  Records are complete
 * (seq/ts/target/flags set by the producer), sorted by ts_ns, 32-byte aligned.
 * watermark_ns >= last ts; becomes the bus clock.  One launch takes up to batch_cap
 * records and a watermark step of up to 32/timers_per_sub periods of the fastest armed
 * timer; a batch beyond either is cut into several launches (the cut reads the records'
 * timestamps back, 8 bytes each: a slow path, counted in cpbus_stats.device_splits).
 * Lossless mode keeps the strict form: CPBUS_EINVAL / CPBUS_EORDER for such a batch. */
int cpbus_publish_device(cpbus_t* bus, const void* d_events, size_t n, uint64_t watermark_ns);
/* (Batches published this way are accounted for by the kernel itself: cpbus_stats.published_by_code,
 * cpbus_publish_counts and cpbus_debug_events see their broadcast events exactly as if they had gone through cpbus_publish.) */
/* Same, but d_events may point into ANOTHER GPU's HBM (the publisher's event stream, peer-mapped over
 * NVLink, e.g. through CUDA IPC): one CTA of the fan-out kernel pulls the batch across the link, stages it
 * locally and hands it to the other CTAs together with the batch descriptor — the broadcast of SURVEY.md §8e
 * fused into the fan-out launch, no collective call.  If d_next/n_next name a LATER batch (the next one, or better
 * the one after it), the same launch also pulls that batch (the NVLink transfer hides under this launch's stores) and
 * a later call given that pointer as its d_events starts from local memory; a batch pulled two launches earlier also
 * lets that launch's prologue overlap its predecessor (programmatic dependent launch).  The caller guarantees the peer batches are complete and stable while the
 * launch runs (throughput mode only). */
int cpbus_publish_device_staged(cpbus_t* bus, const void* d_events, size_t n, uint64_t watermark_ns,
                                const void* d_next, size_t n_next);

/* ---- the publisher's event stream across the GPUs of one box (one process per GPU) ----------------------------------
 * The subscriber set partitions into contiguous shards, one bus per GPU (cpbus_config.sub_id_base); every shard must see
 * the identical, totally ordered batch sequence (SURVEY.md §8e).  A stream is a ring of n_slots batch slots in the
 * PUBLISHER GPU's HBM, exported with CUDA IPC.  cpbus_stream_put copies a batch into the next slot and then releases it
 * by writing the slot header {seq, watermark, n} (stream-ordered after the payload).  cpbus_stream_fanout, called by
 * every rank including the publisher's, launches the ordinary fan-out kernel for the next batch of the stream: its lead
 * CTA acquires the header across NVLink (ld.acquire.sys, bounded wait), pulls the 32-byte records over the peer mapping,
 * stages them locally for the other CTAs and acknowledges the slot (st.release.sys into the publisher's memory) — the
 * broadcast is fused into the fan-out launch; there is no collective, no copy-engine op and no cross-stream wait on the
 * consumers' data path.  When the publisher runs >= 2 batches ahead, the lead CTA of batch q also pulls batch q+2 while
 * its own stores are in flight, so later launches start from local memory and keep their prologue overlapped with the
 * previous launch (programmatic dependent launch).  Throughput (overwrite-oldest) mode only.
 *   publisher rank : cpbus_stream_create(bus, n_slots, n_consumers, &st, handle); send `handle` to the other ranks
 *   other ranks    : cpbus_stream_open(bus, handle, consumer_index (1..n_consumers-1), &st)
 *   every step     : [publisher] cpbus_stream_put(st, events, n, now_ns, flags)   (may run ahead by < n_slots batches)
 *                    [all ranks] cpbus_stream_fanout(st, n, now_ns)
 * The consumers must be told n and now_ns of every batch by the caller: SPMD drivers know them; others ask cpbus_stream_poll,
 * which reads them from the slot header (the kernel cross-checks n either way).  CPBUS_EAGAIN from _put: the slot's previous batch is still not acknowledged by every
 * consumer after the stream timeout (or at once with CPBUS_PUT_NOWAIT) — call again after the consumers have advanced.  CPBUS_ETIMEDOUT from _fanout/_status: an earlier stream
 * launch gave up waiting for its batch (bounded in-kernel wait, cpbus_stream_set_timeout) and delivered nothing. */
typedef struct cpbus_stream cpbus_stream_t;
#define CPBUS_PUT_STAMP 0x0u /* records are stamped like cpbus_publish: seq = running publish ordinal, ts = now_ns,
                                target = ALL, flags = 0; only code/source_id are read from the caller's records */
#define CPBUS_PUT_RAW   0x1u /* records are complete (as for cpbus_publish_device): copied verbatim */
#define CPBUS_PUT_NOWAIT 0x2u /* if the slot's previous batch is not yet acknowledged by every consumer, return
                                CPBUS_EAGAIN at once.  Default: wait for the consumers (their launches are queued, the
                                GPUs are busy) up to the stream timeout, then CPBUS_EAGAIN.  A single thread that drives
                                the publisher AND consumers (LocalShardedBus) must use NOWAIT or never run more than
                                n_slots batches ahead of its own fan-outs. */
int cpbus_stream_create(cpbus_t* bus, uint32_t n_slots, uint32_t n_consumers, cpbus_stream_t** out, unsigned char handle[64]);
int cpbus_stream_open(cpbus_t* bus, const unsigned char handle[64], uint32_t consumer_index, cpbus_stream_t** out);
/* same-process consumer (one host process driving several GPUs, as the cgo shim does): no IPC handle, the owner's ring is
 * used through peer access (enabled here if the two buses live on different GPUs) */
int cpbus_stream_attach(cpbus_t* bus, cpbus_stream_t* owner, uint32_t consumer_index, cpbus_stream_t** out);
int cpbus_stream_put(cpbus_stream_t* st, const cpbus_event* events, size_t n, uint64_t now_ns, uint32_t flags);
int cpbus_stream_fanout(cpbus_stream_t* st, size_t n, uint64_t now_ns);
/* For a consumer whose driver does not know the batches' shapes: *ready = 1 and {n, now_ns} of the NEXT batch if the publisher
 * has released it, *ready = 0 otherwise (one 32-byte read of the slot header, synchronous).  Then cpbus_stream_fanout(st, n, now_ns). */
int cpbus_stream_poll(cpbus_stream_t* st, int* ready, size_t* n, uint64_t* now_ns);
int cpbus_stream_status(cpbus_stream_t* st);                       /* CPBUS_OK or the sticky error */
int cpbus_stream_set_timeout(cpbus_stream_t* st, uint32_t microseconds);   /* in-kernel wait bound; default 2 s */
int cpbus_stream_close(cpbus_stream_t* st);                        /* importers close before the owner */

/* Buffers shared between the GPUs (processes) of one box, for the publisher's event stream: _alloc makes a
 * device buffer on this bus's GPU and returns a 64-byte CUDA IPC handle; _open, called on ANOTHER bus (another
 * process/GPU), maps it over NVLink and returns a pointer valid for cpbus_publish_device_staged there.
 * _close frees (owner) or unmaps (importer); cpbus_destroy closes what is left. */
int cpbus_shared_alloc(cpbus_t* bus, size_t bytes, void** dptr, unsigned char handle[64]);
int cpbus_shared_open(cpbus_t* bus, const unsigned char handle[64], void** dptr);
int cpbus_shared_close(cpbus_t* bus, void* dptr);

/* ---- consumer side ---- */
/* Mailbox -> host, FIFO (`<-sub.Rx`).  *lost = records overwritten before they
 * could be drained (always 0 in lossless mode). */
int cpbus_drain(cpbus_t* bus, uint32_t sub_id, cpbus_event* out, size_t cap, size_t* n, uint64_t* lost);
/* Bulk drain of mailboxes [first_sub, first_sub+n): one kernel gathers every undrained record into a staging
 * buffer (one atomic per mailbox), two D2H copies bring them back.  out[offsets[i] .. offsets[i]+counts[i]) is mailbox
 * i's run, FIFO.  A mailbox whose run does not fit into `cap` is left untouched (counts[i] = 0) for the next call;
 * *total = records returned.  This is what the `chan Event` pump of a shim with many subscribers calls. */
int cpbus_drain_many(cpbus_t* bus, uint32_t first_sub, uint32_t n, cpbus_event* out, size_t cap,
                     uint32_t* offsets, uint32_t* counts, size_t* total);
/* Device-side consumer: every mailbox is read to the end and its records are discarded (head = tail), ordered behind
 * every earlier fan-out on the bus stream.  For subscribers nobody reads, and for measuring the lossless mode with
 * consumers that keep up. */
int cpbus_consume_all(cpbus_t* bus);
/* Last min(cap, ring_cap, count) delivered records, oldest first, without consuming. */
int cpbus_peek_window(cpbus_t* bus, uint32_t sub_id, cpbus_event* out, size_t cap, size_t* n);
int cpbus_digest(cpbus_t* bus, uint32_t first_sub, uint32_t n, cpbus_digest_t* out);
/* XOR-fold / sum of (count, digest) over [first_sub, first_sub+n) computed on the
 * device: one 32-byte D2H instead of 16 B per subscriber. */
int cpbus_digest_fold(cpbus_t* bus, uint32_t first_sub, uint32_t n, uint64_t out[4]);
/* Split form: _begin enqueues the fold + the 32-byte D2H on the bus stream and returns a ticket
 * (up to 8 outstanding); _end waits for that ticket only.  Lets a caller read step i's result
 * while step i+1 is already running. */
int cpbus_digest_fold_begin(cpbus_t* bus, uint32_t first_sub, uint32_t n, uint32_t* ticket);
int cpbus_digest_fold_end(cpbus_t* bus, uint32_t ticket, uint64_t out[4]);

/* Result of the LAST fan-out launch, written by the kernel itself: out = {records delivered by that launch,
 * ticks among them, sum over every mailbox it appended to of fold32(new digest) with
 * fold32(x) = low32(x ^ (x >> 32)), launch ordinal}.
 * _begin enqueues a 256-byte D2H on the bus stream (up to 8 outstanding tickets), _end waits for it. */
int cpbus_step_result_begin(cpbus_t* bus, uint32_t* ticket);
int cpbus_step_result_end(cpbus_t* bus, uint32_t ticket, uint64_t out[4]);

/* ---- observation ---- */
/* DebugEvents (events/bus.go:34-54): drains the 10-slot ring of the last published
 * events, oldest first, stopping at a NonEvent.  Host-side, no 100 ms sleep. */
int cpbus_debug_events(cpbus_t* bus, cpbus_event* out, size_t cap, size_t* n);
int cpbus_stats(cpbus_t* bus, cpbus_stats_t* out);
/* Publish counts by {code, source}: the label set of the reference's `containerpilot_events` counter
 * (events/bus.go:60-68,130-132; code Metric is excluded there and here).  Covers both host publishes and batches that
 * reached the bus in device memory (counted by the kernel).  Writes at most cap entries, *n = entries available.
 * Call it from the publisher's thread (or with the publisher quiescent): it reads the table cpbus_publish updates. */
typedef struct cpbus_pair_count { uint32_t code, source_id; uint64_t count; } cpbus_pair_count;
int cpbus_publish_counts(cpbus_t* bus, cpbus_pair_count* out, size_t cap, size_t* n);
/* HBM layout, for zero-copy inspection by tests/bench: `ring` = n_max_subs mailboxes of
 * ring_cap records each (mailbox s starts at ring + s*ring_cap*32 bytes; slot of the j-th
 * delivered record = j mod ring_cap); `ctl` = n_max_subs control blocks of 32 bytes:
 * {u64 tail (records ever delivered); u64 head (consumer cursor); u64 digest; u32 mask
 * (bit 31 = subscribed, bits 24..27 = timer slots in use); u32 pad}. */
int cpbus_device_ptrs(cpbus_t* bus, void** ring, void** ctl);

/* ---- names: EventCode.String (events/eventcode_string.go:9-15), FromString (events/events.go:52-86) ---- */
const char* cpbus_code_name(int code);               /* NULL if out of range      */
int cpbus_code_from_string(const char* name);        /* code, or -1 if not valid  */

const char* cpbus_strerror(int status);
const char* cpbus_last_cuda_error(void);
uint32_t cpbus_abi_version(void);
/* 64-bit record hash and digest multiplier used by the in-kernel digest (so the
 * oracle and external checkers can reproduce it without reading kernel code) */
uint64_t cpbus_record_hash(const cpbus_event* ev);
uint64_t cpbus_digest_multiplier(void);
/* How cpbus_publish_device cuts a batch one launch cannot take, as a pure host function (no device needed): ts[0..n) = the
 * records' timestamps (sorted), now_ns = the bus clock, window_ns = the widest watermark step of one launch (UINT64_MAX: no
 * timer armed).  Slice k = records [ends[k-1], ends[k]) with watermark watermarks[k]; *n_slices = how many there are (the
 * first `cap` are written).  CPBUS_EORDER: unsorted, a record beyond watermark_ns, or watermark_ns < now_ns. */
int cpbus_split_plan(const uint64_t* ts, size_t n, uint32_t batch_cap, uint64_t now_ns, uint64_t watermark_ns, uint64_t window_ns,
                     size_t* ends, uint64_t* watermarks, size_t cap, size_t* n_slices);
/* The order in which the filtered (ORDERED) fan-out walks the mailboxes, as a pure host function (no device needed):
 * out[] receives the indices i < n with active[i] != 0 (active == NULL: all), grouped per block of `block` consecutive
 * subscribers (0 = the library's policy from n and ring_cap: one block up to 16 GiB of rings, 8-GiB blocks beyond;
 * 0xFFFFFFFF = one block), inside a block by code mask — equal masks adjacent — and, with heavy_first, masks with more
 * codes first.  out must have room for n indices; returns how many were written (0 on bad arguments).  Delivery
 * results never depend on this order. */
size_t cpbus_mask_order(const uint32_t* masks, const uint8_t* active, uint32_t n, uint32_t ring_cap, uint32_t block,
                        int heavy_first, uint32_t* out);

#ifdef __cplusplus
}
#endif
#endif /* CPBUS_H */
