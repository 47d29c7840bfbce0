// dingest.cu — host side of the device record-batch decode (include/sgr.h "device ingest"; kernels: dingest_kernels.cu).
//
// The host keeps exactly what is sequential and tiny: the walk over the 61-byte RecordBatch headers of a fetch (boundaries, a
// trailing partial batch, magic), the read_committed bookkeeping of org.apache.kafka consumers (control batches, the aborted
// transactions a fetch response announces) and the partition positions for the lag gate
// (modules/command-engine/core/src/main/scala/surge/internal/kafka/KafkaProducerActorImpl.scala:684-708). The wire bytes go to
// the device as they are; CRC, lz4, record parsing, id interning and the fold never touch the CPU.
//
// Call sequence per poll:   sgr_dingest_submit(partition, fetch bytes)*  ->  sgr_dingest_fold()
// submit = header walk + one asynchronous H2D copy of the fetch (page-locked source memory makes it a single DMA). Whenever
//          `group_batches` data batches have accumulated, their whole chain
//              descriptors up -> crc_size (claims each batch's arena slot) -> decode_walk -> parse + intern
//          is enqueued on one of a few streams behind the copy that brought the group's last byte: no host round trip inside
//          the chain, so groups decode while later fetches are still crossing PCIe and while the host walks their headers.
// fold   = the chain of the remainder, one synchronisation, the verdicts (any error: nothing of the poll is applied), table
//          growth, new ids to the engine's key table, the sort-free fold of the decoded records onto the live table; only
//          then do the partitions' positions advance. All or nothing.
// The arena the batches decompress into is sized from the wire bytes (3x); if a poll compresses better than that the claims
// overflow, the flag comes back with the verdicts and the poll is decoded again from an exact host-side layout.
// SGR_DINGEST_V1=1 selects the first generation (memory-walking kernels, arena laid out on the host between two
// synchronisations) for A/B runs.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <map>
#include <string>
#include <thread>
#include <unordered_set>
#include <vector>

#include "../../include/sgr.h"
#include "devbuf.h"
#include "dingest_kernels.cuh"

using namespace sgr;

namespace {
inline uint16_t be16(const uint8_t* p) { return (uint16_t)((p[0] << 8) | p[1]); }
inline uint32_t be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }
inline uint64_t be64(const uint8_t* p) { return ((uint64_t)be32(p) << 32) | be32(p + 4); }
constexpr uint64_t kBatchHeader = 61;

struct PartState {
  int64_t decoded_next = 0, folded_next = 0;
  bool seen = false;
  std::vector<std::pair<int64_t, int64_t>> aborted;   // (first_offset, producer_id), ascending, not yet reached
  std::unordered_set<int64_t> aborting;               // producers inside an aborted transaction right now
};

// growable device buffer that keeps its content (the staged fetches of one poll accumulate in it)
struct KeepBuf {
  DevBuf b;
  uint64_t used = 0;
  cudaError_t ensure(uint64_t extra, cudaStream_t st) {
    if (used + extra <= b.cap) return cudaSuccess;
    DevBuf nb;
    uint64_t cap = b.cap ? b.cap : (1ull << 20);
    while (cap < used + extra) cap *= 2;
    cudaError_t e = nb.reserve(cap);
    if (e != cudaSuccess) return e;
    if (used) { e = cudaMemcpyAsync(nb.p, b.p, used, cudaMemcpyDeviceToDevice, st); if (e == cudaSuccess) e = cudaStreamSynchronize(st); }
    if (e != cudaSuccess) { nb.release(); return e; }
    b.release();
    b = nb;
    return cudaSuccess;
  }
};
}  // namespace

struct sgr_dingest {
  sgr_engine* eng = nullptr;
  cudaStream_t stream = nullptr;
  std::string last_error;
  std::map<int32_t, PartState> parts;       // committed view (after the last successful fold)
  std::map<int32_t, PartState> staged;      // view after the submissions of the current poll
  int32_t null_value_type = -1;
  // staged submissions
  KeepBuf wire;
  // descriptors of the poll's data batches, in PAGE-LOCKED memory: every copy of them is a true asynchronous DMA (a copy from
  // pageable memory makes the host wait for the stream, which serialised the submissions behind each other's CRC kernels)
  struct PinnedBatches {
    DgBatch* p = nullptr; size_t n = 0, cap = 0;
    bool reserve(size_t want) {
      if (want <= cap) return true;
      size_t c = cap ? cap : 4096;
      while (c < want) c *= 2;
      DgBatch* np = nullptr;
      if (cudaHostAlloc((void**)&np, c * sizeof(DgBatch), cudaHostAllocMapped) != cudaSuccess) return false;
      if (n) memcpy(np, p, n * sizeof(DgBatch));
      if (p) cudaFreeHost(p);
      p = np; cap = c;
      return true;
    }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    void clear() { n = 0; }
    DgBatch* data() { return p; }
    DgBatch& operator[](size_t i) { return p[i]; }
    void release() { if (p) cudaFreeHost(p); p = nullptr; n = cap = 0; }
  } batches;
  uint64_t n_record_slots = 0;
  sgr_ingest_stats poll{};                  // statistics of the current poll (host-side parts)
  sgr_ingest_stats total{};
  struct Sub { uint32_t batch_begin, batch_end; uint64_t nbytes; cudaEvent_t copied; };
  std::vector<Sub> subs;                    // the submissions of the current poll, in order
  std::vector<cudaEvent_t> event_pool;
  cudaStream_t copy_stream = nullptr;       // H2D copies of the wire bytes: they overlap the decode of earlier submissions
  // device scratch
  KeepBuf arena, d_batches;
  uint64_t d_batches_used = 0;              // descriptors uploaded by the submissions of this poll
  uint64_t crc_launched = 0;                // ... of which the CRC + size pass (v1) / the whole chain (default) has been launched
  KeepBuf rec_off, rec_batch, out;          // per record slot; they keep their content when a later group needs them larger
  DevBuf key_offs_dev, key_bytes_dev;
  // chains of launches per group of batches
  bool v1 = false;                          // SGR_DINGEST_V1
  uint32_t group_batches = 8192;            // SGR_DINGEST_GROUP
  static constexpr int kGroupStreams = 8;
  cudaStream_t gstream[kGroupStreams] = {};
  std::vector<cudaEvent_t> group_events;    // pool; the first n_groups are this poll's "group done" events
  uint32_t n_groups = 0;
  uint64_t launched_records = 0;            // record slots covered by the launched chains
  // SGR_DINGEST_TIMING: per group the device times (ms since the poll's first copy was queued) at which its bytes had landed,
  // its CRC + size pass, its decode and its parse ended; printed to stderr by sgr_dingest_fold
  std::vector<cudaEvent_t> tl_events;       // 4 per group, + [last] the poll's origin
  cudaEvent_t tl_origin = nullptr;
  void* h_keys = nullptr; uint64_t h_keys_cap = 0;   // page-locked landing area of the new ids
  // device dictionary
  DevBuf tags, slot_idx, key_ref, id_arena, ctl;
  uint64_t slots = 0, max_keys = 0, arena_cap = 0;
  uint64_t keys_on_host = 0;                // ids already appended to the engine's key table
  uint64_t id_bytes_on_host = 0;            // ... and the id-arena bytes they occupy
  uint64_t keys_reported = 0;               // ids counted in the n_new_keys of a successful poll
  cudaEvent_t keys_landed = nullptr;
  uint64_t generation = 0;                  // bumped by sgr_dingest_reset: a new dictionary is a new owner of the engine's key table
  void* h_ctl = nullptr;                    // page-locked landing area
  bool timing_syncs = false;                // SGR_DINGEST_TIMING=1: an extra synchronisation separates decode from parse in ms[]
  float ms[8] = {};                         // last fold: [0] wait for H2D + crc/size [1] decode + walk [2] parse + intern [3] keys to host
                                            //            [4] table growth + fold [5] total
};

namespace {
int32_t dfail(sgr_dingest* g, int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  if (g) g->last_error = buf;
  return code;
}
#define DG_TRY(g, call)                                                                                          \
  do {                                                                                                           \
    cudaError_t _e = (call);                                                                                     \
    if (_e != cudaSuccess) return dfail((g), _e == cudaErrorMemoryAllocation ? SGR_ERR_OOM : SGR_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(_e)); \
  } while (0)

const char* dg_err_text(uint32_t e) {
  switch (e) {
    case DG_CRC: return "CRC-32C mismatch";
    case DG_LZ4_HEADER: return "bad LZ4 frame header";
    case DG_LZ4_BLOCK: return "LZ4 frame / block truncated or inconsistent";
    case DG_LZ4_SEQUENCE: return "malformed LZ4 sequence";
    case DG_LZ4_CHECKSUM: return "LZ4 checksum mismatch";
    case DG_LZ4_TOO_LARGE: return "LZ4 block decodes past its maximum size";
    case DG_RECORD_LENGTH: return "record length runs past the batch";
    case DG_RECORD_MALFORMED: return "record is malformed";
    case DG_RECORD_COUNT: return "recordsCount does not fit the batch";
    case DG_VALUE_LENGTH: return "packed event value outside 8..56 bytes (u32 type, u32 seq, payload)";
    case DG_ID_LENGTH: return "aggregate id too long";
    case DG_STRAY_BYTES: return "stray bytes after the last record";
  }
  return "unknown";
}

cudaError_t sync_all(sgr_dingest* g) {
  cudaError_t e = cudaSuccess, x;
  if (g->copy_stream && (x = cudaStreamSynchronize(g->copy_stream)) != cudaSuccess) e = x;
  for (cudaStream_t s : g->gstream) if (s && (x = cudaStreamSynchronize(s)) != cudaSuccess) e = x;
  if (g->stream && (x = cudaStreamSynchronize(g->stream)) != cudaSuccess) e = x;
  return e;
}

// per-poll device counters back to zero: [2] markers [3] null values [4] duplicates [5] dictionary overflow [6] records written,
// [8] arena bytes claimed, [10] arena overflow; [0] keys / [1] id bytes / [9] arena capacity persist
cudaError_t reset_poll_counters(sgr_dingest* g) {
  cudaError_t e = cudaMemsetAsync((unsigned long long*)g->ctl.p + 2, 0, 5 * 8, g->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync((unsigned long long*)g->ctl.p + 8, 0, 8, g->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync((unsigned long long*)g->ctl.p + 10, 0, 8, g->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(g->stream);   // group streams of the next poll must see it
  return e;
}

void clear_poll(sgr_dingest* g) {
  g->wire.used = 0; g->batches.clear(); g->n_record_slots = 0; g->poll = sgr_ingest_stats{}; g->subs.clear(); g->d_batches_used = 0; g->crc_launched = 0;
  g->n_groups = 0; g->launched_records = 0;
}

void discard_poll(sgr_dingest* g) {
  sync_all(g);   // no copy may still be landing in the buffer the next poll reuses, no chain still running
  reset_poll_counters(g);
  clear_poll(g);
  g->staged = g->parts;
}

DgParse parse_args(sgr_dingest* g) {
  DgParse p{};
  p.wire = (const uint8_t*)g->wire.b.p; p.arena = (const uint8_t*)g->arena.b.p;
  p.batches = (DgBatch*)g->d_batches.b.p;
  p.rec_off = (const uint32_t*)g->rec_off.b.p; p.rec_batch = (const uint32_t*)g->rec_batch.b.p; p.out = (uint8_t*)g->out.b.p; p.null_value_type = g->null_value_type;
  p.dict.tags = (unsigned long long*)g->tags.p; p.dict.slot_idx = (uint32_t*)g->slot_idx.p; p.dict.key_ref = (uint2*)g->key_ref.p;
  p.dict.arena = (uint8_t*)g->id_arena.p; p.dict.ctl = (unsigned long long*)g->ctl.p; p.dict.slots_mask = g->slots - 1;
  p.dict.max_keys = g->max_keys; p.dict.arena_cap = g->arena_cap;
  return p;
}

// grow a content-keeping buffer; anything that moves waits for every stream first (kernels in flight hold the old address)
cudaError_t grow_keeping(sgr_dingest* g, KeepBuf& kb, uint64_t keep_bytes, uint64_t want_bytes) {
  if (want_bytes <= kb.b.cap) return cudaSuccess;
  cudaError_t e = sync_all(g);
  if (e != cudaSuccess) return e;
  kb.used = keep_bytes;
  return kb.ensure(want_bytes - keep_bytes, g->stream);   // (ensure doubles, copies `used` bytes and synchronises)
}

cudaError_t set_arena_capacity(sgr_dingest* g) {
  const unsigned long long cap = g->arena.b.cap >= 512 ? g->arena.b.cap - 512 : 0;   // (the walk's ring reads 256 bytes past a slot)
  return cudaMemcpy((unsigned long long*)g->ctl.p + 9, &cap, 8, cudaMemcpyHostToDevice);
}

// Enqueue descriptors-up -> crc_size (+ arena claim) -> decode_walk -> parse for the batches [crc_launched, batch_end) — record
// slots [launched_records, rec_end) — behind `landed` (the copy of the last fetch that contributes to the group).
int32_t launch_group(sgr_dingest* g, uint64_t batch_end, uint64_t rec_end, cudaEvent_t landed) {
  const uint64_t b0 = g->crc_launched, nb = batch_end - b0;
  if (!nb) return SGR_OK;
  const uint64_t r0 = g->launched_records;
  DG_TRY(g, grow_keeping(g, g->d_batches, b0 * sizeof(DgBatch), batch_end * sizeof(DgBatch) + 64));
  DG_TRY(g, grow_keeping(g, g->rec_off, r0 * 4, rec_end * 4 + 64));
  DG_TRY(g, grow_keeping(g, g->rec_batch, r0 * 4, rec_end * 4 + 64));
  DG_TRY(g, grow_keeping(g, g->out, r0 * 64, rec_end * 64 + 64));
  const uint64_t arena_want = 3 * (uint64_t)g->wire.b.cap + 512;
  if (g->arena.b.cap < arena_want) {
    DG_TRY(g, grow_keeping(g, g->arena, b0 ? g->arena.b.cap : 0, arena_want));
    DG_TRY(g, set_arena_capacity(g));
  }
  if (g->n_groups >= g->group_events.size()) {
    cudaEvent_t ev;
    DG_TRY(g, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    g->group_events.push_back(ev);
  }
  cudaStream_t s = g->gstream[g->n_groups % sgr_dingest::kGroupStreams];
  DG_TRY(g, cudaStreamWaitEvent(s, landed, 0));
  cudaEvent_t* tl = nullptr;
  if (g->timing_syncs) {
    while (g->tl_events.size() < 4 * (size_t)(g->n_groups + 1)) { cudaEvent_t ev; DG_TRY(g, cudaEventCreate(&ev)); g->tl_events.push_back(ev); }
    tl = g->tl_events.data() + 4 * (size_t)g->n_groups;
    DG_TRY(g, cudaEventRecord(tl[0], s));
  }
  DgBatch* db = (DgBatch*)g->d_batches.b.p + b0;
  {
    void* mapped = nullptr;   // the descriptors go up by a kernel: a copy-engine transfer would queue behind every fetch of the poll
    DG_TRY(g, cudaHostGetDevicePointer(&mapped, g->batches.p + b0, 0));
    DG_TRY(g, dg_copy_from_mapped_host(mapped, db, nb * sizeof(DgBatch), s));
  }
  if (rec_end > r0) DG_TRY(g, cudaMemsetAsync((uint32_t*)g->rec_batch.b.p + r0, 0xff, (rec_end - r0) * 4, s));
  DG_TRY(g, dg_launch_crc_size_fast((const uint8_t*)g->wire.b.p, db, (uint32_t)nb, (unsigned long long*)g->ctl.p + 8, s));
  if (tl) DG_TRY(g, cudaEventRecord(tl[1], s));
  DG_TRY(g, dg_launch_decode_walk_fast((const uint8_t*)g->wire.b.p, (uint8_t*)g->arena.b.p, db, (uint32_t)nb, (uint32_t)b0, (uint32_t*)g->rec_off.b.p, (uint32_t*)g->rec_batch.b.p, (unsigned long long*)g->ctl.p + 8, s));
  if (tl) DG_TRY(g, cudaEventRecord(tl[2], s));
  DgParse p = parse_args(g);
  p.n_batches = (uint32_t)batch_end; p.rec_begin = (uint32_t)r0; p.n_records = (uint32_t)rec_end;
  DG_TRY(g, dg_launch_parse(p, s));
  if (tl) DG_TRY(g, cudaEventRecord(tl[3], s));
  DG_TRY(g, cudaEventRecord(g->group_events[g->n_groups], s));
  ++g->n_groups;
  g->crc_launched = batch_end; g->launched_records = rec_end;
  return SGR_OK;
}
}  // namespace

extern "C" {

int32_t sgr_dingest_create(sgr_engine* e, uint64_t max_keys, uint64_t max_id_bytes, sgr_dingest** out) {
  if (!e || !out || !max_keys) return SGR_ERR_INVALID;
  *out = nullptr;
  void* st = nullptr;
  if (sgr_stream(e, &st) != SGR_OK) return SGR_ERR_INVALID;
  sgr_dingest* g = new sgr_dingest();
  g->eng = e; g->stream = (cudaStream_t)st;
  g->timing_syncs = getenv("SGR_DINGEST_TIMING") != nullptr;
  g->v1 = getenv("SGR_DINGEST_V1") != nullptr;
  if (const char* gb = getenv("SGR_DINGEST_GROUP")) { const long v = atol(gb); if (v >= 64 && v <= (1l << 24)) g->group_batches = (uint32_t)v; }
  if (dg_prepare() != cudaSuccess) { delete g; return SGR_ERR_CUDA; }
  if (cudaStreamCreateWithFlags(&g->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { delete g; return SGR_ERR_CUDA; }
  for (cudaStream_t& s : g->gstream)
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) { sgr_dingest_destroy(g); return SGR_ERR_CUDA; }
  g->max_keys = max_keys;
  g->slots = 1024;
  while (g->slots < 2 * max_keys) g->slots *= 2;          // load factor <= 0.5
  g->arena_cap = max_id_bytes ? max_id_bytes : 32 * max_keys;
  cudaError_t ce;
  if ((ce = g->tags.reserve(g->slots * 8)) != cudaSuccess || (ce = g->slot_idx.reserve(g->slots * 4)) != cudaSuccess ||
      (ce = g->key_ref.reserve(max_keys * 8)) != cudaSuccess || (ce = g->id_arena.reserve(g->arena_cap + 64)) != cudaSuccess ||
      (ce = g->ctl.reserve(128)) != cudaSuccess || (ce = cudaHostAlloc(&g->h_ctl, 256, cudaHostAllocDefault)) != cudaSuccess ||
      (ce = cudaMemsetAsync(g->tags.p, 0, g->slots * 8, g->stream)) != cudaSuccess || (ce = cudaMemsetAsync(g->slot_idx.p, 0, g->slots * 4, g->stream)) != cudaSuccess ||
      (ce = cudaMemsetAsync(g->ctl.p, 0, 128, g->stream)) != cudaSuccess || (ce = cudaStreamSynchronize(g->stream)) != cudaSuccess) {
    sgr_dingest_destroy(g);
    return ce == cudaErrorMemoryAllocation ? SGR_ERR_OOM : SGR_ERR_CUDA;
  }
  *out = g;
  return SGR_OK;
}

int32_t sgr_dingest_destroy(sgr_dingest* g) {
  if (!g) return SGR_OK;
  sync_all(g);
  if (g->copy_stream) cudaStreamDestroy(g->copy_stream);
  for (cudaStream_t s : g->gstream) if (s) cudaStreamDestroy(s);
  for (cudaEvent_t ev : g->event_pool) cudaEventDestroy(ev);
  for (cudaEvent_t ev : g->group_events) cudaEventDestroy(ev);
  for (cudaEvent_t ev : g->tl_events) cudaEventDestroy(ev);
  if (g->tl_origin) cudaEventDestroy(g->tl_origin);
  if (g->keys_landed) cudaEventDestroy(g->keys_landed);
  if (g->h_keys) cudaFreeHost(g->h_keys);
  g->batches.release();
  g->wire.b.release(); g->d_batches.b.release(); g->arena.b.release(); g->rec_off.b.release(); g->rec_batch.b.release(); g->out.b.release();
  g->key_offs_dev.release(); g->key_bytes_dev.release();
  g->tags.release(); g->slot_idx.release(); g->key_ref.release(); g->id_arena.release(); g->ctl.release();
  if (g->h_ctl) cudaFreeHost(g->h_ctl);
  delete g;
  return SGR_OK;
}

const char* sgr_dingest_last_error(const sgr_dingest* g) { return g ? g->last_error.c_str() : "null device-ingest handle"; }

int32_t sgr_dingest_set_null_value_type(sgr_dingest* g, int32_t event_type) {
  if (!g || event_type >= (int32_t)SGR_MAX_TYPES) return dfail(g, SGR_ERR_INVALID, "event type out of range");
  g->null_value_type = event_type < 0 ? -1 : event_type;
  return SGR_OK;
}

int32_t sgr_dingest_set_aborted(sgr_dingest* g, int32_t partition, const int64_t* producer_ids, const int64_t* first_offsets, uint64_t n) {
  if (!g || (n && (!producer_ids || !first_offsets))) return dfail(g, SGR_ERR_INVALID, "null argument");
  PartState& ps = g->staged[partition];
  for (uint64_t i = 0; i < n; ++i) ps.aborted.emplace_back(first_offsets[i], producer_ids[i]);
  std::sort(ps.aborted.begin(), ps.aborted.end());
  return SGR_OK;
}

// Walk the batch headers of one fetch; data batches that a read_committed consumer would deliver are queued for the device.
int32_t sgr_dingest_submit(sgr_dingest* g, int32_t partition, const void* data, uint64_t nbytes, sgr_ingest_stats* stats) {
  if (!g || (!data && nbytes)) return dfail(g, SGR_ERR_INVALID, "null argument");
  const uint8_t* buf = (const uint8_t*)data;
  PartState ps = g->staged[partition];   // work on a copy: a malformed fetch leaves the staged view untouched
  sgr_ingest_stats st{};
  std::vector<DgBatch> add;
  uint64_t slots = 0, pos = 0;
  while (nbytes - pos >= 12) {
    const int64_t base_offset = (int64_t)be64(buf + pos);
    const int32_t batch_length = (int32_t)be32(buf + pos + 8);
    if (batch_length < (int32_t)(kBatchHeader - 12)) return dfail(g, SGR_ERR_INVALID, "partition %d offset %lld: batch length %d is smaller than a v2 header", partition, (long long)base_offset, batch_length);
    const uint64_t total = 12ull + (uint32_t)batch_length;
    if (nbytes - pos < total) break;   // a trailing partial batch: the next fetch repeats it
    const uint8_t* b = buf + pos;
    if ((int8_t)b[16] != 2) return dfail(g, SGR_ERR_UNSUPPORTED, "partition %d offset %lld: message format v%d (only RecordBatch magic 2 is decoded)", partition, (long long)base_offset, (int)(int8_t)b[16]);
    const uint16_t attrs = be16(b + 21);
    const int32_t last_offset_delta = (int32_t)be32(b + 23);
    const int64_t producer_id = (int64_t)be64(b + 43);
    const int32_t records_count = (int32_t)be32(b + 57);
    if (last_offset_delta < 0 || records_count < 0) return dfail(g, SGR_ERR_INVALID, "partition %d offset %lld: negative lastOffsetDelta / recordsCount", partition, (long long)base_offset);
    const int64_t last_offset = base_offset + last_offset_delta;
    const int codec = attrs & 7;
    const bool transactional = attrs & 0x10, control = attrs & 0x20;
    ++st.n_batches;
    while (!ps.aborted.empty() && ps.aborted.front().first <= last_offset) { ps.aborting.insert(ps.aborted.front().second); ps.aborted.erase(ps.aborted.begin()); }
    if (control) {
      // tiny and never compressed by the broker: read on the host (CRC included), it only steers the bookkeeping
      ++st.n_control_batches;
      if (sgr_crc32c(b + 21, total - 21) != be32(b + 17)) return dfail(g, SGR_ERR_INVALID, "partition %d offset %lld: CRC-32C mismatch in a control batch", partition, (long long)base_offset);
      if (codec == 0 && total >= kBatchHeader + 8) {
        // record: varint length, attributes, varlong ts delta, varint offset delta, varint key length, key = int16 version, int16 type
        const uint8_t* r = b + kBatchHeader; const uint8_t* end = b + total;
        auto skip_varint = [&]() { while (r < end && (*r & 0x80)) ++r; if (r < end) ++r; };
        skip_varint(); if (r < end) ++r; skip_varint(); skip_varint();
        int32_t kl = 0; { uint32_t v = 0; int sh = 0; while (r < end) { const uint8_t c = *r++; v |= (uint32_t)(c & 0x7f) << sh; if (!(c & 0x80)) break; sh += 7; } kl = (int32_t)(v >> 1) ^ -(int32_t)(v & 1); }
        if (kl >= 4 && r + 4 <= end && be16(r + 2) == 0) ps.aborting.erase(producer_id);   // ABORT marker ends the transaction
      }
    } else if (transactional && ps.aborting.count(producer_id)) {
      ++st.n_aborted_batches; st.n_aborted_records += (uint64_t)records_count;
    } else if (!(ps.seen && last_offset < ps.decoded_next)) {   // (a batch entirely below the position is all duplicates)
      if (codec != 0 && codec != 3) return dfail(g, SGR_ERR_UNSUPPORTED, "partition %d offset %lld: compression codec %d (none and lz4 are decoded)", partition, (long long)base_offset, codec);
      if (total < kBatchHeader) return dfail(g, SGR_ERR_INVALID, "partition %d offset %lld: batch shorter than its header", partition, (long long)base_offset);
      DgBatch d{};
      d.src_off = g->wire.used + pos; d.base_offset = base_offset; d.min_offset = ps.seen ? ps.decoded_next : INT64_MIN;
      d.total_len = (uint32_t)total; d.n_records = (uint32_t)records_count; d.codec = (uint32_t)codec; d.stored_crc = be32(b + 17);
      d.rec_base = (uint32_t)(g->n_record_slots + slots);
      slots += (uint64_t)records_count;
      if (codec == 3) st.n_compressed_bytes += total - kBatchHeader;
      add.push_back(d);
    } else {
      st.n_duplicates += (uint64_t)records_count;
    }
    if (!ps.seen || last_offset + 1 > ps.decoded_next) ps.decoded_next = last_offset + 1;
    ps.seen = true;
    pos += total;
  }
  st.n_bytes = pos; st.n_trailing_bytes = nbytes - pos;
  if (g->n_record_slots + slots >= (1ull << 32)) return dfail(g, SGR_ERR_CAPACITY, "more than 2^32 records in one poll");
  sgr_dingest::Sub sub{};
  sub.batch_begin = (uint32_t)g->batches.size(); sub.batch_end = sub.batch_begin + (uint32_t)add.size(); sub.nbytes = pos;
  if (g->subs.size() >= g->event_pool.size()) {
    cudaEvent_t ev;
    DG_TRY(g, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    g->event_pool.push_back(ev);
  }
  sub.copied = g->event_pool[g->subs.size()];
  if (g->timing_syncs && g->subs.empty()) {
    if (!g->tl_origin) DG_TRY(g, cudaEventCreate(&g->tl_origin));
    DG_TRY(g, cudaEventRecord(g->tl_origin, g->copy_stream));
  }
  if (pos) {
    if (g->wire.used + pos + 272 > g->wire.b.cap) DG_TRY(g, sync_all(g));   // the buffer moves: no copy in flight, no kernel reading it
    DG_TRY(g, g->wire.ensure(pos + 272, g->copy_stream));                     // (the input ring reads up to 256 bytes past a batch)
    DG_TRY(g, cudaMemcpyAsync((uint8_t*)g->wire.b.p + g->wire.used, buf, pos, cudaMemcpyHostToDevice, g->copy_stream));
    g->wire.used += (pos + 15) & ~15ull;
  }
  DG_TRY(g, cudaEventRecord(sub.copied, g->copy_stream));
  g->subs.push_back(sub);
  if (!add.empty()) {
    if (g->batches.n + add.size() > g->batches.cap) {   // the pinned array moves: nothing may still be copying from / into it
      DG_TRY(g, sync_all(g));
      if (!g->batches.reserve(g->batches.n + add.size())) return dfail(g, SGR_ERR_OOM, "page-locked descriptor array");
    }
    memcpy(g->batches.p + g->batches.n, add.data(), add.size() * sizeof(DgBatch));
    const DgBatch* src_desc = g->batches.p + g->batches.n;   // (the first generation uploads them from here right away)
    (void)src_desc;
    g->batches.n += add.size();
    if (!g->v1) {
      g->d_batches_used += add.size();
      if (g->d_batches_used - g->crc_launched >= g->group_batches) {
        const int32_t rc = launch_group(g, g->d_batches_used, g->n_record_slots + slots, sub.copied);
        if (rc) { discard_poll(g); return rc; }
      }
    } else {
      // descriptors go up right away; the CRC + lz4 size pass is launched once >= 32 k batches are waiting (one thread per batch:
      // a small launch takes as long as a large one, it is the serial walk of ONE batch) — it then runs while the host walks
      // the next fetches and the copy engine brings them in; sgr_dingest_fold launches the remainder
      if ((g->d_batches_used + add.size()) * sizeof(DgBatch) > g->d_batches.b.cap) DG_TRY(g, cudaStreamSynchronize(g->stream));
      g->d_batches.used = g->d_batches_used * sizeof(DgBatch);
      DG_TRY(g, g->d_batches.ensure(add.size() * sizeof(DgBatch) + 64, g->stream));
      DgBatch* db = (DgBatch*)g->d_batches.b.p + g->d_batches_used;
      DG_TRY(g, cudaMemcpyAsync(db, src_desc, add.size() * sizeof(DgBatch), cudaMemcpyHostToDevice, g->stream));
      g->d_batches_used += add.size();
      if (g->d_batches_used - g->crc_launched >= 32768) {
        DG_TRY(g, cudaStreamWaitEvent(g->stream, sub.copied, 0));
        DG_TRY(g, dg_launch_crc_size((const uint8_t*)g->wire.b.p, (DgBatch*)g->d_batches.b.p + g->crc_launched, (uint32_t)(g->d_batches_used - g->crc_launched), g->stream));
        g->crc_launched = g->d_batches_used;
      }
    }
  }
  g->n_record_slots += slots;
  g->staged[partition] = ps;
  sgr_ingest_stats& t = g->poll;
  t.n_bytes += st.n_bytes; t.n_batches += st.n_batches; t.n_control_batches += st.n_control_batches; t.n_aborted_batches += st.n_aborted_batches;
  t.n_aborted_records += st.n_aborted_records; t.n_duplicates += st.n_duplicates; t.n_compressed_bytes += st.n_compressed_bytes;
  t.n_trailing_bytes = st.n_trailing_bytes;
  if (stats) *stats = st;
  return SGR_OK;
}

int32_t sgr_dingest_fold(sgr_dingest* g, sgr_ingest_stats* stats) {
  if (!g) return SGR_ERR_INVALID;
  const uint32_t nb = (uint32_t)g->batches.size();
  const uint32_t nrec = (uint32_t)g->n_record_slots;
  sgr_ingest_stats st = g->poll;
  unsigned long long* h = (unsigned long long*)g->h_ctl;
  typedef std::chrono::steady_clock Clk;
  const Clk::time_point t_begin = Clk::now();
  Clk::time_point t_last = t_begin;
  auto lap = [&](int i) { const Clk::time_point now = Clk::now(); g->ms[i] += std::chrono::duration<float, std::milli>(now - t_last).count(); t_last = now; };
  memset(g->ms, 0, sizeof g->ms);
  if (nb) {
    DgParse p = parse_args(g);
    if (!g->v1) {
      // ---- chains: launch the remainder, wait for every group, bring the verdicts back
      { const int32_t rc = launch_group(g, nb, nrec, g->subs.back().copied); if (rc) { discard_poll(g); return rc; } }
      for (uint32_t k = 0; k < g->n_groups; ++k) DG_TRY(g, cudaStreamWaitEvent(g->stream, g->group_events[k], 0));
      DG_TRY(g, cudaMemcpyAsync(g->batches.data(), g->d_batches.b.p, (size_t)nb * sizeof(DgBatch), cudaMemcpyDeviceToHost, g->stream));
      DG_TRY(g, cudaMemcpyAsync(h, g->ctl.p, 128, cudaMemcpyDeviceToHost, g->stream));
      DG_TRY(g, cudaStreamSynchronize(g->stream));
      lap(0);
      if (g->timing_syncs && g->tl_origin) {
        for (uint32_t k = 0; k < g->n_groups; ++k) {
          float t[4] = {0, 0, 0, 0};
          for (int j = 0; j < 4; ++j) cudaEventElapsedTime(&t[j], g->tl_origin, g->tl_events[4 * (size_t)k + j]);
          fprintf(stderr, "[dingest] group %u: landed %.2f  crc+size %.2f  decode+walk %.2f  parse %.2f ms\n", k, t[0], t[1], t[2], t[3]);
        }
      }
      if (h[10]) {
        // the arena claims overflowed (the poll compresses better than 3x): lay the arena out exactly and decode + parse again.
        // Ids the first attempt interned stay (an id is an id); its records are overwritten slot for slot.
        // (exact sizes first: the claim mode never measured them)
        DG_TRY(g, dg_launch_crc_size_fast((const uint8_t*)g->wire.b.p, (DgBatch*)g->d_batches.b.p, nb, nullptr, g->stream));
        DG_TRY(g, cudaMemcpyAsync(g->batches.data(), g->d_batches.b.p, (size_t)nb * sizeof(DgBatch), cudaMemcpyDeviceToHost, g->stream));
        DG_TRY(g, cudaStreamSynchronize(g->stream));
        uint64_t need = 0;
        for (uint32_t i = 0; i < nb; ++i) {
          DgBatch& b = g->batches[i];
          if (b.err == DG_ARENA_FULL) b.err = DG_OK;
          if (b.err) { const int32_t rc = dfail(g, SGR_ERR_INVALID, "offset %lld: %s", (long long)b.base_offset, dg_err_text(b.err)); discard_poll(g); return rc; }
          b.err_record = 0;
          if (b.codec == 3) { b.arena_off = need; need += ((uint64_t)b.dsize + 15) & ~15ull; }
        }
        g->arena.used = 0;
        DG_TRY(g, g->arena.ensure(need + 512, g->stream));
        DG_TRY(g, set_arena_capacity(g));
        p = parse_args(g);
        h[2] = h[3] = h[4] = h[5] = h[6] = 0; h[8] = need; h[10] = 0;
        DG_TRY(g, cudaMemcpyAsync((unsigned long long*)g->ctl.p + 2, h + 2, 5 * 8, cudaMemcpyHostToDevice, g->stream));
        DG_TRY(g, cudaMemcpyAsync((unsigned long long*)g->ctl.p + 8, h + 8, 8, cudaMemcpyHostToDevice, g->stream));
        DG_TRY(g, cudaMemcpyAsync((unsigned long long*)g->ctl.p + 10, h + 10, 8, cudaMemcpyHostToDevice, g->stream));
        DG_TRY(g, cudaMemsetAsync(g->rec_batch.b.p, 0xff, (size_t)nrec * 4 + 4, g->stream));
        DG_TRY(g, cudaMemcpyAsync(g->d_batches.b.p, g->batches.data(), (size_t)nb * sizeof(DgBatch), cudaMemcpyHostToDevice, g->stream));
        DG_TRY(g, dg_launch_decode_walk_fast((const uint8_t*)g->wire.b.p, (uint8_t*)g->arena.b.p, (DgBatch*)g->d_batches.b.p, nb, 0, (uint32_t*)g->rec_off.b.p, (uint32_t*)g->rec_batch.b.p, nullptr, g->stream));
        p.n_batches = nb; p.rec_begin = 0; p.n_records = nrec;
        DG_TRY(g, dg_launch_parse(p, g->stream));
        DG_TRY(g, cudaMemcpyAsync(g->batches.data(), g->d_batches.b.p, (size_t)nb * sizeof(DgBatch), cudaMemcpyDeviceToHost, g->stream));
        DG_TRY(g, cudaMemcpyAsync(h, g->ctl.p, 128, cudaMemcpyDeviceToHost, g->stream));
        DG_TRY(g, cudaStreamSynchronize(g->stream));
        lap(1);
      }
      for (uint32_t i = 0; i < nb; ++i) if (g->batches[i].codec == 3 && !g->batches[i].err) st.n_decompressed_bytes += g->batches[i].dsize;
    } else {
      DG_TRY(g, g->rec_off.b.reserve((size_t)nrec * 4 + 64));
      DG_TRY(g, g->rec_batch.b.reserve((size_t)nrec * 4 + 64));
      DG_TRY(g, g->out.b.reserve((size_t)nrec * 64 + 64));
      p = parse_args(g);
      DG_TRY(g, cudaMemsetAsync(g->rec_batch.b.p, 0xff, (size_t)nrec * 4 + 4, g->stream));
      p.n_batches = nb;
      // ---- the CRC + lz4 size pass: most of it was launched by sgr_dingest_submit behind the copies; the rest now
      if (g->crc_launched < nb) {
        DG_TRY(g, cudaStreamWaitEvent(g->stream, g->subs.back().copied, 0));
        DG_TRY(g, dg_launch_crc_size((const uint8_t*)g->wire.b.p, (DgBatch*)g->d_batches.b.p + g->crc_launched, (uint32_t)(nb - g->crc_launched), g->stream));
        g->crc_launched = nb;
      }
      DG_TRY(g, cudaMemcpyAsync(g->batches.data(), g->d_batches.b.p, (size_t)nb * sizeof(DgBatch), cudaMemcpyDeviceToHost, g->stream));
      DG_TRY(g, cudaStreamSynchronize(g->stream));
      lap(0);
      uint64_t arena_need = 0;
      for (uint32_t i = 0; i < nb; ++i) {
        DgBatch& b = g->batches[i];
        if (b.err) { const int32_t rc = dfail(g, SGR_ERR_INVALID, "offset %lld: %s", (long long)b.base_offset, dg_err_text(b.err)); discard_poll(g); return rc; }
        if (b.codec == 3) { b.arena_off = arena_need; arena_need += ((uint64_t)b.dsize + 15) & ~15ull; st.n_decompressed_bytes += b.dsize; }
      }
      g->arena.used = 0;
      DG_TRY(g, g->arena.ensure(arena_need + 64, g->stream));
      DG_TRY(g, cudaMemcpyAsync(g->d_batches.b.p, g->batches.data(), (size_t)nb * sizeof(DgBatch), cudaMemcpyHostToDevice, g->stream));
      DG_TRY(g, dg_launch_decode_walk((const uint8_t*)g->wire.b.p, (uint8_t*)g->arena.b.p, (DgBatch*)g->d_batches.b.p, nb, 0, (uint32_t*)g->rec_off.b.p, (uint32_t*)g->rec_batch.b.p, g->stream));
      if (g->timing_syncs) { DG_TRY(g, cudaStreamSynchronize(g->stream)); lap(1); }
      p.wire = (const uint8_t*)g->wire.b.p; p.arena = (const uint8_t*)g->arena.b.p; p.rec_begin = 0; p.n_records = nrec;
      DG_TRY(g, dg_launch_parse(p, g->stream));
      DG_TRY(g, cudaMemcpyAsync(g->batches.data(), g->d_batches.b.p, (size_t)nb * sizeof(DgBatch), cudaMemcpyDeviceToHost, g->stream));
      DG_TRY(g, cudaMemcpyAsync(h, g->ctl.p, 128, cudaMemcpyDeviceToHost, g->stream));
      DG_TRY(g, cudaStreamSynchronize(g->stream));
      lap(2);
    }
    for (uint32_t i = 0; i < nb; ++i)
      if (g->batches[i].err) {
        const int32_t rc = dfail(g, SGR_ERR_INVALID, "offset %lld, record %u: %s", (long long)g->batches[i].base_offset, g->batches[i].err_record, dg_err_text(g->batches[i].err));
        // ids interned by this failed poll stay in the dictionary (harmless: an id is an id); the records are dropped
        discard_poll(g); return rc;
      }
    if (h[5]) {
      const int32_t rc = dfail(g, SGR_ERR_CAPACITY, "device id dictionary full (%llu ids / %llu id bytes allowed): create the device ingest with larger bounds", (unsigned long long)g->max_keys, (unsigned long long)g->arena_cap);
      discard_poll(g); return rc;
    }
    st.n_markers = h[2]; st.n_null_values = h[3]; st.n_duplicates += h[4]; st.n_records = h[6]; st.n_new_keys = h[0] - g->keys_reported;   // (ids a failed poll interned are counted by the next good one)
    // ---- grow the table for the new ids, hand their names to the engine's key table, fold
    const uint64_t n_keys = h[0];
    void* d_states = nullptr; uint64_t n_agg = 0; uint32_t sb = 0;
    const int32_t have = sgr_states_device(g->eng, &d_states, &n_agg, &sb);
    if (have != SGR_OK || n_keys > n_agg) {
      uint64_t cap = have == SGR_OK ? n_agg : 0;
      if (cap < 1024) cap = 1024;
      while (cap < n_keys) cap *= 2;
      if (cap > g->max_keys && g->max_keys >= n_keys) cap = g->max_keys;
      int32_t rc = sgr_grow_states(g->eng, cap);
      if (rc) { dfail(g, rc, "engine: %s", sgr_last_error(g->eng)); discard_poll(g); return rc; }
    }
    lap(4);
    // The new ids, gathered on the device into dense-index order, come down in two copies queued BEHIND nothing the fold needs
    // and IN FRONT of the fold's kernels; a helper thread hands them to the engine's key table while this thread runs the fold.
    std::thread appender;
    int32_t rc_append = SGR_OK;
    if (n_keys > g->keys_on_host) {
      const uint64_t add = n_keys - g->keys_on_host;
      const uint64_t id_bytes_max = h[1] - g->id_bytes_on_host;   // (an upper bound: arena entries are padded to 8 bytes)
      DG_TRY(g, g->key_offs_dev.reserve((add + 2) * 4 + (2 * (add / 4096 + 2) + 4 * 4096) * 4));
      DG_TRY(g, g->key_bytes_dev.reserve(id_bytes_max + 64));
      uint32_t* d_offs = (uint32_t*)g->key_offs_dev.p;
      uint32_t* d_tmp = d_offs + add + 2;
      DG_TRY(g, dg_gather_keys(p.dict, g->keys_on_host, (uint32_t)add, d_offs, (uint8_t*)g->key_bytes_dev.p, d_tmp, g->stream));
      if (g->h_keys_cap < (add + 2) * 4 + id_bytes_max + 64) {
        if (g->h_keys) cudaFreeHost(g->h_keys);
        g->h_keys = nullptr; g->h_keys_cap = 0;
        const uint64_t want = 2 * ((add + 2) * 4 + id_bytes_max + 64);
        DG_TRY(g, cudaHostAlloc(&g->h_keys, want, cudaHostAllocDefault));
        g->h_keys_cap = want;
      }
      uint32_t* h_offs = (uint32_t*)g->h_keys;
      uint8_t* h_bytes = (uint8_t*)g->h_keys + (add + 2) * 4;
      DG_TRY(g, cudaMemcpyAsync(h_offs, d_offs, (add + 1) * 4, cudaMemcpyDeviceToHost, g->stream));
      if (id_bytes_max) DG_TRY(g, cudaMemcpyAsync(h_bytes, g->key_bytes_dev.p, id_bytes_max, cudaMemcpyDeviceToHost, g->stream));
      if (!g->keys_landed) DG_TRY(g, cudaEventCreateWithFlags(&g->keys_landed, cudaEventDisableTiming));
      DG_TRY(g, cudaEventRecord(g->keys_landed, g->stream));
      int dev = 0;
      cudaGetDevice(&dev);
      const void* owner = (const char*)g + g->generation;
      appender = std::thread([g, dev, owner, h_offs, h_bytes, add, &rc_append]() {
        cudaSetDevice(dev);
        if (cudaEventSynchronize(g->keys_landed) != cudaSuccess) { rc_append = SGR_ERR_CUDA; return; }
        rc_append = sgr_append_keys(g->eng, owner, h_bytes, h_offs, add);
      });
    }
    lap(3);
    int32_t rc_fold = SGR_OK;
    if (nrec) rc_fold = sgr_fold_incremental_device(g->eng, g->out.b.p, nrec);
    if (appender.joinable()) appender.join();
    // the engine's key table holds these ids now, whatever the fold returned: the next poll appends only what follows them
    if (rc_append == SGR_OK) { g->keys_on_host = n_keys; g->id_bytes_on_host = h[1]; }
    if (rc_fold) { dfail(g, rc_fold, "engine: %s", sgr_last_error(g->eng)); discard_poll(g); return rc_fold; }
    if (rc_append) { dfail(g, rc_append, "engine: %s", sgr_last_error(g->eng)); discard_poll(g); return rc_append; }
    g->keys_reported = n_keys;
  }
  lap(4);
  g->ms[5] = std::chrono::duration<float, std::milli>(Clk::now() - t_begin).count();
  // ---- commit: the staged positions become the live ones and everything decoded is folded
  for (auto& kv : g->staged) { kv.second.folded_next = kv.second.decoded_next; }
  g->parts = g->staged;
  if (nb) DG_TRY(g, reset_poll_counters(g));
  clear_poll(g);
  sgr_ingest_stats& t = g->total;
  t.n_bytes += st.n_bytes; t.n_batches += st.n_batches; t.n_records += st.n_records; t.n_markers += st.n_markers; t.n_null_values += st.n_null_values;
  t.n_control_batches += st.n_control_batches; t.n_aborted_batches += st.n_aborted_batches; t.n_aborted_records += st.n_aborted_records;
  t.n_duplicates += st.n_duplicates; t.n_new_keys += st.n_new_keys; t.n_compressed_bytes += st.n_compressed_bytes; t.n_decompressed_bytes += st.n_decompressed_bytes;
  if (stats) *stats = st;
  return SGR_OK;
}

int32_t sgr_dingest_reset(sgr_dingest* g) {
  if (!g) return SGR_ERR_INVALID;
  discard_poll(g);
  g->parts.clear(); g->staged.clear(); g->total = sgr_ingest_stats{}; g->keys_on_host = 0; g->id_bytes_on_host = 0; g->keys_reported = 0; ++g->generation;
  DG_TRY(g, cudaMemsetAsync(g->tags.p, 0, g->slots * 8, g->stream));
  DG_TRY(g, cudaMemsetAsync(g->slot_idx.p, 0, g->slots * 4, g->stream));
  DG_TRY(g, cudaMemsetAsync(g->ctl.p, 0, 9 * 8, g->stream));                                  // ([9], the arena's capacity, stays)
  DG_TRY(g, cudaMemsetAsync((unsigned long long*)g->ctl.p + 10, 0, 8, g->stream));
  DG_TRY(g, cudaStreamSynchronize(g->stream));                                                   // the group streams must see it
  return SGR_OK;
}

int32_t sgr_dingest_offsets(sgr_dingest* g, int32_t partition, int64_t* decoded_next, int64_t* folded_next) {
  if (!g) return SGR_ERR_INVALID;
  auto it = g->parts.find(partition);
  if (decoded_next) *decoded_next = it == g->parts.end() ? 0 : it->second.decoded_next;
  if (folded_next) *folded_next = it == g->parts.end() ? 0 : it->second.folded_next;
  return SGR_OK;
}

int32_t sgr_dingest_last_timing(sgr_dingest* g, float* ms8) {
  if (!g || !ms8) return SGR_ERR_INVALID;
  memcpy(ms8, g->ms, sizeof g->ms);
  return SGR_OK;
}

int32_t sgr_dingest_get_stats(sgr_dingest* g, sgr_ingest_stats* out) {
  if (!g || !out) return SGR_ERR_INVALID;
  *out = g->total;
  return SGR_OK;
}

}  // extern "C"
