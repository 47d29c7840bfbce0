// engine.cu — the C ABI of include/sgr.h over the CUDA kernels (host side of the boundary).
//
// No CPU fallback lives here: every compute entry point launches a kernel on the engine's
// device or fails with a status code. Nothing in this file includes or links oracle/.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/sgr.h"
#include "bulk_fold.cuh"
#include "devbuf.h"
#include "dist.cuh"
#include "fold_kernels.cuh"
#include "fold_rows.cuh"
#include "group_kernels.cuh"
#include "incremental.cuh"
#include "keytable.h"
#include "route_push.cuh"

using namespace sgr;

namespace {
thread_local std::string g_create_error;
thread_local std::string t_last_error;
thread_local const sgr_engine* t_last_engine = nullptr;

// host snapshot of the state table that sgr_get reads (published after a fold)
struct Snapshot {
  std::vector<uint8_t> states;
  uint64_t n_agg = 0;
  uint32_t state_bytes = 0;
};
}  // namespace

struct sgr_engine {
  int device = 0;
  int num_sms = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;

  bool has_program = false;
  sgr_fold_program program{};
  DevProgram dprog{};

  // CSR event log: owned buffers or borrowed pointers
  DevBuf own_events, own_offsets, own_rec_offsets;
  const uint64_t* d_rec_offsets = nullptr;   // record directory (variable records), or null
  uint64_t n_rec = 0;
  const uint8_t* d_events = nullptr;
  const uint64_t* d_offsets = nullptr;
  uint64_t event_bytes = 0;
  uint64_t n_agg = 0;
  bool loaded = false;
  uint32_t max_record_bytes = 64;

  DevBuf states;        // n_agg * state_bytes, live table
  bool states_valid = false;  // holds prior states (set_initial_states or a previous fold)
  bool states_invalidated = false;  // a failed in-place fold left the table half-applied: nothing may fold onto it (or grow it)
                                    // until set_initial_states, a full fold or fold_unsorted replaces it
  uint64_t states_n = 0;
  DevBuf counters;      // 8 x u64
  GroupScratch group;   // K5 scratch
  DevBuf inc_records, inc_offsets, inc_ids, inc_prev_ids;  // K6
  uint64_t inc_prev_n = 0;
  // sort-free K6 (incremental.cu)
  DevBuf inc_scratch, inc_touched[2], inc_err_ids, inc_counters;
  uint64_t inc_scratch_slots = 0;
  int inc_flip = 0;
  bool inc_atomic_prev_valid = false;   // inc_touched[inc_flip^1] / its counter describe the previous batch
  uint32_t inc_prev_upper = 0;

  // record-parallel path (fold_rows.cu)
  bool row_ok = false;            // program is inside the transformer algebra
  RowProgram row_prog{};
  int row_max_grid = 0;
  int run_max_grid = 0, run_max_grid_variant = -1;
  int64_t opt_run_variant = 0;
  DevBuf part_flags, part_data, redo_ids;
  DevBuf run_counters;            // 2 x 8 u64, ping-pong; the runs kernel zeroes the other block itself
  int run_counter_idx = 0;
  const void* pending_counters = nullptr;
  uint32_t epoch = 0;
  size_t part_flags_cap_seen = 0;
  bool offsets_aligned64 = false; // every segment offset == log_begin (mod 64)
  uint64_t log_begin = 0, log_end = 0, max_seg_bytes = 0;
  bool fold_pending = false;      // a fold was enqueued and not yet finished
  bool pending_rows_v1 = false, pending_var = false;
  bool pending_used_rows = false, pending_prior = false, pending_timed_group = false;
  uint64_t pending_n_seg = 0, pending_event_bytes = 0;
  const uint8_t* pending_events = nullptr; const uint64_t* pending_offsets = nullptr; const uint32_t* pending_ids = nullptr;
  cudaEvent_t ev2 = nullptr, ev3 = nullptr;

  int64_t opt_kernel = 0;         // 0 auto (runs if the program allows), 1 lane-sequential TMA kernel (fold_kernels.cu),
                                  // 2 force runs (fold_runs.cu), 3 record-per-lane rows (fold_rows.cu)
  int64_t opt_variant = -1;
  int64_t opt_long_threshold = 0;
  int64_t opt_var_stages = 1;     // measured: 1 stage x 16 warps/SM (5.0 TB/s) beats 2 x 9 (4.4) and 3 x 6 (3.2) on configs[3]
  int64_t opt_var_stage_bytes = 12288;  // smem bytes staged per 32-record step of the variable-record kernel
  int64_t opt_replay_budget = 1ll << 24;  // K6: in-kernel replay of throwing slots only while n_err * n stays below this
                                          // (measured ~15 ps per slot-record; beyond it one group-by of the batch is cheaper)
  int64_t opt_force_route = 0;    // profiling aid: run K4 even on a single rank
  int64_t opt_incremental = 0;    // 0 auto (sort-free K6 when the program allows), 1 force the sort-based path
  int64_t opt_max_record_bytes = 528;

  // sort-free fold of large arrival-order logs (bulk_fold.cu)
  bool bulk_ok = false;
  BulkLayout bulk_lay{};
  DevBuf bulk_scratch, bulk_err_ids, bulk_counters, hash_out;
  uint64_t bulk_scratch_slots = 0;
  int64_t opt_bulk = 1;           // 0: keep arrival-order logs on the single-launch micro-batch kernel (incremental.cu)
  int64_t opt_push_ordered = 0;   // 1: positions inside the exchange regions follow the log from the first attempt (look-back)
  int64_t opt_push_chunks = 16;   // chunks of the pipelined route + exchange + fold (route_push.cu); the same on every rank

  sgr_stats stats{};

  DistState* dist = nullptr;
  sgr_dist_stats dstats{};

  std::shared_ptr<const KeyTable> keys;   // swapped atomically: sgr_get readers never see a table being rebuilt
  // ids handed over by sgr_fold_ingested: appended per poll (the dictionary is append-only), hashed lazily by the first
  // sgr_get that follows — a restore polls thousands of times before anybody reads
  std::mutex keys_mu;
  std::vector<uint8_t> ing_key_bytes;
  std::vector<uint32_t> ing_key_offs;
  const void* ing_keys_from = nullptr;      // whose dictionary the appended ids mirror (an sgr_ingest or an sgr_dingest)
  std::atomic<bool> keys_stale{false};
  // Every call that changes the engine (loads, folds, table growth) and the snapshot refresh of a reader hold op_mu:
  // a reader never sees a table being freed or swapped, and a snapshot is only marked clean for the generation it copied.
  std::recursive_mutex op_mu;
  std::atomic<uint64_t> generation{0};
  std::shared_ptr<Snapshot> snapshot;
  std::atomic<bool> snapshot_dirty{true};
};

namespace {

// serialises engine mutation against the snapshot refresh of concurrent readers (ADVICE r1: reader threads touched a table
// the stream thread was freeing); recursive because public entry points call each other (sgr_fold_ingested)
struct OpLock {
  std::unique_lock<std::recursive_mutex> l;
  explicit OpLock(sgr_engine* e) { if (e) l = std::unique_lock<std::recursive_mutex>(e->op_mu); }
};

int32_t fail(sgr_engine* e, int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  // errno-style: the message belongs to the calling thread (sgr_get runs on a 32-thread pool in the reference; two failing
  // readers must not race on one string). sgr_last_error(e) answers for the last failure of THIS thread on e.
  if (e) { t_last_error = buf; t_last_engine = e; } else g_create_error = buf;
  return code;
}
#define CUDA_TRY(e, call)                                                                         \
  do {                                                                                            \
    cudaError_t _err = (call);                                                                    \
    if (_err != cudaSuccess)                                                                      \
      return fail((e), _err == cudaErrorMemoryAllocation ? SGR_ERR_OOM : SGR_ERR_CUDA, "%s: %s", #call, \
                  cudaGetErrorString(_err));                                                      \
  } while (0)

int32_t use_device(sgr_engine* e) {
  CUDA_TRY(e, cudaSetDevice(e->device));
  return SGR_OK;
}

int32_t compile_program(sgr_engine* e, const sgr_fold_program* p, DevProgram* d) {
  if (p->state_bytes < 16 || p->state_bytes > SGR_MAX_STATE_BYTES || p->state_bytes % 16)
    return fail(e, SGR_ERR_INVALID, "state_bytes %u must be a multiple of 16 in [16,%u]", p->state_bytes, SGR_MAX_STATE_BYTES);
  if (p->record_kind != SGR_REC_FIXED64 && p->record_kind != SGR_REC_VAR16)
    return fail(e, SGR_ERR_INVALID, "unknown record_kind %u", p->record_kind);
  if (p->n_types == 0 || p->n_types > SGR_MAX_TYPES) return fail(e, SGR_ERR_INVALID, "n_types %u out of range", p->n_types);
  if (p->n_f64_fields > 8) return fail(e, SGR_ERR_INVALID, "n_f64_fields %u > 8", p->n_f64_fields);
  memset(d, 0, sizeof *d);
  d->state_words = p->state_bytes / 4;
  d->user_words = d->state_words - 2;
  d->record_kind = p->record_kind;
  d->n_types = p->n_types;
  d->n_f64 = p->n_f64_fields;
  const uint32_t user_bytes = p->state_bytes - 8;
  for (uint32_t f = 0; f < p->n_f64_fields; ++f) {
    if (p->f64_field_off[f] % 4 || p->f64_field_off[f] + 8u > user_bytes)
      return fail(e, SGR_ERR_INVALID, "f64 field %u at offset %u outside the program area", f, p->f64_field_off[f]);
    d->f64_word[f] = p->f64_field_off[f] / 4;
  }
  const uint32_t max_src = p->record_kind == SGR_REC_FIXED64 ? 64u : 0xfffcu;
  for (uint32_t t = 0; t < p->n_types; ++t) {
    const sgr_rule& r = p->rules[t];
    if (r.exists_rule > SGR_THROW) return fail(e, SGR_ERR_INVALID, "rule %u: bad exists_rule %u", t, r.exists_rule);
    if (r.n_ops > SGR_MAX_OPS) return fail(e, SGR_ERR_INVALID, "rule %u: n_ops %u > %u", t, r.n_ops, SGR_MAX_OPS);
    DevRule& dr = d->rules[t];
    dr.exists_rule = r.exists_rule;
    dr.n_ops = (r.exists_rule == SGR_TOMBSTONE || r.exists_rule == SGR_THROW) ? 0 : r.n_ops;
    dr.min_len = 16;
    for (uint32_t i = 0; i < dr.n_ops; ++i) {
      const sgr_op& o = r.ops[i];
      if (o.opcode > SGR_OP_SUB_I64) return fail(e, SGR_ERR_UNSUPPORTED, "rule %u op %u: opcode %u", t, i, o.opcode);
      uint32_t len = o.len;
      if (o.opcode == SGR_OP_ADD_I32 || o.opcode == SGR_OP_SUB_I32) { if (len != 4) return fail(e, SGR_ERR_INVALID, "rule %u op %u: i32 op needs len 4", t, i); }
      else if (o.opcode == SGR_OP_ADD_I64 || o.opcode == SGR_OP_SUB_I64) { if (len != 8) return fail(e, SGR_ERR_INVALID, "rule %u op %u: i64 op needs len 8", t, i); }
      if (len == 0 || len % 4 || o.dst_off % 4 || o.src_off % 4)
        return fail(e, SGR_ERR_INVALID, "rule %u op %u: offsets and length must be non-zero multiples of 4", t, i);
      if (o.dst_off + len > user_bytes) return fail(e, SGR_ERR_INVALID, "rule %u op %u: writes past the program area", t, i);
      if (o.src_off + len > max_src) return fail(e, SGR_ERR_INVALID, "rule %u op %u: reads past the record", t, i);
      if (o.src_off + len > dr.min_len) dr.min_len = o.src_off + len;
      dr.ops[i] = pack_op(o.opcode, len / 4, o.dst_off / 4, o.src_off / 4);
    }
  }
  return SGR_OK;
}

int32_t finish_fold(sgr_engine* e);

void mark_dirty(sgr_engine* e) { e->generation.fetch_add(1, std::memory_order_acq_rel); e->snapshot_dirty.store(true, std::memory_order_release); }

int32_t ensure_states(sgr_engine* e, uint64_t n_agg) {
  const size_t need = (size_t)n_agg * e->program.state_bytes;
  if (e->states_n != n_agg || e->states.cap < need) {
    CUDA_TRY(e, e->states.reserve(need));
    e->states_n = n_agg;
    e->states_valid = false;
  }
  return SGR_OK;
}

// publish a host snapshot of the live state table for sgr_get
int32_t refresh_snapshot(sgr_engine* e, std::shared_ptr<Snapshot>* out) {
  // readers (sgr_get on the store's 32-thread pool) and the stream thread's loads/folds exclude each other here
  std::lock_guard<std::recursive_mutex> g(e->op_mu);
  if (!e->snapshot_dirty.load(std::memory_order_acquire) && e->snapshot) { *out = e->snapshot; return SGR_OK; }
  const uint64_t gen = e->generation.load(std::memory_order_acquire);
  if (!e->states_valid) return fail(e, SGR_ERR_STATE, "state store is not readable: no fold has completed");
  int32_t rc = use_device(e); if (rc) return rc;
  rc = finish_fold(e); if (rc) return rc;
  auto s = std::make_shared<Snapshot>();
  s->n_agg = e->states_n; s->state_bytes = e->program.state_bytes;
  s->states.resize((size_t)s->n_agg * s->state_bytes);
  CUDA_TRY(e, cudaMemcpyAsync(s->states.data(), e->states.p, s->states.size(), cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  std::atomic_store(&e->snapshot, s);
  // clean only for the generation that was copied (op_mu makes a concurrent bump impossible today; the check keeps it so)
  if (e->generation.load(std::memory_order_acquire) == gen) e->snapshot_dirty.store(false, std::memory_order_release);
  *out = s;
  return SGR_OK;
}

constexpr uint64_t kRedoCap = 1u << 20;

// Enqueue one fold on the engine's stream (no host synchronisation).
int32_t enqueue_fold(sgr_engine* e, const uint8_t* d_events, const uint64_t* d_offsets, const uint32_t* d_ids,
                     uint64_t n_seg, bool use_prior, uint64_t event_bytes, bool aligned64, uint64_t log_begin, uint64_t log_end) {
  const uint8_t* states_in = use_prior ? (const uint8_t*)e->states.p : nullptr;
  // 64-byte states: the transformer scan moves 16 registers per lane per step and the lane-per-aggregate TMA kernel is
  // faster on balanced logs (measured 2.47 vs 1.76 TB/s on BankAccount); the record-parallel kernel is taken when a
  // long segment would otherwise serialise one lane
  const bool wide_balanced = e->row_prog.user_words == 14 && e->opt_kernel == 0 && d_offsets == e->d_offsets && e->max_seg_bytes <= (256u << 10);
  bool use_rows = e->row_ok && !wide_balanced && e->program.record_kind == SGR_REC_FIXED64 && aligned64 && e->opt_kernel != 1 && n_seg < (1ull << 32) && n_seg > 0;
  if ((e->opt_kernel == 2 || e->opt_kernel == 3) && !use_rows && n_seg > 0)
    return fail(e, SGR_ERR_UNSUPPORTED, "record-parallel kernel cannot take this program/log");
  if (use_rows && e->opt_kernel == 3 && (e->row_prog.user_words != 2 || e->row_prog.cls != 0 || e->row_prog.n_slots > 6 || e->row_prog.f64_mask))
    return fail(e, SGR_ERR_UNSUPPORTED, "the record-per-lane kernel takes 16-byte class-0 programs only");
  const bool runs = use_rows && e->opt_kernel != 3;
  unsigned long long* counters = (unsigned long long*)e->counters.p;
  if (runs) {
    if (!e->run_counters.p) {
      CUDA_TRY(e, e->run_counters.reserve(256));
      CUDA_TRY(e, cudaMemsetAsync(e->run_counters.p, 0, 256, e->stream));
    }
    counters = (unsigned long long*)e->run_counters.p + 8 * e->run_counter_idx;
  } else {
    CUDA_TRY(e, cudaMemsetAsync(e->counters.p, 0, 64, e->stream));
  }
  e->pending_counters = counters;
  e->pending_var = false;
  CUDA_TRY(e, cudaEventRecord(e->ev0, e->stream));
  uint32_t launches = 0;
  const bool use_var = e->row_ok && e->row_prog.user_words == 2 && e->row_prog.cls == 0 && e->program.record_kind == SGR_REC_VAR16 && e->d_rec_offsets && d_offsets == e->d_offsets && !use_prior &&
                       !d_ids && e->opt_kernel != 1 && n_seg > 0 && n_seg < (1ull << 32) && e->n_rec > 0;
  if (use_var) {
    int threads = 0; size_t smem = 0; uint32_t stage = 0;
    const int max_grid = vruns_config(e->num_sms, e->max_record_bytes, (uint32_t)e->opt_var_stage_bytes, (int)e->opt_var_stages, &threads, &smem, &stage);
    if (max_grid > 0) {
      const uint64_t n_warps_max = (uint64_t)max_grid * (threads / 32);
      CUDA_TRY(e, e->part_flags.reserve(n_warps_max * 4 + 256));
      CUDA_TRY(e, e->part_data.reserve(n_warps_max * 8 * 4 + 256));
      CUDA_TRY(e, e->redo_ids.reserve(kRedoCap * 4));
      if (e->epoch == 0 || e->part_flags_cap_seen != e->part_flags.cap) {
        CUDA_TRY(e, cudaMemsetAsync(e->part_flags.p, 0, e->part_flags.cap, e->stream));
        e->part_flags_cap_seen = e->part_flags.cap;
      }
      ++e->epoch;
      if (e->epoch == 0) { CUDA_TRY(e, cudaMemsetAsync(e->part_flags.p, 0, e->part_flags.cap, e->stream)); e->epoch = 1; }
      CUDA_TRY(e, cudaMemsetAsync(e->states.p, 0, (size_t)n_seg * e->program.state_bytes, e->stream));
      VarArgs v{};
      v.events = d_events; v.rec_offsets = e->d_rec_offsets; v.n_rec = e->n_rec; v.seg_offsets = d_offsets; v.n_seg = n_seg;
      v.states_out = (uint8_t*)e->states.p; v.counters = counters; v.redo_ids = (uint32_t*)e->redo_ids.p; v.redo_cap = kRedoCap;
      v.part_flags = (uint32_t*)e->part_flags.p; v.part_data = (uint32_t*)e->part_data.p; v.epoch = e->epoch; v.stage_bytes = stage;
      const uint64_t steps = (e->n_rec + 31) / 32;
      uint64_t want = (steps + (threads / 32) - 1) / (threads / 32);
      const int grid = (int)(want < (uint64_t)max_grid ? want : (uint64_t)max_grid);
      cudaError_t le = launch_fold_vruns(v, e->row_prog, (int)e->opt_var_stages, grid, threads, smem, e->stream);
      if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "fold_vruns launch: %s", cudaGetErrorString(le));
      // exact replay of throwing / malformed segments (count lives on the device)
      FoldArgs a{};
      a.events = d_events; a.seg_offsets = d_offsets; a.n_seg = kRedoCap; a.seg_list = (const uint32_t*)e->redo_ids.p;
      a.n_seg_dev = counters + 3; a.states_in = nullptr; a.states_out = (uint8_t*)e->states.p; a.counters = counters;
      FoldLaunchInfo info{};
      le = launch_fold_stream(a, e->dprog, -1, 8, e->max_record_bytes, e->stream, &info);
      if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "replay launch: %s", cudaGetErrorString(le));
      launches = 2;
      e->pending_var = true;
    }
  }
  if (n_seg && !e->pending_var) {
    FoldArgs a{};
    a.events = d_events; a.seg_offsets = d_offsets; a.seg_ids = d_ids; a.n_seg = n_seg;
    a.states_in = states_in; a.states_out = (uint8_t*)e->states.p;
    a.counters = counters;
    a.long_threshold = (uint64_t)e->opt_long_threshold;
    FoldLaunchInfo info{};
    if (use_rows) {
      const bool v1 = e->opt_kernel == 3;
      const int rv = (int)e->opt_run_variant;
      if (v1 && !e->row_max_grid) e->row_max_grid = row_kernel_max_grid(e->num_sms, e->row_prog);
      if (!v1 && e->run_max_grid_variant != rv) { e->run_max_grid = run_kernel_max_grid(e->num_sms, rv, e->row_prog); e->run_max_grid_variant = rv; }
      const int max_grid = v1 ? e->row_max_grid : e->run_max_grid;
      const int wpc = v1 ? kRowThreads / 32 : run_warps_per_cta();
      const uint64_t step_bytes = v1 ? 2048 : (uint64_t)run_variant_step_bytes(rv, e->row_prog);
      const uint64_t n_warps_max = (uint64_t)max_grid * wpc;
      CUDA_TRY(e, e->part_flags.reserve(n_warps_max * 4 + 256));
      CUDA_TRY(e, e->part_data.reserve(n_warps_max * (e->row_prog.user_words + 2) * 4 + 256));
      CUDA_TRY(e, e->redo_ids.reserve(kRedoCap * 4));
      if (e->epoch == 0 || e->part_flags_cap_seen != e->part_flags.cap) {
        CUDA_TRY(e, cudaMemsetAsync(e->part_flags.p, 0, e->part_flags.cap, e->stream));
        e->part_flags_cap_seen = e->part_flags.cap;
      }
      ++e->epoch;
      if (e->epoch == 0) { CUDA_TRY(e, cudaMemsetAsync(e->part_flags.p, 0, e->part_flags.cap, e->stream)); e->epoch = 1; }
      RowArgs r{};
      r.events = d_events; r.seg_offsets = d_offsets; r.seg_ids = d_ids; r.n_seg = n_seg;
      r.log_begin = log_begin; r.log_end = log_end;
      r.states_in = states_in; r.states_out = (uint8_t*)e->states.p;
      r.counters = counters;
      r.counters_next = runs ? (unsigned long long*)e->run_counters.p + 8 * (e->run_counter_idx ^ 1) : nullptr;
      r.redo_ids = (uint32_t*)e->redo_ids.p; r.redo_cap = kRedoCap;
      r.part_flags = (uint32_t*)e->part_flags.p; r.part_data = (uint32_t*)e->part_data.p; r.epoch = e->epoch;
      const uint64_t steps = (log_end - log_begin + step_bytes - 1) / step_bytes;
      uint64_t want = (steps + wpc - 1) / wpc;
      if (want == 0) want = 1;  // all segments empty: one CTA still writes every (None) state
      const int grid = (int)(want < (uint64_t)max_grid ? want : (uint64_t)max_grid);
      cudaError_t le = v1 ? launch_fold_rows(r, e->row_prog, grid, e->stream) : launch_fold_runs(r, e->row_prog, rv, grid, e->stream);
      if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "fold launch: %s", cudaGetErrorString(le));
      if (runs) {
        e->run_counter_idx ^= 1;  // the kernel replays throwing segments itself and cleans the other block
        launches = 1;
      } else {
        // rows kernel: exact replay of the segments whose handler threw (count lives on the device)
        a.seg_list = (const uint32_t*)e->redo_ids.p;
        a.n_seg = kRedoCap;
        a.n_seg_dev = counters + 3;
        a.long_threshold = 0;
        le = launch_fold_stream(a, e->dprog, -1, 8, e->max_record_bytes, e->stream, &info);
        if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "replay launch: %s", cudaGetErrorString(le));
        launches = 2;
      }
    } else {
      cudaError_t le = launch_fold_stream(a, e->dprog, (int)e->opt_variant, e->num_sms, e->max_record_bytes, e->stream, &info);
      if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "fold launch: %s", cudaGetErrorString(le));
      launches = 1;
    }
  }
  CUDA_TRY(e, cudaEventRecord(e->ev1, e->stream));
  e->fold_pending = true; e->pending_used_rows = use_rows; e->pending_rows_v1 = use_rows && e->opt_kernel == 3; e->pending_prior = use_prior;
  e->pending_n_seg = n_seg; e->pending_event_bytes = event_bytes;
  e->pending_events = d_events; e->pending_offsets = d_offsets; e->pending_ids = d_ids;
  e->stats.fold_launches = launches;
  return SGR_OK;
}

// Wait for the enqueued fold and collect its statistics.
int32_t finish_fold(sgr_engine* e) {
  if (!e->fold_pending) return SGR_OK;
  e->fold_pending = false;
  unsigned long long h[8];
  CUDA_TRY(e, cudaMemcpyAsync(h, e->pending_counters, 64, cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_fold, e->ev0, e->ev1));
  if (e->pending_var && (h[7] != 0 || h[3] > kRedoCap)) {
    // the directory/header view disagreed with the CSR (or too many throwing segments): the CSR is the source of truth,
    // fold everything on the sequential kernel
    e->pending_var = false;
    FoldArgs a{};
    a.events = e->pending_events; a.seg_offsets = e->pending_offsets; a.n_seg = e->pending_n_seg;
    a.states_out = (uint8_t*)e->states.p; a.counters = (unsigned long long*)e->counters.p;
    CUDA_TRY(e, cudaMemsetAsync(e->counters.p, 0, 64, e->stream));
    CUDA_TRY(e, cudaEventRecord(e->ev2, e->stream));
    FoldLaunchInfo info{};
    cudaError_t le = launch_fold_stream(a, e->dprog, -1, e->num_sms, e->max_record_bytes, e->stream, &info);
    if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "fold launch: %s", cudaGetErrorString(le));
    CUDA_TRY(e, cudaEventRecord(e->ev3, e->stream));
    CUDA_TRY(e, cudaMemcpyAsync(h, e->counters.p, 64, cudaMemcpyDeviceToHost, e->stream));
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    float ms2 = 0; CUDA_TRY(e, cudaEventElapsedTime(&ms2, e->ev2, e->ev3));
    e->stats.ms_fold += ms2; e->stats.fold_launches += 1;
  }
  if (e->pending_used_rows && h[3] > kRedoCap) {
    // more throwing aggregates than the replay list holds: redo everything on the sequential kernel
    FoldArgs a{};
    a.events = e->pending_events; a.seg_offsets = e->pending_offsets; a.seg_ids = e->pending_ids; a.n_seg = e->pending_n_seg;
    a.states_in = e->pending_prior ? (const uint8_t*)e->states.p : nullptr; a.states_out = (uint8_t*)e->states.p;
    a.counters = (unsigned long long*)e->counters.p;
    if (e->pending_prior) {
      // the kernel has already overwritten the non-throwing aggregates in place: the table is half-applied. It must not be
      // served, and a retry must not double-apply — invalidate it (reads fail with SGR_ERR_STATE until the next full fold)
      e->states_valid = false; e->states_invalidated = true; mark_dirty(e);
      return fail(e, SGR_ERR_UNSUPPORTED, "replay list overflow on an in-place incremental fold: state table invalidated, rebuild it");
    }
    CUDA_TRY(e, cudaMemsetAsync(e->counters.p, 0, 64, e->stream));
    CUDA_TRY(e, cudaEventRecord(e->ev2, e->stream));
    FoldLaunchInfo info{};
    cudaError_t le = launch_fold_stream(a, e->dprog, -1, e->num_sms, e->max_record_bytes, e->stream, &info);
    if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "fold launch: %s", cudaGetErrorString(le));
    CUDA_TRY(e, cudaEventRecord(e->ev3, e->stream));
    CUDA_TRY(e, cudaMemcpyAsync(h, e->counters.p, 64, cudaMemcpyDeviceToHost, e->stream));
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    float ms2 = 0; CUDA_TRY(e, cudaEventElapsedTime(&ms2, e->ev2, e->ev3));
    e->stats.ms_fold += ms2; e->stats.fold_launches += 1;
    e->pending_used_rows = false;   // h now holds the sequential kernel's counts
  }
  const uint64_t n_seg = e->pending_n_seg;
  e->stats.n_aggregates = n_seg;
  // runs kernel counts every record, the replay takes back what followed a throw; the rows kernel skips
  // throwing segments, the replay adds what preceded the throw
  e->stats.n_events = e->pending_var ? h[0] - h[4] + h[5] : !e->pending_used_rows ? h[0] : (e->pending_rows_v1 ? h[0] + h[5] : h[0] - h[4]);
  e->stats.n_errors = h[1];
  e->stats.n_long_segments = h[2];
  e->stats.event_bytes = e->pending_event_bytes;
  e->stats.algorithmic_bytes = e->pending_event_bytes + 8 * (n_seg + 1) +
                               (uint64_t)e->program.state_bytes * n_seg * (e->pending_prior ? 2 : 1) + (e->pending_ids ? 4 * n_seg : 0);
  return SGR_OK;
}

}  // namespace

// ================================================================== C ABI
extern "C" {

int32_t sgr_abi_version(void) { return SGR_ABI_VERSION; }

const char* sgr_last_error(const sgr_engine* e) {
  if (!e) return g_create_error.c_str();
  return t_last_engine == e ? t_last_error.c_str() : "";
}

int32_t sgr_create(const sgr_config* cfg, sgr_engine** out) {
  if (!out) return fail(nullptr, SGR_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0)
    return fail(nullptr, SGR_ERR_NO_DEVICE, "no CUDA device (%s); the replay engine has no CPU fallback",
                ce != cudaSuccess ? cudaGetErrorString(ce) : "device count 0");
  const int dev = cfg ? cfg->device : 0;
  if (dev < 0 || dev >= ndev) return fail(nullptr, SGR_ERR_NO_DEVICE, "device %d out of range (have %d)", dev, ndev);
  cudaDeviceProp prop;
  if ((ce = cudaGetDeviceProperties(&prop, dev)) != cudaSuccess)
    return fail(nullptr, SGR_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(ce));
  if (prop.major != 10)
    return fail(nullptr, SGR_ERR_NO_DEVICE, "device %d is sm_%d%d; kernels are built for sm_100a only", dev, prop.major, prop.minor);
  std::unique_ptr<sgr_engine> e(new sgr_engine());
  e->device = dev;
  e->num_sms = prop.multiProcessorCount;
  if ((ce = cudaSetDevice(dev)) != cudaSuccess) return fail(nullptr, SGR_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(ce));
  if ((ce = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (ce = cudaEventCreate(&e->ev0)) != cudaSuccess || (ce = cudaEventCreate(&e->ev1)) != cudaSuccess ||
      (ce = cudaEventCreate(&e->ev2)) != cudaSuccess || (ce = cudaEventCreate(&e->ev3)) != cudaSuccess ||
      (ce = e->counters.reserve(64)) != cudaSuccess)
    return fail(nullptr, SGR_ERR_CUDA, "engine setup: %s", cudaGetErrorString(ce));
  *out = e.release();
  return SGR_OK;
}

int32_t sgr_destroy(sgr_engine* e) {
  if (!e) return SGR_OK;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  e->own_events.release(); e->own_offsets.release(); e->own_rec_offsets.release(); e->states.release(); e->counters.release();
  e->inc_records.release(); e->inc_offsets.release(); e->inc_ids.release(); e->inc_prev_ids.release();
  e->inc_scratch.release(); e->inc_touched[0].release(); e->inc_touched[1].release(); e->inc_err_ids.release(); e->inc_counters.release();
  e->group.release();
  e->bulk_scratch.release(); e->bulk_err_ids.release(); e->bulk_counters.release(); e->hash_out.release();
  if (e->dist) dist_destroy(e->dist);
  e->part_flags.release(); e->part_data.release(); e->redo_ids.release(); e->run_counters.release();
  cudaEventDestroy(e->ev0); cudaEventDestroy(e->ev1); cudaEventDestroy(e->ev2); cudaEventDestroy(e->ev3);
  cudaStreamDestroy(e->stream);
  delete e;
  return SGR_OK;
}

int32_t sgr_register_program(sgr_engine* e, const sgr_fold_program* prog) {
  OpLock op_lock(e);
  if (!e || !prog) return fail(e, SGR_ERR_INVALID, "null argument");
  DevProgram d;
  int32_t rc = compile_program(e, prog, &d);
  if (rc) return rc;
  e->program = *prog; e->dprog = d; e->has_program = true;
  e->row_ok = build_row_program(d, &e->row_prog);
  e->bulk_ok = e->row_ok && prog->record_kind == SGR_REC_FIXED64 && bulk_layout_for(e->row_prog, &e->bulk_lay);
  e->bulk_scratch_slots = 0;
  e->row_max_grid = 0; e->run_max_grid_variant = -1;
  e->states_valid = false; e->states_n = 0;
  mark_dirty(e);
  return SGR_OK;
}

static int32_t before_load(sgr_engine* e) {
  int32_t rc = use_device(e); if (rc) return rc;
  return finish_fold(e);
}

static int32_t after_load(sgr_engine* e, const uint8_t* d_events, const uint64_t* d_offsets, uint64_t nbytes, uint64_t n_agg) {
  e->d_events = d_events; e->d_offsets = d_offsets; e->event_bytes = nbytes; e->n_agg = n_agg; e->loaded = true;
  e->d_rec_offsets = nullptr; e->n_rec = 0;
  // variable records: the format caps a record at 16+512 bytes unless the caller raises
  // "max_record_bytes"; a longer record is flagged as a malformed event by the kernel, never mis-parsed
  e->max_record_bytes = e->program.record_kind == SGR_REC_VAR16 ? (uint32_t)e->opt_max_record_bytes : 64u;
  e->offsets_aligned64 = false; e->log_begin = 0; e->log_end = nbytes;
  if (e->program.record_kind == SGR_REC_FIXED64) {
    cudaError_t ce = inspect_offsets(d_offsets, n_agg, (unsigned long long*)e->counters.p, e->stream, &e->offsets_aligned64,
                                     &e->log_begin, &e->log_end, &e->max_seg_bytes);
    if (ce != cudaSuccess) return fail(e, SGR_ERR_CUDA, "offset inspection: %s", cudaGetErrorString(ce));
  }
  return SGR_OK;
}

int32_t sgr_load_events(sgr_engine* e, const void* events, uint64_t nbytes, const uint64_t* seg_offsets, uint64_t n_agg) {
  OpLock op_lock(e);
  if (!e || (!events && nbytes) || !seg_offsets) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program before loading events");
  if (seg_offsets[n_agg] > nbytes) return fail(e, SGR_ERR_INVALID, "seg_offsets[n_agg]=%llu exceeds nbytes=%llu",
                                               (unsigned long long)seg_offsets[n_agg], (unsigned long long)nbytes);
  for (uint64_t i = 0; i <= n_agg; ++i) {
    if (seg_offsets[i] % 16) return fail(e, SGR_ERR_INVALID, "seg_offsets[%llu] is not a multiple of 16", (unsigned long long)i);
    if (i && seg_offsets[i] < seg_offsets[i - 1]) return fail(e, SGR_ERR_INVALID, "seg_offsets not monotone at %llu", (unsigned long long)i);
  }
  int32_t rc = before_load(e); if (rc) return rc;
  CUDA_TRY(e, e->own_events.reserve(nbytes));
  CUDA_TRY(e, e->own_offsets.reserve((n_agg + 1) * 8));
  CUDA_TRY(e, cudaEventRecord(e->ev0, e->stream));
  CUDA_TRY(e, cudaMemcpyAsync(e->own_events.p, events, nbytes, cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(e, cudaMemcpyAsync(e->own_offsets.p, seg_offsets, (n_agg + 1) * 8, cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(e, cudaEventRecord(e->ev1, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_h2d, e->ev0, e->ev1));
  e->stats.ms_group = 0;
  return after_load(e, (const uint8_t*)e->own_events.p, (const uint64_t*)e->own_offsets.p, nbytes, n_agg);
}

int32_t sgr_load_events_device(sgr_engine* e, const void* d_events, uint64_t nbytes, const uint64_t* d_seg_offsets, uint64_t n_agg) {
  OpLock op_lock(e);
  if (!e || (!d_events && nbytes) || !d_seg_offsets) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program before loading events");
  if (((uintptr_t)d_events) % 16) return fail(e, SGR_ERR_INVALID, "device event log must be 16-byte aligned");
  int32_t rc = before_load(e); if (rc) return rc;
  e->stats.ms_h2d = 0; e->stats.ms_group = 0;
  return after_load(e, (const uint8_t*)d_events, d_seg_offsets, nbytes, n_agg);
}

int32_t sgr_load_events_indexed(sgr_engine* e, const void* events, uint64_t nbytes, const uint64_t* seg_offsets, uint64_t n_agg,
                                const uint64_t* rec_offsets, uint64_t n_records) {
  OpLock op_lock(e);
  if (!rec_offsets) return fail(e, SGR_ERR_INVALID, "null record directory");
  int32_t rc = sgr_load_events(e, events, nbytes, seg_offsets, n_agg);
  if (rc) return rc;
  for (uint64_t i = 0; i < n_records; ++i)
    if (rec_offsets[i + 1] < rec_offsets[i] || rec_offsets[i] % 16) return fail(e, SGR_ERR_INVALID, "record directory is not monotone / 16-byte aligned at %llu", (unsigned long long)i);
  if (rec_offsets[0] != seg_offsets[0] || rec_offsets[n_records] != seg_offsets[n_agg]) return fail(e, SGR_ERR_INVALID, "record directory and CSR cover different byte ranges");
  CUDA_TRY(e, e->own_rec_offsets.reserve((n_records + 1) * 8));
  CUDA_TRY(e, cudaMemcpyAsync(e->own_rec_offsets.p, rec_offsets, (n_records + 1) * 8, cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  e->d_rec_offsets = (const uint64_t*)e->own_rec_offsets.p; e->n_rec = n_records;
  return SGR_OK;
}

int32_t sgr_load_events_indexed_device(sgr_engine* e, const void* d_events, uint64_t nbytes, const uint64_t* d_seg_offsets, uint64_t n_agg,
                                       const uint64_t* d_rec_offsets, uint64_t n_records) {
  OpLock op_lock(e);
  if (!d_rec_offsets) return fail(e, SGR_ERR_INVALID, "null record directory");
  int32_t rc = sgr_load_events_device(e, d_events, nbytes, d_seg_offsets, n_agg);
  if (rc) return rc;
  e->d_rec_offsets = d_rec_offsets; e->n_rec = n_records;   // consistency with the CSR is checked by the kernel at every segment head
  return SGR_OK;
}

static int32_t load_unsorted_impl(sgr_engine* e, const void* d_records, uint64_t n_records, uint64_t n_agg) {
  if (e->program.record_kind != SGR_REC_FIXED64) return fail(e, SGR_ERR_UNSUPPORTED, "unsorted loads take fixed 64-byte records");
  if (n_agg >= (1ull << 32) || n_records >= (1ull << 32)) return fail(e, SGR_ERR_UNSUPPORTED, "group-by is limited to 2^32 records/aggregates");
  CUDA_TRY(e, e->own_events.reserve(n_records * 64));
  CUDA_TRY(e, e->own_offsets.reserve((n_agg + 1) * 8));
  CUDA_TRY(e, cudaEventRecord(e->ev0, e->stream));
  unsigned long long bad = 0, holes = 0;
  cudaError_t ce = group_by_agg_stable(e->group, (const uint8_t*)d_records, n_records, n_agg, (uint8_t*)e->own_events.p,
                                       (uint64_t*)e->own_offsets.p, nullptr, nullptr, (unsigned long long*)e->counters.p, e->stream, &bad, &holes);
  if (ce != cudaSuccess) return fail(e, SGR_ERR_CUDA, "group-by: %s", cudaGetErrorString(ce));
  CUDA_TRY(e, cudaEventRecord(e->ev1, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_group, e->ev0, e->ev1));
  if (bad) return fail(e, SGR_ERR_INVALID, "%llu records carry an aggregate index >= n_agg", bad);
  // the holes were sorted behind the last segment: the log ends before them
  return after_load(e, (const uint8_t*)e->own_events.p, (const uint64_t*)e->own_offsets.p, (n_records - holes) * 64, n_agg);
}

int32_t sgr_load_unsorted_device(sgr_engine* e, const void* d_records, uint64_t n_records, uint64_t n_agg) {
  OpLock op_lock(e);
  if (!e || (!d_records && n_records)) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program before loading events");
  int32_t rc = before_load(e); if (rc) return rc;
  e->stats.ms_h2d = 0;
  return load_unsorted_impl(e, d_records, n_records, n_agg);
}

int32_t sgr_load_unsorted(sgr_engine* e, const void* records, uint64_t n_records, uint64_t n_agg) {
  OpLock op_lock(e);
  if (!e || (!records && n_records)) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program before loading events");
  int32_t rc = before_load(e); if (rc) return rc;
  CUDA_TRY(e, e->inc_records.reserve(n_records * 64));
  CUDA_TRY(e, cudaEventRecord(e->ev0, e->stream));
  CUDA_TRY(e, cudaMemcpyAsync(e->inc_records.p, records, n_records * 64, cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(e, cudaEventRecord(e->ev1, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_h2d, e->ev0, e->ev1));
  return load_unsorted_impl(e, e->inc_records.p, n_records, n_agg);
}

int32_t sgr_set_initial_states(sgr_engine* e, const void* states, uint64_t n_agg) {
  OpLock op_lock(e);
  if (!e) return SGR_ERR_INVALID;
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program first");
  // NULL only says "the next fold starts from None everywhere": no device work, no wait
  if (!states) { e->states_valid = false; e->states_invalidated = false; mark_dirty(e); return SGR_OK; }
  int32_t rc = before_load(e); if (rc) return rc;
  rc = ensure_states(e, n_agg); if (rc) return rc;
  CUDA_TRY(e, cudaMemcpyAsync(e->states.p, states, (size_t)n_agg * e->program.state_bytes, cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  e->states_valid = true; e->states_invalidated = false;
  e->inc_atomic_prev_valid = false; e->inc_prev_n = 0;
  mark_dirty(e);
  return SGR_OK;
}

static int32_t fold_begin(sgr_engine* e, bool pipelined) {
  if (!e) return SGR_ERR_INVALID;
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "no fold program registered");
  if (!e->loaded) return fail(e, SGR_ERR_NOT_LOADED, "no event log loaded");
  int32_t rc = use_device(e); if (rc) return rc;
  // back-to-back asynchronous folds of the same log are queued without a host round trip;
  // only the last one is waited on (sgr_wait) and has its statistics collected
  if (!pipelined) { rc = finish_fold(e); if (rc) return rc; }
  const bool prior = e->states_valid && e->states_n == e->n_agg;
  rc = ensure_states(e, e->n_agg); if (rc) return rc;
  e->states_invalidated = false;   // a full fold replaces the table (a failed in-place fold left prior states invalid)
  rc = enqueue_fold(e, e->d_events, e->d_offsets, nullptr, e->n_agg, prior, e->event_bytes, e->offsets_aligned64, e->log_begin, e->log_end);
  if (rc) return rc;
  e->states_valid = true;
  e->inc_prev_n = 0;
  e->inc_atomic_prev_valid = false;
  mark_dirty(e);
  return SGR_OK;
}

int32_t sgr_fold(sgr_engine* e) {
  OpLock op_lock(e);
  int32_t rc = fold_begin(e, false); if (rc) return rc;
  return finish_fold(e);
}

int32_t sgr_fold_async(sgr_engine* e) { OpLock op_lock(e); return fold_begin(e, true); }

int32_t sgr_wait(sgr_engine* e) {
  OpLock op_lock(e);
  if (!e) return SGR_ERR_INVALID;
  int32_t rc = use_device(e); if (rc) return rc;
  return finish_fold(e);
}

static int32_t replay_throwing_slots(sgr_engine* e, const void* d_records, uint64_t n_records, uint64_t n_agg, const uint32_t* d_err_ids,
                                     uint64_t n_err, unsigned long long* h_throwing, unsigned long long* h_dropped);

// sort-free path for programs inside the transformer algebra (incremental.cu)
static int32_t fold_incremental_atomic(sgr_engine* e, const void* d_records, uint64_t n_records) {
  const uint64_t n_agg = e->states_n;
  if (n_records >= (1ull << 32)) return fail(e, SGR_ERR_UNSUPPORTED, "micro-batches are limited to 2^32 records");
  if (e->inc_scratch_slots != n_agg) {
    CUDA_TRY(e, e->inc_scratch.reserve(inc_scratch_bytes(n_agg)));
    CUDA_TRY(e, cudaMemsetAsync(e->inc_scratch.p, 0, inc_scratch_bytes(n_agg), e->stream));
    e->inc_scratch_slots = n_agg;
  }
  // sized by the table, not by the batch: the previous batch's list must survive a larger next batch
  CUDA_TRY(e, e->inc_touched[0].reserve((n_agg + 1) * 4)); CUDA_TRY(e, e->inc_touched[1].reserve((n_agg + 1) * 4));
  CUDA_TRY(e, e->inc_err_ids.reserve((n_agg + 1) * 4));
  CUDA_TRY(e, e->inc_counters.reserve(256));
  unsigned long long* cur = (unsigned long long*)e->inc_counters.p + 8 * e->inc_flip;
  unsigned long long* prev = (unsigned long long*)e->inc_counters.p + 8 * (e->inc_flip ^ 1);
  CUDA_TRY(e, cudaEventRecord(e->ev0, e->stream));
  CUDA_TRY(e, cudaMemsetAsync(cur, 0, 64, e->stream));
  uint32_t prev_upper = 0;
  if (!e->inc_atomic_prev_valid) {
    // first batch after a full fold / set_initial_states / a sort-based batch: every slot may carry per-batch flags
    clear_batch_flags((uint8_t*)e->states.p, e->program.state_bytes, nullptr, n_agg, e->stream);
  } else {
    prev_upper = e->inc_prev_upper;
  }
  cudaError_t le = launch_incremental_atomic((const uint8_t*)d_records, (uint32_t)n_records, n_agg, e->inc_scratch.p, (uint8_t*)e->states.p,
                                             (uint32_t*)e->inc_touched[e->inc_flip].p, (uint32_t*)e->inc_err_ids.p,
                                             (const uint32_t*)e->inc_touched[e->inc_flip ^ 1].p, prev + 5, prev_upper, e->row_prog, cur, (unsigned long long)e->opt_replay_budget, e->stream);
  if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "incremental launch: %s", cudaGetErrorString(le));
  CUDA_TRY(e, cudaEventRecord(e->ev1, e->stream));
  unsigned long long h[8];
  CUDA_TRY(e, cudaMemcpyAsync(h, cur, 64, cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_fold, e->ev0, e->ev1));
  if (h[4]) return fail(e, SGR_ERR_INVALID, "%llu records carry an aggregate index >= n_agg; the batch was not applied", h[4]);
  if (h[2]) {
    // too many throwing slots to re-scan the batch for each: group the batch once and replay exactly those slots
    // on the sequential kernel (their states are still the pre-batch ones)
    unsigned long long thr = 0, drop = 0;
    int32_t rr = replay_throwing_slots(e, d_records, n_records, n_agg, (const uint32_t*)e->inc_err_ids.p, h[3], &thr, &drop);
    if (rr) return rr;
    h[1] = thr; h[6] = drop;   // throwing slots, events dropped after their throw
  }
  e->inc_atomic_prev_valid = true;
  e->inc_prev_upper = (uint32_t)(h[5]);
  e->inc_flip ^= 1;
  e->inc_prev_n = 0;
  e->stats.ms_group = 0;
  e->stats.n_aggregates = h[5]; e->stats.n_errors = h[1]; e->stats.n_events = n_records - h[0] - h[6];   // [0] holes
  e->stats.event_bytes = n_records * 64; e->stats.n_long_segments = 0;
  e->stats.algorithmic_bytes = n_records * 64 + 2 * (uint64_t)e->program.state_bytes * h[5];
  e->stats.fold_launches = 1;
  mark_dirty(e);
  return SGR_OK;
}

static int32_t fold_incremental_impl(sgr_engine* e, const void* d_records, uint64_t n_records) {
  if (e->program.record_kind != SGR_REC_FIXED64) return fail(e, SGR_ERR_UNSUPPORTED, "incremental batches take fixed 64-byte records");
  if (!e->states_valid) return fail(e, SGR_ERR_NOT_LOADED, "incremental fold needs a live state table (fold or set_initial_states first)");
  { int32_t rc0 = finish_fold(e); if (rc0) return rc0; }
  // (a 16-byte state that is one JVM Double compares with ==, not bitwise: it takes the sort-based path)
  if (e->row_ok && e->row_prog.user_words == 2 && e->row_prog.cls == 0 && !e->row_prog.f64_mask && e->opt_kernel != 1 && e->opt_kernel != 3 && e->opt_incremental != 1)
    return fold_incremental_atomic(e, d_records, n_records);
  e->inc_atomic_prev_valid = false;
  const uint64_t n_agg = e->states_n;
  CUDA_TRY(e, e->inc_offsets.reserve((n_records + 2) * 8));
  CUDA_TRY(e, e->inc_ids.reserve((n_records + 1) * 4));
  DevBuf& grouped = e->group.batch_records;
  CUDA_TRY(e, grouped.reserve(n_records * 64));
  CUDA_TRY(e, cudaEventRecord(e->ev2, e->stream));
  // per-batch flags (CHANGED/ERROR) of the aggregates touched by the previous batch are cleared
  if (e->inc_prev_n) clear_batch_flags((uint8_t*)e->states.p, e->program.state_bytes, (const uint32_t*)e->inc_prev_ids.p, e->inc_prev_n, e->stream);
  else clear_batch_flags((uint8_t*)e->states.p, e->program.state_bytes, nullptr, n_agg, e->stream);
  unsigned long long bad = 0, holes = 0;
  uint64_t n_touched = 0;
  cudaError_t ce = group_by_agg_stable(e->group, (const uint8_t*)d_records, n_records, n_agg, (uint8_t*)grouped.p,
                                       (uint64_t*)e->inc_offsets.p, (uint32_t*)e->inc_ids.p, &n_touched,
                                       (unsigned long long*)e->counters.p, e->stream, &bad, &holes);
  if (ce != cudaSuccess) return fail(e, SGR_ERR_CUDA, "group-by: %s", cudaGetErrorString(ce));
  CUDA_TRY(e, cudaEventRecord(e->ev3, e->stream));
  if (bad) return fail(e, SGR_ERR_INVALID, "%llu records carry an aggregate index >= n_agg", bad);
  const uint64_t real_bytes = (n_records - holes) * 64;   // the holes were sorted behind the last segment
  int32_t rc = enqueue_fold(e, (const uint8_t*)grouped.p, (const uint64_t*)e->inc_offsets.p, (const uint32_t*)e->inc_ids.p, n_touched, true,
                            real_bytes, true, 0, real_bytes);
  if (rc) return rc;
  rc = finish_fold(e); if (rc) return rc;
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_group, e->ev2, e->ev3));
  // remember who was touched so the next batch can clear their per-batch flags
  std::swap(e->inc_ids, e->inc_prev_ids);
  e->inc_prev_n = n_touched;
  mark_dirty(e);
  return SGR_OK;
}

int32_t sgr_fold_incremental_device(sgr_engine* e, const void* d_records, uint64_t n_records) {
  OpLock op_lock(e);
  if (!e || (!d_records && n_records)) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "no fold program registered");
  int32_t rc = use_device(e); if (rc) return rc;
  e->stats.ms_h2d = 0;
  return fold_incremental_impl(e, d_records, n_records);
}

int32_t sgr_fold_incremental(sgr_engine* e, const void* records, uint64_t n_records) {
  OpLock op_lock(e);
  if (!e || (!records && n_records)) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "no fold program registered");
  int32_t rc = use_device(e); if (rc) return rc;
  CUDA_TRY(e, e->inc_records.reserve(n_records * 64));
  CUDA_TRY(e, cudaMemcpyAsync(e->inc_records.p, records, n_records * 64, cudaMemcpyHostToDevice, e->stream));
  return fold_incremental_impl(e, e->inc_records.p, n_records);
}

int32_t sgr_load_keys(sgr_engine* e, const uint8_t* keys, const uint32_t* key_offsets, uint64_t n_agg) {
  if (!e || !key_offsets || (!keys && n_agg && key_offsets[n_agg])) return fail(e, SGR_ERR_INVALID, "null argument");
  std::string err;
  auto kt = std::make_shared<KeyTable>();
  if (!kt->build(keys, key_offsets, n_agg, &err)) return fail(e, SGR_ERR_INVALID, "%s", err.c_str());
  std::lock_guard<std::mutex> lk(e->keys_mu);
  e->ing_keys_from = nullptr; e->ing_key_bytes.clear(); e->ing_key_offs.clear();
  e->keys_stale.store(false, std::memory_order_release);
  std::atomic_store(&e->keys, std::shared_ptr<const KeyTable>(kt));
  return SGR_OK;
}

int32_t sgr_grow_states(sgr_engine* e, uint64_t n_agg) {
  OpLock op_lock(e);
  if (!e) return SGR_ERR_INVALID;
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program first");
  int32_t rc = use_device(e); if (rc) return rc;
  rc = before_load(e); if (rc) return rc;
  if (e->states_invalidated) return fail(e, SGR_ERR_STATE, "state table invalidated by a failed fold: reset it (set_initial_states) or rebuild it");
  if (e->states_valid && n_agg <= e->states_n) return SGR_OK;
  const size_t sb = e->program.state_bytes;
  if (!e->states_valid && e->states.p && e->states.cap >= (size_t)n_agg * sb) {
    // a table that was reset (sgr_set_initial_states(NULL)) and is large enough: all None, no reallocation, no device-wide
    // synchronisation by cudaFree
    CUDA_TRY(e, cudaMemsetAsync(e->states.p, 0, (size_t)n_agg * sb, e->stream));
    e->states_n = n_agg; e->states_valid = true;
    e->inc_atomic_prev_valid = false; e->inc_prev_n = 0;
    mark_dirty(e);
    return SGR_OK;
  }
  struct Guard { DevBuf b; ~Guard() { b.release(); } } guard;   // frees the old table on success, the new one on failure
  DevBuf& nb = guard.b;
  CUDA_TRY(e, nb.reserve((size_t)n_agg * sb));
  const size_t keep = e->states_valid ? (size_t)e->states_n * sb : 0;
  if (keep) CUDA_TRY(e, cudaMemcpyAsync(nb.p, e->states.p, keep, cudaMemcpyDeviceToDevice, e->stream));
  CUDA_TRY(e, cudaMemsetAsync((uint8_t*)nb.p + keep, 0, (size_t)n_agg * sb - keep, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  std::swap(e->states, nb);
  e->states_n = n_agg;
  e->states_valid = true;
  e->inc_atomic_prev_valid = false; e->inc_prev_n = 0;
  mark_dirty(e);
  return SGR_OK;
}

static void* pinned_alloc(size_t n) { void* p = nullptr; return cudaHostAlloc(&p, n, cudaHostAllocPortable) == cudaSuccess ? p : nullptr; }
static void pinned_free(void* p) { cudaFreeHost(p); }

// the key table follows an append-only id dictionary kept elsewhere (host ingest, device ingest): ids [have, n_keys) are appended,
// the hash index is rebuilt lazily by the first sgr_get that follows (a restore polls thousands of times before anybody reads)
static int32_t sgr_append_keys_upto(sgr_engine* e, const void* owner, const uint8_t* keys, const uint32_t* key_offsets, uint64_t n_keys) {
  std::lock_guard<std::mutex> lk(e->keys_mu);
  if (e->ing_keys_from != owner) { e->ing_keys_from = owner; e->ing_key_bytes.clear(); e->ing_key_offs.assign(1, 0u); }
  const uint64_t have = e->ing_key_offs.size() - 1;
  if (n_keys > have) {
    e->ing_key_bytes.insert(e->ing_key_bytes.end(), keys + key_offsets[have], keys + key_offsets[n_keys]);
    const uint32_t shift = e->ing_key_offs.back() - key_offsets[have];
    for (uint64_t i = have + 1; i <= n_keys; ++i) e->ing_key_offs.push_back(key_offsets[i] + shift);
    e->keys_stale.store(true, std::memory_order_release);
  }
  return SGR_OK;
}

int32_t sgr_append_keys(sgr_engine* e, const void* owner, const uint8_t* keys, const uint32_t* key_offsets, uint64_t n_new) {
  if (!e || !key_offsets || (!keys && n_new && key_offsets[n_new])) return fail(e, SGR_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> lk(e->keys_mu);
  if (e->ing_keys_from != owner) { e->ing_keys_from = owner; e->ing_key_bytes.clear(); e->ing_key_offs.assign(1, 0u); }
  if (n_new) {
    e->ing_key_bytes.insert(e->ing_key_bytes.end(), keys + key_offsets[0], keys + key_offsets[n_new]);
    const uint32_t shift = e->ing_key_offs.back() - key_offsets[0];
    const size_t old = e->ing_key_offs.size();
    e->ing_key_offs.resize(old + n_new);
    uint32_t* dst = e->ing_key_offs.data() + old;
    for (uint64_t i = 0; i < n_new; ++i) dst[i] = key_offsets[i + 1] + shift;
    e->keys_stale.store(true, std::memory_order_release);
  }
  return SGR_OK;
}

int32_t sgr_fold_ingested(sgr_engine* e, sgr_ingest* g) {
  OpLock op_lock(e);
  if (!e || !g) return fail(e, SGR_ERR_INVALID, "null argument");
  { int32_t rc0 = use_device(e); if (rc0) return rc0; }
  if (e->states_invalidated) return fail(e, SGR_ERR_STATE, "state table invalidated by a failed fold: reset it (set_initial_states) or rebuild it");
  // from now on the ingest decodes straight into page-locked memory (what is pending right now is moved once)
  if (sgr_ingest_set_allocator(g, pinned_alloc, pinned_free)) return fail(e, SGR_ERR_OOM, "ingest: %s", sgr_ingest_last_error(g));
  const void* recs = nullptr; uint64_t n_records = 0;
  const uint8_t* keys = nullptr; const uint32_t* key_offsets = nullptr; uint64_t n_keys = 0;
  if (sgr_ingest_pending(g, &recs, &n_records) || sgr_ingest_keys(g, &keys, &key_offsets, &n_keys))
    return fail(e, SGR_ERR_INVALID, "ingest: %s", sgr_ingest_last_error(g));
  if (!e->states_valid || n_keys > e->states_n) {
    // amortised doubling, like a hash table: the resize copies the table device to device
    uint64_t cap = e->states_valid ? e->states_n : 0;
    if (cap < 1024) cap = 1024;
    while (cap < n_keys) cap *= 2;
    int32_t rc = sgr_grow_states(e, cap); if (rc) return rc;
  }
  if (n_records) { int32_t rc = sgr_fold_incremental(e, recs, n_records); if (rc) return rc; }
  if (n_keys) { int32_t rc = sgr_append_keys_upto(e, g, keys, key_offsets, n_keys); if (rc) return rc; }
  sgr_ingest_mark_folded(g);
  return SGR_OK;
}

int32_t sgr_get_index(sgr_engine* e, uint64_t agg, void* out, uint32_t cap, uint32_t* outlen, int32_t* exists,
                      uint32_t* flags, uint32_t* err_idx) {
  if (!e) return SGR_ERR_INVALID;
  std::shared_ptr<Snapshot> s = std::atomic_load(&e->snapshot);
  if (!s || e->snapshot_dirty.load(std::memory_order_acquire)) {
    int32_t rc = refresh_snapshot(e, &s); if (rc) return rc;
  }
  if (agg >= s->n_agg) return fail(e, SGR_ERR_INVALID, "aggregate index %llu out of range", (unsigned long long)agg);
  const uint8_t* st = s->states.data() + agg * s->state_bytes;
  uint32_t fl, ei;
  memcpy(&fl, st + s->state_bytes - 8, 4); memcpy(&ei, st + s->state_bytes - 4, 4);
  const uint32_t user = s->state_bytes - 8;
  if (flags) *flags = fl;
  if (err_idx) *err_idx = ei;
  if (exists) *exists = (fl & SGR_ST_EXISTS) ? 1 : 0;
  if (outlen) *outlen = (fl & SGR_ST_EXISTS) ? user : 0;
  if ((fl & SGR_ST_EXISTS) && out) {
    if (cap < user) return fail(e, SGR_ERR_CAPACITY, "buffer of %u bytes is smaller than the state (%u)", cap, user);
    memcpy(out, st, user);
  }
  return SGR_OK;
}

// dense index of an aggregate id in the key table (rebuilt first if ids were appended since), or -1
static int32_t find_key(sgr_engine* e, const uint8_t* key, uint32_t klen, int64_t* idx) {
  if (e->keys_stale.load(std::memory_order_acquire)) {
    std::lock_guard<std::mutex> lk(e->keys_mu);
    if (e->keys_stale.load(std::memory_order_relaxed)) {
      auto fresh = std::make_shared<KeyTable>();
      std::string err;
      if (!fresh->build(e->ing_key_bytes.data(), e->ing_key_offs.data(), e->ing_key_offs.size() - 1, &err)) return fail(e, SGR_ERR_INVALID, "%s", err.c_str());
      std::atomic_store(&e->keys, std::shared_ptr<const KeyTable>(fresh));
      e->keys_stale.store(false, std::memory_order_release);
    }
  }
  std::shared_ptr<const KeyTable> kt = std::atomic_load(&e->keys);
  *idx = kt ? kt->find(key, klen) : -1;
  return SGR_OK;
}

int32_t sgr_key_index(sgr_engine* e, const uint8_t* key, uint32_t klen, uint64_t* agg) {
  if (!e || (!key && klen) || !agg) return fail(e, SGR_ERR_INVALID, "null argument");
  int64_t idx = -1;
  int32_t rc = find_key(e, key, klen, &idx); if (rc) return rc;
  *agg = idx < 0 ? UINT64_MAX : (uint64_t)idx;
  return SGR_OK;
}

int32_t sgr_get(sgr_engine* e, const uint8_t* key, uint32_t klen, void* out, uint32_t cap, uint32_t* outlen, int32_t* exists) {
  if (!e || (!key && klen)) return fail(e, SGR_ERR_INVALID, "null argument");
  int64_t idx = -1;
  { int32_t rc = find_key(e, key, klen, &idx); if (rc) return rc; }
  if (idx < 0) {  // unknown aggregate id: Option.empty, like a KTable miss
    if (exists) *exists = 0;
    if (outlen) *outlen = 0;
    // still surface "store not readable" the way the reference does
    std::shared_ptr<Snapshot> s = std::atomic_load(&e->snapshot);
    if (!s || e->snapshot_dirty.load(std::memory_order_acquire)) { int32_t rc = refresh_snapshot(e, &s); if (rc) return rc; }
    return SGR_OK;
  }
  return sgr_get_index(e, (uint64_t)idx, out, cap, outlen, exists, nullptr, nullptr);
}

int32_t sgr_export_states(sgr_engine* e, void* out, uint64_t cap, uint8_t* exists_bits, uint8_t* changed_bits, uint8_t* error_bits) {
  OpLock op_lock(e);
  if (!e) return SGR_ERR_INVALID;
  if (!e->states_valid) return fail(e, SGR_ERR_STATE, "no folded state table to export");
  int32_t rc = use_device(e); if (rc) return rc;
  rc = finish_fold(e); if (rc) return rc;
  const uint64_t n = e->states_n; const uint32_t sb = e->program.state_bytes;
  const uint64_t need = n * sb;
  std::vector<uint8_t> tmp;
  uint8_t* host = (uint8_t*)out;
  if (out) { if (cap < need) return fail(e, SGR_ERR_CAPACITY, "export needs %llu bytes, buffer has %llu", (unsigned long long)need, (unsigned long long)cap); }
  else { tmp.resize(need); host = tmp.data(); }
  CUDA_TRY(e, cudaEventRecord(e->ev0, e->stream));
  CUDA_TRY(e, cudaMemcpyAsync(host, e->states.p, need, cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(e, cudaEventRecord(e->ev1, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_d2h, e->ev0, e->ev1));
  if (exists_bits || changed_bits || error_bits) {
    const uint64_t nb = (n + 7) / 8;
    if (exists_bits) memset(exists_bits, 0, nb);
    if (changed_bits) memset(changed_bits, 0, nb);
    if (error_bits) memset(error_bits, 0, nb);
    for (uint64_t i = 0; i < n; ++i) {
      uint32_t fl; memcpy(&fl, host + i * sb + sb - 8, 4);
      if (exists_bits && (fl & SGR_ST_EXISTS)) exists_bits[i >> 3] |= (uint8_t)(1u << (i & 7));
      if (changed_bits && (fl & SGR_ST_CHANGED)) changed_bits[i >> 3] |= (uint8_t)(1u << (i & 7));
      if (error_bits && (fl & SGR_ST_ERROR)) error_bits[i >> 3] |= (uint8_t)(1u << (i & 7));
    }
  }
  return SGR_OK;
}

int32_t sgr_states_device(sgr_engine* e, void** d_states, uint64_t* n_agg, uint32_t* state_bytes) {
  OpLock op_lock(e);
  if (!e) return SGR_ERR_INVALID;
  if (!e->states_valid) return fail(e, SGR_ERR_STATE, "no folded state table");
  if (d_states) *d_states = e->states.p;
  if (n_agg) *n_agg = e->states_n;
  if (state_bytes) *state_bytes = e->program.state_bytes;
  return SGR_OK;
}

int32_t sgr_events_device(sgr_engine* e, void** d_events, uint64_t* nbytes, uint64_t** d_seg_offsets) {
  if (!e) return SGR_ERR_INVALID;
  if (!e->loaded) return fail(e, SGR_ERR_NOT_LOADED, "no event log loaded");
  if (d_events) *d_events = (void*)e->d_events;
  if (nbytes) *nbytes = e->event_bytes;
  if (d_seg_offsets) *d_seg_offsets = (uint64_t*)e->d_offsets;
  return SGR_OK;
}

int32_t sgr_get_stats(sgr_engine* e, sgr_stats* out) {
  OpLock op_lock(e);
  if (!e || !out) return SGR_ERR_INVALID;
  if (e->fold_pending) { int32_t rc = use_device(e); if (rc) return rc; rc = finish_fold(e); if (rc) return rc; }
  *out = e->stats;
  return SGR_OK;
}

// Exact replay of the slots that saw a throwing event in a sort-free fold: the batch is grouped once (K5) and exactly those
// slots are folded sequentially onto their untouched prior states (exact err_idx, state kept: PersistentActor.scala:260-263).
// h_throwing / h_dropped: aggregates in error, events dropped after their throw.
static int32_t replay_throwing_slots(sgr_engine* e, const void* d_records, uint64_t n_records, uint64_t n_agg, const uint32_t* d_err_ids,
                                     uint64_t n_err, unsigned long long* h_throwing, unsigned long long* h_dropped) {
  DevBuf& grouped = e->group.batch_records;
  CUDA_TRY(e, grouped.reserve(n_records * 64));
  CUDA_TRY(e, e->inc_offsets.reserve((n_agg + 2) * 8));
  unsigned long long bad = 0;
  cudaError_t ce = group_by_agg_stable(e->group, (const uint8_t*)d_records, n_records, n_agg, (uint8_t*)grouped.p, (uint64_t*)e->inc_offsets.p,
                                       nullptr, nullptr, (unsigned long long*)e->counters.p, e->stream, &bad, nullptr);
  if (ce != cudaSuccess) return fail(e, SGR_ERR_CUDA, "group-by (replay): %s", cudaGetErrorString(ce));
  CUDA_TRY(e, cudaMemsetAsync(e->counters.p, 0, 64, e->stream));
  FoldArgs a{};
  a.events = (const uint8_t*)grouped.p; a.seg_offsets = (const uint64_t*)e->inc_offsets.p; a.n_seg = n_err;
  a.seg_list = d_err_ids; a.states_in = (const uint8_t*)e->states.p; a.states_out = (uint8_t*)e->states.p;
  a.counters = (unsigned long long*)e->counters.p;
  FoldLaunchInfo info{};
  cudaError_t le2 = launch_fold_stream(a, e->dprog, -1, e->num_sms, e->max_record_bytes, e->stream, &info);
  if (le2 != cudaSuccess) return fail(e, SGR_ERR_CUDA, "replay launch: %s", cudaGetErrorString(le2));
  unsigned long long h2[8];
  CUDA_TRY(e, cudaMemcpyAsync(h2, e->counters.p, 64, cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  *h_throwing = h2[1]; *h_dropped = h2[4];
  return SGR_OK;
}

static int32_t ensure_bulk_buffers(sgr_engine* e, uint64_t n_agg) {
  if (e->bulk_scratch_slots != n_agg || !e->bulk_scratch.p) {
    const size_t need = bulk_scratch_bytes(e->bulk_lay, n_agg);
    CUDA_TRY(e, e->bulk_scratch.reserve(need));
    CUDA_TRY(e, cudaMemsetAsync(e->bulk_scratch.p, 0, need, e->stream));   // the finish pass leaves it zero again
    e->bulk_scratch_slots = n_agg;
  }
  CUDA_TRY(e, e->bulk_err_ids.reserve((n_agg + 1) * 4));
  CUDA_TRY(e, e->bulk_counters.reserve(64));
  return SGR_OK;
}

// sort-free fold of a large arrival-order log onto the (zeroed or prior) state table: accumulate + finish (bulk_fold.cu)
static int32_t fold_bulk(sgr_engine* e, const uint8_t* d_records, uint64_t n_records, uint64_t n_agg) {
  int32_t rc = ensure_bulk_buffers(e, n_agg); if (rc) return rc;
  unsigned long long* cnt = (unsigned long long*)e->bulk_counters.p;
  CUDA_TRY(e, cudaEventRecord(e->ev0, e->stream));
  CUDA_TRY(e, cudaMemsetAsync(cnt, 0, 64, e->stream));
  BulkSrc src{};
  src.n_regions = 1; src.base[0] = d_records; src.count[0] = n_records; src.rec_bytes = 64;
  cudaError_t le = launch_bulk_accumulate(src, n_agg, e->bulk_scratch.p, e->row_prog, e->bulk_lay, cnt, e->num_sms, e->stream);
  if (le == cudaSuccess) le = launch_bulk_finish(n_agg, e->bulk_scratch.p, (uint8_t*)e->states.p, (uint32_t*)e->bulk_err_ids.p, e->bulk_lay, cnt, e->stream);
  if (le != cudaSuccess) return fail(e, SGR_ERR_CUDA, "bulk fold launch: %s", cudaGetErrorString(le));
  CUDA_TRY(e, cudaEventRecord(e->ev1, e->stream));
  unsigned long long h[8];
  CUDA_TRY(e, cudaMemcpyAsync(h, cnt, 64, cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_fold, e->ev0, e->ev1));
  if (h[4]) { e->states_valid = false; return fail(e, SGR_ERR_INVALID, "%llu records carry an aggregate index >= n_agg; nothing was applied", h[4]); }
  unsigned long long throwing = 0, dropped = 0;
  if (h[3]) { rc = replay_throwing_slots(e, d_records, n_records, n_agg, (const uint32_t*)e->bulk_err_ids.p, h[3], &throwing, &dropped); if (rc) return rc; }
  e->stats.ms_group = 0;
  e->stats.n_aggregates = n_agg; e->stats.n_errors = throwing; e->stats.n_events = n_records - h[0] - dropped;   // [0] holes
  e->stats.event_bytes = n_records * 64; e->stats.n_long_segments = 0;
  e->stats.algorithmic_bytes = n_records * 64 + (uint64_t)(16 + 2 * e->program.state_bytes) * n_agg;
  e->stats.fold_launches = 2;
  mark_dirty(e);
  return SGR_OK;
}

// Fold an arrival-order log (aggregates interleaved, per-aggregate order kept) from None.
// class-0 programs need no grouping at all: the records are folded with integer atomics (bulk_fold.cu / incremental.cu);
// other programs are grouped stably (K5) and folded from the CSR.
static int32_t fold_arrival_order(sgr_engine* e, const uint8_t* d_records, uint64_t n_records, uint64_t n_agg) {
  const bool sort_free = e->row_ok && e->row_prog.user_words == 2 && e->row_prog.cls == 0 && !e->row_prog.f64_mask && e->opt_kernel != 1 && e->opt_kernel != 3 &&
                         e->opt_incremental != 1 && n_records > 0;
  int32_t rc;
  if (sort_free) {
    rc = ensure_states(e, n_agg); if (rc) return rc;
    CUDA_TRY(e, cudaMemsetAsync(e->states.p, 0, (size_t)n_agg * e->program.state_bytes, e->stream));
    e->states_valid = true; e->states_invalidated = false;
    e->loaded = false;
    if (e->bulk_ok && e->opt_bulk && n_records < (1ull << 30)) {
      e->inc_atomic_prev_valid = false; e->inc_prev_n = 0;   // the next micro-batch clears every slot's per-batch flags
      return fold_bulk(e, d_records, n_records, n_agg);
    }
    e->inc_atomic_prev_valid = true; e->inc_prev_upper = 0;   // a fresh all-None table: no per-batch flags to clear
    rc = fold_incremental_atomic(e, d_records, n_records);
    if (rc) return rc;
    e->stats.ms_group = 0;
    return SGR_OK;
  }
  rc = load_unsorted_impl(e, d_records, n_records, n_agg);
  if (rc) return rc;
  e->states_valid = false;
  return sgr_fold(e);
}

int32_t sgr_fold_unsorted_device(sgr_engine* e, const void* d_records, uint64_t n_records, uint64_t n_agg) {
  OpLock op_lock(e);
  if (!e || (!d_records && n_records)) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program first");
  if (e->program.record_kind != SGR_REC_FIXED64) return fail(e, SGR_ERR_UNSUPPORTED, "arrival-order logs take fixed 64-byte records");
  int32_t rc = before_load(e); if (rc) return rc;
  e->stats.ms_h2d = 0;
  return fold_arrival_order(e, (const uint8_t*)d_records, n_records, n_agg);
}

int32_t sgr_fold_unsorted(sgr_engine* e, const void* records, uint64_t n_records, uint64_t n_agg) {
  OpLock op_lock(e);
  if (!e || (!records && n_records)) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program first");
  if (e->program.record_kind != SGR_REC_FIXED64) return fail(e, SGR_ERR_UNSUPPORTED, "arrival-order logs take fixed 64-byte records");
  int32_t rc = before_load(e); if (rc) return rc;
  CUDA_TRY(e, e->inc_records.reserve(n_records * 64));
  CUDA_TRY(e, cudaEventRecord(e->ev2, e->stream));
  CUDA_TRY(e, cudaMemcpyAsync(e->inc_records.p, records, n_records * 64, cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(e, cudaEventRecord(e->ev3, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  CUDA_TRY(e, cudaEventElapsedTime(&e->stats.ms_h2d, e->ev2, e->ev3));
  return fold_arrival_order(e, (const uint8_t*)e->inc_records.p, n_records, n_agg);
}

// ------------------------------------------------------------------ multi-GPU
int32_t sgr_dist_unique_id(void* out128) {
  if (!out128) return SGR_ERR_INVALID;
  std::string err;
  int rc = dist_unique_id(out128, &err);
  if (rc) return fail(nullptr, rc, "%s", err.c_str());
  return SGR_OK;
}

int32_t sgr_dist_init(sgr_engine* e, int32_t rank, int32_t nranks, const void* unique_id128, uint64_t recv_capacity_records) {
  OpLock op_lock(e);
  if (!e) return fail(e, SGR_ERR_INVALID, "null argument");   // unique_id128 == NULL with nranks > 1: a loopback rank (sgr.h)
  int32_t rc = use_device(e); if (rc) return rc;
  if (e->dist) { dist_destroy(e->dist); e->dist = nullptr; }
  e->dist = dist_create();
  std::string err;
  int r = dist_init(e->dist, rank, nranks, unique_id128, recv_capacity_records, e->stream, &err);
  if (r) return fail(e, r, "%s", err.c_str());
  return SGR_OK;
}

int32_t sgr_dist_set_partitions(sgr_engine* e, const uint32_t* partition_of_agg, uint64_t n_global_agg) {
  OpLock op_lock(e);
  if (!e || !partition_of_agg) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->dist) return fail(e, SGR_ERR_NOT_LOADED, "call sgr_dist_init first");
  int32_t rc = before_load(e); if (rc) return rc;
  std::string err;
  int r = dist_set_partitions(e->dist, partition_of_agg, n_global_agg, e->stream, &err);
  if (r) return fail(e, r, "%s", err.c_str());
  return SGR_OK;
}

int32_t sgr_dist_ipc_export(sgr_engine* e, void* out64) {
  OpLock op_lock(e);
  if (!e || !out64 || !e->dist) return fail(e, SGR_ERR_INVALID, "null argument / no dist state");
  int32_t rc = use_device(e); if (rc) return rc;
  std::string err;
  int r = dist_ipc_export(e->dist, out64, &err);
  if (r) return fail(e, r, "%s", err.c_str());
  return SGR_OK;
}

int32_t sgr_dist_ipc_import(sgr_engine* e, const void* handles64_by_rank) {
  OpLock op_lock(e);
  if (!e || !handles64_by_rank || !e->dist) return fail(e, SGR_ERR_INVALID, "null argument / no dist state");
  int32_t rc = use_device(e); if (rc) return rc;
  std::string err;
  int r = dist_ipc_import(e->dist, handles64_by_rank, &err);
  if (r) return fail(e, r, "%s", err.c_str());
  return SGR_OK;
}

int32_t sgr_dist_route_and_fold(sgr_engine* e, const void* d_records, uint64_t n_records, int32_t fused) {
  OpLock op_lock(e);
  if (!e || (!d_records && n_records)) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program first");
  if (!e->dist) return fail(e, SGR_ERR_NOT_LOADED, "call sgr_dist_init first");
  if (e->program.record_kind != SGR_REC_FIXED64) return fail(e, SGR_ERR_UNSUPPORTED, "routing takes fixed 64-byte records");
  int32_t rc = before_load(e); if (rc) return rc;
  std::string err;
  uint64_t n_recv = 0;
  e->stats.ms_h2d = 0;
  const bool routed = dist_nranks(e->dist) > 1 || e->opt_force_route;
  // fused >= 2: pipelined push (route + exchange + fold overlapped, route_push.cu); 3 = exchange only the words the program reads.
  // Programs outside the sort-free formulation take the scatter + group-by path below (every rank holds the same program).
  if (routed && fused >= 2 && e->bulk_ok && e->opt_incremental != 1) {
    const uint64_t n_local = dist_n_local(e->dist);
    rc = ensure_states(e, n_local); if (rc) return rc;
    rc = ensure_bulk_buffers(e, n_local); if (rc) return rc;
    CUDA_TRY(e, cudaMemsetAsync(e->states.p, 0, (size_t)n_local * e->program.state_bytes, e->stream));
    e->states_valid = true; e->states_invalidated = false; e->loaded = false; e->inc_atomic_prev_valid = false; e->inc_prev_n = 0;
    PushFoldArgs pf{};
    pf.prog = &e->row_prog; pf.lay = &e->bulk_lay; pf.scratch = e->bulk_scratch.p; pf.states = (uint8_t*)e->states.p;
    pf.err_ids = (uint32_t*)e->bulk_err_ids.p; pf.counters = (unsigned long long*)e->bulk_counters.p; pf.n_slots = n_local;
    pf.n_chunks = (uint32_t)e->opt_push_chunks; pf.compact = fused == 3; pf.num_sms = e->num_sms;
    // First attempt: CTAs place their records with atomics and the records carry their own arrival index — nothing waits for
    // anything. The exact replay of a throwing aggregate needs the records in POSITIONAL log order, so if any rank saw one,
    // every rank runs the exchange again in ordered mode (look-back) and replays from that. Throwing events are the exception.
    pf.ordered = e->opt_push_ordered != 0;
    PushFoldResult res;
    int r = dist_push_fold(e->dist, (const uint8_t*)d_records, n_records, pf, e->stream, &res, &err);
    if (r) { e->states_valid = false; e->bulk_scratch_slots = 0; return fail(e, r, "%s", err.c_str()); }
    if (!pf.ordered && res.any_err_slots) {
      if (dist_is_loopback(e->dist)) {   // loopback ranks have no collective to agree over: the caller does (sgr.h)
        e->states_valid = false;
        return fail(e, SGR_ERR_AGAIN, "throwing aggregates: every rank must repeat the call with option push_ordered = 1");
      }
      CUDA_TRY(e, cudaMemsetAsync(e->states.p, 0, (size_t)n_local * e->program.state_bytes, e->stream));
      pf.ordered = true;
      r = dist_push_fold(e->dist, (const uint8_t*)d_records, n_records, pf, e->stream, &res, &err);
      if (r) { e->states_valid = false; e->bulk_scratch_slots = 0; return fail(e, r, "%s", err.c_str()); }
    }
    unsigned long long throwing = 0, dropped = 0;
    if (res.n_err_slots) {
      const uint8_t* contiguous = nullptr;
      r = dist_gather_regions(e->dist, res, e->row_prog, e->stream, &contiguous, &err);
      if (r) return fail(e, r, "%s", err.c_str());
      rc = replay_throwing_slots(e, contiguous, res.n_recv, n_local, (const uint32_t*)e->bulk_err_ids.p, res.n_err_slots, &throwing, &dropped);
      if (rc) return rc;
    }
    e->stats.ms_group = 0; e->stats.ms_fold = res.ms_total - res.ms_push;   // what the fold adds behind the last push
    e->stats.n_aggregates = n_local; e->stats.n_errors = throwing; e->stats.n_events = res.n_recv - dropped;
    e->stats.event_bytes = res.n_recv * 64; e->stats.n_long_segments = 0; e->stats.fold_launches = 2 * (uint32_t)e->opt_push_chunks + 1;
    e->stats.algorithmic_bytes = res.n_recv * 64 + (uint64_t)(16 + 2 * e->program.state_bytes) * n_local;
    mark_dirty(e);
    const DistStats* ds = dist_stats(e->dist);
    e->dstats = sgr_dist_stats{};
    e->dstats.n_sent = ds->n_sent; e->dstats.n_sent_remote = ds->n_sent_remote; e->dstats.n_recv = ds->n_recv;
    e->dstats.n_local_aggregates = n_local;
    e->dstats.ms_scatter = res.ms_push; e->dstats.ms_fold = e->stats.ms_fold;
    e->dstats.ms_pipeline = res.ms_total; e->dstats.exchange_record_bytes = res.out_bytes;
    return SGR_OK;
  }
  if (fused >= 2) fused = dist_nranks(e->dist) > 1 ? 1 : 0;
  if (!routed) {
    // one rank owns everything and local index == global index: no exchange
    dist_clear_stats(e->dist, n_records);
  } else {
    int r = dist_route(e->dist, (const uint8_t*)d_records, n_records, fused != 0, (unsigned long long*)e->counters.p, e->stream, &n_recv, &err);
    if (r) return fail(e, r, "%s", err.c_str());
  }
  const uint8_t* arrived = !routed ? (const uint8_t*)d_records : dist_recv_buffer(e->dist);
  const uint64_t n_arrived = !routed ? n_records : n_recv;
  rc = fold_arrival_order(e, arrived, n_arrived, dist_n_local(e->dist));
  if (rc) return rc;
  const DistStats* ds = dist_stats(e->dist);
  e->dstats = sgr_dist_stats{};
  e->dstats.n_sent = ds->n_sent; e->dstats.n_sent_remote = ds->n_sent_remote; e->dstats.n_recv = ds->n_recv;
  e->dstats.n_local_aggregates = dist_n_local(e->dist);
  e->dstats.ms_count = ds->ms_count; e->dstats.ms_counts_exchange = ds->ms_counts_exchange;
  e->dstats.ms_scatter = ds->ms_scatter; e->dstats.ms_exchange = ds->ms_exchange;
  e->dstats.ms_group = e->stats.ms_group; e->dstats.ms_fold = e->stats.ms_fold;
  return SGR_OK;
}

int32_t sgr_dist_get_stats(sgr_engine* e, sgr_dist_stats* out) {
  if (!e || !out) return SGR_ERR_INVALID;
  *out = e->dstats;
  return SGR_OK;
}

int32_t sgr_dist_local_aggregates(sgr_engine* e, uint32_t* out, uint64_t cap, uint64_t* n_local) {
  OpLock op_lock(e);
  if (!e || !e->dist) return fail(e, SGR_ERR_INVALID, "no dist state");
  const uint64_t n = dist_n_local(e->dist);
  if (n_local) *n_local = n;
  if (out) {
    if (cap < n) return fail(e, SGR_ERR_CAPACITY, "need room for %llu indices", (unsigned long long)n);
    int32_t rc = use_device(e); if (rc) return rc;
    CUDA_TRY(e, cudaMemcpyAsync(out, dist_global_of_local(e->dist), n * 4, cudaMemcpyDeviceToHost, e->stream));
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  }
  return SGR_OK;
}

int32_t sgr_dist_set_peers(sgr_engine* e, void* const* recv_bases_by_rank) {
  OpLock op_lock(e);
  if (!e || !recv_bases_by_rank || !e->dist) return fail(e, SGR_ERR_INVALID, "null argument / no dist state");
  std::string err;
  int r = dist_set_peers(e->dist, recv_bases_by_rank, &err);
  if (r) return fail(e, r, "%s", err.c_str());
  return SGR_OK;
}

int32_t sgr_dist_reserve(sgr_engine* e, uint64_t max_records) {
  OpLock op_lock(e);
  if (!e || !e->dist) return fail(e, SGR_ERR_INVALID, "null argument / no dist state");
  if (!e->has_program) return fail(e, SGR_ERR_NO_PROGRAM, "register a fold program first");
  int32_t rc = use_device(e); if (rc) return rc;
  rc = before_load(e); if (rc) return rc;
  const uint64_t n_local = dist_n_local(e->dist);
  rc = ensure_states(e, n_local); if (rc) return rc;
  if (e->bulk_ok) { rc = ensure_bulk_buffers(e, n_local); if (rc) return rc; }
  std::string err;
  int r = dist_push_reserve(e->dist, max_records, (uint32_t)e->opt_push_chunks, &err);
  if (r) return fail(e, r, "%s", err.c_str());
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  return SGR_OK;
}

int32_t sgr_dist_recv_base(sgr_engine* e, void** base) {
  if (!e || !base || !e->dist) return fail(e, SGR_ERR_INVALID, "null argument / no dist state");
  *base = dist_recv_base(e->dist);
  return SGR_OK;
}

int32_t sgr_states_hash(sgr_engine* e, uint64_t* out) {
  OpLock op_lock(e);
  if (!e || !out) return fail(e, SGR_ERR_INVALID, "null argument");
  if (!e->states_valid) return fail(e, SGR_ERR_STATE, "no folded state table");
  int32_t rc = use_device(e); if (rc) return rc;
  rc = finish_fold(e); if (rc) return rc;
  CUDA_TRY(e, e->hash_out.reserve(64));
  // a routed table is hashed under its GLOBAL aggregate indices, so the sum over the ranks does not depend on their number
  const uint32_t* gids = (e->dist && (dist_nranks(e->dist) > 1 || e->opt_force_route) && dist_n_local(e->dist) == e->states_n) ? dist_global_of_local(e->dist) : nullptr;
  cudaError_t ce = launch_states_hash((const uint8_t*)e->states.p, e->states_n, e->program.state_bytes, gids, (unsigned long long*)e->hash_out.p, e->stream);
  if (ce != cudaSuccess) return fail(e, SGR_ERR_CUDA, "hash launch: %s", cudaGetErrorString(ce));
  unsigned long long h = 0;
  CUDA_TRY(e, cudaMemcpyAsync(&h, e->hash_out.p, 8, cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(e, cudaStreamSynchronize(e->stream));
  *out = h;
  return SGR_OK;
}

int32_t sgr_set_option(sgr_engine* e, const char* name, int64_t value) {
  if (!e || !name) return SGR_ERR_INVALID;
  if (!strcmp(name, "fold_variant")) { e->opt_variant = value; return SGR_OK; }
  if (!strcmp(name, "kernel")) { e->opt_kernel = value; return SGR_OK; }
  if (!strcmp(name, "incremental")) { e->opt_incremental = value; return SGR_OK; }
  if (!strcmp(name, "force_route")) { e->opt_force_route = value; return SGR_OK; }
  if (!strcmp(name, "bulk")) { e->opt_bulk = value; return SGR_OK; }
  if (!strcmp(name, "bulk_unroll")) { bulk_tuning().unroll = (int)value; return SGR_OK; }
  if (!strcmp(name, "bulk_hints")) { bulk_tuning().hints = (int)value; return SGR_OK; }
  if (!strcmp(name, "bulk_blocks_per_sm")) { bulk_tuning().blocks_per_sm = (int)value; return SGR_OK; }
  if (!strcmp(name, "push_tile")) {
    if (value != 256 && value != 512 && value != 1024) return fail(e, SGR_ERR_INVALID, "push_tile must be 256, 512 or 1024");
    push_tuning().tile = (int)value; return SGR_OK;
  }
  if (!strcmp(name, "push_fold_blocks_per_sm")) { push_tuning().fold_blocks_per_sm = (int)value; return SGR_OK; }
  if (!strcmp(name, "push_ordered")) { e->opt_push_ordered = value ? 1 : 0; return SGR_OK; }
  if (!strcmp(name, "push_staged")) { push_tuning().staged = (int)value; return SGR_OK; }
  if (!strcmp(name, "push_pull")) { push_tuning().pull = value ? 1 : 0; return SGR_OK; }
  if (!strcmp(name, "push_chunks")) {
    if (value < 1 || value > 256) return fail(e, SGR_ERR_INVALID, "push_chunks must be in [1, 256]");
    e->opt_push_chunks = value; return SGR_OK;
  }
  if (!strcmp(name, "replay_budget")) { e->opt_replay_budget = value; return SGR_OK; }
  if (!strcmp(name, "var_stage_bytes")) { e->opt_var_stage_bytes = value; return SGR_OK; }
  if (!strcmp(name, "var_stages")) { e->opt_var_stages = (value >= 1 && value <= 3) ? value : 2; return SGR_OK; }
  if (!strcmp(name, "run_variant")) {
    if (value < 0 || value >= run_variant_count()) return fail(e, SGR_ERR_INVALID, "run_variant out of range");
    e->opt_run_variant = value; return SGR_OK;
  }
  if (!strcmp(name, "long_threshold")) { e->opt_long_threshold = value; return SGR_OK; }
  if (!strcmp(name, "max_record_bytes")) {
    if (value < 16 || value > 2048 + 16) return fail(e, SGR_ERR_INVALID, "max_record_bytes must be in [16, 2064]");
    e->opt_max_record_bytes = value; return SGR_OK;
  }
  return fail(e, SGR_ERR_INVALID, "unknown option '%s'", name);
}

int32_t sgr_stream(sgr_engine* e, void** stream) {
  if (!e || !stream) return SGR_ERR_INVALID;
  *stream = (void*)e->stream;
  return SGR_OK;
}

}  // extern "C"
