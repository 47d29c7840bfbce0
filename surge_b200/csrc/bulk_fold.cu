// bulk_fold.cu — sort-free fold of a LARGE arrival-order log (sm_100a): the K6 formulation of incremental.cu as two
// plain launches, for logs much larger than the state table (a whole Kafka partition log, or what arrives from the
// other ranks after routing).
//
// Contract: events.foldLeft(state)(handleEvent) per aggregate (modules/command-engine/scaladsl/src/main/scala/surge/
// scaladsl/command/CommandModels.scala:25-28) with the actor rules of PersistentActor.doApplyEvent
// (modules/command-engine/core/src/main/scala/surge/internal/persistence/PersistentActor.scala:245-264) on a log in which
// aggregates are interleaved but every aggregate's own events keep their order (one key -> one Kafka partition).
//
// For 16-byte class-0 programs whose state words are each add-only or set-only the left fold has the closed form
//     add-only word' = old + sum of the ADDs              (i32 wrap-adds commute)
//     set-only word' = value of the LAST SET, else old    (last by arrival index)
//     exists'        = exists-op of the aggregate's LAST event
// so integer atomics on a small per-slot scratch entry give the exact result in any execution order:
//   accumulate   one pass over the records, 64 B read per record (streamed through L2 with evict-first), 2-3 RED ops on
//                the slot's 16-byte entry (kept in L2 with evict-last): no sort, no grouped copy of the log
//   finish       one pass over the SLOTS: entry + prior state -> state, CHANGED, entry zeroed for the next fold
// A slot that saw a throwing event (handler exception / MatchError) keeps its state and is queued; the caller replays
// exactly those slots sequentially (exact err_idx), see engine.cu.
//
// Algorithmic bytes per launch: 64 * n_records (accumulate) + (16 scratch + 16 state in + 16 state out) * n_slots (finish).
#include "bulk_fold.cuh"

#include "../../include/sgr.h"

namespace sgr {
namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// HINTS: records stream through L2 (evict-first), the scratch entries are asked to stay (evict-last)
template <bool HINTS>
__device__ __forceinline__ uint4 ldg_stream(const void* p, uint64_t pol) {
  uint4 v;
  if (HINTS) asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                          : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
  else asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
// one 32-byte sector in one request (LDG.256): the two halves of a record's first sector never travel twice — matters when
// the records are read from a peer over NVLink
template <bool HINTS>
__device__ __forceinline__ void ldg_stream32(const void* p, uint64_t pol, uint4& a, uint4& b) {
  if (HINTS) asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                          : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p), "l"(pol));
  else asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                    : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}
template <bool HINTS>
__device__ __forceinline__ void red_add_u32(uint32_t* p, uint32_t v, uint64_t pol) {
  if (HINTS) asm volatile("red.relaxed.gpu.global.add.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
  else asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
template <bool HINTS>
__device__ __forceinline__ void red_max_u32(uint32_t* p, uint32_t v, uint64_t pol) {
  if (HINTS) asm volatile("red.relaxed.gpu.global.max.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
  else asm volatile("red.relaxed.gpu.global.max.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
template <bool HINTS>
__device__ __forceinline__ void red_max_u64(unsigned long long* p, unsigned long long v, uint64_t pol) {
  if (HINTS) asm volatile("red.relaxed.gpu.global.max.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(p), "l"(v), "l"(pol) : "memory");
  else asm volatile("red.relaxed.gpu.global.max.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// word w (0..7) of the 32 bytes held in (a, b)
__device__ __forceinline__ uint32_t pick8(const uint4& a, const uint4& b, uint32_t w) {
  const uint32_t lo = (w & 2u) ? ((w & 1u) ? a.w : a.z) : ((w & 1u) ? a.y : a.x);
  const uint32_t hi = (w & 2u) ? ((w & 1u) ? b.w : b.z) : ((w & 1u) ? b.y : b.x);
  return (w & 4u) ? hi : lo;
}

struct BulkArgs {
  BulkSrc src;
  uint64_t n_slots;
  uint8_t* scr;
  uint32_t* throw_bits;
  unsigned long long* counters;
  BulkLayout lay;
};

struct RecView {
  uint4 q0, q1;
  const uint8_t* p;
  bool live;
};

template <bool HINTS>
__device__ __forceinline__ void load_rec(RecView& r, const uint8_t* p, bool live, bool two, uint64_t pol) {
  r.p = p; r.live = live;
  if (live) {
    if (two) ldg_stream32<HINTS>(p, pol, r.q0, r.q1);
    else { r.q0 = ldg_stream<HINTS>(p, pol); r.q1 = make_uint4(0, 0, 0, 0); }
  }
}

template <bool COMPACT, bool HINTS>
__device__ __forceinline__ void apply_rec(const RecView& r, uint32_t idx1, uint32_t ib, const BulkArgs& a, const RowProgram& pg,
                                          const uint32_t* tab, uint64_t pol_last) {
  if (!r.live) return;
  unsigned long long slot;
  uint32_t type;
  if (COMPACT) { slot = r.q0.x; type = r.q0.y >> 27; idx1 = ib + (r.q0.y & 0x07ffffffu); }
  else if (a.src.carried) { slot = r.q0.z; type = r.q0.x; idx1 = ib + r.q0.w; }
  else { slot = ((unsigned long long)r.q0.w << 32) | r.q0.z; type = r.q0.x; }
  if (slot == ~0ull) { atomicAdd(a.counters + 0, 1ull); return; }   // a hole: a record the device decode dropped in place (flush marker, duplicate, null value)
  if (slot >= a.n_slots) { atomicAdd(a.counters + 4, 1ull); return; }
  uint8_t* entry = a.scr + (slot << a.lay.entry_shift);
  const uint32_t fl = type < 16u ? tab[type * kTabStride] : 0u;
  if (!(fl & 1u)) {   // handler exception / MatchError: sticky mark, the slot is replayed exactly afterwards
    atomicOr(a.throw_bits + (slot >> 5), 1u << (slot & 31u));
    return;
  }
#pragma unroll
  for (int w = 0; w < 2; ++w) {
    const uint32_t spec = tab[type * kTabStride + 1 + w];
    const uint32_t mode = spec & 3u, s = spec >> 3;
    if (!mode) continue;
    uint32_t v = 0;
    if (s) {
      const uint32_t rw = COMPACT ? 1u + s : pg.slot_word[s];
      v = rw < 8u ? pick8(r.q0, r.q1, rw) : __ldg(reinterpret_cast<const uint32_t*>(r.p) + rw);
    }
    if (spec & 4u) v = 0u - v;
    if (mode == 1u) { if (v) red_add_u32<HINTS>(reinterpret_cast<uint32_t*>(entry + a.lay.word_off[w]), v, pol_last); }
    else red_max_u64<HINTS>(reinterpret_cast<unsigned long long*>(entry + a.lay.word_off[w]), ((unsigned long long)idx1 << 32) | v, pol_last);
  }
  if ((a.lay.last_needed_mask >> type) & 1u)
    red_max_u32<HINTS>(reinterpret_cast<uint32_t*>(entry), (idx1 << 2) | ((fl & 2u) ? 2u : 1u), pol_last);
}

template <bool COMPACT, bool HINTS, int kUnroll>
__global__ void __launch_bounds__(kThreads) bulk_accumulate_kernel(const __grid_constant__ BulkArgs a, const __grid_constant__ RowProgram pg) {
  __shared__ uint32_t tab[16 * kTabStride];
  for (int i = threadIdx.x; i < 16 * kTabStride; i += kThreads) tab[i] = pg.tab[i];
  __syncthreads();
  const uint64_t pol_first = policy_evict_first(), pol_last = policy_evict_last();
  const uint32_t stride = a.src.rec_bytes;
  // the second 16 bytes are needed when a slot word lies there (full records: `by` at word 4; compact: records wider than 16 B)
  bool two = COMPACT ? stride > 16u : false;
  if (!COMPACT) for (uint32_t s = 1; s < pg.n_slots; ++s) two |= pg.slot_word[s] >= 4u;
  // record counts of the regions (given, or published by the sender in an arrival flag)
  __shared__ uint64_t n_of[kMaxRanks];
  __shared__ uint64_t n_max;
  if (threadIdx.x < a.src.n_regions) {
    const uint32_t rg = threadIdx.x;
    uint64_t n = a.src.count[rg];
    if (a.src.count_flag[rg]) {   // (epoch << 32) | count + 1; 0xffffffff = the sender gave up on this region
      const uint32_t f = (uint32_t)ld_acquire_sys_u64(a.src.count_flag[rg]);
      const uint64_t got = (f == 0xffffffffu || f == 0u) ? 0ull : (uint64_t)(f - 1u);
      n = got < n ? got : n;
    }
    n_of[rg] = n;
  }
  __syncthreads();
  if (threadIdx.x == 0) { uint64_t m = 0; for (uint32_t rg = 0; rg < a.src.n_regions; ++rg) m = n_of[rg] > m ? n_of[rg] : m; n_max = m; }
  __syncthreads();
  // tiles of kThreads * kUnroll records; consecutive tiles rotate over the regions (starting at `rotate`), so the regions —
  // one per source rank when they are read over NVLink — are all in flight together instead of one peer at a time
  constexpr uint32_t kTile = kThreads * kUnroll;
  const uint32_t R = a.src.n_regions;
  const uint64_t tiles_per_region = (n_max + kTile - 1) / kTile, total = tiles_per_region * R;
  for (uint64_t T = blockIdx.x; T < total; T += gridDim.x) {
    const uint32_t rg = (uint32_t)((T + a.src.rotate) % R);
    const uint64_t n = n_of[rg], i0 = (T / R) * kTile + threadIdx.x;
    if ((T / R) * kTile >= n) continue;
    const uint8_t* base = a.src.base[rg];
    const uint32_t ib = a.src.idx_base[rg] + 1u;
    RecView r[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint64_t i = i0 + (uint64_t)u * kThreads;
      load_rec<HINTS>(r[u], base + i * stride, i < n, two, pol_first);
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) apply_rec<COMPACT, HINTS>(r[u], ib + (uint32_t)(i0 + (uint64_t)u * kThreads), ib, a, pg, tab, pol_last);
  }
}

struct FinishArgs {
  uint64_t n_slots;
  uint8_t* scr;
  uint32_t* throw_bits;
  uint8_t* states;
  uint32_t* err_ids;
  unsigned long long* counters;
  BulkLayout lay;
};

__global__ void __launch_bounds__(kThreads) bulk_finish_kernel(const __grid_constant__ FinishArgs a) {
  const uint64_t nthreads = (uint64_t)gridDim.x * kThreads;
  const int lane = threadIdx.x & 31;
  const uint64_t n_round = (a.n_slots + 31) & ~31ull;   // whole warps: a warp covers exactly one word of the throw bitmap
  const bool rejected = a.counters[4] != 0;             // a record with a slot out of range: nothing is applied
  for (uint64_t slot = (uint64_t)blockIdx.x * kThreads + threadIdx.x; slot < n_round; slot += nthreads) {
    uint32_t tw = 0;
    if (lane == 0) { tw = a.throw_bits[slot >> 5]; if (tw) a.throw_bits[slot >> 5] = 0u; }
    tw = __shfl_sync(0xffffffffu, tw, 0);
    if (slot >= a.n_slots) continue;
    const bool threw = (tw >> lane) & 1u;
    uint8_t* entry = a.scr + (slot << a.lay.entry_shift);
    uint4 e0 = *reinterpret_cast<const uint4*>(entry), e1 = make_uint4(0, 0, 0, 0);
    if (a.lay.entry_shift == 5) e1 = reinterpret_cast<const uint4*>(entry)[1];
    const bool touched = (e0.x | e0.y | e0.z | e0.w | e1.x | e1.y | e1.z | e1.w) != 0u;
    if (!touched && !threw) continue;
    if (touched) {
      *reinterpret_cast<uint4*>(entry) = make_uint4(0, 0, 0, 0);
      if (a.lay.entry_shift == 5) reinterpret_cast<uint4*>(entry)[1] = make_uint4(0, 0, 0, 0);
    }
    if (rejected) continue;
    if (threw) { a.err_ids[atomicAdd(a.counters + 3, 1ull)] = (uint32_t)slot; continue; }
    const uint32_t ew[8] = {e0.x, e0.y, e0.z, e0.w, e1.x, e1.y, e1.z, e1.w};
    uint4* st = reinterpret_cast<uint4*>(a.states + slot * 16);
    const uint4 old = *st;
    const uint32_t ex0 = old.z & SGR_ST_EXISTS;
    const uint32_t exn = (a.lay.has_none && (e0.x & 3u) == 2u) ? 0u : SGR_ST_EXISTS;
    const uint32_t b[2] = {ex0 ? old.x : 0u, ex0 ? old.y : 0u};
    uint32_t nv[2];
#pragma unroll
    for (int w = 0; w < 2; ++w) {
      const uint32_t c = a.lay.word_off[w] >> 2;   // cell's first word inside the entry
      uint32_t lo = 0, hi = 0;
#pragma unroll
      for (int k = 1; k < 8; ++k) { if ((uint32_t)k == c) lo = ew[k]; if ((uint32_t)k == c + 1u) hi = ew[k]; }
      nv[w] = ((a.lay.set_only_mask >> w) & 1u) ? (hi ? lo : b[w]) : b[w] + lo;
    }
    if (!exn) { nv[0] = 0; nv[1] = 0; }
    uint32_t changed = exn != ex0;
    if (exn && ex0) changed |= (nv[0] != old.x) | (nv[1] != old.y);
    *st = make_uint4(nv[0], nv[1], exn | (changed ? SGR_ST_CHANGED : 0u), 0u);
  }
}

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void __launch_bounds__(kThreads) states_hash_kernel(const uint8_t* __restrict__ states, uint64_t n, uint32_t state_bytes,
                                                               const uint32_t* __restrict__ gids, unsigned long long* __restrict__ out) {
  unsigned long long acc = 0;
  const uint64_t nthreads = (uint64_t)gridDim.x * kThreads;
  for (uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += nthreads) {
    unsigned long long h = splitmix64(gids ? (unsigned long long)gids[i] : i);
    const unsigned long long* p = reinterpret_cast<const unsigned long long*>(states + i * state_bytes);
    for (uint32_t k = 0; k < state_bytes / 8; ++k) h = splitmix64(h ^ p[k]);
    acc += h;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

int grid_for(int num_sms, uint64_t work_items, int per_sm) {
  uint64_t want = (work_items + kThreads - 1) / kThreads;
  const uint64_t cap = (uint64_t)num_sms * per_sm;
  if (want > cap) want = cap;
  return want ? (int)want : 1;
}

}  // namespace

BulkTuning& bulk_tuning() { static BulkTuning t; return t; }

cudaError_t bulk_preload_kernels() {
  cudaFuncAttributes fa;
  cudaError_t e;
#define SGR_TOUCH(...) if ((e = cudaFuncGetAttributes(&fa, __VA_ARGS__)) != cudaSuccess) return e;
#define SGR_TOUCH_U(C, H) SGR_TOUCH(bulk_accumulate_kernel<C, H, 1>) SGR_TOUCH(bulk_accumulate_kernel<C, H, 2>) SGR_TOUCH(bulk_accumulate_kernel<C, H, 4>)
  SGR_TOUCH_U(true, true) SGR_TOUCH_U(true, false) SGR_TOUCH_U(false, true) SGR_TOUCH_U(false, false)
  SGR_TOUCH(bulk_finish_kernel) SGR_TOUCH(states_hash_kernel)
#undef SGR_TOUCH_U
#undef SGR_TOUCH
  return cudaSuccess;
}

bool bulk_layout_for(const RowProgram& prog, BulkLayout* out) {
  if (prog.user_words != 2 || prog.cls != 0 || prog.f64_mask || prog.slot_word[0] != 0) return false;
  uint32_t has_add = 0, has_set = 0, has_none = 0;
  for (int t = 0; t < 16; ++t) {
    const uint32_t fl = prog.tab[t * kTabStride];
    if (!(fl & 1u)) continue;
    if (fl & 2u) has_none = 1;
    for (int w = 0; w < 2; ++w) {
      const uint32_t mode = prog.tab[t * kTabStride + 1 + w] & 3u;
      if (mode == 1u) has_add |= 1u << w;
      if (mode == 2u) has_set |= 1u << w;
    }
  }
  if (has_add & has_set) return false;
  BulkLayout l{};
  l.set_only_mask = has_set; l.has_none = has_none;
  // cells: `last` at +0; add-only words take 4 bytes, set-only words 8 (8-byte aligned)
  const int n_set = __builtin_popcount(has_set & 3u);
  if (n_set == 2) { l.entry_shift = 5; l.word_off[0] = 8; l.word_off[1] = 16; }
  else if (n_set == 1) {
    l.entry_shift = 4;
    const int ws = (has_set & 1u) ? 0 : 1;
    l.word_off[ws] = 8; l.word_off[ws ^ 1] = 4;
  } else { l.entry_shift = 4; l.word_off[0] = 4; l.word_off[1] = 8; }
  for (int t = 0; t < 16; ++t) {
    const uint32_t fl = prog.tab[t * kTabStride];
    if (!(fl & 1u)) continue;
    bool sets = false;
    for (int w = 0; w < 2; ++w) sets |= (prog.tab[t * kTabStride + 1 + w] & 3u) == 2u;
    if (has_none || !sets) l.last_needed_mask |= 1u << t;
  }
  *out = l;
  return true;
}

size_t bulk_scratch_bytes(const BulkLayout& lay, uint64_t n_slots) {
  return ((size_t)n_slots << lay.entry_shift) + ((n_slots + 31) / 32) * 4 + 256;
}

static uint32_t* throw_bits_of(void* scratch, const BulkLayout& lay, uint64_t n_slots) {
  return reinterpret_cast<uint32_t*>((uint8_t*)scratch + ((((size_t)n_slots << lay.entry_shift) + 127) & ~(size_t)127));
}

cudaError_t launch_bulk_accumulate(const BulkSrc& src, uint64_t n_slots, void* d_scratch, const RowProgram& prog, const BulkLayout& lay,
                                   unsigned long long* d_counters, int num_sms, cudaStream_t st) {
  BulkArgs a{};
  a.src = src; a.n_slots = n_slots; a.scr = (uint8_t*)d_scratch; a.throw_bits = throw_bits_of(d_scratch, lay, n_slots);
  a.counters = d_counters; a.lay = lay;
  uint64_t work = 0;
  for (uint32_t r = 0; r < src.n_regions; ++r) work += src.count[r];
  if (!work) return cudaSuccess;
  const BulkTuning& t = bulk_tuning();
  const int unroll = t.unroll == 1 || t.unroll == 2 ? t.unroll : 4;
  // blocks_per_sm == ~0: one tile per CTA (many short CTAs: a low-priority launch then yields to a concurrent high-priority kernel
  // at CTA granularity instead of squatting on the SMs with a persistent grid)
  int grid;
  if (src.blocks_per_sm == 0xffffffffu) {
    uint64_t mx = 0;
    for (uint32_t r = 0; r < src.n_regions; ++r) mx = mx > src.count[r] ? mx : src.count[r];
    const uint64_t tiles = (mx + (uint64_t)kThreads * unroll - 1) / ((uint64_t)kThreads * unroll) * src.n_regions;
    grid = (int)(tiles < 0x7fffffffull ? (tiles ? tiles : 1) : 0x7fffffffull);
  } else {
    grid = grid_for(num_sms, (work + unroll - 1) / unroll, src.blocks_per_sm ? (int)src.blocks_per_sm : (t.blocks_per_sm > 0 ? t.blocks_per_sm : 8));
  }
#define SGR_BULK_LAUNCH(C, H, U) bulk_accumulate_kernel<C, H, U><<<grid, kThreads, 0, st>>>(a, prog)
#define SGR_BULK_U(C, H) (unroll == 1 ? SGR_BULK_LAUNCH(C, H, 1) : unroll == 2 ? SGR_BULK_LAUNCH(C, H, 2) : SGR_BULK_LAUNCH(C, H, 4))
  if (src.compact) { if (t.hints) SGR_BULK_U(true, true); else SGR_BULK_U(true, false); }
  else { if (t.hints) SGR_BULK_U(false, true); else SGR_BULK_U(false, false); }
#undef SGR_BULK_U
#undef SGR_BULK_LAUNCH
  return cudaGetLastError();
}

cudaError_t launch_bulk_finish(uint64_t n_slots, void* d_scratch, uint8_t* d_states, uint32_t* d_err_ids, const BulkLayout& lay,
                               unsigned long long* d_counters, cudaStream_t st) {
  if (!n_slots) return cudaSuccess;
  FinishArgs a{};
  a.n_slots = n_slots; a.scr = (uint8_t*)d_scratch; a.throw_bits = throw_bits_of(d_scratch, lay, n_slots); a.states = d_states;
  a.err_ids = d_err_ids; a.counters = d_counters; a.lay = lay;
  uint64_t want = (n_slots + kThreads - 1) / kThreads;
  if (want > 148ull * 16) want = 148ull * 16;
  bulk_finish_kernel<<<(int)want, kThreads, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_states_hash(const uint8_t* d_states, uint64_t n_slots, uint32_t state_bytes, const uint32_t* d_global_ids,
                               unsigned long long* d_out, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(d_out, 0, 8, st);
  if (e != cudaSuccess || !n_slots) return e;
  uint64_t want = (n_slots + kThreads - 1) / kThreads;
  if (want > 148ull * 8) want = 148ull * 8;
  states_hash_kernel<<<(int)want, kThreads, 0, st>>>(d_states, n_slots, state_bytes, d_global_ids, d_out);
  return cudaGetLastError();
}

}  // namespace sgr
