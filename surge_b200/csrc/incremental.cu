// incremental.cu — K6: append a micro-batch (arrival order) to the live state table without sorting (sm_100a).
//
// Contract: for every aggregate touched by the batch, ApplyEvents(id, its events in arrival order) on the live
// actor state — PersistentActor.doApplyEvent, modules/command-engine/core/src/main/scala/surge/internal/persistence/
// PersistentActor.scala:245-264 (publish iff changed :257, handler exception => state kept :260-263).
//
// For programs inside the transformer algebra (fold_rows.cuh) the left-to-right fold of one aggregate's events has
// a closed form that needs no grouping:
//     word' = (a SET exists ? value of the LAST SET : old) + sum of the ADDs that come AFTER the last SET   (i32 wrap)
//     exists' = exists-op of the aggregate's LAST event
// "last" is by arrival index, wrap-adds commute, so integer atomics give the exact result in any execution order:
//   pass A   atomicMax(last_event[slot]), atomicMax(last_set[slot][w])            (arrival index + 1)
//   pass B   ADD after the last SET -> atomicAdd(acc[slot][w]); the unique last SET stores its value;
//            the unique last event stores its exists-op
//   pass C   the unique last event of each touched slot finishes it: applies (set, acc) to the prior state, sets
//            CHANGED, appends the slot to the touched list (whose per-batch flags the NEXT batch clears) and zeroes
//            the slot's scratch. A slot that saw a throwing event is queued instead and replayed strictly
//            sequentially by one warp (exact err_idx, state kept), pass D.
// The scratch (32 B per slot) and the table stay L2-resident for config 5 (1 M live aggregates); a 100 k-event batch
// is ONE persistent launch (phases separated by grid barriers) instead of the ~22 launches of the sort-based path.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/sgr.h"
#include "fold_rows.cuh"
#include "incremental.cuh"

namespace sgr {
namespace {

constexpr int W = 2;  // state words of the instantiated width (16-byte states)
struct Scratch {      // 32 bytes, zero between batches
  uint32_t last_event;   // arrival index + 1 of the slot's last event (0: untouched)
  uint32_t flags;        // bit0 a throwing event was seen, bit1 last event makes None, bit2 last event makes Some
  uint32_t last_set[W];  // arrival index + 1 of the last SET per word
  uint32_t acc[W];       // sum of ADDs after the last SET
  uint32_t set_val[W];   // value of the last SET
};
static_assert(sizeof(Scratch) == 32, "scratch entry");

__device__ __forceinline__ bool decode(const uint32_t* tab, const RowProgram& pg, const uint8_t* rec, uint32_t* fl, uint32_t mode[W], uint32_t val[W]) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(rec);
  const uint32_t type = r[pg.slot_word[0]];
  *fl = type < 16u ? tab[type * kTabStride] : 0u;
  if (!(*fl & 1u)) return false;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const uint32_t spec = tab[type * kTabStride + 1 + w];
    mode[w] = spec & 3u;
    uint32_t v = (spec >> 3) ? r[pg.slot_word[spec >> 3]] : 0u;
    if (spec & 4u) v = 0u - v;
    val[w] = mode[w] ? v : 0u;
  }
  return true;
}

__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}
// every block of the grid is resident (grid <= occupancy * SMs), so a counter barrier cannot deadlock
__device__ __forceinline__ void grid_barrier(unsigned long long* bar, unsigned long long target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(bar, 1ull);
    while (ld_volatile_u64(bar) < target) { __nanosleep(32); }
    __threadfence();
  }
  __syncthreads();
}

struct IncArgs {
  const uint8_t* rec; uint32_t n; uint64_t n_slots;
  Scratch* scr; uint8_t* states;
  uint32_t* touched_ids; uint32_t* err_ids;
  const uint32_t* prev_ids; const unsigned long long* prev_n;   // previous batch's touched list (prev_n may be null)
  unsigned long long* counters;  // [0] holes [1] throwing slots [3] error list [4] bad records [5] touched [6] dropped events [7] barrier
  uint32_t fast2;                    // every state word is add-only or set-only across the program: phases A and B fuse
  uint32_t set_only_mask;            // bit w: word w is only ever SET (otherwise, in fast2 mode, only ever ADDed)
  unsigned long long replay_budget;  // phase D runs only if n_err * n <= budget (it re-scans the batch per throwing slot); beyond
                                     // that the host replays the queued slots through the sort-based path ([2] is set to 1)
};

__global__ void __launch_bounds__(256) inc_fused_kernel(const __grid_constant__ IncArgs a, const __grid_constant__ RowProgram pg) {
  __shared__ uint32_t tab[16 * kTabStride];
  for (int i = threadIdx.x; i < 16 * kTabStride; i += 256) tab[i] = pg.tab[i];
  __syncthreads();
  const uint64_t tid = (uint64_t)blockIdx.x * 256 + threadIdx.x, nthreads = (uint64_t)gridDim.x * 256;
  unsigned long long* bar = a.counters + 7;

  // ---- phase 0: per-batch flags (CHANGED / ERROR / err_idx) of the previous batch's slots
  if (a.prev_n) {
    const uint64_t np = *a.prev_n;
    for (uint64_t i = tid; i < np; i += nthreads) {
      uint2* p = reinterpret_cast<uint2*>(a.states + (uint64_t)a.prev_ids[i] * ((W + 2) * 4) + W * 4);
      uint2 v = *p;
      v.x &= SGR_ST_EXISTS; v.y = 0;
      *p = v;
    }
  }
  if (a.fast2) {
    // ---- phase A+B fused. Scratch words are reinterpreted: [0] (arrival index + 1) << 2 | exists-op of the last event,
    //      [1] flags, then one u64 per state word: add-only word -> low half accumulates; set-only word -> max of
    //      (arrival index + 1) << 32 | value, i.e. the value of the LAST set. No second pass is needed because no word
    //      ever sees both a SET and an ADD.
    for (uint64_t i = tid; i < a.n; i += nthreads) {
      const uint8_t* r = a.rec + i * 64;
      const unsigned long long slot = *reinterpret_cast<const unsigned long long*>(r + 8);
      if (slot == ~0ull) { atomicAdd(a.counters + 0, 1ull); continue; }   // hole left by the device decode
      if (slot >= a.n_slots) { atomicAdd(a.counters + 4, 1ull); continue; }
      uint32_t* sw = reinterpret_cast<uint32_t*>(a.scr + slot);
      unsigned long long* s64 = reinterpret_cast<unsigned long long*>(sw + 2);
      uint32_t fl, mode[W], val[W];
      if (!decode(tab, pg, r, &fl, mode, val)) { atomicOr(sw + 1, 1u); atomicMax(sw, (((uint32_t)i + 1) << 2) | 3u); continue; }
      atomicMax(sw, (((uint32_t)i + 1) << 2) | ((fl & 2u) ? 2u : 1u));
#pragma unroll
      for (int w = 0; w < W; ++w) {
        if (mode[w] == 1u) { if (val[w]) atomicAdd(reinterpret_cast<uint32_t*>(s64 + w), val[w]); }
        else if (mode[w] == 2u) atomicMax(s64 + w, ((unsigned long long)((uint32_t)i + 1) << 32) | val[w]);
      }
    }
    grid_barrier(bar, gridDim.x);
    const bool rejected2 = ld_volatile_u64(a.counters + 4) != 0;
    // finishing pass: by record (the slot's last event finishes it) for a micro-batch, by slot when the batch is larger
    // than the table — touching a record's aggregate index costs a full 64-byte DRAM burst, the 32-byte scratch entry is
    // L2-resident
    const bool by_slot = (uint64_t)a.n > a.n_slots;
    const uint64_t c_end = by_slot ? a.n_slots : (uint64_t)a.n;
    for (uint64_t i = tid; i < c_end; i += nthreads) {
      unsigned long long slot = i;
      if (!by_slot) {
        slot = *reinterpret_cast<const unsigned long long*>(a.rec + i * 64 + 8);
        if (slot >= a.n_slots) continue;
      }
      Scratch* sp = a.scr + slot;
      const uint4 s0 = *reinterpret_cast<const uint4*>(sp);        // last_event|ex, flags, word0 (lo, hi)
      if (by_slot ? (s0.x == 0u) : ((s0.x >> 2) != (uint32_t)i + 1)) continue;   // untouched slot / not the slot's last event
      const uint4 s1 = reinterpret_cast<const uint4*>(sp)[1];      // word1 (lo, hi), unused
      reinterpret_cast<uint4*>(sp)[0] = make_uint4(0, 0, 0, 0);
      reinterpret_cast<uint4*>(sp)[1] = make_uint4(0, 0, 0, 0);
      if (rejected2) continue;
      a.touched_ids[atomicAdd(a.counters + 5, 1ull)] = (uint32_t)slot;
      if (s0.y & 1u) { a.err_ids[atomicAdd(a.counters + 3, 1ull)] = (uint32_t)slot; continue; }
      uint4* st = reinterpret_cast<uint4*>(a.states + slot * ((W + 2) * 4));
      const uint4 old = *st;
      const uint32_t ex0 = old.z & SGR_ST_EXISTS;
      const uint32_t exn = ((s0.x & 3u) == 2u) ? 0u : SGR_ST_EXISTS;
      const uint32_t b0 = ex0 ? old.x : 0u, b1 = ex0 ? old.y : 0u;
      uint32_t n0 = (a.set_only_mask & 1u) ? (s0.w ? s0.z : b0) : b0 + s0.z;
      uint32_t n1 = (a.set_only_mask & 2u) ? (s1.y ? s1.x : b1) : b1 + s1.x;
      if (!exn) { n0 = 0; n1 = 0; }
      uint32_t changed = exn != ex0;
      if (exn && ex0) changed |= (n0 != old.x) | (n1 != old.y);
      *st = make_uint4(n0, n1, exn | (changed ? SGR_ST_CHANGED : 0u), 0u);
    }
    grid_barrier(bar, 2ull * gridDim.x);
  } else {
  // ---- phase A: last event and last SET per slot
  for (uint64_t i = tid; i < a.n; i += nthreads) {
    const uint8_t* r = a.rec + i * 64;
    const unsigned long long slot = *reinterpret_cast<const unsigned long long*>(r + 8);
    if (slot == ~0ull) { atomicAdd(a.counters + 0, 1ull); continue; }   // hole left by the device decode
      if (slot >= a.n_slots) { atomicAdd(a.counters + 4, 1ull); continue; }
    Scratch* s = a.scr + slot;
    uint32_t fl, mode[W], val[W];
    atomicMax(&s->last_event, (uint32_t)i + 1);
    if (!decode(tab, pg, r, &fl, mode, val)) { atomicOr(&s->flags, 1u); continue; }
#pragma unroll
    for (int w = 0; w < W; ++w) if (mode[w] == 2u) atomicMax(&s->last_set[w], (uint32_t)i + 1);
  }
  grid_barrier(bar, gridDim.x);
  const bool rejected = ld_volatile_u64(a.counters + 4) != 0;  // an out-of-range slot: nothing is applied
  // ---- phase B: ADDs after the last SET, the last SET's value, the last event's exists-op
  if (!rejected) {
    for (uint64_t i = tid; i < a.n; i += nthreads) {
      const uint8_t* r = a.rec + i * 64;
      const unsigned long long slot = *reinterpret_cast<const unsigned long long*>(r + 8);
      if (slot == ~0ull) continue;   // hole left by the device decode
      Scratch* s = a.scr + slot;
      uint32_t fl, mode[W], val[W];
      if (!decode(tab, pg, r, &fl, mode, val)) continue;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const uint32_t ls = s->last_set[w];
        if (mode[w] == 1u) { if ((uint32_t)i + 1 > ls && val[w]) atomicAdd(&s->acc[w], val[w]); }
        else if (mode[w] == 2u) { if ((uint32_t)i + 1 == ls) s->set_val[w] = val[w]; }
      }
      if ((uint32_t)i + 1 == s->last_event) atomicOr(&s->flags, (fl & 2u) ? 2u : 4u);
    }
  }
  grid_barrier(bar, 2ull * gridDim.x);
  // ---- phase C: the slot's last event finishes it and cleans its scratch (by slot when the batch exceeds the table)
  const bool by_slot = (uint64_t)a.n > a.n_slots;
  const uint64_t c_end = by_slot ? a.n_slots : (uint64_t)a.n;
  for (uint64_t i = tid; i < c_end; i += nthreads) {
    unsigned long long slot = i;
    if (!by_slot) {
      slot = *reinterpret_cast<const unsigned long long*>(a.rec + i * 64 + 8);
      if (slot >= a.n_slots) continue;
    }
    Scratch* sp = a.scr + slot;
    const uint4 s0 = *reinterpret_cast<const uint4*>(sp);        // last_event, flags, last_set[0..1]
    if (by_slot ? (s0.x == 0u) : (s0.x != (uint32_t)i + 1)) continue;   // untouched slot / not the slot's last event
    const uint4 s1 = reinterpret_cast<const uint4*>(sp)[1];      // acc[0..1], set_val[0..1]
    reinterpret_cast<uint4*>(sp)[0] = make_uint4(0, 0, 0, 0);
    reinterpret_cast<uint4*>(sp)[1] = make_uint4(0, 0, 0, 0);
    if (rejected) continue;                                      // rejected batch: only the scratch is cleaned
    a.touched_ids[atomicAdd(a.counters + 5, 1ull)] = (uint32_t)slot;
    if (s0.y & 1u) { a.err_ids[atomicAdd(a.counters + 3, 1ull)] = (uint32_t)slot; continue; }
    uint4* st = reinterpret_cast<uint4*>(a.states + slot * ((W + 2) * 4));
    const uint4 old = *st;
    const uint32_t ex0 = old.z & SGR_ST_EXISTS;
    const uint32_t exn = (s0.y & 2u) ? 0u : SGR_ST_EXISTS;
    const uint32_t b0 = ex0 ? old.x : 0u, b1 = ex0 ? old.y : 0u;
    uint32_t n0 = (s0.z ? s1.z : b0) + s1.x, n1 = (s0.w ? s1.w : b1) + s1.y;
    if (!exn) { n0 = 0; n1 = 0; }
    uint32_t changed = exn != ex0;
    if (exn && ex0) changed |= (n0 != old.x) | (n1 != old.y);
    *st = make_uint4(n0, n1, exn | (changed ? SGR_ST_CHANGED : 0u), 0u);
  }
  grid_barrier(bar, 3ull * gridDim.x);
  }  // general (three-phase) mode
  // ---- phase D: one warp per throwing slot walks the batch in arrival order (exact err_idx, state kept)
  const unsigned long long n_err = ld_volatile_u64(a.counters + 3);
  if (n_err == 0) return;
  if (n_err * (unsigned long long)a.n > a.replay_budget) { if (tid == 0) a.counters[2] = 1ull; return; }
  const int lane = threadIdx.x & 31;
  const uint64_t warps = (uint64_t)gridDim.x * 8;
  for (uint64_t e = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5); e < n_err; e += warps) {
    const uint32_t slot = a.err_ids[e];
    uint4* stp = reinterpret_cast<uint4*>(a.states + (uint64_t)slot * ((W + 2) * 4));
    const uint4 old = *stp;
    const uint32_t ex0 = old.z & SGR_ST_EXISTS;
    uint32_t st[W] = {ex0 ? old.x : 0u, ex0 ? old.y : 0u}, exn = ex0, k = 0, total = 0;
    bool threw = false;
    for (uint32_t base = 0; base < a.n; base += 32) {
      const uint32_t i = base + lane;
      const uint8_t* r = a.rec + (uint64_t)i * 64;
      const bool mine = i < a.n && *reinterpret_cast<const unsigned long long*>(r + 8) == (unsigned long long)slot;
      uint32_t fl = 0, mode[W] = {0, 0}, val[W] = {0, 0};
      const bool ok = mine && decode(tab, pg, r, &fl, mode, val);
      uint32_t m = __ballot_sync(0xffffffffu, mine);
      total += __popc(m);
      while (m && !threw) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        const bool okb = __shfl_sync(0xffffffffu, (int)ok, b) != 0;
        if (!okb) { threw = true; break; }
        const uint32_t flb = __shfl_sync(0xffffffffu, fl, b);
#pragma unroll
        for (int w = 0; w < W; ++w) {
          const uint32_t mo = __shfl_sync(0xffffffffu, mode[w], b), va = __shfl_sync(0xffffffffu, val[w], b);
          const uint32_t cur = exn ? st[w] : 0u;
          st[w] = mo == 2u ? va : (mo == 1u ? cur + va : cur);
        }
        exn = (flb & 2u) ? 0u : SGR_ST_EXISTS;
        if (!exn) { st[0] = 0; st[1] = 0; }
        ++k;
      }
    }
    if (lane == 0) {
      if (threw) {
        *stp = make_uint4(old.x, old.y, ex0 | SGR_ST_ERROR, k);
        atomicAdd(a.counters + 1, 1ull);
        atomicAdd(a.counters + 6, (unsigned long long)(total - k));  // events dropped after the throw
      } else {
        uint32_t changed = exn != ex0;
        if (exn && ex0) changed |= (st[0] != old.x) | (st[1] != old.y);
        *stp = make_uint4(st[0], st[1], exn | (changed ? SGR_ST_CHANGED : 0u), 0u);
      }
    }
  }
}

}  // namespace

size_t inc_scratch_bytes(uint64_t n_slots) { return (size_t)n_slots * sizeof(Scratch); }

// counters (8 x u64, zeroed by the caller before): [1] throwing slots, [3] error list length, [4] records with slot >= n_slots,
// [5] touched slots, [6] events dropped after a throw. prev_n points at the previous batch's [5] (kept in a separate buffer).
cudaError_t launch_incremental_atomic(const uint8_t* d_records, uint32_t n, uint64_t n_slots, void* d_scratch, uint8_t* d_states,
                                      uint32_t* d_touched_ids, uint32_t* d_err_ids, const uint32_t* d_prev_ids,
                                      const unsigned long long* d_prev_n, uint32_t prev_n_upper, const RowProgram& prog,
                                      unsigned long long* d_counters, unsigned long long replay_budget, cudaStream_t st) {
  static int max_grid = 0;
  if (!max_grid) {
    int per_sm = 0, dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, inc_fused_kernel, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    max_grid = per_sm * sms;
  }
  IncArgs a{};
  a.rec = d_records; a.n = n; a.n_slots = n_slots; a.scr = reinterpret_cast<Scratch*>(d_scratch); a.states = d_states;
  a.touched_ids = d_touched_ids; a.err_ids = d_err_ids; a.prev_ids = d_prev_ids; a.prev_n = prev_n_upper ? d_prev_n : nullptr;
  a.counters = d_counters; a.replay_budget = replay_budget;
  // add-only / set-only analysis over every valid event type
  uint32_t has_add = 0, has_set = 0;
  for (int t = 0; t < 16; ++t) {
    if (!(prog.tab[t * kTabStride] & 1u)) continue;
    for (int w = 0; w < W; ++w) {
      const uint32_t mode = prog.tab[t * kTabStride + 1 + w] & 3u;
      if (mode == 1u) has_add |= 1u << w;
      if (mode == 2u) has_set |= 1u << w;
    }
  }
  a.fast2 = ((has_add & has_set) == 0 && n < (1u << 30)) ? 1u : 0u;
  a.set_only_mask = has_set;
  const uint32_t work = n > prev_n_upper ? n : prev_n_upper;  // (the by-slot finishing pass is grid-stride over n_slots < n)
  if (!work) return cudaSuccess;
  uint32_t g = (work + 255) / 256;
  if (g > (uint32_t)max_grid) g = (uint32_t)max_grid;
  inc_fused_kernel<<<g, 256, 0, st>>>(a, prog);
  return cudaGetLastError();
}

}  // namespace sgr
