// fold_runs.cu — K1/K3 (primary): segmented fold of fixed 64-byte records, lane-runs + warp scan (sm_100a).
//
// Contract: for every aggregate, events.foldLeft(state)(handleEvent)
// (modules/command-engine/scaladsl/src/main/scala/surge/scaladsl/command/CommandModels.scala:25-28) with the
// actor's publish rule (modules/command-engine/core/src/main/scala/surge/internal/persistence/
// PersistentActor.scala:252-257). Exactness comes from the transformer algebra of fold_rows.cuh:
// an event is a per-word (KEEP | ADD v | SET v) map, composition is associative, so any
// bracketing of the log-ordered product equals the sequential fold bit for bit.
//
// Shape (HBM-bound byte parse + segmented scan; no tensor cores):
//   * the log is cut into byte-balanced spans, one per warp — a hot aggregate (Zipf skew) is
//     spread over many warps instead of serialising one lane;
//   * a warp walks its span in steps of 32*R records. The step's 2048*R bytes are staged into
//     shared memory with coalesced 16-byte cp.async copies (512 contiguous bytes per warp
//     instruction), NSTAGE steps deep, no register staging;
//   * the staging layout XOR-swizzles each record's 16-byte chunks with (record/R)&7, so that
//     lane i reading its run of R consecutive records [R*i, R*i+R) is bank-conflict free;
//   * lane i folds its R records left to right into a running transformer (the only per-record
//     work: 1 table read + the needed record words); segments that start and end inside the
//     run are finished on the spot;
//   * once per step the 32 lane-transformers are combined by a 5-step segmented warp-shuffle
//     scan in log order; the lane holding the first segment head of its run finishes the segment
//     that flows into it; the scan's tail is the carry into the next step;
//   * segment heads come from the CSR offsets: a window of 32 boundaries is read with coalesced
//     8-byte loads and scattered into a per-step head bitmap + segment-id table in smem;
//   * a segment that crosses a span boundary is finished by the warp that sees its end, after a
//     decoupled look-back over the predecessors' published open transformers.
#include <stdio.h>

#include "../../include/sgr.h"
#include "fold_rows.cuh"

namespace sgr {
namespace {

constexpr uint32_t M_ERR = 0x80000000u;  // some event in the range threw
constexpr uint32_t M_COPY = 0x40000000u; // some applied event built a new state instance (tab flag 8u << 27), see finish_segment
constexpr uint32_t EX_SOME = 1u, EX_NONE = 2u;
constexpr int kRunThreads = 128;
constexpr int kRunWarps = kRunThreads / 32;

template <int W>
struct Xf {
  uint32_t m;     // bits [2w+1:2w]: mode of word w (bit0 ADD, bit1 SET; OR-composable), bit30 copy, bit31 error
  uint32_t ex;    // exists-op of the LAST event in the range: 0 = no event, EX_SOME, EX_NONE
  uint32_t v[W];  // KEEP => 0
};

template <int W>
__device__ __forceinline__ Xf<W> identity() {
  Xf<W> r;
  r.m = 0; r.ex = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) r.v[w] = 0;
  return r;
}
// later . earlier  (apply `a` first, then `b`)
template <int W, int CLS = 1>
__device__ __forceinline__ Xf<W> compose(const Xf<W>& a, const Xf<W>& b) {
  // class 1: b.ex == 0 means b holds only IF_EXISTS events (or nothing); they apply iff the state exists after a — a
  // tombstoned prefix absorbs them. (In class 0, b.ex == 0 only for the identity, where the plain rule gives a too.)
  // A throwing event sets no exists-op either: its error bit must survive, or the segment is never replayed.
  if (CLS == 1 && b.ex == 0u && a.ex == EX_NONE) {
    Xf<W> r = a;
    r.m |= b.m & M_ERR;
    return r;
  }
  Xf<W> r;
  r.m = a.m | b.m;
  r.ex = b.ex ? b.ex : a.ex;
#pragma unroll
  for (int w = 0; w < W; ++w) r.v[w] = (b.m & (2u << (2 * w))) ? b.v[w] : a.v[w] + b.v[w];
  return r;
}
template <int W>
__device__ __forceinline__ Xf<W> shfl_xf(const Xf<W>& t, int src) {
  Xf<W> r;
  r.m = __shfl_sync(0xffffffffu, t.m, src);
  r.ex = __shfl_sync(0xffffffffu, t.ex, src);
#pragma unroll
  for (int w = 0; w < W; ++w) r.v[w] = __shfl_sync(0xffffffffu, t.v[w], src);
  return r;
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// Finish one segment: apply the composed transformer to the prior state, write the state struct.
template <int W>
__device__ __forceinline__ void finish_segment(const RowArgs& a, uint32_t f64_mask, uint32_t seg, const Xf<W>& ts) {
  if (ts.m & M_ERR) {
    // the handler threw somewhere in the segment: exact replay by the sequential phase
    const unsigned long long pos = atomicAdd(a.counters + 3, 1ull);
    if (pos < a.redo_cap) a.redo_ids[pos] = seg;
    return;
  }
  const uint64_t slot = a.seg_ids ? (uint64_t)a.seg_ids[seg] : (uint64_t)seg;
  uint32_t old[W], ex0 = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) old[w] = 0;
  if (a.states_in) {
    const uint4* sp = reinterpret_cast<const uint4*>(a.states_in + slot * (uint64_t)(W + 2) * 4);
    uint32_t raw[W + 2];
#pragma unroll
    for (int q = 0; q < (W + 2) / 4; ++q) { const uint4 v4 = __ldg(sp + q); raw[4 * q] = v4.x; raw[4 * q + 1] = v4.y; raw[4 * q + 2] = v4.z; raw[4 * q + 3] = v4.w; }
    ex0 = raw[W] & SGR_ST_EXISTS;
#pragma unroll
    for (int w = 0; w < W; ++w) old[w] = ex0 ? raw[w] : 0u;
  }
  // ts.ex: SOME / NONE = exists-op of the last CREATE/MATERIALISE/TOMBSTONE-class event; 0 = only IF_EXISTS events
  // (or none at all): the words apply iff the prior state exists
  const uint32_t exn = ts.ex == EX_NONE ? 0u : (ts.ex == EX_SOME ? (uint32_t)SGR_ST_EXISTS : ex0);
  uint32_t nw[W];
#pragma unroll
  for (int w = 0; w < W; ++w) {
    nw[w] = (ts.m & (2u << (2 * w))) ? ts.v[w] : old[w] + ts.v[w];
    if (!exn) nw[w] = 0u;
  }
  uint32_t changed = exn != ex0;
  if (exn && ex0) {
#pragma unroll
    for (int w = 0; w < W; ++w) {
      const bool f_lo = (f64_mask >> w) & 1u, f_hi = w > 0 && ((f64_mask >> (w - 1)) & 1u);
      if (f_lo) {
        // JVM Double ==: numeric (0.0 == -0.0, NaN != NaN), as Scala case-class equality does — after its `this eq that`
        // shortcut: if no applied event built a new instance the state is the old object, equal to itself even with a NaN
        const uint32_t xh = nw[w + 1 < W ? w + 1 : w], yh = old[w + 1 < W ? w + 1 : w];
        const double x = __hiloint2double((int)xh, (int)nw[w]);
        const double y = __hiloint2double((int)yh, (int)old[w]);
        changed |= !(x == y) && ((ts.m & M_COPY) != 0u || nw[w] != old[w] || xh != yh);
      } else if (!f_hi) {
        changed |= (nw[w] != old[w]);
      }
    }
  }
  uint32_t outw[W + 2];
#pragma unroll
  for (int w = 0; w < W; ++w) outw[w] = nw[w];
  outw[W] = exn | (changed ? SGR_ST_CHANGED : 0u);
  outw[W + 1] = 0u;
  uint4* dp = reinterpret_cast<uint4*>(a.states_out + slot * (uint64_t)(W + 2) * 4);
#pragma unroll
  for (int q = 0; q < (W + 2) / 4; ++q) dp[q] = make_uint4(outw[4 * q], outw[4 * q + 1], outw[4 * q + 2], outw[4 * q + 3]);
}

// state of an aggregate that received no event in this batch: unchanged, per-batch flags cleared
template <int W>
__device__ __forceinline__ void finish_empty(const RowArgs& a, uint32_t seg) {
  const uint64_t slot = a.seg_ids ? (uint64_t)a.seg_ids[seg] : (uint64_t)seg;
  uint4* dp = reinterpret_cast<uint4*>(a.states_out + slot * (uint64_t)(W + 2) * 4);
  if (a.states_in) {
    const uint4* sp = reinterpret_cast<const uint4*>(a.states_in + slot * (uint64_t)(W + 2) * 4);
#pragma unroll
    for (int q = 0; q < (W + 2) / 4; ++q) {
      uint4 v4 = __ldg(sp + q);
      if (q == (W + 2) / 4 - 1) { v4.z &= SGR_ST_EXISTS; v4.w = 0u; }
      dp[q] = v4;
    }
  } else {
#pragma unroll
    for (int q = 0; q < (W + 2) / 4; ++q) dp[q] = make_uint4(0, 0, 0, 0);
  }
}

template <int R, int NSTAGE>
__host__ __device__ constexpr int warp_smem_bytes() {
  return NSTAGE * 2048 * R   // staged steps
         + 2 * 32 * R * 4    // segment ids at head positions: starting segment, ending segment
         + 32 * 4;           // head bitmap (R words used) + pad
}

// DIRECT: programs with many source words read each state word's source straight from the staged record instead of
// pre-fetching NS slots and selecting (NS is then unused)
template <int W, int R, int NSTAGE, int NS, int MINB, bool DIRECT, int CLS>
__global__ void __launch_bounds__(kRunThreads, MINB) fold_runs_kernel(const __grid_constant__ RowArgs a, const __grid_constant__ RowProgram pg) {
  static_assert(R % 2 == 0 && 8 % R == 0, "R in {2,4,8}");
  constexpr int STEP_BYTES = 2048 * R;
  constexpr int STEP_RECS = 32 * R;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ __align__(16) uint32_t tab[16 * kTabStride];
  for (int i = threadIdx.x; i < 16 * kTabStride; i += kRunThreads) tab[i] = pg.tab[i];
  const uint32_t f64_mask = pg.f64_mask;
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* wsm = smem_raw + (size_t)warp * warp_smem_bytes<R, NSTAGE>();
  const uint32_t stage0 = smem_u32(wsm);
  uint32_t* hs_start = reinterpret_cast<uint32_t*>(wsm + NSTAGE * STEP_BYTES);  // segment starting at a head
  uint32_t* hs_end = hs_start + STEP_RECS;                                       // segment ending at a head (0xffffffff: none)
  uint32_t* hmask = hs_end + STEP_RECS;                                          // head bitmap, R words

  const uint64_t gw = (uint64_t)blockIdx.x * kRunWarps + warp;  // global warp id
  const uint64_t n_warps = (uint64_t)gridDim.x * kRunWarps;
  const uint64_t n_seg = a.n_seg;
  const uint64_t base = a.log_begin;
  const uint64_t total_bytes = a.log_end - base;
  const uint64_t total_steps = (total_bytes + STEP_BYTES - 1) / STEP_BYTES;
  const uint64_t spw = (total_steps + n_warps - 1) / n_warps;  // steps per warp
  const uint64_t step0 = gw * spw;
  const uint64_t step_end = step0 + spw < total_steps ? step0 + spw : total_steps;
  const bool has_span = step0 < step_end;
  const uint64_t wb = base + step0 * STEP_BYTES;
  // the warp that owns the end of the log also finishes the last segment and trailing empty ones;
  // with an empty log that is warp 0
  const bool owns_end = has_span ? (step_end == total_steps) : (total_steps == 0 && gw == 0);

  // ---- first boundary of the span: kc = first k in [0, n_seg] with off[k] >= wb (32-ary search)
  uint64_t kc = 0;
  if (has_span && gw != 0) {
    uint64_t lo = 0, hi = n_seg + 1;  // answer in [lo, hi]; hi == n_seg+1: no such boundary
    while (lo < hi) {
      const uint64_t chunk = (hi - lo + 31) / 32;
      const uint64_t p = lo + (uint64_t)lane * chunk;
      const bool valid = p < hi;
      const bool ge = !valid || a.seg_offsets[p] >= wb;  // monotone in lane
      const uint32_t bal = __ballot_sync(0xffffffffu, ge);
      if (bal == 0) { lo = lo + 31 * chunk + 1; continue; }
      const int f = __ffs(bal) - 1;
      if (f == 0) { hi = lo; break; }
      const uint64_t pf = lo + (uint64_t)f * chunk;
      lo = lo + (uint64_t)(f - 1) * chunk + 1;
      hi = pf < hi ? pf : hi;
    }
    kc = lo;
  }

  bool span_has_head = false;          // a segment head was seen in this span
  bool inh_pending = false;            // the segment flowing into the span awaits the look-back (held by lane 0)
  uint32_t inh_seg = 0;
  Xf<W> inh_t = identity<W>();
  Xf<W> carry = identity<W>();         // open transformer at the end of the previous step

  // ---- staging: lane l, copy q of a step moves the 16-byte chunk g = q*32 + l (source order) to its
  //      swizzled place: record j = g>>2, chunk c = g&3 -> line j>>1, position (4*(j&1)+c) ^ ((j/R)&7)
  const uint8_t* src_lane = a.events + base + (uint64_t)lane * 16;
  const uint32_t low_pos = (uint32_t)(4 * ((lane >> 2) & 1) + (lane & 3));
  const uint32_t lane_jr = (uint32_t)(lane >> 2) / R;
  uint32_t dst_q[4 * R];  // smem offset (within a stage) of copy q
#pragma unroll
  for (int q = 0; q < 4 * R; ++q)
    dst_q[q] = (uint32_t)q * 512u + (uint32_t)(lane >> 3) * 128u + ((low_pos ^ (((uint32_t)(q * 8) / R + lane_jr) & 7u)) << 4);
  auto issue_step = [&](uint64_t s, int stage) {
    const uint64_t sbyte = s * (uint64_t)STEP_BYTES;
    const uint8_t* src = src_lane + sbyte;
    const uint32_t dst = stage0 + (uint32_t)stage * STEP_BYTES;
    if (sbyte + STEP_BYTES <= total_bytes) {  // uniform: the whole step lies inside the log
#pragma unroll
      for (int q = 0; q < 4 * R; ++q) cp_async16(dst + dst_q[q], src + q * 512);
    } else {
#pragma unroll
      for (int q = 0; q < 4 * R; ++q)
        if (sbyte + (uint64_t)q * 512 + (uint64_t)lane * 16 < total_bytes) cp_async16(dst + dst_q[q], src + q * 512);
    }
  };
  // prologue: NSTAGE-1 steps in flight
  if (has_span) {
#pragma unroll
    for (int s = 0; s < NSTAGE - 1; ++s) {
      if (step0 + s < step_end) issue_step(step0 + s, s);
      cp_async_commit();
    }
  }

  // where lane i finds word (c,k) of a record of parity par: byte (((4*par + c) ^ (i&7)) << 4) + 4k of its 128-byte line
  constexpr int NSOFF = DIRECT ? 1 : NS;
  uint32_t soff[2][NSOFF];
#pragma unroll
  for (int s = 0; s < NSOFF; ++s) {
    const uint32_t c = pg.slot_word[s] >> 2, k = pg.slot_word[s] & 3u;
    soff[0][s] = ((c ^ (uint32_t)(lane & 7)) << 4) + (k << 2);
    soff[1][s] = (((4u + c) ^ (uint32_t)(lane & 7)) << 4) + (k << 2);
  }
  // boundary window: lane j holds off[kc+j] and off[kc+j+1]; reloaded right after boundaries are consumed,
  // so the values a step needs were requested one step earlier
  uint64_t win_b = ~0ull, win_bn = ~0ull;
  auto load_window = [&]() {
    const uint64_t k = kc + lane;
    win_b = k <= n_seg ? a.seg_offsets[k] : ~0ull;
    win_bn = k < n_seg ? a.seg_offsets[k + 1] : ~0ull;
  };
  if (has_span) load_window();

  int stage = 0;
  for (uint64_t step = step0; step < step_end; ++step) {
    // keep NSTAGE-1 steps in flight
    {
      const uint64_t ahead = step + (NSTAGE - 1);
      int st = stage + (NSTAGE - 1); if (st >= NSTAGE) st -= NSTAGE;
      if (ahead < step_end) issue_step(ahead, st);
      cp_async_commit();
    }
    const uint64_t sb = base + step * (uint64_t)STEP_BYTES;
    const uint64_t rem = a.log_end - sb;
    const uint32_t span = rem < (uint64_t)STEP_BYTES ? (uint32_t)rem : (uint32_t)STEP_BYTES;
    const int nvalid = (int)(span >> 6);

    // ---- segment heads of this step: boundaries k with off[k] in [sb, sb+span) ----------------------
#pragma unroll
    for (int i = 0; i < R; ++i) { hs_end[i * 32 + lane] = 0xffffffffu; hs_start[i * 32 + lane] = 0u; }
    if (lane < R) hmask[lane] = 0u;
    __syncwarp();
    while (true) {
      const uint64_t k = kc + lane;
      const uint64_t b = win_b, bn = win_bn;  // window at kc, loaded one step ahead
      const uint64_t d = b - sb;  // >= 0 for every unconsumed boundary
      const bool in = d < (uint64_t)span;
      if (in) {
        const uint32_t pos = (uint32_t)d >> 6;
        atomicOr(&hmask[pos >> 5], 1u << (pos & 31));
        atomicMax(&hs_start[pos], (uint32_t)k);                       // the last boundary at this offset starts the live segment
        if (k > 0) atomicMin(&hs_end[pos], (uint32_t)k - 1u);         // the first one ends the previous segment
        if (bn == b) finish_empty<W>(a, (uint32_t)k);                 // segment k is empty
      }
      const int cnt = __popc(__ballot_sync(0xffffffffu, in));
      kc += cnt;
      if (cnt) load_window();
      if (cnt < 32) break;
    }
    __syncwarp();

    // ---- wait for this step's bytes --------------------------------------------------------------------
    cp_async_wait<NSTAGE - 1>();
    __syncwarp();

    // ---- lane run: R consecutive records, left to right -------------------------------------------------
    const uint32_t sbase = stage0 + (uint32_t)stage * STEP_BYTES;
    uint32_t hbits;
    if (R >= 32) hbits = hmask[lane];
    else hbits = (hmask[(lane * R) >> 5] >> ((lane * R) & 31)) & ((R >= 32) ? 0xffffffffu : ((1u << R) - 1u));
    Xf<W> cur = identity<W>();
    Xf<W> first = identity<W>();
    uint32_t first_seg = 0xffffffffu;
    bool have_first = false;
#pragma unroll
    for (int t = 0; t < R; ++t) {
      const int p = lane * R + t;
      if (hbits & (1u << t)) {
        const uint32_t eseg = hs_end[p];
        if (!have_first) { first = cur; first_seg = eseg; have_first = true; }
        else if (eseg != 0xffffffffu) finish_segment<W>(a, f64_mask, eseg, cur);  // began and ended inside this run
        cur = identity<W>();
      }
      if (p < nvalid) {
        const uint32_t rec = sbase + (uint32_t)(p >> 1) * 128u;
        const uint32_t lane7 = (uint32_t)(lane & 7), par4 = (uint32_t)(t & 1) * 4u;  // p&1 == t&1: R is even
        uint32_t sv[DIRECT ? 1 : NS];
        if (DIRECT) {
          sv[0] = lds32(rec + soff[t & 1][0]);
        } else {
#pragma unroll
          for (int s = 0; s < NS; ++s) sv[s] = lds32(rec + soff[t & 1][s]);
        }
        const uint32_t type = sv[0];
        uint4 e0 = make_uint4(0, 0, 0, 0);
        if (type < 16u) e0 = *reinterpret_cast<const uint4*>(tab + type * kTabStride);
        if (!(e0.x & 1u)) {
          cur.m |= M_ERR;  // THROW rule or scala.MatchError
        } else if (CLS == 1 && (e0.x & 4u) && cur.ex == EX_NONE) {
          // IF_EXISTS event after a tombstone in this run: the state does not exist, the event is a no-op
        } else {
          if (CLS == 0 || !(e0.x & 4u)) cur.ex = (e0.x & 2u) ? EX_NONE : EX_SOME;  // an IF_EXISTS event leaves the exists-op as it is
          uint32_t spec[W];
          spec[0] = e0.y;
          if (W > 1) spec[1] = e0.z;
          if (W > 2) spec[2] = e0.w;
#pragma unroll
          for (int w = 3; w < W; ++w) spec[w] = tab[type * kTabStride + 1 + w];
#pragma unroll
          for (int w = 0; w < W; ++w) {
            uint32_t val = 0;
            if (DIRECT) {
              const uint32_t sl = spec[w] >> 3;
              if (sl) { const uint32_t sw = pg.slot_word[sl]; val = lds32(rec + ((((par4 + (sw >> 2)) ^ lane7) << 4) | ((sw & 3u) << 2))); }
            } else {
#pragma unroll
              for (int s = 1; s < NS; ++s) val = ((spec[w] >> 3) == (uint32_t)s) ? sv[s] : val;
            }
            if (spec[w] & 4u) val = 0u - val;
            const uint32_t mode = spec[w] & 3u;
            if (mode == 2u) cur.v[w] = val;
            else if (mode == 1u) cur.v[w] += val;
            cur.m |= mode << (2 * w);
          }
          cur.m |= (e0.x & 8u) << 27;   // M_COPY: this rule builds a new instance (CREATE, or any field op)
        }
      }
    }
    // cur = transformer of the records after the run's last head (the whole run if it has none)

    // ---- once per step: segmented inclusive scan of the 32 lane transformers, in log order -------------
    const uint32_t lane_heads = __ballot_sync(0xffffffffu, have_first);
    Xf<W> sc = cur;
    if (lane == 0 && !have_first) sc = compose<W, CLS>(carry, sc);
#pragma unroll
    for (int dd = 1; dd < 32; dd <<= 1) {
      const Xf<W> o = shfl_xf(sc, lane - dd);  // wraps for lane < dd; masked below
      const int sh = lane >= dd ? lane - dd + 1 : 0;
      const uint32_t window = (lane_heads >> sh) & ((1u << dd) - 1u);  // a head in lanes (lane-dd, lane]?
      if (lane >= dd && window == 0) sc = compose<W, CLS>(o, sc);
    }
    // what flows INTO each lane's run: the scan value of the previous lane (lane 0: the carry)
    Xf<W> cin = shfl_xf(sc, lane - 1);
    if (lane == 0) cin = carry;
    carry = shfl_xf(sc, 31);

    // ---- the segment that ends at a run's first head needs what flowed in ----------------------------------
    if (have_first && first_seg != 0xffffffffu) {
      const Xf<W> tot = compose<W, CLS>(cin, first);
      // the very first head of the span ends a segment that began in an earlier span: look-back needed
      const bool is_span_first = !span_has_head && (lane_heads & ((1u << lane) - 1u)) == 0;
      if (is_span_first && gw != 0) { inh_t = tot; inh_seg = first_seg; inh_pending = true; }
      else finish_segment<W>(a, f64_mask, first_seg, tot);
    }
    if (lane_heads) {
      // the pending look-back lives in the lane that saw the span's first head: move it to lane 0
      if (!span_has_head) {
        const int src = __ffs(lane_heads) - 1;
        inh_t = shfl_xf(inh_t, src);
        inh_seg = __shfl_sync(0xffffffffu, inh_seg, src);
        inh_pending = __shfl_sync(0xffffffffu, (int)inh_pending, src) != 0;
      }
      span_has_head = true;
    }
    __syncwarp();
    if (++stage == NSTAGE) stage = 0;
  }
  cp_async_wait<0>();

  // ---- end of the log: the open segment and any trailing empty segments --------------------------------
  // boundaries with off[k] == log_end were never a head inside a step; kc is the first of them.
  bool end_needs_lookback = false;
  if (owns_end) {
    for (uint64_t k = kc + lane; k < n_seg; k += 32) finish_empty<W>(a, (uint32_t)k);  // segments kc..n_seg-1 are empty
    if (kc >= 1 && total_steps > 0) {
      // segment kc-1 is the last non-empty one; its transformer is the carry
      if (span_has_head || gw == 0) { if (lane == 0) finish_segment<W>(a, f64_mask, (uint32_t)(kc - 1), carry); }
      else end_needs_lookback = true;  // the whole span lies inside that segment
    }
  }

  // ---- publish this span's open transformer, then finish what needs the predecessors ---------------------
  if (has_span) {
    uint32_t* part_data = a.part_data + gw * (W + 2);
    if (lane == 0) {
      part_data[0] = carry.m;
#pragma unroll
      for (int w = 0; w < W; ++w) part_data[1 + w] = carry.v[w];
      part_data[W + 1] = carry.ex | (span_has_head ? 4u : 0u);
      __threadfence();
      asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(a.part_flags + gw), "r"(a.epoch) : "memory");
    }
    if (lane == 0 && (inh_pending || end_needs_lookback)) {
      // decoupled look-back: compose predecessors' open transformers until one that contains a head
      Xf<W> pre = identity<W>();
      uint64_t p = gw;
      while (p > 0) {
        --p;
        const uint32_t* pf = a.part_flags + p;
        while (ld_volatile_u32(pf) != a.epoch) { __nanosleep(64); }
        __threadfence();
        const uint32_t* pd = a.part_data + p * (W + 2);
        Xf<W> e;
        e.m = ld_volatile_u32(pd);
#pragma unroll
        for (int w = 0; w < W; ++w) e.v[w] = ld_volatile_u32(pd + 1 + w);
        const uint32_t tailw = ld_volatile_u32(pd + W + 1);
        e.ex = tailw & 3u;
        pre = compose<W, CLS>(e, pre);
        if (tailw & 4u) break;
      }
      if (inh_pending) finish_segment<W>(a, f64_mask, inh_seg, compose<W, CLS>(pre, inh_t));
      if (end_needs_lookback) finish_segment<W>(a, f64_mask, (uint32_t)(kc - 1), compose<W, CLS>(pre, carry));
    }
  }
  // every record of the span was applied; records of throwing segments are taken back by the replay below
  if (lane == 0 && has_span) {
    const uint64_t we = base + step_end * (uint64_t)STEP_BYTES < a.log_end ? base + step_end * (uint64_t)STEP_BYTES : a.log_end;
    atomicAdd(a.counters + 0, (unsigned long long)((we - wb) >> 6));
  }

  // ---- grid barrier (every warp of the grid is resident), then exact replay of the throwing segments ----
  // A segment whose handler threw keeps its pre-batch state and reports the index of the throwing event
  // (PersistentActor.scala:260-263); that needs the strictly sequential walk, done here one lane per segment.
  if (lane == 0) {
    __threadfence();
    atomicAdd(a.counters + 6, 1ull);
    while (ld_volatile_u64(a.counters + 6) < n_warps) { __nanosleep(128); }
    __threadfence();
  }
  __syncwarp();
  if (gw == 0 && lane < 8) a.counters_next[lane] = 0ull;  // the next fold starts from clean counters without a memset
  unsigned long long n_redo = ld_volatile_u64(a.counters + 3);
  if (n_redo == 0) return;
  if (n_redo > a.redo_cap) n_redo = a.redo_cap;  // overflow: the host re-runs the whole fold sequentially
  unsigned long long n_err = 0, n_dropped = 0;
  for (unsigned long long i = gw * 32 + lane; i < n_redo; i += n_warps * 32) {
    const uint32_t seg = a.redo_ids[i];
    const uint64_t b = a.seg_offsets[seg], e = a.seg_offsets[(uint64_t)seg + 1];
    const uint64_t slot = a.seg_ids ? (uint64_t)a.seg_ids[seg] : (uint64_t)seg;
    uint32_t st[W], ex0 = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) st[w] = 0;
    if (a.states_in) {
      const uint32_t* sp = reinterpret_cast<const uint32_t*>(a.states_in + slot * (uint64_t)(W + 2) * 4);
      ex0 = sp[W] & SGR_ST_EXISTS;
#pragma unroll
      for (int w = 0; w < W; ++w) st[w] = ex0 ? sp[w] : 0u;
    }
    uint32_t old[W];
#pragma unroll
    for (int w = 0; w < W; ++w) old[w] = st[w];
    uint32_t exn = ex0, k = 0;
    bool threw = false;
    for (uint64_t pos = b; pos < e; pos += 64, ++k) {
      const uint32_t* rec = reinterpret_cast<const uint32_t*>(a.events + pos);
      const uint32_t type = rec[pg.slot_word[0]];
      const uint32_t fl = type < 16u ? tab[type * kTabStride] : 0u;
      if (!(fl & 1u)) { threw = true; break; }
      if (fl & 2u) { exn = 0u; for (int w = 0; w < W; ++w) st[w] = 0u; continue; }  // tombstone
      if ((fl & 4u) && !exn) continue;                                                // IF_EXISTS on None: no-op
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const uint32_t spec = tab[type * kTabStride + 1 + w];
        const uint32_t mode = spec & 3u;
        uint32_t val = (spec >> 3) ? rec[pg.slot_word[spec >> 3]] : 0u;
        if (spec & 4u) val = 0u - val;
        if (mode == 2u) st[w] = val; else if (mode == 1u) st[w] = (exn ? st[w] : 0u) + val;
        else if (!exn) st[w] = 0u;
      }
      exn = SGR_ST_EXISTS;
    }
    uint32_t* dp = reinterpret_cast<uint32_t*>(a.states_out + slot * (uint64_t)(W + 2) * 4);
    if (threw) {
#pragma unroll
      for (int w = 0; w < W; ++w) dp[w] = old[w];
      dp[W] = ex0 | SGR_ST_ERROR;
      dp[W + 1] = k;
      ++n_err;
      n_dropped += ((e - b) >> 6) - k;
    } else {
      uint32_t changed = exn != ex0;
#pragma unroll
      for (int w = 0; w < W; ++w) { if (!exn) st[w] = 0u; if (exn && ex0) changed |= st[w] != old[w]; dp[w] = st[w]; }  // (a replayed segment that did not throw cannot occur)
      dp[W] = exn | (changed ? SGR_ST_CHANGED : 0u);
      dp[W + 1] = 0u;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    n_err += __shfl_xor_sync(0xffffffffu, n_err, o);
    n_dropped += __shfl_xor_sync(0xffffffffu, n_dropped, o);
  }
  if (lane == 0) {
    if (n_err) atomicAdd(a.counters + 1, n_err);
    if (n_dropped) atomicAdd(a.counters + 4, n_dropped);
  }
}

typedef void (*RunKernel)(const RowArgs, const RowProgram);
struct RunVariant { RunKernel k[3]; int r, nstage; const char* name; };  // 16-byte states; k[i]: NS = 2, 3, 6
#define RUN_VARIANT(R, ST, MINB) {{fold_runs_kernel<2, R, ST, 2, MINB, false, 0>, fold_runs_kernel<2, R, ST, 3, MINB, false, 0>, fold_runs_kernel<2, R, ST, 6, MINB, false, 0>}, R, ST, "runs W2 R" #R " st" #ST}
const RunVariant kRunVariants[] = {
    RUN_VARIANT(4, 2, 3), RUN_VARIANT(4, 1, 5), RUN_VARIANT(2, 2, 5), RUN_VARIANT(2, 1, 5), RUN_VARIANT(4, 3, 2), RUN_VARIANT(8, 1, 3), RUN_VARIANT(2, 3, 4),
};
constexpr int kNumRunVariants = sizeof(kRunVariants) / sizeof(kRunVariants[0]);
// wider states / many source words: one configuration each (R = 4, 2 stages, direct word reads)
constexpr int kWideR = 4, kWideStages = 2;

size_t variant_smem(int v, const RowProgram& prog) {
  const bool wide = prog.user_words != 2 || prog.n_slots > 6 || prog.cls != 0;
  const int r = wide ? kWideR : kRunVariants[v].r, ns = wide ? kWideStages : kRunVariants[v].nstage;
  return (size_t)kRunWarps * ((size_t)ns * 2048 * r + 2 * 32 * r * 4 + 32 * 4);
}
RunKernel variant_kernel(int v, const RowProgram& prog) {
  if (prog.user_words == 14) return fold_runs_kernel<14, kWideR, kWideStages, 1, 1, true, 1>;
  if (prog.user_words == 6) return fold_runs_kernel<6, kWideR, kWideStages, 1, 2, true, 1>;
  if (prog.n_slots > 6 || prog.cls != 0) return fold_runs_kernel<2, kWideR, kWideStages, 1, 3, true, 1>;
  return kRunVariants[v].k[prog.n_slots <= 2 ? 0 : (prog.n_slots <= 3 ? 1 : 2)];
}

}  // namespace

int run_variant_count() { return kNumRunVariants; }
const char* run_variant_name(int v) { return (v >= 0 && v < kNumRunVariants) ? kRunVariants[v].name : "?"; }

int run_kernel_max_grid(int num_sms, int variant, const RowProgram& prog) {
  if (variant < 0 || variant >= kNumRunVariants) variant = 0;
  const size_t smem = variant_smem(variant, prog);
  RunKernel k = variant_kernel(variant, prog);
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, kRunThreads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  return per_sm * num_sms;
}

int run_variant_step_bytes(int variant, const RowProgram& prog) {
  if (variant < 0 || variant >= kNumRunVariants) variant = 0;
  const bool wide = prog.user_words != 2 || prog.n_slots > 6 || prog.cls != 0;
  return 2048 * (wide ? kWideR : kRunVariants[variant].r);
}
int run_warps_per_cta() { return kRunWarps; }

cudaError_t launch_fold_runs(const RowArgs& args, const RowProgram& prog, int variant, int grid, cudaStream_t stream) {
  if (variant < 0 || variant >= kNumRunVariants) variant = 0;
  const size_t smem = variant_smem(variant, prog);
  RunKernel k = variant_kernel(variant, prog);  // its smem attribute was set by run_kernel_max_grid
  k<<<grid, kRunThreads, smem, stream>>>(args, prog);
  return cudaGetLastError();
}

}  // namespace sgr
