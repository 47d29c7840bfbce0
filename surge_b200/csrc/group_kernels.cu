// group_kernels.cu — K5: stable group-by of arrival-ordered 64-byte records into CSR form (sm_100a).
//
// A Kafka partition log interleaves aggregates; the fold wants each aggregate's events
// contiguous and in log order. The reference gets that from the broker + KTable keyed store
// (modules/common/src/main/scala/surge/kafka/streams/SurgeStateStoreConsumer.scala:57-76);
// here it is a stable LSD radix sort of (aggregate index, arrival index) pairs — 8 bytes per
// record instead of 64 — followed by ONE gather of the 64-byte records into CSR order:
//   extract keys -> [hist -> scan -> stable scatter] x ceil(bits/8) -> offsets -> gather
// Stability of every pass keeps per-aggregate arrival order, which is the only order the
// fold depends on. All kernels are plain HBM-bound integer kernels (no tensor cores).
#include "group_kernels.cuh"

#include <stdio.h>

#include "../../include/sgr.h"

namespace sgr {
namespace {

constexpr int kThreads = 256;
constexpr int kItems = 16;
constexpr int kTile = kThreads * kItems;  // 4096 keys per block
constexpr int kWarps = kThreads / 32;
constexpr int kPerWarp = kTile / kWarps;  // 512 keys per warp
constexpr int kRounds = kPerWarp / 32;    // 16

// ---------------------------------------------------------------- keys
// A hole (agg == UINT64_MAX: a record the device decode dropped in place) gets the sentinel key n_agg, which sorts after every
// real key; any other agg >= n_agg is counted as bad.
__global__ void extract_keys_kernel(const uint8_t* __restrict__ rec, uint32_t n, uint64_t n_agg,
                                    uint32_t* __restrict__ keys, unsigned long long* __restrict__ bad, unsigned long long* __restrict__ holes) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long agg = *reinterpret_cast<const unsigned long long*>(rec + (size_t)i * 64 + 8);
  if (agg == ~0ull) { atomicAdd(holes, 1ull); keys[i] = (uint32_t)n_agg; return; }
  if (agg >= n_agg) atomicAdd(bad, 1ull);
  keys[i] = (uint32_t)agg;
}

// ---------------------------------------------------------------- exclusive scan (u32), three-kernel, recursive on block sums
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total, uint32_t* smem /*[kWarps]*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) smem[warp] = x;
  __syncthreads();
  uint32_t base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) {
    const uint32_t s = smem[w];
    if (w < warp) base += s;
    tot += s;
  }
  __syncthreads();
  *total = tot;
  return base + x - v;
}

__global__ void __launch_bounds__(kThreads) scan_reduce_kernel(const uint32_t* __restrict__ in, uint32_t n, uint32_t* __restrict__ sums) {
  __shared__ uint32_t sm[kWarps];
  const uint32_t base = blockIdx.x * kTile + threadIdx.x * kItems;
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < kItems; ++j) s += (base + j < n) ? in[base + j] : 0u;
  uint32_t total;
  block_exclusive_scan(s, &total, sm);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kThreads) scan_down_kernel(const uint32_t* __restrict__ in, uint32_t n, const uint32_t* __restrict__ sums_ex,
                                                             uint32_t* __restrict__ out) {
  __shared__ uint32_t sm[kWarps];
  const uint32_t base = blockIdx.x * kTile + threadIdx.x * kItems;
  uint32_t v[kItems];
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < kItems; ++j) { v[j] = (base + j < n) ? in[base + j] : 0u; s += v[j]; }
  uint32_t total;
  uint32_t run = block_exclusive_scan(s, &total, sm) + (sums_ex ? sums_ex[blockIdx.x] : 0u);
#pragma unroll
  for (int j = 0; j < kItems; ++j) { if (base + j < n) out[base + j] = run; run += v[j]; }
}

// exclusive scan of in[0..n) into out (may alias in). tmp must hold >= 2*ceil(n/kTile)+ 2*kTile u32.
cudaError_t exclusive_scan_u32(const uint32_t* in, uint32_t* out, uint32_t n, uint32_t* tmp, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  const uint32_t nb = (n + kTile - 1) / kTile;
  if (nb == 1) {
    scan_down_kernel<<<1, kThreads, 0, st>>>(in, n, nullptr, out);
    return cudaGetLastError();
  }
  scan_reduce_kernel<<<nb, kThreads, 0, st>>>(in, n, tmp);
  cudaError_t e = exclusive_scan_u32(tmp, tmp, nb, tmp + nb, st);
  if (e != cudaSuccess) return e;
  scan_down_kernel<<<nb, kThreads, 0, st>>>(in, n, tmp, out);
  return cudaGetLastError();
}

// lanes holding the same 8-bit digit; invalid lanes match nobody. (Measured on B200: MATCH.ANY beats the
// 8-ballot formulation here, 3.10 ms vs 4.13 ms for the whole group-by of 33.5 M records.)
__device__ __forceinline__ uint32_t match_digit(uint32_t d, bool valid) {
  const uint32_t m = __match_any_sync(0xffffffffu, valid ? d : (256u + (threadIdx.x & 31)));
  return valid ? m : 0u;
}

// ---------------------------------------------------------------- radix pass
// Per-block digit histogram: hist[digit * nblocks + block]
__global__ void __launch_bounds__(kThreads) radix_hist_kernel(const uint32_t* __restrict__ keys, uint32_t n, int shift,
                                                              uint32_t* __restrict__ hist, uint32_t nblocks) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t base = blockIdx.x * kTile;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const uint32_t i = base + j * kThreads + threadIdx.x;
    if (i < n) atomicAdd(&h[(keys[i] >> shift) & 255u], 1u);
  }
  __syncthreads();
  hist[threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];
}

// Stable scatter. Warp w of the block owns keys [w*512, (w+1)*512) of the tile, in 16 rounds of 32.
// A key's place inside the tile's digit-sorted order = (keys of smaller digits in the tile) + keys with the same
// digit in earlier warps + in this warp's earlier rounds + in lower lanes of this round. The (key, index) pairs are
// first reordered in shared memory and then written out in that order, so every digit's run of the tile goes to
// consecutive global addresses (coalesced) instead of 32 scattered 4-byte stores per warp instruction.
__global__ void __launch_bounds__(kThreads) radix_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ idx_in,
                                                                 uint32_t* __restrict__ keys_out, uint32_t* __restrict__ idx_out, uint32_t n,
                                                                 int shift, const uint32_t* __restrict__ base, uint32_t nblocks) {
  __shared__ uint32_t wh[kWarps][256];
  __shared__ uint32_t skey[kTile];
  __shared__ uint32_t sidx[kTile];
  __shared__ uint32_t gbase[256];
  __shared__ uint32_t scan_sm[kWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < kWarps * 256; i += kThreads) (&wh[0][0])[i] = 0;
  __syncthreads();
  const uint32_t tile0 = blockIdx.x * kTile;
  const uint32_t start = tile0 + warp * kPerWarp;
  uint32_t key[kRounds];
  uint16_t pre[kRounds];   // keys with the same digit in this warp's earlier rounds + in lower lanes of this round
  const uint32_t lt = (1u << lane) - 1u;
  // phase 1: this warp's digit counts, and every key's rank among the warp's keys of its digit — ONE match per key: the second
  // MATCH.ANY of the placement phase (r01: 32 per warp and tile, the kernel's main cost) is replaced by a register
#pragma unroll
  for (int r = 0; r < kRounds; ++r) {
    const uint32_t i = start + r * 32 + lane;
    const bool valid = i < n;
    key[r] = valid ? keys_in[i] : 0u;
    const uint32_t d = (key[r] >> shift) & 255u;
    const uint32_t m = match_digit(d, valid);
    const uint32_t earlier = valid ? wh[warp][d] : 0u;    // read by every lane of the digit before its leader adds this round
    pre[r] = (uint16_t)(earlier + __popc(m & lt));
    __syncwarp();
    if (valid && (m & lt) == 0) wh[warp][d] = earlier + __popc(m);
    __syncwarp();
  }
  __syncthreads();
  // phase 2: per digit, exclusive prefix over warps; then exclusive scan over digits = start of the digit's run in the tile
  {
    const uint32_t d = threadIdx.x;
    uint32_t off = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) { const uint32_t c = wh[w][d]; wh[w][d] = off; off += c; }
    uint32_t total;
    const uint32_t tile_start = block_exclusive_scan(off, &total, scan_sm);
#pragma unroll
    for (int w = 0; w < kWarps; ++w) wh[w][d] += tile_start;
    gbase[d] = base[d * nblocks + blockIdx.x] - tile_start;  // global position = gbase[digit] + place in tile
  }
  __syncthreads();
  // phase 3: place every pair at its digit-sorted position in shared memory
#pragma unroll
  for (int r = 0; r < kRounds; ++r) {
    const uint32_t i = start + r * 32 + lane;
    if (i < n) {
      const uint32_t pos = wh[warp][(key[r] >> shift) & 255u] + pre[r];
      skey[pos] = key[r]; sidx[pos] = idx_in ? idx_in[i] : i;
    }
  }
  __syncthreads();
  // phase 4: write the tile out in sorted order
  const uint32_t tile_n = n - tile0 < (uint32_t)kTile ? n - tile0 : (uint32_t)kTile;
  for (uint32_t j = threadIdx.x; j < tile_n; j += kThreads) {
    const uint32_t k = skey[j];
    const uint32_t pos = gbase[(k >> shift) & 255u] + j;
    keys_out[pos] = k;
    idx_out[pos] = sidx[j];
  }
}

// ---------------------------------------------------------------- CSR offsets from sorted keys
// full mode: offsets[a] = 64 * lower_bound(sorted, a) for a in [0, n_agg] (the holes' sentinel run starts at offsets[n_agg])
__global__ void offsets_full_kernel(const uint32_t* __restrict__ sorted, uint32_t n, uint64_t n_agg, uint64_t* __restrict__ offsets) {
  const uint64_t a = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a > n_agg) return;
  uint32_t lo = 0, hi = n;
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if ((uint64_t)sorted[mid] < a) lo = mid + 1; else hi = mid;
  }
  offsets[a] = (uint64_t)lo * 64;
}

// compact mode: heads[j] = 1 where a new aggregate (or the holes' sentinel run, which comes last) starts in the sorted order
__global__ void heads_kernel(const uint32_t* __restrict__ sorted, uint32_t n, uint32_t* __restrict__ heads) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  heads[j] = (j == 0 || sorted[j] != sorted[j - 1]) ? 1u : 0u;
}
__global__ void compact_kernel(const uint32_t* __restrict__ sorted, uint32_t n, const uint32_t* __restrict__ heads,
                               const uint32_t* __restrict__ pos, uint32_t* __restrict__ ids, uint64_t* __restrict__ offsets,
                               uint32_t hole_key, unsigned long long* __restrict__ n_touched) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  if (sorted[j] == hole_key) {
    // the holes' run ends the real records: no touched id of its own
    if (heads[j]) { offsets[pos[j]] = (uint64_t)j * 64; *n_touched = pos[j]; }
    return;
  }
  if (heads[j]) { ids[pos[j]] = sorted[j]; offsets[pos[j]] = (uint64_t)j * 64; }
  if (j == n - 1) {
    const uint32_t t = pos[j] + heads[j];
    offsets[t] = (uint64_t)n * 64;
    *n_touched = t;
  }
}

// ---------------------------------------------------------------- gather: out[j] = rec[idx[j]], 4 lanes x 16 bytes per record
__global__ void gather_records_kernel(const uint8_t* __restrict__ rec, const uint32_t* __restrict__ idx, uint32_t n, uint8_t* __restrict__ out) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t j = t >> 2;
  if (j >= n) return;
  const uint32_t part = (uint32_t)t & 3u;
  const uint4 v = __ldg(reinterpret_cast<const uint4*>(rec + (size_t)idx[j] * 64) + part);
  reinterpret_cast<uint4*>(out + j * 64)[part] = v;
}

__global__ void clear_flags_kernel(uint8_t* __restrict__ states, uint32_t state_bytes, const uint32_t* __restrict__ ids, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t slot = ids ? (uint64_t)ids[i] : i;
  uint2* p = reinterpret_cast<uint2*>(states + slot * state_bytes + state_bytes - 8);
  uint2 v = *p;
  v.x &= SGR_ST_EXISTS; v.y = 0;
  *p = v;
}

inline uint32_t cdiv(uint64_t a, uint32_t b) { return (uint32_t)((a + b - 1) / b); }

}  // namespace

cudaError_t exclusive_scan_u32_public(const uint32_t* in, uint32_t* out, uint32_t n, uint32_t* tmp, cudaStream_t st) {
  return exclusive_scan_u32(in, out, n, tmp, st);
}

void clear_batch_flags(uint8_t* d_states, uint32_t state_bytes, const uint32_t* d_ids, uint64_t n, cudaStream_t stream) {
  if (!n) return;
  clear_flags_kernel<<<cdiv(n, 256), 256, 0, stream>>>(d_states, state_bytes, d_ids, n);
}

cudaError_t group_by_agg_stable(GroupScratch& sc, const uint8_t* d_records, uint64_t n64, uint64_t n_agg,
                                uint8_t* d_out_records, uint64_t* d_out_offsets, uint32_t* d_touched_ids,
                                uint64_t* n_touched, unsigned long long* d_counters, cudaStream_t st,
                                unsigned long long* bad_out, unsigned long long* holes_out) {
  const uint32_t n = (uint32_t)n64;
  cudaError_t e;
  *bad_out = 0;
  if (holes_out) *holes_out = 0;
  if (n_touched) *n_touched = 0;
  if (n == 0) {
    // empty batch: every aggregate has an empty segment
    if (!d_touched_ids) {
      if ((e = cudaMemsetAsync(d_out_offsets, 0, (n_agg + 1) * 8, st)) != cudaSuccess) return e;
    } else if ((e = cudaMemsetAsync(d_out_offsets, 0, 8, st)) != cudaSuccess) return e;
    return cudaStreamSynchronize(st);
  }
  const uint32_t nblocks = cdiv(n, kTile);
  if ((e = sc.keys_a.reserve((size_t)n * 4)) != cudaSuccess || (e = sc.keys_b.reserve((size_t)n * 4)) != cudaSuccess ||
      (e = sc.idx_a.reserve((size_t)n * 4)) != cudaSuccess || (e = sc.idx_b.reserve((size_t)n * 4)) != cudaSuccess ||
      (e = sc.hist.reserve((size_t)256 * nblocks * 4)) != cudaSuccess ||
      (e = sc.scan_tmp.reserve(((size_t)2 * cdiv((uint64_t)256 * nblocks > n ? (uint64_t)256 * nblocks : n, kTile) + 4 * kTile) * 4)) != cudaSuccess)
    return e;
  uint32_t *ka = (uint32_t*)sc.keys_a.p, *kb = (uint32_t*)sc.keys_b.p, *ia = (uint32_t*)sc.idx_a.p, *ib = (uint32_t*)sc.idx_b.p;
  uint32_t* hist = (uint32_t*)sc.hist.p;
  uint32_t* tmp = (uint32_t*)sc.scan_tmp.p;

  if ((e = cudaMemsetAsync(d_counters, 0, 64, st)) != cudaSuccess) return e;
  extract_keys_kernel<<<cdiv(n, 256), 256, 0, st>>>(d_records, n, n_agg, ka, d_counters + 4, d_counters + 6);

  // keys 0..n_agg (n_agg: the holes' sentinel) must all be told apart, or a hole lands in slot n_agg-1's bucket
  int bits = 1;
  while (bits < 32 && (1ull << bits) <= n_agg) ++bits;
  for (int shift = 0; shift < bits; shift += 8) {
    radix_hist_kernel<<<nblocks, kThreads, 0, st>>>(ka, n, shift, hist, nblocks);
    if ((e = exclusive_scan_u32(hist, hist, 256 * nblocks, tmp, st)) != cudaSuccess) return e;
    // first pass: the arrival index is the position itself
    radix_scatter_kernel<<<nblocks, kThreads, 0, st>>>(ka, shift == 0 ? nullptr : ia, kb, ib, n, shift, hist, nblocks);
    uint32_t* t;
    t = ka; ka = kb; kb = t;
    t = ia; ia = ib; ib = t;
  }
  // ka/ia now hold the sorted keys and the arrival indices in CSR order
  if (!d_touched_ids) {
    offsets_full_kernel<<<cdiv(n_agg + 1, 256), 256, 0, st>>>(ka, n, n_agg, d_out_offsets);
  } else {
    if ((e = sc.flags.reserve((size_t)n * 8)) != cudaSuccess) return e;
    uint32_t* heads = (uint32_t*)sc.flags.p;
    uint32_t* pos = heads + n;
    heads_kernel<<<cdiv(n, 256), 256, 0, st>>>(ka, n, heads);
    if ((e = exclusive_scan_u32(heads, pos, n, tmp, st)) != cudaSuccess) return e;
    compact_kernel<<<cdiv(n, 256), 256, 0, st>>>(ka, n, heads, pos, d_touched_ids, d_out_offsets, (uint32_t)n_agg, d_counters + 5);
  }
  gather_records_kernel<<<cdiv((uint64_t)n * 4, 256), 256, 0, st>>>(d_records, ia, n, d_out_records);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  unsigned long long h[3];
  if ((e = cudaMemcpyAsync(h, d_counters + 4, 24, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  *bad_out = h[0];
  if (holes_out) *holes_out = h[2];
  if (n_touched) *n_touched = h[1];
  return cudaSuccess;
}

}  // namespace sgr
