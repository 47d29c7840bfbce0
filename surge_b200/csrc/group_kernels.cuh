// group_kernels.cuh — K5: stable group-by of arrival-ordered records into CSR form.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "devbuf.h"

namespace sgr {

struct GroupScratch {
  DevBuf keys_a, keys_b, idx_a, idx_b;  // radix-sort ping-pong buffers (u32 each)
  DevBuf hist;                          // per-(digit, block) counts
  DevBuf scan_tmp;                      // block sums of the scans (all levels)
  DevBuf flags;                         // segment-head flags / positions (compact mode)
  DevBuf batch_records;                 // grouped records of an incremental batch
  void release() {
    keys_a.release(); keys_b.release(); idx_a.release(); idx_b.release(); hist.release(); scan_tmp.release();
    flags.release(); batch_records.release();
  }
};

// Stable group-by of n fixed 64-byte records by their aggregate index (u64 at +8, < n_agg). A record with index UINT64_MAX is
// a hole (a record the device decode dropped in place): holes are sorted behind every real record and belong to no segment,
// so the grouped output holds the n - holes real records first.
// Replaces what the Kafka broker + KTable do in the reference: per-key log order is kept
// (modules/common/src/main/scala/surge/kafka/streams/SurgeStateStoreConsumer.scala:57-76).
//   full mode    (d_touched_ids == nullptr): d_out_offsets gets n_agg+1 byte offsets;
//   compact mode (d_touched_ids != nullptr): d_out_offsets gets n_touched+1 byte offsets over the
//                 aggregates that own at least one record, whose indices go to d_touched_ids
//                 (ascending); *n_touched is returned to the host.
// d_counters: >= 8 u64 of scratch. *bad_out = number of records with n_agg <= agg < UINT64_MAX (nothing else is valid then);
// *holes_out (may be null) = number of holes.
cudaError_t group_by_agg_stable(GroupScratch& sc, const uint8_t* d_records, uint64_t n, uint64_t n_agg,
                                uint8_t* d_out_records, uint64_t* d_out_offsets, uint32_t* d_touched_ids,
                                uint64_t* n_touched, unsigned long long* d_counters, cudaStream_t stream,
                                unsigned long long* bad_out, unsigned long long* holes_out);

// Clear the per-batch flags (CHANGED, ERROR, err_idx) of the listed state slots (ids == nullptr: all n slots).
void clear_batch_flags(uint8_t* d_states, uint32_t state_bytes, const uint32_t* d_ids, uint64_t n, cudaStream_t stream);

}  // namespace sgr
