// bulk_fold.cuh — sort-free fold of a large arrival-order log (K6 formulation, separate launches, L2-resident scratch).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dist.cuh"
#include "fold_rows.cuh"

namespace sgr {

// Scratch entry layout chosen from the program (16-byte states, class 0, every state word add-only or set-only):
//   +0  u32 last   (arrival index + 1) << 2 | exists-op of the slot's last event (1 Some, 2 None, 3 threw); 0 = untouched
//   add-only word  u32 accumulator
//   set-only word  u64 max of (arrival index + 1) << 32 | value  = the value of the LAST set
// 16 bytes per slot when at most one word is set-only (Counter: count added, version set), else 32.
struct BulkLayout {
  uint32_t entry_shift;      // 4 or 5
  uint32_t word_off[2];      // byte offset of each state word's cell inside the entry
  uint32_t set_only_mask;    // bit w: word w is only ever SET
  uint32_t has_none;         // some rule produces None (TOMBSTONE): the last event's exists-op decides
  uint32_t last_needed_mask; // bit t: events of type t must record themselves in `last` (has_none, or the rule has no SET op
                             // that would mark the slot as touched)
};

// measurement knobs (sgr_set_option "bulk_unroll" / "bulk_hints" / "bulk_blocks_per_sm"); the defaults are the measured best
struct BulkTuning { int unroll = 4; int hints = 1; int blocks_per_sm = 8; };
BulkTuning& bulk_tuning();
cudaError_t bulk_preload_kernels();   // force the (lazy) load of every kernel of this file

// false when the program is outside the sort-free formulation (a word both added and set, wide state, class 1, f64 fields)
bool bulk_layout_for(const RowProgram& prog, BulkLayout* out);
size_t bulk_scratch_bytes(const BulkLayout& lay, uint64_t n_slots);   // entries + the throw bitmap behind them

// Where the records of one accumulate launch live: up to kMaxRanks regions (one per source rank for a routed chunk, one for a
// plain log). A region's record count is either given, or read on the device from an arrival flag
// ((epoch << 32) | count + 1, written by the sender once the region is complete).
struct BulkSrc {
  const uint8_t* base[kMaxRanks];
  const unsigned long long* count_flag[kMaxRanks];
  uint64_t count[kMaxRanks];
  uint32_t idx_base[kMaxRanks];   // arrival index of the region's first record: monotone per aggregate across launches
  uint32_t n_regions;
  uint32_t blocks_per_sm;         // 0: the tuning default; else the grid cap of this launch (a fold that reads peers over NVLink
                                  // must leave the SMs to the partition kernel running beside it)
  uint32_t rotate;                // region the first tile starts with (the reader's rank: staggers the peers)
  uint32_t carried;               // routed records: the arrival index is idx_base + the index the record carries (full records:
                                  // upper half of the agg field; projected: low 27 bits of word 1), not its position
  uint32_t compact;               // 0: 64-byte records (agg u64 at +8); 1: projected records: u32 local agg, type << 27 | index,
                                  //    then the slot words 1..
  uint32_t rec_bytes;             // record stride
};

// counters (u64): [0] holes (agg == UINT64_MAX, skipped) [1] throwing slots (after finish) [3] error list length [4] records with slot >= n_slots
cudaError_t launch_bulk_accumulate(const BulkSrc& src, uint64_t n_slots, void* d_scratch, const RowProgram& prog, const BulkLayout& lay,
                                   unsigned long long* d_counters, int num_sms, cudaStream_t st);
// by slot: applies (last, accumulators) to the prior state, sets EXISTS/CHANGED, zeroes the slot's scratch; slots that saw a
// throwing event keep their state and are appended to d_err_ids (counters[3]) for the exact replay
cudaError_t launch_bulk_finish(uint64_t n_slots, void* d_scratch, uint8_t* d_states, uint32_t* d_err_ids, const BulkLayout& lay,
                               unsigned long long* d_counters, cudaStream_t st);

// 64-bit order-independent hash of a state table: sum over slots of mix(global id, state words) mod 2^64.
// d_global_ids == nullptr: the slot index is the id. Used by the multi-GPU parity check (bench.py, tests).
cudaError_t launch_states_hash(const uint8_t* d_states, uint64_t n_slots, uint32_t state_bytes, const uint32_t* d_global_ids,
                               unsigned long long* d_out, cudaStream_t st);

}  // namespace sgr
