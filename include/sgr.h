/*
 * sgr.h — C ABI of the B200 batched event-replay engine ("surge gpu replay").
 *
 * This is the drop-in boundary for ONE path of UltimateSoftware/surge: rebuilding
 * aggregate state by folding each aggregate's ordered event log through the model's
 * event handler, and the AggregateStateStore recovery read that consumes the result.
 * The reference has no FFI of its own (pure Scala/JVM); each entry point below names
 * the JVM interface a JNI stub would bind it behind (paths relative to the reference
 * checkout, see INTEGRATION.md for the stubs):
 *
 *   CORE  = modules/command-engine/core/src/main/scala/surge
 *   SDSL  = modules/command-engine/scaladsl/src/main/scala/surge/scaladsl
 *   COMMON= modules/common/src/main/scala/surge
 *
 * Conventions
 *   - plain C, no C++/CUDA/torch types cross this boundary;
 *   - every function returns an int32 status (SGR_OK == 0, negative == error class);
 *     the message for the calling thread's last error on an engine is sgr_last_error(engine)
 *     (errno-style, thread-local: concurrent readers never share a message buffer);
 *   - buffers are caller-allocated and caller-owned in both directions; the engine
 *     never frees caller memory and only sgr_destroy frees engine memory;
 *   - "_device" variants take CUDA device pointers on the engine's device and BORROW
 *     them (no copy) — the caller keeps them alive until the next load or destroy;
 *   - load/fold calls are serialised by the caller (the Kafka Streams stream thread in
 *     the reference, COMMON/kafka/streams/KafkaStreamManagerActor.scala:106-133);
 *     sgr_get / sgr_get_index may be called concurrently from many threads (the
 *     reference reads the store from a 32-thread pool,
 *     COMMON/kafka/streams/ThreadPools.scala:9-11).
 *   - there is NO CPU fallback: without a usable CUDA device sgr_create fails.
 */
#ifndef SGR_H
#define SGR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGR_ABI_VERSION 1

/* ------------------------------------------------------------------ status codes */
#define SGR_OK                 0
#define SGR_ERR_INVALID       -1   /* bad argument / malformed buffer (IllegalArgumentException) */
#define SGR_ERR_NO_DEVICE     -2   /* no CUDA device / extension unusable: fail loudly, never fall back */
#define SGR_ERR_CUDA          -3   /* a CUDA call failed; message carries cudaGetErrorString */
#define SGR_ERR_NO_PROGRAM    -4   /* fold requested before sgr_register_program */
#define SGR_ERR_NOT_LOADED    -5   /* fold/get requested before any load */
#define SGR_ERR_UNSUPPORTED   -6   /* model cannot be expressed as a fold program: decline the plugin */
#define SGR_ERR_OOM           -7
#define SGR_ERR_STATE         -8   /* store not readable now (maps to InvalidStateStoreException,
                                      COMMON/kafka/streams/SurgeAggregateStore.scala:31-46) */
#define SGR_ERR_DIST          -9   /* NCCL / peer-memory failure */
#define SGR_ERR_CAPACITY     -10   /* caller buffer too small */
#define SGR_ERR_AGAIN        -11   /* loopback ranks only: repeat the call on every rank with option "push_ordered" = 1 */

/* ------------------------------------------------------------------ packed formats
 *
 * Fixed record (SGR_REC_FIXED64): 64 bytes, little-endian, 64-byte aligned in the log
 *   +0  u32 type      event type = index into the program's rule table
 *   +4  u32 seq       sequence number (Counter: sequenceNumber)
 *   +8  u64 agg       dense aggregate index (or global index before routing)
 *   +16 u8  payload[48]  program-defined view (Counter: i32 by @16;
 *                        BankAccount: uuid @16, f64 balance @32, owner @40, code @56)
 *
 * Variable record (SGR_REC_VAR16): 16-byte header + payload padded to 16 bytes
 *   +0  u32 type   +4 u32 seq   +8 u32 payload_len (unpadded)   +12 u32 agg
 *   +16 payload, padded with zeros up to a multiple of 16
 *
 * CSR: u64 seg_offsets[n_agg+1], BYTE offsets into the event log; segment i is
 *   [seg_offsets[i], seg_offsets[i+1]); every offset is a multiple of 16 so that
 *   each segment is a legal source for a 1-D TMA bulk copy.
 *
 * State table: n_agg structs of state_bytes (multiple of 16, <= SGR_MAX_STATE_BYTES).
 *   The program owns bytes [0, state_bytes-8); the engine owns the trailing 8:
 *   +state_bytes-8  u32 flags   (SGR_ST_EXISTS | SGR_ST_CHANGED | SGR_ST_ERROR)
 *   +state_bytes-4  u32 err_idx (index, within the aggregate's batch, of the event that
 *                                threw; 0 when no error)
 *   A state that does not exist (Scala None) has all program bytes zero.
 */
#define SGR_REC_FIXED64 0u
#define SGR_REC_VAR16   1u

#define SGR_ST_EXISTS   1u
#define SGR_ST_CHANGED  2u   /* newState != oldState: the publish rule of
                                CORE/internal/persistence/PersistentActor.scala:252-257 */
#define SGR_ST_ERROR    4u   /* handler threw: state kept at its pre-batch value
                                (PersistentActor.scala:260-263,303-309) */

#define SGR_MAX_STATE_BYTES 128u
#define SGR_MAX_TYPES        16u
#define SGR_MAX_OPS           8u

/* ------------------------------------------------------------------ fold program
 *
 * Declarative form of AggregateCommandModel.handleEvent(Option[Agg], Evt): Option[Agg]
 * (SDSL/command/CommandModels.scala:14). A JVM closure cannot run on a GPU, so a model
 * registers, next to its handler, one rule per event type:
 *
 *   exists_rule   what happens to Option-ness before the field ops run
 *     SGR_IF_EXISTS    None stays None and the ops are skipped   (aggregate.map(_.copy(..)))
 *     SGR_MATERIALISE  None becomes the all-zero default state    (agg.getOrElse(State(id,0,0)))
 *     SGR_CREATE       state is reset to the default, then ops    (Some(Agg(evt fields)))
 *     SGR_TOMBSTONE    state becomes None                          (handler returns None)
 *     SGR_THROW        the handler throws                          (ExceptionThrowingEvent)
 *   ops           word-granular field transfers record -> state, applied in order.
 *                 All offsets/lengths are byte counts and multiples of 4.
 *
 * An event whose type is >= n_types is a scala.MatchError, i.e. SGR_THROW.
 *
 * Instance identity: a rule with field ops, SGR_CREATE, and SGR_MATERIALISE on None build a NEW state instance
 * (Scala constructor / copy); SGR_IF_EXISTS / SGR_MATERIALISE without ops on an existing state hand the same instance
 * back (`current`). The publish rule compares with the case-class equals, which starts with `this eq that`: an
 * aggregate with no events in the fold, or only instance-preserving ones, is never SGR_ST_CHANGED — even if one of its
 * Double fields holds a NaN — while a new instance compares field by field (NaN != NaN, 0.0 == -0.0).
 */
#define SGR_IF_EXISTS    0u
#define SGR_MATERIALISE  1u
#define SGR_CREATE       2u
#define SGR_TOMBSTONE    3u
#define SGR_THROW        4u

#define SGR_OP_SET      0u  /* state[dst .. dst+len) = record[src .. src+len)   (bit copy; f64, strings) */
#define SGR_OP_ADD_I32  1u  /* state.i32[dst] += record.i32[src]   two's-complement wrap (JVM Int)  */
#define SGR_OP_SUB_I32  2u  /* state.i32[dst] -= record.i32[src]                                     */
#define SGR_OP_ADD_I64  3u  /* state.i64[dst] += record.i64[src]   wrap (JVM Long)                    */
#define SGR_OP_SUB_I64  4u

typedef struct sgr_op {
  uint8_t  opcode;     /* SGR_OP_* */
  uint8_t  reserved;
  uint16_t dst_off;    /* byte offset into the state struct (program area) */
  uint16_t src_off;    /* byte offset into the record, header included */
  uint16_t len;        /* bytes; SET: any multiple of 4; I32 ops: 4; I64 ops: 8 */
} sgr_op;

typedef struct sgr_rule {
  uint8_t exists_rule; /* SGR_IF_EXISTS .. SGR_THROW */
  uint8_t n_ops;       /* <= SGR_MAX_OPS */
  uint8_t reserved[6];
  sgr_op  ops[SGR_MAX_OPS];
} sgr_rule;

typedef struct sgr_fold_program {
  uint32_t state_bytes;   /* multiple of 16, 16..SGR_MAX_STATE_BYTES, includes the 8 engine bytes */
  uint32_t record_kind;   /* SGR_REC_FIXED64 | SGR_REC_VAR16 */
  uint32_t n_types;       /* <= SGR_MAX_TYPES */
  uint32_t n_f64_fields;  /* <= 8: state fields that are JVM Doubles; they are bit-copied by SGR_OP_SET
                             but compare with == for the publish rule (0.0 == -0.0, NaN != NaN), as
                             Scala case-class equality does in PersistentActor.scala:257 */
  uint16_t f64_field_off[8];
  sgr_rule rules[SGR_MAX_TYPES];
} sgr_fold_program;

/* ------------------------------------------------------------------ engine */
typedef struct sgr_engine sgr_engine;   /* opaque */

typedef struct sgr_config {
  int32_t  device;          /* CUDA device ordinal */
  uint32_t flags;           /* reserved, 0 */
  uint64_t reserved[6];
} sgr_config;

typedef struct sgr_stats {
  uint64_t n_aggregates;    /* segments folded by the last fold */
  uint64_t n_events;        /* events consumed by the last fold */
  uint64_t event_bytes;     /* stored event-record bytes read by the last fold */
  uint64_t algorithmic_bytes;/* event_bytes + 8*(n_agg+1) + state_bytes*n_agg (+ prior states read) */
  uint64_t n_errors;        /* aggregates whose handler threw */
  uint64_t n_long_segments; /* aggregates taken by the split (long-segment) path */
  float    ms_h2d;          /* host->device copy of the last load (0 for _device loads) */
  float    ms_group;        /* stable group-by of the last unsorted load */
  float    ms_fold;         /* device time of the last fold (all its kernels) */
  float    ms_d2h;          /* device->host copy of the last export */
  uint32_t fold_launches;   /* kernels launched by the last fold */
  uint32_t reserved[7];
} sgr_stats;

int32_t sgr_abi_version(void);

/* Create an engine bound to one CUDA device. Replaces the construction of the state
 * store inside the engine pipeline (CORE/internal/domain/SurgeMessagePipeline.scala:68-78). */
int32_t sgr_create(const sgr_config* cfg, sgr_engine** out);
int32_t sgr_destroy(sgr_engine* e);
const char* sgr_last_error(const sgr_engine* e);   /* e may be NULL: last create error */

/* Register the declarative form of the model's event handler
 * (SDSL/command/CommandModels.scala:14; core entry
 * CORE/internal/domain/AggregateProcessingModel.scala:21). */
int32_t sgr_register_program(sgr_engine* e, const sgr_fold_program* prog);

/* Load a CSR-ordered event log (host buffers; copied to HBM). The log is what
 * AggregateRef.applyEvents would be handed per aggregate, for every aggregate at once
 * (SDSL/common/AggregateRefBaseTrait.scala:23-28). */
int32_t sgr_load_events(sgr_engine* e, const void* events, uint64_t nbytes,
                        const uint64_t* seg_offsets, uint64_t n_agg);
int32_t sgr_load_events_device(sgr_engine* e, const void* d_events, uint64_t nbytes,
                               const uint64_t* d_seg_offsets, uint64_t n_agg);

/* Variable records with a record directory: rec_offsets[n_records+1] are the byte offsets of every record in log order
 * (the packer knows them for free). With it the log is cut into record-balanced spans, so skewed (Zipf) keys do not
 * serialise one lane; without it (sgr_load_events) variable records are folded one lane per aggregate. */
int32_t sgr_load_events_indexed(sgr_engine* e, const void* events, uint64_t nbytes, const uint64_t* seg_offsets, uint64_t n_agg,
                                const uint64_t* rec_offsets, uint64_t n_records);
int32_t sgr_load_events_indexed_device(sgr_engine* e, const void* d_events, uint64_t nbytes, const uint64_t* d_seg_offsets,
                                       uint64_t n_agg, const uint64_t* d_rec_offsets, uint64_t n_records);

/* Load records in ARRIVAL order (a Kafka partition log interleaves aggregates) and group
 * them, stably, by aggregate index into CSR form on the device. n_agg is the number of
 * dense aggregate indices (records carry agg < n_agg). Fixed 64-byte records only.
 * Holes: a record with agg == UINT64_MAX is a hole (what the device ingest leaves in place of a dropped record) and is
 * skipped by every arrival-order entry point (sgr_load_unsorted*, sgr_fold_unsorted*, sgr_fold_incremental*): the outcome,
 * statistics included, is that of the same records without the holes. Any other agg >= n_agg fails the call with
 * SGR_ERR_INVALID and nothing is applied. */
int32_t sgr_load_unsorted(sgr_engine* e, const void* records, uint64_t n_records, uint64_t n_agg);
int32_t sgr_load_unsorted_device(sgr_engine* e, const void* d_records, uint64_t n_records, uint64_t n_agg);

/* Rebuild every state from an arrival-order log in one call (the shape of a Kafka partition log: aggregates
 * interleaved, each aggregate's own order kept), without exposing a CSR log afterwards. Programs inside the
 * transformer algebra with add-only / set-only words need no grouping at all (integer-atomic fold); others are grouped
 * and folded as sgr_load_unsorted + sgr_fold would. */
int32_t sgr_fold_unsorted(sgr_engine* e, const void* records, uint64_t n_records, uint64_t n_agg);
int32_t sgr_fold_unsorted_device(sgr_engine* e, const void* d_records, uint64_t n_records, uint64_t n_agg);

/* Prior states for an incremental fold (None everywhere if never called):
 * the actor's state before ApplyEvents, PersistentActor.scala:245-264. states may be NULL to reset. */
int32_t sgr_set_initial_states(sgr_engine* e, const void* states, uint64_t n_agg);

/* Fold every aggregate's segment left to right in event order:
 * events.foldLeft(state)(handleEvent), SDSL/command/CommandModels.scala:25-28. */
int32_t sgr_fold(sgr_engine* e);

/* The same fold without host synchronisation: sgr_fold_async enqueues the kernels on the engine's
 * stream and returns; sgr_wait blocks until they finish and collects the statistics. Any call that
 * reads results (get/export/stats) waits implicitly. */
int32_t sgr_fold_async(sgr_engine* e);
int32_t sgr_wait(sgr_engine* e);

/* Append one micro-batch (arrival order, fixed records, holes skipped) to the live state table: group by
 * aggregate, fold onto the current states, write back (PersistentActor.doApplyEvent on a
 * live actor, PersistentActor.scala:245-264). Requires a prior fold or set_initial_states.
 * A fold that fails half-applied (more throwing aggregates than the replay list holds on an in-place fold) invalidates the
 * table: reads, sgr_grow_states, sgr_fold_ingested and sgr_dingest_fold fail with SGR_ERR_STATE until sgr_set_initial_states
 * (NULL included), a full fold or sgr_fold_unsorted replaces it. */
int32_t sgr_fold_incremental(sgr_engine* e, const void* records, uint64_t n_records);
int32_t sgr_fold_incremental_device(sgr_engine* e, const void* d_records, uint64_t n_records);

/* Key table: UTF-8 aggregate ids, key i = keys[key_offsets[i] .. key_offsets[i+1]).
 * Not read by the fold; only by sgr_get. */
int32_t sgr_load_keys(sgr_engine* e, const uint8_t* keys, const uint32_t* key_offsets, uint64_t n_agg);

/* Point lookup of folded state bytes by aggregate id: the recovery read
 * AggregateStateStoreKafkaStreams.getAggregateBytes(aggregateId): Future[Option[Array[Byte]]]
 * (COMMON/kafka/streams/AggregateStateStoreKafkaStreams.scala:83-85). *exists == 0 is None.
 * Thread-safe against a published snapshot. Copies the program bytes (state_bytes-8). */
int32_t sgr_get(sgr_engine* e, const uint8_t* key, uint32_t klen,
                void* out, uint32_t cap, uint32_t* outlen, int32_t* exists);
int32_t sgr_get_index(sgr_engine* e, uint64_t agg, void* out, uint32_t cap,
                      uint32_t* outlen, int32_t* exists, uint32_t* flags, uint32_t* err_idx);
/* The dense aggregate index sgr_get resolves an id to (*agg = UINT64_MAX for an unknown id). The device ingest hands out
 * indices from an atomic counter, so this is how a caller reaches an id's flags and err_idx through sgr_get_index. */
int32_t sgr_key_index(sgr_engine* e, const uint8_t* key, uint32_t klen, uint64_t* agg);

/* Export the whole state table (n_agg * state_bytes) and, optionally, bitmaps
 * (bit i of byte i/8, LSB first). Any out pointer may be NULL. */
int32_t sgr_export_states(sgr_engine* e, void* out, uint64_t cap,
                          uint8_t* exists_bits, uint8_t* changed_bits, uint8_t* error_bits);
/* Device pointer to the live state table (borrowed; valid until the next load/destroy). */
int32_t sgr_states_device(sgr_engine* e, void** d_states, uint64_t* n_agg, uint32_t* state_bytes);
/* Device pointers to the engine's CSR event log (after any load). */
int32_t sgr_events_device(sgr_engine* e, void** d_events, uint64_t* nbytes, uint64_t** d_seg_offsets);

int32_t sgr_get_stats(sgr_engine* e, sgr_stats* out);

/* Tuning knob for measurements: which fold kernel variant to launch
 * (0 = default; see DESIGN.md "kernel variants"). */
int32_t sgr_set_option(sgr_engine* e, const char* name, int64_t value);

/* The CUDA stream (cudaStream_t) the engine launches on, so callers can record events. */
int32_t sgr_stream(sgr_engine* e, void** stream);

/* ------------------------------------------------------------------ multi-GPU (one process per GPU, one node)
 * Aggregates are hash-partitioned across ranks exactly as Surge shards them across nodes
 * (aggregateId -> partition -> owner): partition_of_agg[g] is
 * KafkaPartitionProvider.partitionForKey of global aggregate g (COMMON/kafka/KafkaPartitioner.scala:7-9)
 * and the owner rank is partition % nranks. Each rank feeds the records of ITS source partitions in arrival
 * order (records carry the GLOBAL aggregate index at +8); one exchange over NVLink replaces the broker
 * shuffle (KafkaProducerHelperCommon.getPartitionFor, COMMON/kafka/KafkaProducer.scala:45-57). */
typedef struct sgr_dist_stats {
  uint64_t n_sent, n_sent_remote, n_recv, n_local_aggregates;
  float ms_count, ms_counts_exchange, ms_scatter, ms_exchange, ms_group, ms_fold;
  float ms_pipeline;               /* fused >= 2: device time of the whole overlapped route + exchange + fold */
  uint32_t exchange_record_bytes;  /* bytes per record that crossed NVLink (64, or the projected size with fused == 3) */
  uint32_t reserved[4];
} sgr_dist_stats;

int32_t sgr_dist_unique_id(void* out128);                       /* rank 0: a 128-byte NCCL unique id to hand to the others */
int32_t sgr_dist_init(sgr_engine* e, int32_t rank, int32_t nranks, const void* unique_id128,
                      uint64_t recv_capacity_records);
int32_t sgr_dist_set_partitions(sgr_engine* e, const uint32_t* partition_of_agg, uint64_t n_global_agg);
/* fused path: every rank exports its receive buffer (64-byte CUDA IPC handle), the host exchanges the
 * handles, every rank imports all nranks of them (own slot ignored). */
int32_t sgr_dist_ipc_export(sgr_engine* e, void* out64);
int32_t sgr_dist_ipc_import(sgr_engine* e, const void* handles64_by_rank);
/* Route + exchange + (group-by) + fold.
 *   fused == 0  count + pack, one NCCL all-to-all (grouped ncclSend/ncclRecv), then the fold;
 *   fused == 1  count, then the route kernel writes each record straight into its owner's receive buffer over NVLink;
 *   fused == 2  ONE pass, pipelined: the log is cut into chunks (option "push_chunks", the same on every rank); a push kernel
 *               partitions each chunk in shared memory and writes every owner's run contiguously into that owner's receive
 *               region over NVLink, an arrival flag per (source, chunk) follows, and the owner folds chunk c while chunk c+1 is
 *               still in flight. No count pass, no send buffer, no host synchronisation inside. Needs the peers' receive buffers
 *               (IPC import) and a program in the sort-free class (16-byte state, class 0, every word add-only or set-only) —
 *               other programs silently take fused == 1. Receive regions have a fixed capacity of
 *               recv_capacity / (nranks * push_chunks) records per (source, chunk): a region that would overflow fails the call
 *               with SGR_ERR_CAPACITY on EVERY rank (nothing is written out of bounds); retry with fused <= 1 or more capacity.
 *               Option "push_pull" (default 1): the source partitions into ITS OWN buffer and the owner's fold reads those
 *               regions over NVLink (remote loads: only the 32-byte sectors the fold touches cross the link); 0: the source
 *               writes into the owner's buffer (remote stores). By default a CTA takes its place inside a region with one
 *               atomicAdd per owner and every record carries its index within the chunk, which is the only order the
 *               sort-free fold needs; when any rank meets a throwing aggregate (the exact replay wants positional log order)
 *               every rank repeats the exchange in ordered mode (decoupled look-back) — automatically on real ranks, by
 *               SGR_ERR_AGAIN + option "push_ordered" on loopback ranks.
 *   fused == 3  as 2, but only the record words the fold program reads cross NVLink (u32 local index + slot words:
 *               16 bytes per record for the Counter model). */
int32_t sgr_dist_route_and_fold(sgr_engine* e, const void* d_records, uint64_t n_records, int32_t fused);
/* Several ranks inside ONE process on one device ("loopback", for single-GPU tests of the multi-rank logic): sgr_dist_init with
 * unique_id128 == NULL and nranks > 1 creates such a rank; the ranks hand each other their receive allocation as plain device
 * pointers (sgr_dist_recv_base -> sgr_dist_set_peers) and the caller runs every rank's sgr_dist_route_and_fold(fused >= 2)
 * concurrently (one host thread per rank), with a barrier of its own between calls. fused <= 1 needs NCCL and is refused. */
int32_t sgr_dist_recv_base(sgr_engine* e, void** base);
/* Allocate everything sgr_dist_route_and_fold(fused >= 2) needs for logs of up to max_records records now (after
 * sgr_dist_set_partitions and the "push_chunks" option), so that the call itself allocates nothing. Optional for real ranks;
 * loopback ranks share one device, where an allocation can wait for another rank's kernel: call it on every rank first. */
int32_t sgr_dist_reserve(sgr_engine* e, uint64_t max_records);
int32_t sgr_dist_set_peers(sgr_engine* e, void* const* recv_bases_by_rank);
/* 64-bit order-independent hash of the live state table: sum over slots of mix(aggregate index, state bytes) mod 2^64, the
 * index being the GLOBAL aggregate index on a routed engine — so the sum of the ranks' hashes does not depend on how many ranks
 * there are. The parity check of the multi-GPU runs (bench.py, tests/test_gpu_dist.py; twin: surge_b200/dist.py states_hash). */
int32_t sgr_states_hash(sgr_engine* e, uint64_t* out);
int32_t sgr_dist_get_stats(sgr_engine* e, sgr_dist_stats* out);
/* global aggregate index of each local state slot (host copy, n_local u32) */
int32_t sgr_dist_local_aggregates(sgr_engine* e, uint32_t* out, uint64_t cap, uint64_t* n_local);

/* ------------------------------------------------------------------ ingest: Kafka record batches -> packed records (SURVEY §8 f1, f2)
 * What feeds the store today is a Kafka consumer in read_committed mode
 * (COMMON/kafka/streams/SurgeStateStoreConsumer.scala:38; the plain wrapper is COMMON/kafka/KafkaConsumer.scala:48-105,120-132)
 * over a topic whose producer compresses with lz4 (modules/common/src/main/resources/reference.conf:124) and writes inside
 * transactions. sgr_ingest decodes the raw bytes of a fetch response / log segment — a concatenation of RecordBatch
 * (magic 2) structures — into the engine's fixed 64-byte records in arrival order, interning aggregate ids
 * (key.takeWhile(_ != ':'), COMMON/kafka/KafkaPartitioner.scala:38-42) as dense indices in first-seen order.
 *   - verifies each batch's CRC-32C; decodes compression none and lz4 (gzip/snappy/zstd: SGR_ERR_UNSUPPORTED);
 *   - skips control batches, and data batches of aborted transactions announced with sgr_ingest_set_aborted
 *     (the fetch response's abortedTransactions list), the way a read_committed consumer does;
 *   - drops records with a null/empty key: the producer's flush markers
 *     (CORE/internal/kafka/KafkaProducerActorImpl.scala:321-329);
 *   - a trailing partial batch is left undecoded (n_trailing_bytes), as fetch responses may end with one;
 *   - records below the partition's decoded position are counted as duplicates and skipped (refetch after restart);
 *   - record value = the model's packed event: u32 type, u32 seq (little endian) + up to 48 payload bytes — as is, inside the
 *     multilanguage protobuf Event, or produced from a flat JSON object by a registered member table (sgr_ingest_set_value_framing).
 * A malformed batch fails the whole call and leaves the pending log and the partition position untouched.
 * The RecordBatch framing is third-party (org.apache.kafka:kafka-clients:3.2.3) and the reference holds no broker bytes:
 * its byte-level parity is UNPINNED (see oracle/kafka_batch.py); lz4, xxHash32, CRC-32C and the protobuf framing are pinned
 * against real implementations.
 *
 * Lag gate (f2): actors trust the store only once the consumer group of the streams applicationId has no lag
 * (CORE/internal/kafka/KafkaProducerActorImpl.scala:530-540,684-708; COMMON/kafka/KafkaAdminClient.scala:36-56).
 * sgr_ingest_offsets reports, per partition, the next offset to fetch (decoded_next) and the offset below which every
 * record is inside the state table (folded_next) — the value whoever consumes on the store's behalf commits. */
typedef struct sgr_ingest sgr_ingest;

typedef struct sgr_ingest_stats {
  uint64_t n_bytes;              /* bytes consumed (whole batches) */
  uint64_t n_trailing_bytes;     /* bytes of a trailing partial batch left undecoded (last call only) */
  uint64_t n_batches;
  uint64_t n_records;            /* packed records appended to the pending log */
  uint64_t n_markers;            /* null/empty-key records dropped */
  uint64_t n_null_values;        /* keyed records with a null value: dropped, or turned into tombstone events
                                    (sgr_ingest_set_null_value_type) */
  uint64_t n_control_batches;
  uint64_t n_aborted_batches, n_aborted_records;
  uint64_t n_duplicates;         /* records below the partition's decoded position */
  uint64_t n_new_keys;
  uint64_t n_compressed_bytes, n_decompressed_bytes;
  uint64_t reserved[3];
} sgr_ingest_stats;

int32_t sgr_ingest_create(sgr_ingest** out);
int32_t sgr_ingest_destroy(sgr_ingest* g);
const char* sgr_ingest_last_error(const sgr_ingest* g);
/* How the record value wraps the packed event. SGR_VALUE_PACKED (default): the value IS `u32 type, u32 seq, payload`.
 * SGR_VALUE_PROTOBUF_EVENT: the value is the multilanguage module's protobuf `Event { string aggregateId = 1; bytes payload = 2; }`
 * (modules/multilanguage-protocol/src/main/protobuf/multilanguage-protocol.proto:17-20, written by
 * modules/multilanguage/src/main/scala/com/ukg/surge/multilanguage/GenericSurgeCommandBusinessLogic.scala:30-33) and the packed
 * event is its payload. The framing is pinned against the protobuf runtime in tests/test_ingest_cpu.py. */
#define SGR_VALUE_PACKED          0
#define SGR_VALUE_PROTOBUF_EVENT  1
#define SGR_VALUE_JSON            2
int32_t sgr_ingest_set_value_framing(sgr_ingest* g, int32_t framing);

/* SGR_VALUE_JSON: the value is a flat JSON object as the reference's sample models write their events with play-json,
 * e.g. {"_type":"...CountIncremented","aggregateId":"a","incrementBy":1,"sequenceNumber":4}
 * (modules/command-engine/core/src/test/scala/surge/core/TestBoundedContext.scala:44-56 formats, :159-161 writer).
 * The model registers the discriminator member, the event type index of each class name and where each numeric member
 * lands in the packed record (record byte offsets: 4 = the sequence number, 16..63 = payload). Members are found by name —
 * order, whitespace and extra members do not matter; with an empty discriminator exactly one class is registered and every
 * value is that class (a state topic: Json.toJson(agg) carries no discriminator); an unknown class name becomes event type `unknown_type` (a
 * scala.MatchError in the handler) or, with -1, fails the call. Doubles are parsed correctly rounded (strtod), as
 * java.lang.Double.parseDouble does. The exact bytes play-json writes are NOT pinned (no JVM here); the parser is checked
 * against Python's json module on both well-formed and hostile input. */
#define SGR_JSON_I32  0u
#define SGR_JSON_I64  1u
#define SGR_JSON_F64  2u
#define SGR_JSON_UUID 3u   /* "8-4-4-4-12" string (java.util.UUID.toString) -> 16 bytes, most significant first */
#define SGR_JSON_PSTR 4u   /* string -> length byte + UTF-8 bytes, zero padded to `len` bytes (must fit: len - 1 bytes at most) */
#define SGR_JSON_MAX_FIELDS 8u
typedef struct sgr_json_field { const char* name; uint8_t kind; uint8_t reserved; uint16_t dst_off; uint32_t len; /* PSTR slot */ } sgr_json_field;
typedef struct sgr_json_event {
  const char* type_name;     /* value of the discriminator member */
  uint32_t event_type;       /* index into the fold program's rules */
  uint32_t n_fields;
  sgr_json_field fields[SGR_JSON_MAX_FIELDS];
} sgr_json_event;
int32_t sgr_ingest_set_json_packer(sgr_ingest* g, const char* discriminator, const sgr_json_event* events, uint32_t n_events,
                                   int32_t unknown_type);
/* Compacted STATE topic (what the reference restores from today, COMMON/kafka/streams/SurgeStateStoreConsumer.scala:57-76): a keyed
 * record with a null value deletes the key (CORE/internal/SurgeModel.scala:62-64). With event_type >= 0 such a record becomes an
 * event of that type (the program's SGR_TOMBSTONE rule) instead of being dropped; -1 (default) drops it. */
int32_t sgr_ingest_set_null_value_type(sgr_ingest* g, int32_t event_type);
/* The id dictionary holds at most 2^31 ids and 4 GiB of id bytes (32-bit fields). A call that could exceed a bound fails with
 * SGR_ERR_CAPACITY before anything is applied (every id of the call is counted as new: conservative). Lower bounds can be set
 * to fail earlier (operators; tests). */
int32_t sgr_ingest_set_dictionary_limits(sgr_ingest* g, uint64_t max_ids, uint64_t max_id_bytes);
/* aborted transactions of the next fetch of `partition`: (producerId, firstOffset) pairs */
int32_t sgr_ingest_set_aborted(sgr_ingest* g, int32_t partition, const int64_t* producer_ids, const int64_t* first_offsets, uint64_t n);
int32_t sgr_ingest_record_batches(sgr_ingest* g, int32_t partition, const void* data, uint64_t nbytes, sgr_ingest_stats* stats);
/* n fetches in one call. CRC, decompression and parsing run on up to `threads` host threads (the fetches of one partition
 * stay on one thread, in call order); ids are interned and records appended afterwards in call order, so the outcome is
 * identical to n single calls. All or nothing: one malformed fetch and nothing is applied. stats: n entries or NULL. */
int32_t sgr_ingest_record_batches_mt(sgr_ingest* g, uint32_t n, const int32_t* partitions, const void* const* datas,
                                     const uint64_t* nbytes, uint32_t threads, sgr_ingest_stats* stats);
/* Where the pending log lives (default malloc/free). sgr_fold_ingested installs page-locked host memory so that the copy of
 * a poll to the device is one DMA at full PCIe rate; content already pending is carried over. */
int32_t sgr_ingest_set_allocator(sgr_ingest* g, void* (*alloc_fn)(size_t), void (*free_fn)(void*));
/* the pending packed records (borrowed until the next ingest call) and the id dictionary (key i = dense index i) */
int32_t sgr_ingest_pending(sgr_ingest* g, const void** records, uint64_t* n_records);
int32_t sgr_ingest_keys(sgr_ingest* g, const uint8_t** keys, const uint32_t** key_offsets, uint64_t* n_keys);
/* the pending records are inside the state table now: drop them, advance folded_next to decoded_next */
int32_t sgr_ingest_mark_folded(sgr_ingest* g);
int32_t sgr_ingest_offsets(sgr_ingest* g, int32_t partition, int64_t* decoded_next, int64_t* folded_next);
int32_t sgr_ingest_get_stats(sgr_ingest* g, sgr_ingest_stats* out);   /* totals since create */

/* Resize the live state table to n_agg slots on the device, keeping its content; new slots are None.
 * (A KTable grows as new keys appear; never shrinks.) */
int32_t sgr_grow_states(sgr_engine* e, uint64_t n_agg);
/* Fold everything pending in `g` onto the live table (growing it for new aggregate ids), publish the id dictionary
 * to sgr_get, and mark the ingest folded: poll -> sgr_ingest_record_batches -> sgr_fold_ingested is the whole restore loop. */
int32_t sgr_fold_ingested(sgr_engine* e, sgr_ingest* g);

/* Append ids to the key table sgr_get reads: the ids of dense indices [n, n + n_new) where n is the number of ids `owner` has
 * appended so far (a different owner starts a new table). owner is an opaque tag: the id dictionary the table mirrors. */
int32_t sgr_append_keys(sgr_engine* e, const void* owner, const uint8_t* keys, const uint32_t* key_offsets, uint64_t n_new);

/* ------------------------------------------------------------------ device ingest: the same decode ON THE GPU
 * Same input (raw bytes of fetch responses, RecordBatch magic 2, compression none / lz4, read_committed semantics) and the same
 * outcome as sgr_ingest_* + sgr_fold_ingested, but only the WIRE bytes cross PCIe: CRC-32C, lz4, record parsing, id interning and
 * the fold run on the engine's device (csrc/dingest_kernels.cu); the host walks the 61-byte batch headers and keeps the
 * read_committed bookkeeping (control batches, aborted transactions, partition positions). csrc/ingest.cpp is its checker
 * (tests/test_gpu_dingest.py: identical states, ids, offsets and statistics on the same bytes).
 *   - value framing: SGR_VALUE_PACKED only (protobuf / JSON values: use the host ingest);
 *   - dropped records (markers, duplicates, null values) stay in place as holes (aggregate index UINT64_MAX) the fold skips;
 *   - dense indices are stable per id but follow no arrival-order promise (they come from an atomic counter);
 *   - polls are processed in groups of SGR_DINGEST_GROUP (default 8192) batches, each group one chain of launches on one of eight
 *     streams; batches decompress into an arena of 3x the wire bytes (a poll that compresses better is decoded a second time from
 *     an exact layout — correct, slower); SGR_DINGEST_TIMING=1 prints each group's device timeline to stderr;
 *   - the id dictionary is sized at creation: max_keys ids, max_id_bytes id bytes (0 = 32 per id); exceeding either fails the
 *     poll with SGR_ERR_CAPACITY and applies nothing.
 * poll loop:  sgr_dingest_set_aborted* -> sgr_dingest_submit(partition, bytes)* -> sgr_dingest_fold.
 * `data` of a submit must stay valid until the fold returns (with page-locked memory the copy is one asynchronous DMA). */
typedef struct sgr_dingest sgr_dingest;
int32_t sgr_dingest_create(sgr_engine* e, uint64_t max_keys, uint64_t max_id_bytes, sgr_dingest** out);
int32_t sgr_dingest_destroy(sgr_dingest* g);
const char* sgr_dingest_last_error(const sgr_dingest* g);
int32_t sgr_dingest_set_null_value_type(sgr_dingest* g, int32_t event_type);
int32_t sgr_dingest_set_aborted(sgr_dingest* g, int32_t partition, const int64_t* producer_ids, const int64_t* first_offsets, uint64_t n);
int32_t sgr_dingest_submit(sgr_dingest* g, int32_t partition, const void* data, uint64_t nbytes, sgr_ingest_stats* stats);
/* decode + intern + fold everything submitted since the last fold onto the engine's live table (grown as ids appear), publish
 * the new ids to sgr_get, advance the partitions' positions. All or nothing. stats (optional): this poll's totals. */
int32_t sgr_dingest_fold(sgr_dingest* g, sgr_ingest_stats* stats);
int32_t sgr_dingest_offsets(sgr_dingest* g, int32_t partition, int64_t* decoded_next, int64_t* folded_next);
/* Forget everything (dictionary, partition positions, statistics): the next poll starts a rebuild from offset 0 with dense
 * indices from 0. The engine's table is the caller's to reset (sgr_set_initial_states(e, NULL, 0)). */
int32_t sgr_dingest_reset(sgr_dingest* g);
/* host-clock milliseconds of the last sgr_dingest_fold: [0] wait for the copies and for every group's chain (CRC, lz4 decode +
 * record walk, record parse + id interning — launched by the submits behind the copies), [1] a repeat from an exact arena
 * layout when the 3x estimate was too small (normally 0), [2] unused, [3] launch of the new ids' gather and download,
 * [4] table growth + fold, with the ids handed to the key table by a helper thread meanwhile, [5] the whole call.
 * (SGR_DINGEST_V1=1, the first generation: [0] copies + CRC / size pass, [1] decode + walk, [2] parse + intern.) */
int32_t sgr_dingest_last_timing(sgr_dingest* g, float* ms8);
int32_t sgr_dingest_get_stats(sgr_dingest* g, sgr_ingest_stats* out);

/* building blocks, exported for the known-answer tests */
uint32_t sgr_crc32c(const void* data, uint64_t nbytes);            /* RFC 3720 CRC-32C (SSE4.2 when present) */
uint32_t sgr_crc32c_portable(const void* data, uint64_t nbytes);   /* table-driven twin */
uint32_t sgr_xxh32(const void* data, uint64_t nbytes, uint32_t seed);
int32_t sgr_lz4_frame_decode(const void* src, uint64_t nbytes, void* out, uint64_t cap, uint64_t* out_len);

/* ------------------------------------------------------------------ partitioner
 * KafkaPartitionProvider.partitionForKey = abs(MurmurHash3.stringHash(s) % n)
 * (COMMON/kafka/KafkaPartitioner.scala:7-9) over key.takeWhile(_ != ':')
 * (PartitionStringUpToColon, :38-42). Host-side, UTF-16 code units. */
int32_t sgr_string_hash_utf16(const uint16_t* units, uint32_t n);
int32_t sgr_partition_for_key_utf8(const uint8_t* key, uint32_t klen, uint32_t num_partitions,
                                   int32_t up_to_colon, int32_t* partition);
int32_t sgr_partitions_for_keys(const uint8_t* keys, const uint32_t* key_offsets, uint64_t n, uint32_t num_partitions,
                                int32_t up_to_colon, uint32_t* partition_of);

#ifdef __cplusplus
}
#endif
#endif /* SGR_H */
