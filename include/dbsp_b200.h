/*
 * dbsp_b200.h — C ABI of the B200-native Z-set delta hot path.
 *
 * This is the drop-in boundary for the path BASELINE.json's north_star names:
 * the reference's `Batch` / `Batcher` / `Builder` / `Merger` / `Trace` trait
 * family (crates/dbsp/src/trace/mod.rs:86-396) and the `eval` bodies of the
 * relational operators that consume it.  A Rust `dbsp-b200-sys` crate binds
 * exactly these symbols (see INTEGRATION.md); all arguments are plain
 * pointers, sizes and POD structs — no torch / C++ types cross the boundary.
 *
 * Conventions (mirroring SURVEY.md §8b):
 *   - every call returns int32 status, 0 = DBSP_OK; no exception crosses;
 *   - a `dbsp_ctx` is bound to one GPU + one CUDA stream and must be used
 *     from one host thread at a time (the reference confines a circuit
 *     replica to its worker thread, circuit_builder.rs:1439-1450);
 *   - batches are immutable, reference counted values (the reference's
 *     batches are immutable values too, zset_batch.rs:27);
 *   - every *_free is a no-op on NULL.
 *
 * Data model.  A row is `n_key_lanes + n_val_lanes` 64-bit lanes plus one
 * int64 weight.  Lanes are u64 or i64 and compare lexicographically, which
 * is Rust's derived `Ord` on tuples of integers.  `n_val_lanes == 0` is an
 * `OrdZSet<K,R>` (zset_batch.rs:28-31); otherwise an
 * `OrdIndexedZSet<K,V,R>` (indexed_zset_batch.rs:27-41).  On the device a
 * batch is column-major: one contiguous u64 array per lane plus the weight
 * array, rows sorted by (key lanes, val lanes), consolidated (no duplicate
 * rows, no zero weights).  `dbsp_batch_download_csr` returns the
 * reference's canonical `keys / offs / vals / diffs` vectors.
 */
#ifndef DBSP_B200_H
#define DBSP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DBSP_MAX_LANES 8
#define DBSP_MAX_PREDS 4

enum dbsp_status {
  DBSP_OK = 0,
  DBSP_ERR_INVALID = 1,   /* bad argument / schema mismatch                */
  DBSP_ERR_CUDA = 2,      /* CUDA runtime error (see dbsp_last_error)      */
  DBSP_ERR_NO_DEVICE = 3, /* no usable CUDA device: there is NO CPU fallback */
  DBSP_ERR_UNSUPPORTED = 4
};

enum dbsp_lane_type { DBSP_U64 = 0, DBSP_I64 = 1 };

/* Row schema.  Replaces the `K: DBData, V: DBData` type parameters of
 * `Batch` (trace/mod.rs:49-76, 237-300) for the supported key/value set:
 * tuples of <= 8 integer lanes in total. */
typedef struct dbsp_schema {
  uint8_t n_key_lanes;
  uint8_t n_val_lanes;
  uint8_t lane_types[DBSP_MAX_LANES]; /* key lanes first, then val lanes */
} dbsp_schema;

/* ---- declarative row expressions (replace the Rust closures passed to
 * join / flat_map_index / map_index, join.rs:187, filter_map.rs:143-152) -- */
enum dbsp_src_kind {
  DBSP_SRC_KEY = 0,   /* lane `idx` of the (join) key                       */
  DBSP_SRC_LVAL = 1,  /* lane `idx` of the left value (v1 of join_func);
                         for map_index / raw tables: value lane / column    */
  DBSP_SRC_RVAL = 2,  /* lane `idx` of the right value (v2 of join_func)    */
  DBSP_SRC_CONST = 3  /* the constant `cst`                                 */
};
enum dbsp_expr_op {
  DBSP_OP_COPY = 0, DBSP_OP_NEG = 1, DBSP_OP_ADD = 2, DBSP_OP_SUB = 3,
  DBSP_OP_MUL = 4, DBSP_OP_DIV = 5 /* signed, truncating (Rust isize `/`) */
};
enum dbsp_cmp_op {
  DBSP_CMP_EQ = 0, DBSP_CMP_NE = 1, DBSP_CMP_LT = 2, DBSP_CMP_LE = 3,
  DBSP_CMP_GT = 4, DBSP_CMP_GE = 5,
  DBSP_CMP_IN = 6 /* a < 64 && bit a of b is set: membership in a small code
                     set, e.g. STATES_OF_INTEREST.contains (nexmark q3.rs:44) */
};
typedef struct dbsp_src {
  uint8_t kind;
  uint8_t idx;
  uint8_t pad_[6];
  int64_t cst;
} dbsp_src;
typedef struct dbsp_expr {
  uint8_t op;
  uint8_t pad_[7];
  dbsp_src a, b;
} dbsp_expr;
typedef struct dbsp_pred {
  uint8_t cmp;
  uint8_t is_signed;
  uint8_t pad_[6];
  dbsp_src a, b;
} dbsp_pred;
/* Projection + filter: output row = (out[0..n_out_key+n_out_val)), kept iff
 * every predicate holds. */
typedef struct dbsp_proj {
  dbsp_schema out_schema;
  uint8_t n_pred;
  uint8_t pad_[5];
  dbsp_expr out[DBSP_MAX_LANES];
  dbsp_pred pred[DBSP_MAX_PREDS];
} dbsp_proj;

/* Aggregators (operator/aggregate/{max,min,fold}.rs, mod.rs:129-156). */
enum dbsp_agg_kind {
  DBSP_AGG_MAX = 0,        /* Max over the value tuple  (max.rs:36-55)       */
  DBSP_AGG_MIN = 1,        /* Min                       (min.rs:38-57)       */
  DBSP_AGG_FOLD_COUNT = 2, /* Fold: # values with non-zero weight            */
  DBSP_AGG_FOLD_SUM = 3,   /* Fold: sum of value lane 0 over such values     */
  DBSP_AGG_WCOUNT = 4,     /* WeightedCount over OrdZSet<K> (mod.rs:129-156) */
  DBSP_AGG_WCOUNT2 = 5     /* WeightedCount over the (sum,count) pair weight
                              of `average` (average.rs:26-29): delta is
                              OrdZSet<(K.., which)>, which in {0,1}          */
};
enum dbsp_weigh_mode {
  DBSP_WEIGH_LINEAR = 0, /* weigh(f): weight_k = sum f(k,v)*w (mod.rs:297-323) */
  DBSP_WEIGH_AVG = 1     /* f = Avg(value,1): rows (k,0)->sum v*w, (k,1)->sum w */
};

typedef struct dbsp_ctx dbsp_ctx;
typedef struct dbsp_batch dbsp_batch;
typedef struct dbsp_spine dbsp_spine;

/* ---- context -------------------------------------------------------- */
/* One context per GPU / circuit replica (runtime.rs:137-180: one worker =
 * one replica).  Fails with DBSP_ERR_NO_DEVICE when no CUDA device is
 * usable — there is no CPU path behind this ABI. */
int32_t dbsp_ctx_create(int32_t device, dbsp_ctx** out);
int32_t dbsp_ctx_destroy(dbsp_ctx* ctx);
int32_t dbsp_ctx_sync(dbsp_ctx* ctx);
const char* dbsp_last_error(void);
/* Counters: kernels launched by this library and bytes it copied H2D/D2H
 * since the last reset (bench.py's gpu_launches / e2e byte counts). */
int32_t dbsp_ctx_stats(dbsp_ctx* ctx, uint64_t* kernel_launches,
                       uint64_t* h2d_bytes, uint64_t* d2h_bytes, int32_t reset);
/* Optional per-kernel timing (CUDA events on the stream of the execution lane that runs the
 * library's own kernels).  enable == 1 starts a fresh collection, enable == 2
 * pauses it (what was collected stays readable, nothing more is recorded —
 * a sampling window inside a longer timed region), enable == 0 ends it.  _read
 * returns, for kernel class `kernel_id` (0,1,2,... until DBSP_ERR_INVALID),
 * its name, launch count, summed device time and algorithmic bytes (the
 * per-kernel byte formulas of DESIGN.md). */
int32_t dbsp_ctx_profile(dbsp_ctx* ctx, int32_t enable);
int32_t dbsp_ctx_profile_read(dbsp_ctx* ctx, int32_t kernel_id, char* name32,
                              uint64_t* launches, double* ms,
                              uint64_t* alg_bytes);
/* CUDA stream the context launches on (cudaStream_t as void*), so a host
 * can order its own work / CUDA events on it.  This is execution lane 0; the
 * work a grouped call runs on lane 1 is joined back into it before the call
 * returns. */
void* dbsp_ctx_stream(dbsp_ctx* ctx);

/* ---- batches -------------------------------------------------------- */
/* Batch::from_tuples (trace/mod.rs:259-263) = MergeBatcher + consolidate
 * (merge_batcher/mod.rs:65-80,155-197; consolidation/mod.rs:32-52) + Builder
 * (ordered/mod.rs:874-888): sort, sum equal rows, drop zero weights.
 * `cols[l]` points to n u64 per lane (key lanes then val lanes); `weights`
 * may be NULL (all +1).  `on_device` != 0: the pointers are device memory. */
int32_t dbsp_batch_from_tuples(dbsp_ctx* ctx, const dbsp_schema* schema,
                               const uint64_t* const* cols,
                               const int64_t* weights, uint64_t n,
                               int32_t on_device, dbsp_batch** out);
/* flat_map_index over a raw (unsorted, column-major) event table followed by
 * from_tuples (filter_map.rs:700-724): SRC_LVAL idx = column index. */
int32_t dbsp_batch_from_table(dbsp_ctx* ctx, const uint64_t* const* cols,
                              uint32_t n_cols, const int64_t* weights,
                              uint64_t n, int32_t on_device,
                              const dbsp_proj* proj, dbsp_batch** out);
/* Pipelined ingest of a raw event table: start copying the host columns of a
 * *future* step to the device on the context's copy stream (pinned host
 * memory makes it overlap with the kernels of the current step); the handle
 * is then consumed by dbsp_batch_from_upload.  `col_mask` bit l = column l is
 * needed (the others are not copied).  The host buffers must stay valid until
 * the upload is consumed or freed.  This is the double-buffered input queue of
 * the reference's source operators (crates/nexmark/src/lib.rs:105-231 feeds
 * batches ahead of the circuit) moved to the PCIe boundary. */
typedef struct dbsp_upload dbsp_upload;
int32_t dbsp_upload_begin(dbsp_ctx* ctx, const uint64_t* const* cols,
                          uint32_t n_cols, uint32_t col_mask,
                          const int64_t* weights, uint64_t n,
                          dbsp_upload** out);
int32_t dbsp_batch_from_upload(dbsp_ctx* ctx, dbsp_upload* up,
                               const dbsp_proj* proj, dbsp_batch** out);
int32_t dbsp_upload_free(dbsp_upload* up);
/* flat_map_index of k raw tables in one call.  Each job is either a table of
 * columns (`upload` NULL; cols / weights / n / n_cols / on_device as for
 * dbsp_batch_from_table) or an upload (the other fields are ignored).  outs[i]
 * is the batch dbsp_batch_from_table / dbsp_batch_from_upload would return for
 * jobs[i].  With k >= 2 the jobs are spread over the context's two execution
 * lanes (DESIGN.md §3) and run side by side; with k == 1 the job runs inline.
 * On failure no batch is returned. */
typedef struct dbsp_table_job {
  const uint64_t* const* cols;
  const int64_t* weights;
  uint64_t n;
  dbsp_upload* upload;
  const dbsp_proj* proj;
  uint32_t n_cols;
  int32_t on_device;
} dbsp_table_job;
int32_t dbsp_batches_from_tables(dbsp_ctx* ctx, uint32_t k,
                                 const dbsp_table_job* jobs, dbsp_batch** outs);
/* Columns of the table a projection reads (bit l = SRC_LVAL idx l). */
uint32_t dbsp_proj_table_mask(const dbsp_proj* proj);
int32_t dbsp_batch_empty(dbsp_ctx* ctx, const dbsp_schema* schema,
                         dbsp_batch** out);
/* Batch::merge / Merger::work run to completion (trace/mod.rs:371-396;
 * column_layer/builders.rs:98-169; ordered/mod.rs:344-396,806-834). */
int32_t dbsp_batch_merge(dbsp_ctx* ctx, const dbsp_batch* a,
                         const dbsp_batch* b, dbsp_batch** out);
/* Batcher (trace/mod.rs:316-335) = MergeBatcher (trace/ord/merge_batcher/mod.rs:22-81,
 * 155-260): push_batch consolidates the pushed tuples and queues them, merging
 * the two newest queue entries while the newer is at least half the older;
 * push_consolidated skips the consolidation (rows already sorted, unique, non-zero);
 * seal merges what is left into one batch and frees the batcher. */
typedef struct dbsp_batcher dbsp_batcher;
int32_t dbsp_batcher_new(dbsp_ctx* ctx, const dbsp_schema* schema,
                         dbsp_batcher** out);
int32_t dbsp_batcher_push(dbsp_ctx* ctx, dbsp_batcher* b,
                          const uint64_t* const* cols, const int64_t* weights,
                          uint64_t n, int32_t on_device);
int32_t dbsp_batcher_push_consolidated(dbsp_ctx* ctx, dbsp_batcher* b,
                                       const uint64_t* const* cols,
                                       const int64_t* weights, uint64_t n,
                                       int32_t on_device);
int32_t dbsp_batcher_tuples(const dbsp_batcher* b, uint64_t* n_tuples);
int32_t dbsp_batcher_seal(dbsp_ctx* ctx, dbsp_batcher* b, dbsp_batch** out);
int32_t dbsp_batcher_free(dbsp_batcher* b);
/* Merger::work with a lower value bound, run to completion
 * (trace/ord/indexed_zset_batch.rs:359-382 -> ordered/mod.rs:587-746
 * push_merge_truncate_values_fueled): values below `val_lower_bound`
 * (n_val_lanes u64; NULL = no bound) are dropped, keys left without values
 * vanish.  OrdZSet batches (n_val_lanes == 0) ignore the bound
 * (zset_batch.rs:307-318). */
int32_t dbsp_batch_merge_bounded(dbsp_ctx* ctx, const dbsp_batch* a,
                                 const dbsp_batch* b,
                                 const uint64_t* val_lower_bound,
                                 dbsp_batch** out);
/* The fuelled Merger (trace/mod.rs:371-396: new_merger / work / done).
 * work() spends at most *fuel units (here: input rows) and subtracts what it
 * used; *fuel > 0 after the call <=> the merge is complete (:388-395).
 * done() requires a complete merge, returns the batch and frees the merger. */
typedef struct dbsp_merger dbsp_merger;
int32_t dbsp_merger_new(dbsp_ctx* ctx, const dbsp_batch* a, const dbsp_batch* b,
                        const uint64_t* val_lower_bound, dbsp_merger** out);
int32_t dbsp_merger_work(dbsp_ctx* ctx, dbsp_merger* m, int64_t* fuel);
int32_t dbsp_merger_done(dbsp_ctx* ctx, dbsp_merger* m, dbsp_batch** out);
int32_t dbsp_merger_free(dbsp_merger* m);
/* BatchReader::truncate_keys_below (trace/mod.rs:227-233;
 * column_layer/mod.rs:316-319): zero-copy suffix view, key = n_key_lanes u64. */
int32_t dbsp_batch_truncate_keys_below(dbsp_ctx* ctx, const dbsp_batch* b,
                                       const uint64_t* key, dbsp_batch** out);
/* neg (column_layer/mod.rs:452-480). */
int32_t dbsp_batch_neg(dbsp_ctx* ctx, const dbsp_batch* a, dbsp_batch** out);
/* Same rows, different key/value split: `index()` (operator/index.rs:128-157)
 * and its inverse are free in the flat column-major layout. */
int32_t dbsp_batch_reindex(dbsp_ctx* ctx, const dbsp_batch* a,
                           uint32_t n_key_lanes, dbsp_batch** out);
/* BatchReader::len / key_count (trace/mod.rs:179-234). */
int32_t dbsp_batch_len(const dbsp_batch* b, uint64_t* n_tuples);
int32_t dbsp_batch_key_count(dbsp_ctx* ctx, const dbsp_batch* b,
                             uint64_t* n_keys);
int32_t dbsp_batch_schema(const dbsp_batch* b, dbsp_schema* out);
/* Canonical vectors of the reference's batch structs.  Any pointer may be
 * NULL (skipped).  keys[l]: n_keys u64 (n_tuples when n_val_lanes == 0);
 * offs: n_keys+1 (only when n_val_lanes > 0); vals[l], diffs: n_tuples. */
int32_t dbsp_batch_download_csr(dbsp_ctx* ctx, const dbsp_batch* b,
                                uint64_t* const* keys, uint64_t* offs,
                                uint64_t* const* vals, int64_t* diffs);
/* Asynchronous read of a batch's flat rows (the output handle of a circuit
 * drained while the next step runs — the reference's OutputHandle is read by
 * the client thread between steps, operator/output.rs:20-75).  _begin queues,
 * on the context's read stream (its own: PCIe is full duplex, uploads are not
 * delayed) and ordered after the work already queued on the compute stream, the copy of lane l (n_tuples u64) into cols[l] and of
 * the weights into diffs (NULL entries are skipped); the destinations should
 * be pinned host memory and must stay valid until _finish, which waits for
 * the copy and releases the handle (and its reference on the batch). */
typedef struct dbsp_download dbsp_download;
int32_t dbsp_batch_download_begin(dbsp_ctx* ctx, const dbsp_batch* b,
                                  uint64_t* const* cols, int64_t* diffs,
                                  dbsp_download** out);
int32_t dbsp_download_finish(dbsp_download* d);
/* Host synchronisation counters: how many times the host waited for a count
 * published by the device (mailbox read-backs) and for how long in total,
 * since the last reset. */
int32_t dbsp_ctx_sync_stats(dbsp_ctx* ctx, uint64_t* n_waits, double* wait_us,
                            int32_t reset);
/* Device pointers of the flat column-major rows (lane l, weights). */
int32_t dbsp_batch_device_columns(const dbsp_batch* b, const uint64_t** cols,
                                  const int64_t** weights);
/* Largest key (first key lane set) of the batch — `fast_forward_keys` +
 * `get_key` as used by watermark_monotonic (watermark.rs:38-45).
 * *valid = 0 when the batch is empty. */
int32_t dbsp_batch_last_key(dbsp_ctx* ctx, const dbsp_batch* b, uint64_t* key,
                            int32_t* valid);
int32_t dbsp_batch_clone(const dbsp_batch* b, dbsp_batch** out);
int32_t dbsp_batch_free(dbsp_batch* b);

/* ---- spine (trace) -------------------------------------------------- */
/* Spine (trace/spine_fueled.rs:107-119): LSM of immutable batches. */
int32_t dbsp_spine_new(dbsp_ctx* ctx, const dbsp_schema* schema,
                       dbsp_spine** out);
/* Trace::insert (spine_fueled.rs:605-634): the batch is shared, not copied. */
int32_t dbsp_spine_insert(dbsp_ctx* ctx, dbsp_spine* s, const dbsp_batch* b);
/* Trace::consolidate (spine_fueled.rs:583-600): merge everything. */
int32_t dbsp_spine_consolidate(dbsp_ctx* ctx, dbsp_spine* s, dbsp_batch** out);
/* truncate_keys_below (spine_fueled.rs:223-233); `key` = n_key_lanes u64. */
int32_t dbsp_spine_truncate_keys_below(dbsp_ctx* ctx, dbsp_spine* s,
                                       const uint64_t* key);
/* Trace::truncate_values_below (trace/mod.rs:150-169; spine_fueled.rs:644-656):
 * the bound only grows and is applied by later merges and by consolidate;
 * values below it are undefined until then (as in the reference). */
int32_t dbsp_spine_truncate_values_below(dbsp_ctx* ctx, dbsp_spine* s,
                                         const uint64_t* val);
/* Trace::exert (trace/mod.rs:104-113; spine_fueled.rs:627-634).  This spine
 * merges eagerly on insert, so no merge is ever in progress; effort buys extra
 * compaction instead: the two newest batches are merged while their combined
 * length fits *effort (decremented by the rows merged). */
int32_t dbsp_spine_exert(dbsp_ctx* ctx, dbsp_spine* s, int64_t* effort);
int32_t dbsp_spine_len(const dbsp_spine* s, uint64_t* n_tuples,
                       uint32_t* n_batches);
int32_t dbsp_spine_free(dbsp_spine* s);

/* Checkpoint / resume of a trace (SURVEY.md §8(f)4): the device-side replacement of the RocksDB-backed
 * PersistentTrace (crates/dbsp/src/trace/persistent/) for snapshots.  One little-endian file: magic "DBSPSPN1",
 * the schema, key / value bounds, effort, then every layer of the spine (spine_fueled.rs:1012-1027: Vacant /
 * Single / Double{InProgress, Complete}) with its batches as flat lanes + weights and, for a merge in progress,
 * the fuel still owed — so a loaded spine resumes the same merge schedule.  The format is shared with the oracle. */
int32_t dbsp_spine_save(dbsp_ctx* ctx, const dbsp_spine* s, const char* path);
int32_t dbsp_spine_load(dbsp_ctx* ctx, const char* path, dbsp_spine** out);

/* ---- operators ------------------------------------------------------ */
/* JoinTrace::eval (operator/join.rs:732-863), Time = (): delta joined with
 * every batch of the trace, weights multiplied, join_func = proj, result
 * consolidated.  `delta_is_left` != 0: delta rows feed SRC_LVAL and trace
 * rows SRC_RVAL; 0: swapped (the flipped closure of join.rs:279-284). */
int32_t dbsp_join_delta_trace(dbsp_ctx* ctx, const dbsp_batch* delta,
                              const dbsp_spine* trace, const dbsp_proj* proj,
                              int32_t delta_is_left, dbsp_batch** out);
/* One step of the incremental join operator (join.rs:180-292):
 *   insert(right_trace, d_right); o1 = d_left |x| right_trace;
 *   o2 = d_right |x| left_trace (flipped, = z^-1 of the left integral);
 *   insert(left_trace, d_left); out = o1 + o2.
 * The two halves run side by side on the context's two execution lanes; the
 * result and both traces equal those of that sequence of calls. */
int32_t dbsp_join_step(dbsp_ctx* ctx, const dbsp_batch* d_left,
                       const dbsp_batch* d_right, dbsp_spine* left_trace,
                       dbsp_spine* right_trace, const dbsp_proj* proj,
                       dbsp_batch** out);
/* Join::eval (join.rs:436-473): stateless batch x batch. */
int32_t dbsp_join_batches(dbsp_ctx* ctx, const dbsp_batch* left,
                          const dbsp_batch* right, const dbsp_proj* proj,
                          dbsp_batch** out);
/* SemiJoinStream::eval (operator/semijoin.rs:100-142). */
int32_t dbsp_semijoin(dbsp_ctx* ctx, const dbsp_batch* pairs,
                      const dbsp_batch* keys, dbsp_batch** out);
/* AggregateIncremental::eval (aggregate/mod.rs:600-684) fused with
 * Upsert::eval (operator/upsert.rs:161-208): for every key of `delta`,
 * aggregate the key's values in `in_trace` (which already contains delta),
 * compare with the key's current value in `out_trace`, emit -1/+1 rows.
 * The caller then inserts *out into out_trace (the TraceAppend of
 * upsert.rs:69-107). */
int32_t dbsp_aggregate_delta(dbsp_ctx* ctx, const dbsp_batch* delta,
                             const dbsp_spine* in_trace,
                             const dbsp_spine* out_trace, int32_t agg_kind,
                             dbsp_batch** out);
/* weigh (aggregate/mod.rs:297-323). `f` gives f(k,v) (SRC_KEY/SRC_LVAL). */
int32_t dbsp_weigh(dbsp_ctx* ctx, const dbsp_batch* b, const dbsp_expr* f,
                   int32_t mode, dbsp_batch** out);
/* DistinctIncrementalTotal::eval (operator/distinct.rs:196-254). */
int32_t dbsp_distinct_delta(dbsp_ctx* ctx, const dbsp_batch* delta,
                            const dbsp_spine* delayed_integral,
                            dbsp_batch** out);
/* IndexedZSet::distinct (algebra/zset/mod.rs:14-38). */
int32_t dbsp_stream_distinct(dbsp_ctx* ctx, const dbsp_batch* b,
                             dbsp_batch** out);
/* Window::eval (operator/time_series/window.rs:144-222).  Bounds are
 * n_key_lanes u64 each; has_prev == 0 on the first step. */
int32_t dbsp_window_delta(dbsp_ctx* ctx, const dbsp_spine* trace,
                          const dbsp_batch* delta, int32_t has_prev,
                          const uint64_t* start0, const uint64_t* end0,
                          const uint64_t* start1, const uint64_t* end1,
                          dbsp_batch** out);
/* Map/FlatMap/Index::eval + from_tuples (filter_map.rs:563-577,700-724). */
int32_t dbsp_map_index(dbsp_ctx* ctx, const dbsp_batch* b,
                       const dbsp_proj* proj, dbsp_batch** out);
/* shard_batch (operator/communication/shard.rs:165-199): split by
 * hash(key) % n_shards into n_shards ordered batches.  The exchange itself
 * (exchange.rs:128-200) is done by the host with its collective library on
 * dbsp_batch_device_columns(); the receiver merges (shard.rs:136-144). */
int32_t dbsp_shard_partition(dbsp_ctx* ctx, const dbsp_batch* b,
                             uint32_t n_shards, dbsp_batch** outs);
/* ---- communication between circuit replicas (one replica = one context = one GPU) ----------------
 * Replaces shard (operator/communication/shard.rs:106-162), Exchange (exchange.rs:128-200), gather
 * (gather.rs:41-103) and the watermark exchange (time_series/watermark.rs:53-70) — the three calls SURVEY.md
 * §8(b) lists as dbsp_shard / dbsp_gather / dbsp_allreduce_max_u64.  There is no collective library on the
 * data path: every context owns a device receive region; peers map it (CUDA IPC between processes, peer
 * access between the contexts of one process) and the partition kernel's stores land in it over NVLink.
 *
 * Bootstrap (replaces the ncclUniqueId of the survey's sketch): every rank calls dbsp_comm_create, which
 * returns a DBSP_COMM_BLOB_BYTES descriptor of its region; the HOST moves the `world` descriptors to every
 * rank by whatever channel it has (the reference's workers are threads of one process: a shared Vec; one
 * process per GPU: any all-gather) and hands the rank-ordered array to dbsp_comm_connect.
 * All replicas must issue the same sequence of exchange calls (they run the same circuit). */
#define DBSP_COMM_MAX_RANKS 32
#define DBSP_COMM_BLOB_BYTES 128
int32_t dbsp_comm_create(dbsp_ctx* ctx, int32_t rank, int32_t world,
                         uint64_t slot_bytes /* capacity of one (source,destination) segment per round; 0 = 512 MiB */,
                         uint8_t* blob_out /* DBSP_COMM_BLOB_BYTES */);
int32_t dbsp_comm_connect(dbsp_ctx* ctx, const uint8_t* blobs /* world * DBSP_COMM_BLOB_BYTES, rank order */);
int32_t dbsp_comm_destroy(dbsp_ctx* ctx);
/* rank / world of the context (0 / 1 without a comm) and payload bytes it has sent to other ranks */
int32_t dbsp_comm_info(dbsp_ctx* ctx, int32_t* rank, int32_t* world, uint64_t* bytes_sent);
/* Stream::shard (shard.rs:106-162): rows re-partitioned by hash(key) % world; returns this replica's shard,
 * consolidated (partition + NVLink scatter + receiver merge in one call; identity when world == 1). */
int32_t dbsp_shard(dbsp_ctx* ctx, const dbsp_batch* b, dbsp_batch** out);
/* shard() of both inputs of a binary operator (join.rs:265-266) in ONE exchange round. */
int32_t dbsp_shard2(dbsp_ctx* ctx, const dbsp_batch* a, const dbsp_batch* b,
                    dbsp_batch** out_a, dbsp_batch** out_b);
/* Stream::gather (gather.rs:41-103): everything to `root`, empty batches elsewhere. */
int32_t dbsp_gather(dbsp_ctx* ctx, const dbsp_batch* b, int32_t root, dbsp_batch** out);
/* max over the replicas of *x (watermark.rs:53-70); every replica gets the result. */
int32_t dbsp_allreduce_max_u64(dbsp_ctx* ctx, uint64_t* x);

/* Builder path (trace/mod.rs:338-368): adopt rows that are already sorted
 * and consolidated (e.g. a segment received from a peer). */
int32_t dbsp_batch_from_sorted(dbsp_ctx* ctx, const dbsp_schema* schema,
                               const uint64_t* const* cols,
                               const int64_t* weights, uint64_t n,
                               int32_t on_device, dbsp_batch** out);

#ifdef __cplusplus
}
#endif
#endif /* DBSP_B200_H */
