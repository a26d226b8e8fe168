/*
 * b200promql.h — C ABI of libb200promql.so: a B200 (sm_100a) evaluator for GreptimeDB's
 * PromQL range-query hot path.  Plain pointers and sizes only (no torch / Arrow C++ types), so
 * the reference's Rust host can bind it with `extern "C"` / cxx (see INTEGRATION.md).
 *
 * What each entry point replaces in the reference (paths relative to the greptimedb tree):
 *
 *   b2p_series_offsets_dev     SeriesDivideStream::poll_next + find_first_diff_row
 *                              src/promql/src/extension_plan/series_divide.rs:540-620, 622-670
 *   b2p_range_eval[_dev]       SeriesNormalizeStream::normalize            normalize.rs:388-431
 *                            + RangeManipulateStream::calculate_range/manipulate
 *                                                                          range_manipulate.rs:636-772
 *                            + Projection(prom_* ScalarUDF):  ExtrapolatedRate::calc
 *                              functions/extrapolate_rate.rs:133-288, IDelta::calc idelta.rs:113-153,
 *                              #[range_fn] loop common/macro/src/range_fn.rs:189-229 over
 *                              aggr_over_time.rs:35-179, resets.rs:33-48, changes.rs:33-48,
 *                              deriv.rs:32-40, predict_linear.rs:163-199, quantile.rs:201-225,
 *                              double_exponential_smoothing.rs:226-258
 *                            + Filter(value IS NOT NULL)  src/query/src/promql/planner.rs:1063
 *                              (expressed as the validity bitmap)
 *   b2p_range_udf[_dev]        one prom_* ScalarUDF call over a RangeArray (packed i64 keys
 *                              offset | len<<32, src/promql/src/range_array.rs:247-254) — the narrow
 *                              boundary: Fn(&[ColumnarValue]) -> ColumnarValue, extrapolate_rate.rs:90-96
 *   b2p_instant_select[_dev]   InstantManipulateStream::manipulate         instant_manipulate.rs:473-585
 *   b2p_group_aggregate[_dev]  DataFusion AggregateExec(Partial+Final) planned by
 *                              prom_aggr_expr_to_plan src/query/src/promql/planner.rs:334-452
 *                              (sum/avg/count/min/max/stddev/stdvar by labels + eval ts)
 *   b2p_histogram_quantile[_dev] HistogramFoldStream::fold_buf + evaluate_row
 *                              histogram_fold.rs:754-820, 1046-1118
 *   b2p_column_reduce_dev      avg_over_time over a wide table (config 5): per-column sum,count
 *
 * Data layout (HBM, struct-of-arrays, all row-sorted by (series id, timestamp) exactly like
 * the reference's required_input_ordering, series_divide.rs:410-440):
 *   ts[n_rows]   int64  ms since epoch (Millisecond = i64, extension_plan.rs:42)
 *   val[n_rows]  f64
 *   sid[n_rows]  uint32 dense series id 0..n_series-1, non-decreasing (host-side renumbering of
 *                __tsid: UInt64 / tag tuples, SURVEY.md appendix C-9)
 *   offsets[n_series+1] uint64 row offset of each series (product of b2p_series_offsets_dev)
 * Result layout: dense grid.  T = b2p_num_steps(start,end,interval) global eval steps
 *   t_k = start + k*interval; out[s*T + k] f64, valid bit k of series s in
 *   valid_words[s*Tw + (k>>5)] bit (k&31), Tw = (T+31)/32.  valid=0 <=> the reference emits no
 *   row for (series, t_k) (trimmed step, empty window, null result, NaN-stale); out is 0.0 there.
 *
 * Conventions: every function returns 0 (B2P_OK) or a negative B2P_E_*; b2p_last_error() gives a
 * thread-local message.  *_dev functions take DEVICE pointers, enqueue on the context's stream and
 * return without synchronising; call b2p_sync() before reading results — it also completes the
 * rare slow-path fix-ups.  Host-pointer functions copy H2D, run, copy D2H and synchronise.
 * A b2p_ctx is bound to one device and one stream; use one context per calling thread/partition
 * (DataFusion calls execute(partition) concurrently — range_manipulate.rs:546-579).
 * All column pointers must be 16-byte aligned.
 */
#ifndef B200PROMQL_H
#define B200PROMQL_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B2P_API __attribute__((visibility("default")))
#else
#define B2P_API
#endif

#define B2P_OK 0
#define B2P_E_INVALID (-1)  /* bad argument */
#define B2P_E_CUDA (-2)     /* CUDA runtime error */
#define B2P_E_UNSORTED (-3) /* sid column not non-decreasing / id >= n_series */
#define B2P_E_NOMEM (-4)
#define B2P_E_TOO_LARGE (-5) /* n_series * T exceeds what the dense grid supports */

/* Range functions (UDF names in the reference: prom_rate, prom_increase, ...). */
enum b2p_fn {
  B2P_FN_RATE = 0,             /* ExtrapolatedRate<true,true>   */
  B2P_FN_INCREASE = 1,         /* ExtrapolatedRate<true,false>  */
  B2P_FN_DELTA = 2,            /* ExtrapolatedRate<false,false> */
  B2P_FN_IRATE = 3,            /* IDelta<true>  */
  B2P_FN_IDELTA = 4,           /* IDelta<false> */
  B2P_FN_RESETS = 5,
  B2P_FN_CHANGES = 6,
  B2P_FN_COUNT_OVER_TIME = 7,
  B2P_FN_SUM_OVER_TIME = 8,
  B2P_FN_AVG_OVER_TIME = 9,
  B2P_FN_MIN_OVER_TIME = 10,
  B2P_FN_MAX_OVER_TIME = 11,
  B2P_FN_LAST_OVER_TIME = 12,
  B2P_FN_PRESENT_OVER_TIME = 13,
  B2P_FN_ABSENT_OVER_TIME = 14,
  B2P_FN_STDVAR_OVER_TIME = 15,
  B2P_FN_STDDEV_OVER_TIME = 16,
  B2P_FN_DERIV = 17,
  B2P_FN_PREDICT_LINEAR = 18,    /* param0 = t (seconds, i64 in the reference) */
  B2P_FN_QUANTILE_OVER_TIME = 19,/* param0 = phi */
  B2P_FN_HOLT_WINTERS = 20,      /* param0 = sf, param1 = tf */
  B2P_FN__COUNT = 21
};

/* Aggregators of the by-label aggregate (create_aggregate_exprs, planner.rs:2808-2897). */
enum b2p_agg { B2P_AGG_SUM = 0, B2P_AGG_AVG = 1, B2P_AGG_COUNT = 2, B2P_AGG_MIN = 3, B2P_AGG_MAX = 4,
               B2P_AGG_STDDEV = 5, B2P_AGG_STDVAR = 6 };

/* Parameters of the fused sub-plan.  Field-for-field the arguments of
 * RangeManipulate::new(start,end,interval,range,..) (range_manipulate.rs:86-110),
 * SeriesNormalize::new(offset,..,need_filter_out_nan,..) (normalize.rs:66-83) and the UDF scalars. */
typedef struct b2p_range_params {
  int32_t fn_id;      /* enum b2p_fn */
  int32_t filter_nan; /* need_filter_out_nan: 1 for every range selector (planner.rs:1383) */
  int64_t start;      /* ms */
  int64_t end;        /* ms, inclusive */
  int64_t interval;   /* ms, > 0 */
  int64_t range;      /* ms; also prom_rate's range_length argument (planner.rs:2438-2474) */
  int64_t offset;     /* ms, added to every timestamp */
  double param0;
  double param1;
} b2p_range_params;

typedef struct b2p_ctx b2p_ctx;

/* ---- context ------------------------------------------------------------------------- */
B2P_API b2p_ctx* b2p_create(int device);            /* NULL on failure (see b2p_last_error) */
B2P_API void b2p_destroy(b2p_ctx* ctx);
B2P_API const char* b2p_last_error(void);
B2P_API const char* b2p_version(void);
/* Enqueue on an existing cudaStream_t (e.g. the caller's current stream); NULL is the legacy default
 * stream.  b2p_use_own_stream() goes back to the context's private non-blocking stream. */
B2P_API int b2p_set_stream(b2p_ctx* ctx, void* cuda_stream);
B2P_API int b2p_use_own_stream(b2p_ctx* ctx);
/* Wait for the stream, finish slow-path fix-ups, surface deferred errors (B2P_E_UNSORTED, ...). */
B2P_API int b2p_sync(b2p_ctx* ctx);
B2P_API int64_t b2p_num_steps(int64_t start, int64_t end, int64_t interval);
/* Series the last range/instant call routed to the exact slow path (diagnostic; after b2p_sync). */
B2P_API int64_t b2p_last_slow_series(b2p_ctx* ctx);
/* bytes the last b2p_range_eval (host-pointer call) copied host -> device: fewer than 20 B/row when chunks of equally
 * spaced series went over as (offsets, first timestamp, cadence) descriptors instead of their timestamp / id columns */
B2P_API int64_t b2p_last_h2d_bytes(b2p_ctx* ctx);
/* Series the thread-per-series tier handed to the warp-per-series kernel in the last call (diagnostic). */
B2P_API int64_t b2p_last_warp_tier_series(b2p_ctx* ctx);
/* CUDA-event time (ms) of the kernels of the last *_dev / host call, by stage index:
 * 0 = series_offsets, 1 = range/instant fast kernel, 2 = slow-path kernel, 3 = aggregate /
 * histogram / reduce kernel.  Valid after b2p_sync(). */
B2P_API double b2p_last_kernel_ms(b2p_ctx* ctx, int stage);
/* Kernels launched by this context since creation (the bench's gpu_launches claim). */
B2P_API int64_t b2p_launch_count(b2p_ctx* ctx);

/* ---- device-pointer API (asynchronous) --------------------------------------------------- */
B2P_API int b2p_series_offsets_dev(b2p_ctx* ctx, const uint32_t* sid, uint64_t n_rows, uint32_t n_series,
                           uint64_t* offsets /* [n_series+1] */);
B2P_API int b2p_range_eval_dev(b2p_ctx* ctx, const b2p_range_params* p, const int64_t* ts, const double* val,
                       const uint64_t* offsets, uint64_t n_rows, uint32_t n_series,
                       double* out /* [n_series*T] */, uint32_t* valid_words /* [n_series*Tw] */);
B2P_API int b2p_range_udf_dev(b2p_ctx* ctx, int32_t fn_id, const int64_t* ts, const double* val, uint64_t n_rows,
                      const int64_t* packed_ranges /* [n_win] offset | len<<32 */,
                      const int64_t* eval_ts /* [n_win] or NULL */, uint64_t n_win, int64_t range_length,
                      double param0, double param1, double* out /* [n_win] */, uint8_t* valid /* [n_win] */);
B2P_API int b2p_instant_select_dev(b2p_ctx* ctx, int64_t start, int64_t end, int64_t interval, int64_t lookback,
                           int64_t offset, const int64_t* ts, const double* val, const uint64_t* offsets,
                           uint64_t n_rows, uint32_t n_series, double* out, uint32_t* valid_words);
/* gid[s] in [0,n_groups) (or >= n_groups to drop the series).  members_* is scratch-free: the
 * library builds the group->series CSR itself.  out_val/out_cnt are [n_groups*T]; cnt==0 <=> the
 * group has no row at that step.  Partial results of several shards/GPUs combine by adding
 * out_val (SUM/COUNT) and out_cnt — see b2p_group_finalize_dev. */
B2P_API int b2p_group_aggregate_dev(b2p_ctx* ctx, int32_t agg, const double* vals, const uint32_t* valid_words,
                            const uint32_t* gid, uint32_t n_series, uint32_t n_groups, uint64_t T,
                            double* out_val, uint32_t* out_cnt);
/* group -> member-series index of one gid[] assignment (the by-labels of a query do not change between
 * its batches): built once (radix sort + read-back of the largest group size; synchronises), reused by
 * b2p_group_aggregate_indexed_dev / b2p_range_group_sum_indexed_dev.  Replaces the hash table of string
 * keys DataFusion's AggregateExec builds per input row (planner.rs:334-452, SURVEY.md 8 a10). */
typedef struct b2p_group_index b2p_group_index;
B2P_API int b2p_group_index_create_dev(b2p_ctx* ctx, const uint32_t* gid /* device, [n_series] */, uint32_t n_series,
                               uint32_t n_groups, b2p_group_index** out_index);
B2P_API void b2p_group_index_destroy(b2p_ctx* ctx, b2p_group_index* index);
B2P_API int b2p_group_aggregate_indexed_dev(b2p_ctx* ctx, int32_t agg, const double* vals, const uint32_t* valid_words,
                                    const b2p_group_index* index, uint64_t T, double* out_val, uint32_t* out_cnt);
/* sum by (..)(fn(..)): range function + by-label partial SUM / COUNT of groups [g_lo, g_hi), ADDED into
 * out_sum / out_cnt [n_groups*T] (zero them first; shards, chunks and group ranges chain by accumulation).
 * rate / increase / delta with the first tier's query shape (32-bit time domain, range >= interval, start >= 0)
 * and reasonably balanced groups run FUSED: series are walked group by group, a group's rows of out_sum / out_cnt
 * belong to one warp and are updated in member order — no [n_series*T] intermediate, no atomics on the common
 * path, asynchronous (b2p_range_group_sum_fused() tells).  At most one fused call is outstanding per context: the
 * next range call synchronises first.  Everything else takes two passes through context scratch of
 * n_series*T*8 + n_series*Tw*4 bytes, synchronises in between, and needs the whole group range [0, n_groups). */
B2P_API int b2p_range_group_sum_indexed_dev(b2p_ctx* ctx, const b2p_range_params* p, const int64_t* ts, const double* val,
                                    const uint64_t* offsets, uint64_t n_rows, uint32_t n_series,
                                    const b2p_group_index* index, uint32_t g_lo, uint32_t g_hi, double* out_sum,
                                    uint32_t* out_cnt);
B2P_API int b2p_range_group_sum_fused(b2p_ctx* ctx, const b2p_range_params* p, const b2p_group_index* index); /* 1/0 */
/* Same with a one-off index built from gid (device, [n_series]); synchronous. */
B2P_API int b2p_range_group_sum_dev(b2p_ctx* ctx, const b2p_range_params* p, const int64_t* ts, const double* val,
                            const uint64_t* offsets, uint64_t n_rows, uint32_t n_series, const uint32_t* gid,
                            uint32_t n_groups, double* out_sum, uint32_t* out_cnt);
/* Partial state of one rank / shard for a later cross-rank merge: SUM / AVG -> (sum, cnt); COUNT -> cnt;
 * MIN / MAX -> (extreme, cnt); STDDEV / STDVAR -> (cnt, mean in out_mean, M2 in out_val). */
B2P_API int b2p_group_aggregate_partial_dev(b2p_ctx* ctx, int32_t agg, const double* vals, const uint32_t* valid_words,
                                    const uint32_t* gid, uint32_t n_series, uint32_t n_groups, uint64_t T,
                                    double* out_val, uint32_t* out_cnt, double* out_mean /* stddev / stdvar, else NULL */);
/* After the cross-GPU merge: AVG = sum/cnt in place; COUNT = (double)cnt; STDVAR = M2/cnt; STDDEV = sqrt(M2/cnt). */
B2P_API int b2p_group_finalize_dev(b2p_ctx* ctx, int32_t agg, double* val, const uint32_t* cnt, uint64_t n);

/* ---- multi-GPU (one process / context per GPU): NCCL communicator owned by the context ----------------
 * Series are hash-sharded over the ranks (SURVEY.md 8e; the reference hash-partitions on the series key,
 * series_divide.rs:396-408) and the by-label partials merge with one all-reduce, the analogue of the reference's
 * __sum_state (datanode) / __sum_merge (frontend) split, src/query/src/dist_plan/commutativity.rs:85-113, 158-191.
 * libnccl.so.2 is bound with dlopen at the first call (no link dependency; B2P_NCCL_LIB overrides the name).
 * Rank 0 calls b2p_comm_unique_id and ships the B2P_COMM_ID_BYTES to the other ranks by any means (the reference
 * would use its own RPC); every rank then calls b2p_comm_init (collective). */
#define B2P_COMM_ID_BYTES 128
B2P_API int b2p_comm_unique_id(void* out_id, size_t bytes);
B2P_API int b2p_comm_init(b2p_ctx* ctx, const void* id, size_t bytes, int n_ranks, int rank);
B2P_API int b2p_comm_destroy(b2p_ctx* ctx);
/* In-place merge of every rank's partials [n] on the context's stream (asynchronous): SUM / AVG / COUNT add val and
 * cnt; MIN / MAX reduce val in the f64::total_cmp order (int64 keys; groups absent on a rank are neutral) and add cnt; STDDEV / STDVAR merge
 * the (cnt, mean, M2 = val) states.  A context without communicator and n_ranks == 1 returns at once. */
B2P_API int b2p_allreduce_partials_dev(b2p_ctx* ctx, int32_t agg, double* val, uint32_t* cnt, double* mean, uint64_t n);
/* Wide avg_over_time (config 5): per-column (sum, count) of every rank added in place. */
B2P_API int b2p_allreduce_columns_dev(b2p_ctx* ctx, double* sum, uint64_t* cnt, uint32_t n_cols);
/* sum by (..)(fn(..)) over ALL ranks: this rank's fused partials, computed in n_tiles group ranges; each range's rows
 * of out_sum / out_cnt are all-reduced on a high-priority communication stream as soon as they are complete, while
 * the next range computes (kernel time of the last tile's all-reduce: b2p_last_kernel_ms(ctx, 4)).  On return
 * (stream order) out_sum / out_cnt hold the merged partials on every rank. */
B2P_API int b2p_range_group_sum_allreduce_dev(b2p_ctx* ctx, const b2p_range_params* p, const int64_t* ts,
                                      const double* val, const uint64_t* offsets, uint64_t n_rows, uint32_t n_series,
                                      const b2p_group_index* index, int32_t n_tiles, double* out_sum, uint32_t* out_cnt);
/* rates is the dense matrix of n_hist*n_buckets series (bucket b of histogram h = series
 * h*n_buckets+b, le ascending, last = +Inf).  out [n_hist*T], out_valid_words [n_hist*Tw]. */
B2P_API int b2p_histogram_quantile_dev(b2p_ctx* ctx, double phi, const double* le, uint32_t n_buckets,
                               const double* rates, const uint32_t* valid_words, uint32_t n_hist, uint64_t T,
                               double* out, uint32_t* out_valid_words);
/* HistogramFold over an explicit index (device pointers): histogram h owns buckets hist_off[h] .. hist_off[h+1] of
 * bucket_series / bucket_le, in ascending le order (NaN bounds last); layouts may differ between histograms.  Per
 * (histogram, step) the buckets that have a sample at that step are folded like the reference's safe mode
 * (histogram_fold.rs:834-846, 930-981): none -> no row; fewer than two or no +Inf bound last -> NaN; else
 * evaluate_row (:1046-1118).  b2p_histogram_quantile_dev is the uniform-layout front end of the same kernel. */
B2P_API int b2p_histogram_fold_dev(b2p_ctx* ctx, double phi, const uint32_t* hist_off, const uint32_t* bucket_series,
                           const double* bucket_le, uint32_t n_hist, const double* rates, const uint32_t* valid_words,
                           uint64_t T, double* out, uint32_t* out_valid_words);
/* cols: n_cols column pointers (device array of device pointers), each n_rows f64; NaN rows are
 * skipped (SeriesNormalize filter).  out_sum[n_cols], out_cnt[n_cols] accumulate. */
B2P_API int b2p_column_reduce_dev(b2p_ctx* ctx, const double* const* cols, uint32_t n_cols, uint64_t n_rows,
                          double* out_sum, uint64_t* out_cnt);

/* ---- host-side helper (no device work) -------------------------------------------------------- */
/* SeriesDivide (series_divide.rs:540-670) plus a cadence scan of one sorted batch on the HOST: series boundaries from
 * the id column `sid` (ids sid_base .. sid_base + n_series - 1, non-decreasing), or copied from `offsets_in`
 * (n_series + 1) when sid is NULL, into offsets_out (n_series + 1); and per series t0 = its first timestamp and
 * cadence = ts[1] - ts[0] (0 for series of fewer than two rows).  *all_regular = 1 iff ts[i] == t0 + i * cadence holds
 * for every row of every series — then the timestamp column is fully described by (offsets, t0, cadence), which is what
 * b2p_range_eval sends over PCIe instead of it (8 B/row less; the device rebuilds the column).  Any of t0 / cadence /
 * all_regular may be NULL.  B2P_E_UNSORTED when the ids are not non-decreasing or out of range. */
B2P_API int b2p_host_scan_series(const int64_t* ts, const uint32_t* sid, const uint64_t* offsets_in, uint64_t n_rows,
                         uint32_t n_series, uint32_t sid_base, uint64_t* offsets_out, int64_t* t0, int64_t* cadence,
                         int32_t* all_regular);

/* ---- host-pointer API (synchronous; H2D + kernels + D2H inside) ----------------------------- */
/* sid may be NULL when offsets_host (n_series+1) is given instead. out_ts (may be NULL) receives
 * the T eval timestamps. Pinned host buffers are copied directly; pageable ones are staged. */
B2P_API int b2p_range_eval(b2p_ctx* ctx, const b2p_range_params* p, const int64_t* ts, const double* val,
                   const uint32_t* sid, const uint64_t* offsets_host, uint64_t n_rows, uint32_t n_series,
                   double* out, uint32_t* valid_words, int64_t* out_ts);
B2P_API int b2p_range_udf(b2p_ctx* ctx, int32_t fn_id, const int64_t* ts, const double* val, uint64_t n_rows,
                  const int64_t* packed_ranges, const int64_t* eval_ts, uint64_t n_win, int64_t range_length,
                  double param0, double param1, double* out, uint8_t* valid);
B2P_API int b2p_instant_select(b2p_ctx* ctx, int64_t start, int64_t end, int64_t interval, int64_t lookback,
                       int64_t offset, const int64_t* ts, const double* val, const uint32_t* sid,
                       const uint64_t* offsets_host, uint64_t n_rows, uint32_t n_series, double* out,
                       uint32_t* valid_words);
B2P_API int b2p_group_aggregate(b2p_ctx* ctx, int32_t agg, const double* vals, const uint32_t* valid_words,
                        const uint32_t* gid, uint32_t n_series, uint32_t n_groups, uint64_t T, double* out_val,
                        uint32_t* out_cnt);
B2P_API int b2p_histogram_quantile(b2p_ctx* ctx, double phi, const double* le, uint32_t n_buckets, const double* rates,
                           const uint32_t* valid_words, uint32_t n_hist, uint64_t T, double* out,
                           uint32_t* out_valid_words);
/* histogram_quantile(phi, fn(bucket series)) in one call: samples in (host), rows [n_hist*T] out (host); the dense
 * per-series matrix stays on the device between the range function and the fold.  Index arrays are host pointers. */
B2P_API int b2p_range_histogram_fold(b2p_ctx* ctx, const b2p_range_params* p, const int64_t* ts, const double* val,
                             const uint32_t* sid, const uint64_t* offsets_host, uint64_t n_rows, uint32_t n_series,
                             double phi, const uint32_t* hist_off, const uint32_t* bucket_series, const double* bucket_le,
                             uint32_t n_hist, double* out, uint32_t* out_valid_words);

/* ---- plan-level API over the Arrow C Data Interface ------------------------------------------------
 * GpuPromRangeExec: the whole sub-tree SeriesDivide -> SeriesNormalize -> RangeManipulate ->
 * Projection(prom_fn) -> Filter(IS NOT NULL) [-> Aggregate(by-labels, ts).sort()] as one node, fed
 * with the RecordBatches the scan produces (arrow-rs `arrow::ffi::to_ffi`, pyarrow `_export_to_c`).
 * Constructor arguments carry the reference's names and meaning (see greptimedb_b200/csrc/b2p_plan.hpp:
 * SeriesDivide::new series_divide.rs:83-110, SeriesNormalize::new normalize.rs:66-83,
 * RangeManipulate::new range_manipulate.rs:86-110, UDF names planner.rs:2183-2221).
 * Input batches must be sorted by (tag columns, time index) — SeriesDivideExec's own requirement.
 * `function` is the UDF name ("prom_rate", ...); p->fn_id is ignored.  tag columns: Utf8, or a single
 * UInt64 id column.  aggregate: NULL/"" or "sum|avg|count|min|max|stddev|stdvar" with by_columns ⊆ tags.
 * b2p_plan_push_batch MOVES the batch (its release callbacks are taken over). b2p_plan_execute
 * fills caller-provided ArrowArray/ArrowSchema structs; the caller releases them. */
#ifndef ARROW_C_DATA_INTERFACE
#define ARROW_C_DATA_INTERFACE
struct ArrowSchema {
  const char* format;
  const char* name;
  const char* metadata;
  int64_t flags;
  int64_t n_children;
  struct ArrowSchema** children;
  struct ArrowSchema* dictionary;
  void (*release)(struct ArrowSchema*);
  void* private_data;
};
struct ArrowArray {
  int64_t length;
  int64_t null_count;
  int64_t offset;
  int64_t n_buffers;
  int64_t n_children;
  const void** buffers;
  struct ArrowArray** children;
  struct ArrowArray* dictionary;
  void (*release)(struct ArrowArray*);
  void* private_data;
};
#endif
typedef struct b2p_plan b2p_plan;
B2P_API b2p_plan* b2p_plan_range_create(b2p_ctx* ctx, const char* function, const b2p_range_params* p,
                                        const char* time_index, const char* field_column,
                                        const char* const* tag_columns, int32_t n_tags, const char* aggregate,
                                        const char* const* by_columns, int32_t n_by);
/* Turn the node into the instant-vector form: InstantManipulate(start, end, lookback_delta, interval, ...)
 * (instant_manipulate.rs:189-208) instead of RangeManipulate + prom_fn; `function` / range are then ignored. */
B2P_API int b2p_plan_set_instant(b2p_plan* plan, int64_t lookback_delta);
/* Add HistogramFold(le_column, field, time_index, quantile) (histogram_fold.rs:104-130) on top of the per-series
 * result: series that agree on every tag except `le` form one histogram. */
B2P_API int b2p_plan_set_histogram_quantile(b2p_plan* plan, const char* le_column, double quantile);
B2P_API int b2p_plan_push_batch(b2p_plan* plan, struct ArrowArray* batch, struct ArrowSchema* schema);
B2P_API int b2p_plan_execute(b2p_plan* plan, struct ArrowArray* out, struct ArrowSchema* out_schema);
B2P_API int64_t b2p_plan_num_series(b2p_plan* plan);
B2P_API void b2p_plan_destroy(b2p_plan* plan);
B2P_API const char* b2p_plan_last_error(void);

/* ---- bench/test utility: synthetic workload generated on the device (BASELINE.md §4) ------- */
B2P_API int b2p_synth_fill_dev(b2p_ctx* ctx, uint64_t series_begin, uint64_t n_series, uint32_t n_samples, int64_t t0,
                       int64_t scrape_ms, uint32_t jitter_ms, int32_t with_resets, uint64_t seed, int64_t* ts,
                       double* val, uint32_t* sid);

#ifdef __cplusplus
}
#endif
#endif
