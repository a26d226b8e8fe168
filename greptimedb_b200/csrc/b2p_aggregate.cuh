// b2p_aggregate.cuh — kernels above the range functions:
//   K3 group_aggregate_kernel  by-label aggregate (DataFusion AggregateExec planned by
//                              prom_aggr_expr_to_plan, src/query/src/promql/planner.rs:334-452)
//   K5 histogram_fold_kernel   HistogramFold: fold_buf + safe mode + evaluate_row (histogram_fold.rs:754-1118)
//   K6 column_reduce_*         per-column sum/count of a wide f64 table (config 5)
#pragma once
#include <cstdint>

#include "b2p_kernels.cuh"

namespace b2p {

// ---------------------------------------------------------------------------------------------
// K3.  Members of group g are series members[goff[g] .. goff[g+1]) in ascending series order
// (stable sort of gid), so every accumulator sees its rows in the same order a single DataFusion
// partition would: plain f64 +=, nulls skipped, group absent (cnt 0) when it receives no row.
// One warp per (group, 32-step tile): each member contributes one coalesced 256-byte segment.
// HBM traffic: reads 8 B + 1 bit per (series, step), writes 12 B per (group, step).
// ---------------------------------------------------------------------------------------------
struct GroupArgs {
  int32_t agg;
  const double* vals;
  const uint32_t* valid;
  const uint32_t* goff;     // [n_groups+1]
  const uint32_t* members;  // [n_member_series]
  uint32_t n_groups;
  uint64_t T;
  uint32_t Tw;
  double* out_val;
  uint32_t* out_cnt;
  int32_t accumulate;  // 1: add into existing out_val/out_cnt (SUM/COUNT partial chaining)
  double* out_mean;    // stddev / stdvar only, may be NULL: when given, out_val receives the raw M2 and out_mean the
                       // mean — the (count, mean, M2) state another rank's partial can be merged with
};

// AGG is a compile-time constant so that the per-member fold is one or two instructions (sum / avg / count) instead
// of a switch inside the inner loop.
template <int AGG>
__global__ void __launch_bounds__(256) group_aggregate_kernel(const GroupArgs a) {
  const int lane = threadIdx.x & 31;
  const uint64_t tiles = (a.T + 31) / 32;
  const uint64_t total = (uint64_t)a.n_groups * tiles;
  const uint32_t tiles32 = (uint32_t)tiles;
  const bool small = total < 0xffffffffull;  // 32-bit task arithmetic (always, in practice)
  for (uint64_t w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total;
       w += ((uint64_t)gridDim.x * blockDim.x) >> 5) {
    uint32_t g;
    uint64_t tile;
    if (small) {
      g = (uint32_t)w / tiles32;
      tile = (uint32_t)w - g * tiles32;
    } else {
      g = (uint32_t)(w / tiles);
      tile = w - (uint64_t)g * tiles;
    }
    const uint64_t k = tile * 32 + lane;
    const bool in = k < a.T;
    const uint32_t m0 = a.goff[g], m1 = a.goff[g + 1];
    double acc = 0.0, mean = 0.0, m2 = 0.0;
    uint32_t cnt = 0;
    auto fold = [&](double x) {
      if constexpr (AGG == B2P_AGG_SUM || AGG == B2P_AGG_AVG) {
        acc += x;
      } else if constexpr (AGG == B2P_AGG_COUNT) {
      } else if constexpr (AGG == B2P_AGG_MIN) {  // f64::total_cmp order (arrow-rs / DataFusion min, max): +NaN is greatest
        if (cnt == 0 || total_key(x) < total_key(acc)) acc = x;
      } else if constexpr (AGG == B2P_AGG_MAX) {
        if (cnt == 0 || total_key(x) > total_key(acc)) acc = x;
      } else {  // Welford, population variance
        const double new_count = (double)cnt + 1.0;
        const double delta1 = x - mean;
        const double new_mean = delta1 / new_count + mean;
        const double delta2 = x - new_mean;
        m2 += delta1 * delta2;
        mean = new_mean;
      }
      ++cnt;
    };
    // Up to 32 members at a time: lane i fetches member i's series id and validity word (two dependent loads for
    // the whole batch instead of two per member), then the 256-byte value segments are requested four members
    // ahead of their use; the fold itself stays in member (= series) order.
    const double* const vals_k = a.vals + k;  // lane's column inside a series' row
    for (uint32_t mb = m0; mb < m1; mb += 32) {
      const uint32_t nm = (m1 - mb < 32u) ? (m1 - mb) : 32u;
      uint32_t s_l = 0, bit_l = 0;
      if ((uint32_t)lane < nm) {
        s_l = a.members[mb + lane];
        bit_l = a.valid[(size_t)s_l * a.Tw + tile];
      }
      for (uint32_t j = 0; j < nm; j += 4) {
        double x[4];
        bool ok[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t src = (j + u < nm) ? j + u : j;  // shuffles stay warp-uniform past the batch end
          const uint32_t s = __shfl_sync(0xffffffffu, s_l, (int)src);
          const uint32_t word = __shfl_sync(0xffffffffu, bit_l, (int)src);
          ok[u] = (j + u < nm) && in && ((word >> lane) & 1u);
          x[u] = 0.0;
          if (ok[u]) x[u] = vals_k[(size_t)s * a.T];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (ok[u]) fold(x[u]);
      }
    }
    if (!in) continue;
    const size_t o = (size_t)g * a.T + k;
    if (a.accumulate) {  // raw partials: SUM-type value and count
      a.out_val[o] += acc;
      a.out_cnt[o] += cnt;
      continue;
    }
    if constexpr (AGG == B2P_AGG_STDVAR || AGG == B2P_AGG_STDDEV) {
      if (a.out_mean) {
        a.out_val[o] = cnt ? m2 : 0.0;
        a.out_mean[o] = cnt ? mean : 0.0;
        a.out_cnt[o] = cnt;
        continue;
      }
    }
    double r = 0.0;
    if (cnt > 0) {
      if constexpr (AGG == B2P_AGG_SUM || AGG == B2P_AGG_MIN || AGG == B2P_AGG_MAX) r = acc;
      else if constexpr (AGG == B2P_AGG_AVG) r = acc / (double)cnt;
      else if constexpr (AGG == B2P_AGG_COUNT) r = (double)cnt;
      else if constexpr (AGG == B2P_AGG_STDVAR) r = m2 / (double)cnt;
      else r = sqrt(m2 / (double)cnt);
    }
    a.out_val[o] = r;
    a.out_cnt[o] = cnt;
  }
}

__global__ void __launch_bounds__(256) group_finalize_kernel(int32_t agg, double* val, const uint32_t* cnt, uint64_t n) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t c = cnt[i];
    if (c == 0) { val[i] = 0.0; continue; }
    if (agg == B2P_AGG_AVG) val[i] = val[i] / (double)c;
    else if (agg == B2P_AGG_COUNT) val[i] = (double)c;
    else if (agg == B2P_AGG_STDVAR) val[i] = val[i] / (double)c;        // merged M2 -> population variance
    else if (agg == B2P_AGG_STDDEV) val[i] = sqrt(val[i] / (double)c);
  }
}

// Cross-rank merge helpers of the by-label partials (b2p_allreduce_partials_dev).  min / max are reduced as total-order
// keys (int64 min / max on the collective), so NaNs of either sign and signed zeros merge exactly like the by-label
// kernel's own fold; an f64 min / max there would depend on the rank order.
// encode: val[i] becomes total_key(val[i]) in place, or the neutral key (INT64_MAX for min, INT64_MIN for max) for a
// group this rank has no row for.  decode (after the all-reduce, cnt = global count): keys turn back into values
// (total_key is its own inverse) and groups absent everywhere read 0.0 again, like a freshly built partial.
__global__ void __launch_bounds__(256) minmax_key_encode_kernel(bool is_min, double* val, const uint32_t* cnt, uint64_t n) {
  long long* key = reinterpret_cast<long long*>(val);
  const long long neutral = is_min ? 0x7fffffffffffffffll : (long long)0x8000000000000000ull;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
    key[i] = cnt[i] ? total_key(val[i]) : neutral;
}
__global__ void __launch_bounds__(256) minmax_key_decode_kernel(double* val, const uint32_t* cnt, uint64_t n) {
  const long long* key = reinterpret_cast<const long long*>(val);
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
    val[i] = cnt[i] ? __longlong_as_double(total_key(__longlong_as_double(key[i]))) : 0.0;
}
// (cnt, mean, M2) states of population variance.  phase 0: wsum = cnt * mean, cnt_r = cnt (kept: cnt becomes global);
// phase 1 (wsum, cnt all-reduced): mean_g = wsum / cnt; M2 += cnt_r * (mean_r - mean_g)^2 — the all-reduce of M2 that
// follows yields the merged M2; mean = mean_g.
__global__ void __launch_bounds__(256) variance_merge_kernel(int phase, double* m2, const uint32_t* cnt, double* mean,
                                                             double* wsum, uint32_t* cnt_r, uint64_t n) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    if (phase == 0) {
      cnt_r[i] = cnt[i];
      wsum[i] = (double)cnt[i] * mean[i];
    } else {
      const double mg = cnt[i] ? wsum[i] / (double)cnt[i] : 0.0;
      const double d = mean[i] - mg;
      m2[i] = cnt_r[i] ? m2[i] + (double)cnt_r[i] * d * d : 0.0;
      mean[i] = mg;
    }
  }
}

__global__ void __launch_bounds__(256) iota_kernel(uint32_t* p, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = i;
}

// goff[g] = lower_bound(sorted_gid, g) for g in [0, n_groups]; series with gid >= n_groups fall off the end.
__global__ void __launch_bounds__(256) group_offsets_kernel(const uint32_t* sorted_gid, uint32_t n, uint32_t n_groups,
                                                            uint32_t* goff) {
  for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g <= n_groups; g += gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (sorted_gid[mid] < g) lo = mid + 1; else hi = mid;
    }
    goff[g] = lo;
  }
}

// ---------------------------------------------------------------------------------------------
// K5 HistogramFold on the device (histogram_fold.rs:754-820 fold_buf, :834-981 safe mode, :1046-1118 evaluate_row).
// A histogram is a list of bucket series ordered by their `le` bound (CSR hist_off / bucket_series / bucket_le, built
// once per query from the labels); layouts may differ between histograms.  For every (histogram, eval step) the row
// the reference folds consists of the buckets that HAVE a sample at that step (rows with a null rate were filtered
// before the fold), in le order:
//   no bucket present            -> no output row
//   fewer than two, or the last present bound is not +Inf -> NaN   (safe mode, :930-944; evaluate_row :1048-1055)
//   otherwise evaluate_row on the present (bound, counter) pairs.
// One warp per (histogram, 32-step tile), lane = step: ONE pass over HBM — each bucket's 32-step segment is read once
// (coalesced 256 bytes), counters are made finite and monotone on the way into shared memory ([slot][lane] columns,
// conflict free; slot = rank among the present buckets of that step), then every lane bisects its own column.
// Algorithmic traffic: 8 B x buckets + 1 bit x buckets read, 8 B + 1 bit written per (histogram, step).  Histograms
// with more than kHistSmemBuckets buckets take the two-pass walk below (second pass from L2).
// ---------------------------------------------------------------------------------------------
struct HistFoldArgs {
  double phi;
  const uint32_t* hist_off;       // [n_hist + 1] into bucket_series / bucket_le
  const uint32_t* bucket_series;  // series id of every bucket, per histogram in ascending le order (NaN bounds last)
  const double* bucket_le;        // parsed bound of every bucket (NaN when the label does not parse, :791-796)
  uint32_t n_hist;
  const double* rates;            // [n_series x T]
  const uint32_t* valid;          // [n_series x Tw]
  uint64_t T;
  uint32_t Tw;
  double* out;                    // [n_hist x T]
  uint32_t* out_valid;            // [n_hist x Tw]
};

constexpr int kHistWarps = 4;          // warps per CTA
constexpr int kHistSmemBuckets = 64;   // rows with up to this many buckets keep their counters in shared memory

// evaluate_row from the quantile checks on (histogram_fold.rs:1062-1118); n >= 2 present buckets whose last bound is
// +Inf and whose bounds are non-decreasing; cnt(i) / le(i) give the i-th present bucket's monotonised counter / bound.
template <class Cnt, class Le>
__device__ __forceinline__ double histogram_row(double phi, uint32_t n, Cnt cnt, Le le) {
  const double kNaN = __longlong_as_double(0x7ff8000000000000ll);
  const double kInf = __longlong_as_double(0x7ff0000000000000ll);
  if (phi < 0.0) return -kInf;
  if (phi > 1.0) return kInf;
  if (isnan(phi)) return kNaN;
  const double total = cnt(n - 1);
  const double expected_pos = total * phi;
  // first present bucket whose counter is >= expected_pos: the counters are non-decreasing, so bisect
  uint32_t lo = 0, hi = n;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (cnt(mid) < expected_pos) lo = mid + 1; else hi = mid;
  }
  const uint32_t fit = lo;
  if (fit >= n - 1) return le(n - 2);
  const double upper_count = cnt(fit), upper_bound = le(fit);
  double lower_bound = fmin(le(0), 0.0), lower_count = 0.0;
  if (fit > 0) {
    lower_bound = le(fit - 1);
    lower_count = cnt(fit - 1);
  }
  if (fabs(upper_count - lower_count) < 1e-10) return kNaN;
  return lower_bound + (upper_bound - lower_bound) / (upper_count - lower_count) * (expected_pos - lower_count);
}

__global__ void __launch_bounds__(kHistWarps * 32) histogram_fold_kernel(const HistFoldArgs a) {
  extern __shared__ __align__(16) unsigned char hist_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* col = reinterpret_cast<double*>(hist_smem) + (size_t)warp * kHistSmemBuckets * 32 + lane;  // col[slot * 32]
  unsigned char* idx = hist_smem + (size_t)kHistWarps * kHistSmemBuckets * 32 * 8 + (size_t)warp * kHistSmemBuckets * 32 + lane;
  const double kNaN = __longlong_as_double(0x7ff8000000000000ll);
  const uint64_t tiles = (a.T + 31) / 32;
  const uint64_t total = (uint64_t)a.n_hist * tiles;
  for (uint64_t w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total;
       w += ((uint64_t)gridDim.x * blockDim.x) >> 5) {
    const uint32_t h = (uint32_t)(w / tiles);
    const uint64_t tile = w - (uint64_t)h * tiles;
    const uint64_t k = tile * 32 + lane;
    const bool in = k < a.T;
    const uint32_t o = a.hist_off[h], nb = a.hist_off[h + 1] - o;
    const uint32_t* bs = a.bucket_series + o;
    const double* ble = a.bucket_le + o;
    uint32_t n = 0;          // present buckets of this lane's step
    double prev = 0.0;       // monotonised counter of the previous present bucket
    double last_le = kNaN, prev_le = -__longlong_as_double(0x7ff0000000000000ll);
    bool sorted = true;      // bucket.windows(2).all(|w| w[0] <= w[1]) over the present bounds
    bool ok = false;
    double r = 0.0;
    // common case first: all buckets of the histogram have samples at the same steps of the tile (normally: at every
    // step) -> a step either has no row or every bucket: no per-lane compaction, slot = bucket
    uint32_t all = 0xffffffffu, any = 0u;
    for (uint32_t b0 = 0; b0 < nb; b0 += 32) {
      const bool has = b0 + lane < nb;
      const uint32_t wv = has ? a.valid[(size_t)bs[b0 + lane] * a.Tw + tile] : 0u;
      all &= __reduce_and_sync(0xffffffffu, has ? wv : 0xffffffffu);
      any |= __reduce_or_sync(0xffffffffu, wv);
    }
    if (nb <= (uint32_t)kHistSmemBuckets && all == any && nb >= 2) {
      const bool present = in && ((all >> lane) & 1u);
      for (uint32_t b0 = 0; b0 < nb; b0 += 8) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
          v[u] = (b0 + u < nb && present) ? __ldcs(a.rates + (size_t)bs[b0 + u] * a.T + k) : 0.0;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (b0 + u < nb) {
            double c = isfinite(v[u]) ? v[u] : prev;
            if (b0 + u > 0 && c < prev) c = prev;
            prev = c;
            col[(b0 + u) * 32] = c;
          }
        }
      }
      // the bounds of the histogram are the same for every lane: sortedness and the +Inf check once per warp
      bool srt = true;
      for (uint32_t b0 = 0; b0 + 1 < nb; b0 += 32) {
        const bool okp = (b0 + lane + 1 < nb) ? (ble[b0 + lane] <= ble[b0 + lane + 1]) : true;
        srt = srt && __all_sync(0xffffffffu, okp);
      }
      const double l_last = ble[nb - 1];
      const bool has_inf = l_last == __longlong_as_double(0x7ff0000000000000ll);
      ok = present;
      if (ok) {
        if (!has_inf) r = kNaN;
        else if (!srt && !(a.phi < 0.0) && !(a.phi > 1.0)) r = kNaN;
        else r = histogram_row(a.phi, nb, [&](uint32_t i) { return col[i * 32]; }, [&](uint32_t i) { return ble[i]; });
      }
    } else if (nb <= (uint32_t)kHistSmemBuckets) {
      for (uint32_t b0 = 0; b0 < nb; b0 += 8) {
        double v[8];
        uint32_t wd[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const bool has = b0 + u < nb;
          const uint32_t s = has ? bs[b0 + u] : 0u;
          wd[u] = has ? a.valid[(size_t)s * a.Tw + tile] : 0u;
          v[u] = (has && in && ((wd[u] >> lane) & 1u)) ? __ldcs(a.rates + (size_t)s * a.T + k) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (b0 + u < nb && in && ((wd[u] >> lane) & 1u)) {
            double c = isfinite(v[u]) ? v[u] : prev;   // non-finite -> previous, decreasing -> previous (:1074-1092)
            if (n > 0 && c < prev) c = prev;
            prev = c;
            col[n * 32] = c;
            idx[n * 32] = (unsigned char)(b0 + u);
            const double l = ble[b0 + u];
            sorted = sorted && (n == 0 || prev_le <= l);
            prev_le = l;
            last_le = l;
            ++n;
          }
        }
      }
      ok = n > 0;
      if (ok) {
        const bool has_inf = !(last_le < __longlong_as_double(0x7ff0000000000000ll)) && !isnan(last_le) && last_le > 0.0;
        if (n < 2 || !has_inf) r = kNaN;
        else if (!sorted && !(a.phi < 0.0) && !(a.phi > 1.0)) r = kNaN;
        else r = histogram_row(a.phi, n, [&](uint32_t i) { return col[i * 32]; }, [&](uint32_t i) { return ble[idx[i * 32]]; });
      }
    } else if (in) {
      // wide histogram: walk the buckets twice (presence, total and checks; then the linear search of the reference)
      for (uint32_t b = 0; b < nb; ++b) {
        const uint32_t s = bs[b];
        if (!((a.valid[(size_t)s * a.Tw + tile] >> lane) & 1u)) continue;
        const double x = a.rates[(size_t)s * a.T + k];
        double c = isfinite(x) ? x : prev;
        if (n > 0 && c < prev) c = prev;
        prev = c;
        const double l = ble[b];
        sorted = sorted && (n == 0 || prev_le <= l);
        prev_le = l;
        last_le = l;
        ++n;
      }
      ok = n > 0;
      if (ok) {
        const double kInf = __longlong_as_double(0x7ff0000000000000ll);
        const bool has_inf = last_le == kInf;
        if (n < 2 || !has_inf) r = kNaN;
        else if (a.phi < 0.0) r = -kInf;
        else if (a.phi > 1.0) r = kInf;
        else if (isnan(a.phi) || !sorted) r = kNaN;
        else {
          const double expected_pos = prev * a.phi;  // prev = total after the first walk
          uint32_t i = 0, fit = n;
          double run = 0.0, run_le = 0.0, le0 = 0.0, le_nm2 = 0.0, lc = 0.0, lb = 0.0, uc = 0.0, ub = 0.0;
          for (uint32_t b = 0; b < nb; ++b) {
            const uint32_t s = bs[b];
            if (!((a.valid[(size_t)s * a.Tw + tile] >> lane) & 1u)) continue;
            const double x = a.rates[(size_t)s * a.T + k];
            double c = isfinite(x) ? x : run;
            if (i > 0 && c < run) c = run;
            const double l = ble[b];
            if (i == 0) le0 = l;
            if (i == n - 2) le_nm2 = l;
            if (fit == n && !(c < expected_pos)) {  // the reference's linear search stops here
              fit = i;
              uc = c;
              ub = l;
              lc = i > 0 ? run : 0.0;
              lb = i > 0 ? run_le : fmin(le0, 0.0);
            }
            run = c;
            run_le = l;
            ++i;
          }
          if (fit >= n - 1) r = le_nm2;
          else if (fabs(uc - lc) < 1e-10) r = kNaN;
          else r = lb + (ub - lb) / (uc - lc) * (expected_pos - lc);
        }
      }
    }
    if (in) a.out[(size_t)h * a.T + k] = ok ? r : 0.0;
    const uint32_t word = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) a.out_valid[(size_t)h * a.Tw + tile] = word;
  }
}

// uniform layout (bucket b of histogram h = series h * B + b, shared bounds le[B]) -> the CSR the fold kernel takes
__global__ void __launch_bounds__(256) histogram_uniform_index_kernel(const double* le, uint32_t B, uint32_t n_hist,
                                                                      uint32_t* hist_off, uint32_t* bucket_series,
                                                                      double* bucket_le) {
  const uint64_t n = (uint64_t)n_hist * B;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    bucket_series[i] = (uint32_t)i;
    bucket_le[i] = le[i % B];
    if (i % B == 0) hist_off[i / B] = (uint32_t)i;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) hist_off[n_hist] = (uint32_t)n;
}

// ---------------------------------------------------------------------------------------------
// K6.  Deterministic two-stage per-column reduction; NaN rows are skipped like SeriesNormalize's
// filter.  Stage 1: grid (blocks_per_col, n_cols), each block reduces a contiguous slab with 128-bit
// loads; stage 2: one warp per column folds the block partials in order.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) column_reduce_stage1(const double* const* cols, uint64_t n_rows,
                                                            double* part_sum, unsigned long long* part_cnt) {
  const double* col = cols[blockIdx.y];
  const uint64_t per = ((n_rows + gridDim.x - 1) / gridDim.x + 1) & ~1ull;
  const uint64_t r0 = (uint64_t)blockIdx.x * per;
  const uint64_t r1 = min(n_rows, r0 + per);
  double s = 0.0;
  unsigned long long c = 0;
  for (uint64_t r = r0 + 2ull * threadIdx.x; r < r1; r += 2ull * blockDim.x) {
    if (r + 1 < r1) {
      const double2 v = __ldcs(reinterpret_cast<const double2*>(col + r));
      if (!isnan(v.x)) { s += v.x; ++c; }
      if (!isnan(v.y)) { s += v.y; ++c; }
    } else {
      const double v = col[r];
      if (!isnan(v)) { s += v; ++c; }
    }
  }
  __shared__ double ss[8];
  __shared__ unsigned long long sc[8];
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_down_sync(0xffffffffu, s, o);
    c += __shfl_down_sync(0xffffffffu, c, o);
  }
  if ((threadIdx.x & 31) == 0) { ss[threadIdx.x >> 5] = s; sc[threadIdx.x >> 5] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    unsigned long long tc = 0;
    for (int i = 0; i < 8; ++i) { t += ss[i]; tc += sc[i]; }
    part_sum[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = t;
    part_cnt[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = tc;
  }
}

__global__ void column_reduce_stage2(const double* part_sum, const unsigned long long* part_cnt, uint32_t blocks,
                                     double* out_sum, unsigned long long* out_cnt) {
  const uint32_t c = blockIdx.x;
  if (threadIdx.x != 0) return;
  double t = 0.0;
  unsigned long long tc = 0;
  for (uint32_t i = 0; i < blocks; ++i) { t += part_sum[(size_t)c * blocks + i]; tc += part_cnt[(size_t)c * blocks + i]; }
  out_sum[c] += t;
  out_cnt[c] += tc;
}

}  // namespace b2p
