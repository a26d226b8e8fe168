"""ctypes binding of the CPU ORACLE (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY — see oracle/promql_oracle.h.  Importable from tests/, from
__graft_entry__.smoke() and from bench.py's cpu_baseline / --impl reference legs; the product
package greptimedb_b200 never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")

FN_IDS = {
    "rate": 0, "increase": 1, "delta": 2, "irate": 3, "idelta": 4, "resets": 5, "changes": 6,
    "count_over_time": 7, "sum_over_time": 8, "avg_over_time": 9, "min_over_time": 10,
    "max_over_time": 11, "last_over_time": 12, "present_over_time": 13, "absent_over_time": 14,
    "stdvar_over_time": 15, "stddev_over_time": 16, "deriv": 17, "predict_linear": 18,
    "quantile_over_time": 19, "holt_winters": 20,
}
AGG_OPS = {"sum": 0, "avg": 1, "count": 2, "min": 3, "max": 4, "stddev": 5, "stdvar": 6}


def _cpu_stamp() -> str:
    """Identity of the host CPU (model + ISA flags): the oracle is compiled -march=native and travels with the
    snapshot, so a library built on another CPU is rebuilt here before it is loaded."""
    try:
        model, flags = "", ""
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name") and not model:
                    model = ln.split(":", 1)[1].strip()
                elif ln.startswith("flags") and not flags:
                    flags = " ".join(sorted(ln.split(":", 1)[1].split()))
                if model and flags:
                    break
        import hashlib
        return model + " " + hashlib.sha1(flags.encode()).hexdigest()
    except OSError:
        return "unknown"


_SOURCES = ("promql_oracle.c", "promql_oracle.h", "Makefile")


def build(force: bool = False) -> str:
    """Compile the oracle with gcc (oracle/Makefile).  Building the checker is not using it.  -> path of the library.
    In a source tree that cannot be written (a read-only checkout) a library that has to be rebuilt is compiled into a
    temporary directory instead, removed again when the process exits."""
    src = [os.path.join(_HERE, f) for f in _SOURCES]
    stamp_path = _SO + ".cpu"
    stamp = _cpu_stamp()
    try:
        same_cpu = open(stamp_path).read() == stamp
    except OSError:
        same_cpu = False
    if force or not same_cpu or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in src):
        if not os.access(_HERE, os.W_OK):
            return _build_private()
        subprocess.check_call(["make", "-s", "-B", "-C", _HERE, "liboracle.so"])
        with open(stamp_path, "w") as f:
            f.write(stamp)
    return _SO


def _build_private() -> str:
    import atexit
    import shutil
    import tempfile
    tmp = tempfile.mkdtemp(prefix="promql_oracle_")
    atexit.register(shutil.rmtree, tmp, True)
    for f in _SOURCES:
        shutil.copy(os.path.join(_HERE, f), tmp)
    subprocess.check_call(["make", "-s", "-B", "-C", tmp, "liboracle.so"])
    return os.path.join(tmp, "liboracle.so")


class Params(C.Structure):
    _fields_ = [("fn_id", C.c_int32), ("filter_nan", C.c_int32), ("start", C.c_int64), ("end", C.c_int64),
                ("interval", C.c_int64), ("range", C.c_int64), ("offset", C.c_int64),
                ("param0", C.c_double), ("param1", C.c_double)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        i64p, f64p, u32p, u64p, u8p = (C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_uint32),
                                       C.POINTER(C.c_uint64), C.POINTER(C.c_uint8))
        L.orc_num_steps.restype = C.c_int64
        L.orc_num_steps.argtypes = [C.c_int64] * 3
        for name in ("orc_calculate_range", "orc_calculate_range_definitional"):
            f = getattr(L, name)
            f.restype = C.c_int64
            f.argtypes = [i64p, C.c_size_t, C.c_int64, C.c_int64, C.c_int64, C.c_int64, u32p, u32p, i64p, i64p]
        L.orc_normalize.restype = C.c_size_t
        L.orc_normalize.argtypes = [i64p, f64p, C.c_size_t, C.c_int64, C.c_int, i64p, f64p]
        L.orc_series_divide.restype = C.c_size_t
        L.orc_series_divide.argtypes = [u32p, C.c_size_t, u64p]
        L.orc_instant_manipulate.restype = C.c_int64
        L.orc_instant_manipulate.argtypes = [i64p, f64p, C.c_size_t, C.c_int64, C.c_int64, C.c_int64, C.c_int64, u64p, i64p]
        L.orc_histogram_evaluate_row.restype = C.c_double
        L.orc_histogram_evaluate_row.argtypes = [C.c_double, f64p, f64p, C.c_size_t, C.POINTER(C.c_int)]
        for name in ("orc_range_udf", "orc_range_udf_rescan"):
            f = getattr(L, name)
            f.restype = None
            f.argtypes = [C.c_int, i64p, f64p, u32p, u32p, i64p, C.c_size_t, C.c_int64, C.c_double, C.c_double, f64p, u8p]
        for name in ("orc_arrow_sum", "orc_arrow_min", "orc_arrow_max"):
            f = getattr(L, name)
            f.restype = C.c_double
            f.argtypes = [f64p, C.c_size_t]
        L.orc_compensated_sum_inc.restype = None
        L.orc_compensated_sum_inc.argtypes = [C.c_double, f64p, f64p]
        L.orc_linear_regression.restype = C.c_int
        L.orc_linear_regression.argtypes = [i64p, f64p, C.c_size_t, C.c_int64, f64p, f64p]
        L.orc_quantile.restype = C.c_double
        L.orc_quantile.argtypes = [f64p, C.c_size_t, C.c_double]
        L.orc_holt_winters.restype = C.c_double
        L.orc_holt_winters.argtypes = [f64p, C.c_size_t, C.c_double, C.c_double]
        L.orc_range_query_faithful.restype = None
        L.orc_range_query_faithful.argtypes = [C.POINTER(Params), i64p, f64p, u32p, u64p, C.c_size_t, C.c_size_t, f64p, u32p]
        L.orc_range_query_flat.restype = None
        L.orc_range_query_flat.argtypes = [C.POINTER(Params), i64p, f64p, u64p, C.c_size_t, C.c_size_t, f64p, u32p]
        L.orc_range_query_mt.restype = C.c_int
        L.orc_range_query_mt.argtypes = [C.POINTER(Params), i64p, f64p, u32p, u64p, C.c_size_t, f64p, u32p, C.c_int, C.c_int]
        L.orc_instant_query.restype = None
        L.orc_instant_query.argtypes = [i64p, f64p, u64p, C.c_size_t, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, f64p, u32p]
        L.orc_group_aggregate.restype = None
        L.orc_group_aggregate.argtypes = [C.c_int, f64p, u32p, u32p, C.c_size_t, C.c_size_t, C.c_size_t, f64p, u32p]
        L.orc_histogram_quantile.restype = None
        L.orc_histogram_quantile.argtypes = [C.c_double, f64p, C.c_size_t, f64p, u32p, C.c_size_t, C.c_size_t, f64p, u32p]
        L.orc_synth_fill.restype = None
        L.orc_synth_fill.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int64, C.c_int64, C.c_uint32, C.c_int, C.c_uint64, i64p, f64p, u32p]
        _lib = L
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def num_steps(start, end, interval):
    return int(lib().orc_num_steps(start, end, interval))


def calculate_range(ts, start, end, interval, rng, definitional=False):
    """-> (off[u32], len[u32], start', end')"""
    ts = _i64(ts)
    cap = max(num_steps(start, end, interval), 0) + 1
    off = np.zeros(cap, np.uint32)
    ln = np.zeros(cap, np.uint32)
    s2, e2 = C.c_int64(0), C.c_int64(0)
    f = lib().orc_calculate_range_definitional if definitional else lib().orc_calculate_range
    n = f(_p(ts, C.c_int64), ts.size, start, end, interval, rng, _p(off, C.c_uint32), _p(ln, C.c_uint32),
          C.byref(s2), C.byref(e2))
    return off[:n].copy(), ln[:n].copy(), s2.value, e2.value


def normalize(ts, val, offset, filter_nan):
    ts, val = _i64(ts), _f64(val)
    ots, oval = np.zeros_like(ts), np.zeros_like(val)
    m = lib().orc_normalize(_p(ts, C.c_int64), _p(val, C.c_double), ts.size, offset, int(filter_nan),
                            _p(ots, C.c_int64), _p(oval, C.c_double))
    return ots[:m].copy(), oval[:m].copy()


def series_divide(sid):
    sid = _u32(sid)
    offs = np.zeros(sid.size + 2, np.uint64)
    ns = lib().orc_series_divide(_p(sid, C.c_uint32), sid.size, _p(offs, C.c_uint64))
    return offs[: ns + 1].copy()


def instant_manipulate(ts, val, start, end, interval, lookback):
    """-> (take_idx, out_ts) like InstantManipulateStream::manipulate (sparse rows)."""
    ts = _i64(ts)
    val = None if val is None else _f64(val)
    if ts.size == 0:
        return np.zeros(0, np.uint64), np.zeros(0, np.int64)
    # bound the capacity by the data-trimmed grid, as the reference does (instant_manipulate.rs:501-511)
    last_useful = ts[-1] + lookback - 1 if lookback > 0 else ts[-1]
    lo = max(int(ts[0]), start)
    hi = min(int(last_useful), end)
    cap = max((hi - lo) // interval + 3, 3)
    take = np.zeros(cap, np.uint64)
    ots = np.zeros(cap, np.int64)
    m = lib().orc_instant_manipulate(_p(ts, C.c_int64), _p(val, C.c_double), ts.size, start, end, interval,
                                     lookback, _p(take, C.c_uint64), _p(ots, C.c_int64))
    return take[:m].copy(), ots[:m].copy()


def histogram_evaluate_row(q, bucket, counter):
    """-> (value, err)"""
    b, c = _f64(bucket), _f64(counter)
    err = C.c_int(0)
    v = lib().orc_histogram_evaluate_row(q, _p(b, C.c_double), _p(c, C.c_double), b.size, C.byref(err))
    return v, bool(err.value)


def range_udf(fn, ts, val, ranges, eval_ts=None, range_length=0, param0=0.0, param1=0.0, rescan=False):
    """Evaluate a prom_* range UDF over explicit windows.  -> (out f64[], valid bool[])."""
    ts, val = _i64(ts), _f64(val)
    ranges = np.asarray(ranges, dtype=np.uint32).reshape(-1, 2)
    off, ln = _u32(ranges[:, 0]), _u32(ranges[:, 1])
    n = off.size
    ets = _i64(eval_ts) if eval_ts is not None else np.zeros(n, np.int64)
    out = np.zeros(n, np.float64)
    valid = np.zeros(n, np.uint8)
    f = lib().orc_range_udf_rescan if rescan else lib().orc_range_udf
    fid = FN_IDS[fn] if isinstance(fn, str) else int(fn)
    f(fid, _p(ts, C.c_int64), _p(val, C.c_double), _p(off, C.c_uint32), _p(ln, C.c_uint32), _p(ets, C.c_int64), n,
      int(range_length), float(param0), float(param1), _p(out, C.c_double), _p(valid, C.c_uint8))
    return out, valid.astype(bool)


def make_params(fn, start, end, interval, rng, offset=0, filter_nan=True, param0=0.0, param1=0.0):
    fid = FN_IDS[fn] if isinstance(fn, str) else int(fn)
    return Params(fid, int(bool(filter_nan)), start, end, interval, rng, offset, float(param0), float(param1))


def range_query(p: Params, ts, val, sid, offsets, mode="flat", threads=1):
    """Whole sub-plan, dense [S x T] + validity words.  mode in {"flat","faithful"}."""
    ts, val = _i64(ts), _f64(val)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    S = offsets.size - 1
    sid = _u32(sid) if sid is not None else np.repeat(np.arange(S, dtype=np.uint32), np.diff(offsets).astype(np.int64))
    T = num_steps(p.start, p.end, p.interval)
    Tw = (T + 31) // 32
    out = np.zeros((S, T), np.float64)
    valid = np.zeros((S, Tw), np.uint32)
    rc = lib().orc_range_query_mt(C.byref(p), _p(ts, C.c_int64), _p(val, C.c_double), _p(sid, C.c_uint32),
                                  _p(offsets, C.c_uint64), S, _p(out, C.c_double), _p(valid, C.c_uint32),
                                  int(threads), 1 if mode == "faithful" else 0)
    if rc != 0:
        raise RuntimeError("orc_range_query_mt failed")
    return out, valid


def instant_query(ts, val, offsets, start, end, interval, lookback, offset=0):
    ts, val = _i64(ts), _f64(val)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    S = offsets.size - 1
    T = num_steps(start, end, interval)
    Tw = (T + 31) // 32
    out = np.zeros((S, T), np.float64)
    valid = np.zeros((S, Tw), np.uint32)
    lib().orc_instant_query(_p(ts, C.c_int64), _p(val, C.c_double), _p(offsets, C.c_uint64), S, start, end, interval,
                            lookback, offset, _p(out, C.c_double), _p(valid, C.c_uint32))
    return out, valid


def group_aggregate(op, vals, valid, gid, n_groups):
    vals = _f64(vals)
    valid = _u32(valid)
    gid = _u32(gid)
    S, T = vals.shape
    out = np.zeros((n_groups, T), np.float64)
    cnt = np.zeros((n_groups, T), np.uint32)
    lib().orc_group_aggregate(AGG_OPS[op] if isinstance(op, str) else int(op), _p(vals, C.c_double),
                              _p(valid, C.c_uint32), _p(gid, C.c_uint32), S, n_groups, T, _p(out, C.c_double),
                              _p(cnt, C.c_uint32))
    return out, cnt


def histogram_quantile(phi, le, rates, valid):
    le, rates, valid = _f64(le), _f64(rates), _u32(valid)
    B = le.size
    S, T = rates.shape
    H = S // B
    Tw = (T + 31) // 32
    out = np.zeros((H, T), np.float64)
    ov = np.zeros((H, Tw), np.uint32)
    lib().orc_histogram_quantile(phi, _p(le, C.c_double), B, _p(rates, C.c_double), _p(valid, C.c_uint32), H, T,
                                 _p(out, C.c_double), _p(ov, C.c_uint32))
    return out, ov


def synth_fill(series_begin, n_series, n_samples, t0, scrape_ms, jitter_ms, with_resets, seed):
    n = n_series * n_samples
    ts = np.zeros(n, np.int64)
    val = np.zeros(n, np.float64)
    sid = np.zeros(n, np.uint32)
    lib().orc_synth_fill(series_begin, n_series, n_samples, t0, scrape_ms, jitter_ms, int(with_resets), seed,
                         _p(ts, C.c_int64), _p(val, C.c_double), _p(sid, C.c_uint32))
    return ts, val, sid


def valid_to_bool(valid_words, T):
    """[S x Tw] u32 words -> [S x T] bool."""
    bits = np.unpackbits(valid_words.view(np.uint8), axis=1, bitorder="little")
    return bits[:, :T].astype(bool)


def arrow_sum(v):
    v = _f64(v)
    return lib().orc_arrow_sum(_p(v, C.c_double), v.size)


def linear_regression(ts, val, intercept_time):
    ts, val = _i64(ts), _f64(val)
    s, i = C.c_double(0), C.c_double(0)
    ok = lib().orc_linear_regression(_p(ts, C.c_int64), _p(val, C.c_double), val.size, intercept_time,
                                     C.byref(s), C.byref(i))
    return (s.value, i.value) if ok else (None, None)


def quantile(v, q):
    v = _f64(v)
    return lib().orc_quantile(_p(v, C.c_double), v.size, q)


def holt_winters(v, sf, tf):
    v = _f64(v)
    return lib().orc_holt_winters(_p(v, C.c_double), v.size, sf, tf)


def compensated_sum(inputs):
    s, c = C.c_double(0.0), C.c_double(0.0)
    for x in inputs:
        lib().orc_compensated_sum_inc(float(x), C.byref(s), C.byref(c))
    return s.value, c.value


# ---------------------------------------------------------------------------------------------------
# HistogramFold, row-literal (small cases only): fold_buf's optimistic mode, the switch to safe mode and the safe-mode
# grouping of histogram_fold.rs:725-981, on rows in scan order.  Used to pin the dense device fold on the reference's
# operator tests (tests/golden/reference_histogram_fold_vectors.json).
# ---------------------------------------------------------------------------------------------------
def parse_f64_rust(s):
    """str::parse::<f64>().unwrap_or(NaN) (histogram_fold.rs:791-796): decimal / exponent forms, inf / infinity / nan
    in any case with an optional sign; no surrounding white space, hex, underscores or decimal commas."""
    import math
    import re
    if s is None:
        return math.nan
    m = re.fullmatch(r"([+-]?)(inf|infinity|nan)", s, flags=re.I)
    if m:
        if m.group(2).lower() == "nan":
            return math.nan
        return -math.inf if m.group(1) == "-" else math.inf
    if re.fullmatch(r"[+-]?(\d+\.?\d*|\.\d+)([eE][+-]?\d+)?", s):
        return float(s)
    return math.nan


def histogram_fold_rows(rows, phi):
    """rows: [(tags tuple, ts, le label, value)] in scan order (sorted by tags, ts, le).  -> [(tags, ts, result)].
    A group is a run of rows with equal (tags, ts) — the reference's `normal` columns are everything but le and the field."""
    import math

    def is_pos_inf(le):
        v = parse_f64_rust(le)
        return math.isinf(v) and v > 0

    def evaluate(buckets, counters):  # evaluate_row(..).unwrap_or(NaN)
        v, err = histogram_evaluate_row(phi, np.array(buckets, np.float64), np.array(counters, np.float64))
        return math.nan if err else v

    n = len(rows)
    out = []
    # find_first_complete_bucket (:725-751): rows from the start of the group that holds the first +Inf row
    bucket_num = None
    group_start = 0
    cur_key = rows[0][:2] if n else None
    for r in range(n):
        if rows[r][:2] != cur_key:  # new group begins
            cur_key = rows[r][:2]
            group_start = r
        if is_pos_inf(rows[r][2]):
            bucket_num = r - group_start + 1
            break
    cursor = 0
    if bucket_num is not None:
        while n - cursor >= bucket_num:  # optimistic mode (:768-812)
            key = rows[cursor][:2]
            ok = is_pos_inf(rows[cursor + bucket_num - 1][2]) and all(rows[cursor + o][:2] == key for o in range(1, bucket_num))
            if not ok:
                break
            grp = rows[cursor:cursor + bucket_num]
            try:
                res = evaluate([parse_f64_rust(g[2]) for g in grp], [g[3] for g in grp])
            except Exception:
                res = math.nan
            out.append((key[0], key[1], res))
            cursor += bucket_num
    # safe mode over what is left (:930-981): variable-length groups
    r = cursor
    while r < n:
        key = rows[r][:2]
        e = r
        while e < n and rows[e][:2] == key:
            e += 1
        b = [parse_f64_rust(g[2]) for g in rows[r:e]]
        c = [g[3] for g in rows[r:e]]
        has_inf = len(b) > 0 and math.isinf(b[-1]) and b[-1] > 0
        res = math.nan if (len(b) < 2 or not has_inf) else evaluate(b, c)
        out.append((key[0], key[1], res))
        r = e
    return out
