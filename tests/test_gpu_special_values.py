"""GPU: special f64 values through every tier — +-Inf, NaNs of both signs and with payloads, signed zeros, subnormals,
values next to overflow, counters starting at exactly 0.0 or near 2^53 — compared with the CPU oracle by bits.

The oracle is C on an x86-64 host, like the reference (Rust) on the x86 hosts B200 systems ship with.  There an
invalid operation (inf - inf, 0 * inf, 0 / 0) yields the default NaN 0xfff8000000000000, whose sign bit is set; the
constant NaNs the reference writes as f64::NAN are 0x7ff8000000000000.  The sign is observable further down:
min by / max by order values by f64::total_cmp, where -NaN is the least and +NaN the greatest value.  So with
filter_nan on (no NaN sample reaches the arithmetic) NaN results must match the oracle bit for bit.  The B200's f64
units produce the same default NaN and propagate NaN operands the same way (measured: inf - inf, 0 * inf and 0 / 0
give 0xfff8000000000000; NaN + NaN returns the first operand), so the kernels need no rewriting of their NaNs; these
tests keep it that way.

With filter_nan off, the pass-through functions (last / min / max / quantile / count / present / changes / resets)
stay bit-exact including NaN payloads.  The arithmetic functions are compared by NaN class only there: x86
propagates the first NaN operand of each operation, and which operand comes first is a detail of the reference's
expression order that is not restated on the device.
"""
import os

import numpy as np
import pytest

from oracle import oracle as orc

pytestmark = pytest.mark.gpu

REL = 1e-9
T0 = 1_700_000_000_000
ALL_FNS = ["rate", "increase", "delta", "irate", "idelta", "resets", "changes", "count_over_time", "sum_over_time",
           "avg_over_time", "min_over_time", "max_over_time", "last_over_time", "present_over_time",
           "absent_over_time", "stdvar_over_time", "stddev_over_time", "deriv", "predict_linear",
           "quantile_over_time", "holt_winters"]
FN_PARAMS = {"predict_linear": (600.0, 0.0), "quantile_over_time": (0.9, 0.0), "holt_winters": (0.3, 0.1)}
BIT_EXACT = {"resets", "changes", "count_over_time", "present_over_time", "absent_over_time", "last_over_time",
             "min_over_time", "max_over_time", "idelta"}
PASS_THROUGH = {"last_over_time", "min_over_time", "max_over_time", "quantile_over_time", "count_over_time",
                "present_over_time", "changes", "resets"}
COUNTERS = {"rate", "increase", "delta"}


def f64(*bits):
    return np.array(bits, np.uint64).view(np.float64)


POS_NAN, NEG_NAN, STALE = f64(0x7FF8000000000000, 0xFFF8000000000000, 0x7FF0000000000002)
MIN_NORMAL = 2.2250738585072014e-308
# members of the by-label tests: both zeros, both infinities, NaNs of both signs, a payload NaN, a subnormal, +-1e308
SPECIAL_MEMBERS = np.concatenate([f64(0x0, 0x8000000000000000, 0x7FF0000000000000, 0xFFF0000000000000,
                                      0x7FF8000000000000, 0xFFF8000000000000, 0x7FF0000000000002, 0x1),
                                  [1e308, -1e308]])


def _make_ctx(**env):
    from greptimedb_b200 import Context
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


# one context per tier configuration; the adaptive back-off of the lean tier is pinned off where the tier must stay
TIERS = {
    "default": dict(B2P_LEAN_ADAPTIVE="0"),                                     # K2L + the uniform-cadence probe
    "no_lean": dict(B2P_DISABLE_LEAN_TIER="1"),                                 # K2 alone
    "lean_flags": dict(B2P_LEAN_FORCE_FLAGS="1", B2P_LEAN_ADAPTIVE="0"),        # K2L bit-word variant
    "thread": dict(B2P_ENABLE_THREAD_TIER="1"),                                 # K2T
    "uniform": dict(B2P_UNIFORM="1", B2P_LEAN_ADAPTIVE="0"),                    # K2L uniform cadence, forced
}


@pytest.fixture(scope="module")
def ctxs():
    cs = {name: _make_ctx(**env) for name, env in TIERS.items()}
    yield cs
    for c in cs.values():
        c.close()


@pytest.fixture(scope="module")
def ctx(ctxs):
    return ctxs["default"]


# ---------------------------------------------------------------------------------------------------
# the value zoo
# ---------------------------------------------------------------------------------------------------
N_RECIPES = 10


def recipe(kind, n, rng):
    """Values of one series: a counter-like base with special values spliced in."""
    base = np.cumsum(rng.random(n) * 10)
    i = np.arange(n)
    if kind == 0:        # single +-Inf samples
        v = base.copy()
        v[rng.integers(0, n, max(n // 40, 1))] = np.inf
        v[rng.integers(0, n, max(n // 40, 1))] = -np.inf
    elif kind == 1:      # runs of +Inf: inf - inf inside one window
        v = base.copy()
        for j in rng.integers(0, max(n - 3, 1), max(n // 60, 1)):
            v[j:j + int(rng.integers(2, 4))] = np.inf
    elif kind == 2:      # a counter that jumps to +Inf and back: the reset correction adds Inf
        v = base.copy()
        v[rng.integers(1, n, max(n // 50, 1))] = np.inf
    elif kind == 3:      # next to overflow: last - first and the corrections overflow
        v = np.where(i % 7 < 3, 1e308, -1e308) * (1.0 - rng.random(n) * 1e-3)
        v[n // 2:] = 1.7e308 - np.cumsum(rng.random(n - n // 2)) * 1e306
    elif kind == 4:      # subnormals and values around the smallest normal
        v = np.cumsum(rng.integers(0, 3, n)) * 5e-324
        v[i % 3 == 1] = MIN_NORMAL + (i[i % 3 == 1] % 5 - 2) * 5e-324
    elif kind == 5:      # runs of +-0.0 with a few ones
        v = np.where((i // 5) % 2 == 0, 0.0, -0.0)
        v[rng.random(n) < 0.1] = 1.0
    elif kind == 6:      # a counter starting at exactly 0.0
        v = base - base[0]
    elif kind == 7:      # a counter near 2^53 that increases by 1
        v = 2.0 ** 53 - n // 2 + i.astype(np.float64)
    elif kind == 8:      # negative counters (decreasing and increasing)
        v = -base if rng.random() < 0.5 else base - 1e6
    else:                # input NaNs of both signs and the stale marker
        v = base.copy()
        v[rng.integers(0, n, max(n // 20, 1))] = POS_NAN
        v[rng.integers(0, n, max(n // 20, 1))] = NEG_NAN
        v[rng.integers(0, n, max(n // 30, 1))] = STALE
    return v.astype(np.float64)


# timestamp layouts: (query, sample spacing, samples per series); each is chosen to route series to a known tier
LAYOUTS = {
    "exact": dict(start=T0, end=T0 + 399 * 15_000, interval=15_000, range=300_000, n=400),      # uniform K2L
    "jitter": dict(start=T0, end=T0 + 399 * 15_000, interval=15_000, range=300_000, n=400),     # general K2L
    "resets": dict(start=T0, end=T0 + 399 * 15_000, interval=15_000, range=300_000, n=400),     # flags / K2 hand-off
    "big": dict(start=T0, end=T0 + 1199 * 15_000, interval=60_000, range=3_600_000, n=1200),    # 240-sample windows
    "slow": dict(start=T0, end=T0 + 2999 * 1_000, interval=50_000, range=2_000_000, n=3000),     # > any ring
    "span24": dict(start=T0, end=T0 + 40 * 86_400_000, interval=6 * 3_600_000, range=2 * 86_400_000, n=240),
    "dup": dict(start=T0 + 5_000, end=T0 + 299 * 15_000, interval=15_000, range=10_000, n=600),  # sampled == 0
}


def make_zoo(layout, seed, n_series=30):
    """-> ts, val, offsets, query dict.  Series s carries recipe s % N_RECIPES."""
    L = LAYOUTS[layout]
    rng = np.random.default_rng(seed)
    ts_l, val_l, offs = [], [], [0]
    for s in range(n_series):
        n = L["n"] - int(rng.integers(0, L["n"] // 4))
        k = np.arange(n, dtype=np.int64)
        if layout in ("exact", "resets", "big"):
            t = T0 + k * 15_000
        elif layout == "jitter":
            t = T0 + k * 15_000 + rng.integers(0, 1000, n)
        elif layout == "slow":
            t = T0 + k * 1_000
        elif layout == "span24":
            t = T0 + k * 4 * 3_600_000 + rng.integers(0, 60_000, n)
        else:  # pairs of samples sharing one timestamp
            t = T0 + (k // 2) * 15_000
        if layout == "resets":
            t = t + rng.integers(0, 1000, n)
        v = recipe(s % N_RECIPES, n, rng)
        if layout == "resets":  # drops to (signed) zero: counter resets in every kind of series
            z = np.flatnonzero(rng.random(n) < 0.03)
            v[z] = np.where(z % 2 == 0, 0.0, -0.0)
        ts_l.append(t.astype(np.int64))
        val_l.append(v)
        offs.append(offs[-1] + n)
    q = {k: L[k] for k in ("start", "end", "interval", "range")}
    return np.concatenate(ts_l), np.concatenate(val_l), np.array(offs, np.uint64), q


def oracle_rescan(fn, q, ts, val, offsets, filter_nan=True, p0=0.0, p1=0.0, offset=0):
    """The oracle's flat driver (normalize, calculate_range, the all-empty veto, the UDF) with the counter correction
    rescanned for every window — the restatement the warp-per-series tiers are bit-identical to."""
    T = orc.num_steps(q["start"], q["end"], q["interval"])
    S = offsets.size - 1
    out = np.zeros((S, T))
    valid = np.zeros((S, T), bool)
    for s in range(S):
        o0, o1 = int(offsets[s]), int(offsets[s + 1])
        nts, nval = orc.normalize(ts[o0:o1], val[o0:o1], offset, filter_nan)
        off, ln, s2, e2 = orc.calculate_range(nts, q["start"], q["end"], q["interval"], q["range"])
        if off.size == 0 or not ln.any():
            continue
        ets = s2 + np.arange(off.size, dtype=np.int64) * q["interval"]
        r, v = orc.range_udf(fn, nts, nval, np.stack([off, ln], 1), ets, q["range"], p0, p1, rescan=True)
        k0 = (s2 - q["start"]) // q["interval"]
        for j in range(off.size):
            if 0 <= k0 + j < T and v[j]:
                out[s, k0 + j] = r[j]
                valid[s, k0 + j] = True
    return out, valid


def assert_special(got, gv, exp, ev, what, exact=False, nan_bits=True):
    """Validity bit-exact; +-Inf and the sign of zero exact; NaN by bits (or by class when nan_bits is False); other
    finite values bit-exact when `exact`, else within 1e-9 relative; null slots hold 0.0."""
    assert (gv == ev).all(), f"{what}: validity differs at {np.argwhere(gv != ev)[:5].tolist()}"
    g, e = got[ev], exp[ev]
    gb, eb = g.view(np.uint64), e.view(np.uint64)
    nan_e = np.isnan(e)
    assert (np.isnan(g) == nan_e).all(), f"{what}: NaN pattern differs at {np.argwhere(np.isnan(g) != nan_e)[:5].tolist()}"
    if nan_bits:
        bad = nan_e & (gb != eb)
        assert not bad.any(), f"{what}: {int(bad.sum())} NaNs differ in bits, first {gb[bad][:3]} vs {eb[bad][:3]}"
    pinned = np.isinf(e) | (e == 0.0)
    bad = pinned & (gb != eb)
    assert not bad.any(), f"{what}: {int(bad.sum())} infinities / zeros differ, first {g[bad][:3]} vs {e[bad][:3]}"
    assert not (np.isinf(g) & ~np.isinf(e)).any(), f"{what}: infinities where the oracle has finite values"
    fin = np.isfinite(e) & ~pinned
    if exact:
        bad = fin & (gb != eb)
    else:
        with np.errstate(invalid="ignore", over="ignore"):
            bad = fin & ~((g == e) | (np.abs(g - e) <= REL * np.maximum(np.abs(g), np.abs(e))))
    assert not bad.any(), f"{what}: {int(bad.sum())} mismatches, first {g[bad][:3]} vs {e[bad][:3]}"
    assert (got[~ev] == 0.0).all() and not np.signbit(got[~ev]).any(), f"{what}: null slots must hold +0.0"


# ---------------------------------------------------------------------------------------------------
# 1. every function x every tier x every layout
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fn", ALL_FNS)
def test_value_zoo_every_function_every_tier(ctxs, fn):
    from greptimedb_b200 import make_params
    p0, p1 = FN_PARAMS.get(fn, (0.0, 0.0))
    for li, layout in enumerate(LAYOUTS):
        ts, val, offsets, q = make_zoo(layout, 100 + li)
        S = offsets.size - 1
        p = make_params(fn, q["start"], q["end"], q["interval"], q["range"], param0=p0, param1=p1)
        op = orc.make_params(fn, q["start"], q["end"], q["interval"], q["range"], param0=p0, param1=p1)
        T = orc.num_steps(q["start"], q["end"], q["interval"])
        flat, flat_w = orc.range_query(op, ts, val, None, offsets, mode="flat", threads=4)
        flat_v = orc.valid_to_bool(flat_w, T)
        resc, resc_v = oracle_rescan(fn, q, ts, val, offsets, p0=p0, p1=p1)
        handed = {}
        for name, c in ctxs.items():
            out, valid, ets = c.range_eval(p, ts, val, offsets=offsets)
            handed[name] = c.last_warp_tier_series()
            slow = c.last_slow_series()
            gv = orc.valid_to_bool(valid, T)
            what = f"{fn} {layout} {name}"
            if name == "thread" and fn in COUNTERS:
                # K2T keeps the reference's sliding counter correction (inf - inf where the rescan adds); the series
                # it hands on take the rescanning tiers: each series matches one of the two restatements
                for s in range(S):
                    try:
                        assert_special(out[s:s + 1], gv[s:s + 1], flat[s:s + 1], flat_v[s:s + 1], f"{what} series {s}")
                    except AssertionError:
                        assert_special(out[s:s + 1], gv[s:s + 1], resc[s:s + 1], resc_v[s:s + 1], f"{what} series {s}",
                                       exact=fn == "rate")
            else:
                assert_special(out, gv, resc, resc_v, what, exact=fn in BIT_EXACT or fn == "rate")
                if fn not in COUNTERS:   # one restatement for everything but the counter correction
                    assert_special(out, gv, flat, flat_v, what + " (flat)", exact=fn in BIT_EXACT)
            # the layout reached the tier it targets
            if layout == "big":
                assert slow == 0, (what, slow)
            if layout == "slow":
                assert slow == S, (what, slow)
        if fn == "rate":
            for name in ("default", "uniform", "lean_flags"):
                if layout in ("exact", "jitter") or (layout == "resets" and name == "lean_flags"):
                    assert handed[name] < S, (layout, name, handed)       # the first tier kept series
            if layout == "resets":
                assert handed["default"] > 0, handed                        # resets leave the plain variant ...
                assert handed["lean_flags"] < handed["default"], handed     # ... the bit-word variant keeps more


@pytest.mark.parametrize("fn", ALL_FNS)
def test_value_zoo_with_nan_filter_off(ctx, fn):
    """need_filter_out_nan = false: NaN samples reach the functions.  Pass-through functions keep every bit, the
    arithmetic ones are compared by NaN class (see the module docstring)."""
    from greptimedb_b200 import make_params
    p0, p1 = FN_PARAMS.get(fn, (0.0, 0.0))
    for layout in ("exact", "jitter", "big"):
        ts, val, offsets, q = make_zoo(layout, 7)
        p = make_params(fn, q["start"], q["end"], q["interval"], q["range"], filter_nan=False, param0=p0, param1=p1)
        out, valid, ets = ctx.range_eval(p, ts, val, offsets=offsets)
        e_out, e_valid = oracle_rescan(fn, q, ts, val, offsets, filter_nan=False, p0=p0, p1=p1)
        assert_special(out, orc.valid_to_bool(valid, ets.size), e_out, e_valid, f"{fn} {layout} nan-off",
                       exact=fn in BIT_EXACT or fn == "rate", nan_bits=fn in PASS_THROUGH)


def test_value_zoo_through_udf_sid_column_and_pipelined_host_path(ctx):
    from greptimedb_b200 import make_params
    # the UDF entry point over explicit windows
    ts, val, offsets, q = make_zoo("jitter", 5, n_series=1)
    rng = np.random.default_rng(5)
    lo = rng.integers(0, ts.size - 40, 300)
    ranges = np.stack([lo, rng.integers(0, 40, 300)], 1).astype(np.uint32)
    ets = ts[lo] + 300_000
    for fn in ALL_FNS:
        p0, p1 = FN_PARAMS.get(fn, (0.0, 0.0))
        for kind in range(N_RECIPES):
            v = recipe(kind, ts.size, np.random.default_rng(kind))
            got, gv = ctx.range_udf(fn, ts, v, ranges, ets, 300_000, p0, p1)
            e, ev = orc.range_udf(fn, ts, v, ranges, ets, 300_000, p0, p1, rescan=True)
            assert_special(got, gv, e, ev, f"udf {fn} recipe {kind}", exact=fn in BIT_EXACT or fn == "rate",
                           nan_bits=fn in PASS_THROUGH)
    # range_eval_n with a series-id column
    ts, val, offsets, q = make_zoo("jitter", 6)
    S = offsets.size - 1
    sid = np.repeat(np.arange(S, dtype=np.uint32), np.diff(offsets).astype(np.int64))
    for fn in ("rate", "delta", "deriv", "stddev_over_time"):
        p = make_params(fn, q["start"], q["end"], q["interval"], q["range"])
        out, valid, ets = ctx.range_eval_n(p, ts, val, sid, None, S)
        e, ev = oracle_rescan(fn, q, ts, val, offsets)
        assert_special(out, orc.valid_to_bool(valid, ets.size), e, ev, f"sid {fn}", exact=fn == "rate")
    # > 6 M rows: the double-buffered host path, special series spread over every chunk
    S, N = 6500, 1000
    ts, val, sid = orc.synth_fill(0, S, N, T0, 15_000, 1000, 1, 0x5EED)
    rng = np.random.default_rng(8)
    for s in range(0, S, 53):
        val[s * N:(s + 1) * N] = recipe(s % N_RECIPES, N, rng)
    offsets = np.arange(S + 1, dtype=np.uint64) * N
    p = make_params("rate", T0, T0 + 999 * 15_000, 60_000, 300_000)
    op = orc.make_params("rate", T0, T0 + 999 * 15_000, 60_000, 300_000)
    e_out, e_valid = orc.range_query(op, ts, val, sid, offsets, threads=8)
    out, valid, ets = ctx.range_eval_n(p, ts, val, sid, None, S)
    assert_special(out, orc.valid_to_bool(valid, ets.size), e_out, orc.valid_to_bool(e_valid, ets.size), "pipelined")


# ---------------------------------------------------------------------------------------------------
# 2. by-label aggregate on special members
# ---------------------------------------------------------------------------------------------------
def _member_table():
    """Columns = every ordered pair and every single member of SPECIAL_MEMBERS, plus runs of all of them: group g of
    column c holds the members of that column, in series order."""
    M = SPECIAL_MEMBERS.size
    cols = [[a] for a in range(M)] + [[a, b] for a in range(M) for b in range(M)]
    rng = np.random.default_rng(3)
    cols += [list(rng.permutation(M)[:int(rng.integers(3, M + 1))]) for _ in range(200)]
    T, width = len(cols), max(len(c) for c in cols)
    vals = np.zeros((width, T))
    valid = np.zeros((width, T), bool)
    for k, c in enumerate(cols):
        vals[:len(c), k] = SPECIAL_MEMBERS[c]
        valid[:len(c), k] = True
    Tw = (T + 31) // 32
    pad = np.zeros((width, Tw * 32), bool)
    pad[:, :T] = valid
    return vals, np.packbits(pad, axis=1, bitorder="little").view(np.uint32).copy(), T


@pytest.mark.parametrize("agg", ["sum", "avg", "count", "min", "max", "stddev", "stdvar"])
def test_group_aggregate_on_special_members_is_bit_exact(ctx, agg):
    """Device twin of the oracle's total-order test: the by-label kernel folds members in series order like a single
    DataFusion partition, so every result — NaN bits, signed zeros and infinities included — equals the oracle's.
    Only stddev / stdvar of a group with a NaN member compare the NaN by class: which member's NaN the Welford
    update carries through on x86 depends on operand order inside each step, which is not restated."""
    vals, valid, T = _member_table()
    S = vals.shape[0]
    for gid in (np.zeros(S, np.uint32), (np.arange(S) % 3).astype(np.uint32)):
        G = int(gid.max()) + 1
        got, gc = ctx.group_aggregate(agg, vals, valid, gid, G)
        exp, ec = orc.group_aggregate(agg, vals, valid, gid, G)
        assert (gc == ec).all()
        bad = got.view(np.uint64) != exp.view(np.uint64)
        if agg in ("stddev", "stdvar"):
            nan_in = orc.group_aggregate("sum", np.isnan(vals).astype(np.float64), valid, gid, G)[0] > 0
            bad &= ~(nan_in & np.isnan(got) & np.isnan(exp))
        assert not bad.any(), (agg, int(bad.sum()), np.argwhere(bad)[:3].tolist(),
                               got[bad][:3].view(np.uint64), exp[bad][:3].view(np.uint64))


# ---------------------------------------------------------------------------------------------------
# 3. compositions that make the NaN sign visible
# ---------------------------------------------------------------------------------------------------
def _composition_series():
    """Counters in four jobs; some series make rate() NaN by arithmetic (windows whose samples share one timestamp:
    0 / 0; a counter at +Inf twice in a row: inf - inf) or +-Inf (differences that overflow).
    -> ts, val, offsets, job of every series, query"""
    N = 200
    k = np.arange(N, dtype=np.int64)
    rng = np.random.default_rng(21)
    series = []
    for job in range(4):
        for m in range(4):
            t = T0 + k * 15_000 + rng.integers(0, 1000, N)
            v = np.cumsum(rng.random(N) * 10)
            kind = (job + m) % 4
            if kind == 1:        # one pair of samples per 10 minutes, both at the same timestamp
                t = T0 + (k // 2) * 600_000
            elif kind == 2:      # +Inf twice in a row, now and then
                for j in range(5, N - 2, 37):
                    v[j:j + 2] = np.inf
            elif kind == 3:      # overflowing differences: +Inf for one series, -Inf for the other
                v = np.where(k % 2 == 0, -1e308, 1e308) if m % 2 else np.where(k % 2 == 0, 1e308, -1e308)
            series.append((job, t.astype(np.int64), v.astype(np.float64)))
    ts = np.concatenate([s[1] for s in series])
    val = np.concatenate([s[2] for s in series])
    offsets = np.concatenate([[0], np.cumsum([s[1].size for s in series])]).astype(np.uint64)
    jobs = np.array([s[0] for s in series], np.uint32)
    q = dict(start=T0, end=T0 + 199 * 15_000, interval=15_000, range=300_000)
    return ts, val, offsets, jobs, q


def test_max_min_by_over_rate_see_the_sign_of_computed_nans(ctx):
    import pyarrow as pa
    import torch
    from greptimedb_b200 import make_params
    from greptimedb_b200.plan import PromRangeExec
    ts, val, offsets, jobs, q = _composition_series()
    S, G = offsets.size - 1, int(jobs.max()) + 1
    T = orc.num_steps(q["start"], q["end"], q["interval"])
    # the warp-per-series tiers rescan the counter correction (see DESIGN.md on +Inf counters)
    e_out, e_vb = oracle_rescan("rate", q, ts, val, offsets)
    Tw = (T + 31) // 32
    pad = np.zeros((S, Tw * 32), bool)
    pad[:, :T] = e_vb
    e_valid = np.packbits(pad, axis=1, bitorder="little").view(np.uint32).copy()
    e_nan = np.isnan(e_out) & e_vb
    assert (e_nan & np.signbit(e_out)).any() and np.isinf(e_out).any()
    p = make_params("rate", q["start"], q["end"], q["interval"], q["range"])
    out, valid, _ = ctx.range_eval(p, ts, val, offsets=offsets)
    names = [f"job{j}" for j in range(G)]
    # plan layer input: rows in scan order (sorted by job, then instance)
    inst = np.arange(S) % 4
    b = pa.record_batch([pa.array(ts, pa.timestamp("ms")), pa.array(val),
                         pa.array(np.repeat([names[j] for j in jobs], np.diff(offsets).astype(np.int64))),
                         pa.array(np.repeat([f"i{i}" for i in inst], np.diff(offsets).astype(np.int64)))],
                        names=["ts", "v", "job", "instance"])
    for agg in ("max", "min"):
        exp, ec = orc.group_aggregate(agg, e_out, e_valid, jobs, G)
        got, gc = ctx.group_aggregate(agg, out, valid, jobs, G)
        assert (gc == ec).all()
        assert (got.view(np.uint64) == exp.view(np.uint64)).all(), (agg, np.argwhere(got.view(np.uint64) != exp.view(np.uint64))[:4].tolist())
        ex = PromRangeExec(ctx, "prom_rate", q["start"], q["end"], q["interval"], q["range"], "ts", "v",
                           ["job", "instance"], aggregate=agg, by_columns=["job"])
        ex.push(b)
        res = ex.execute()
        rows = {(j, int(t.timestamp() * 1000)): v for j, t, v in zip(res.column(0).to_pylist(), res.column(1).to_pylist(),
                                                                     res.column(2).to_pylist())}
        want = {(names[g], q["start"] + k * q["interval"]): exp[g, k] for g in range(G) for k in range(T) if ec[g, k]}
        assert set(rows) == set(want), agg
        for key, e in want.items():
            assert np.float64(rows[key]).view(np.uint64) == np.float64(e).view(np.uint64), (agg, key, rows[key], e)
    # sum by, fused into the range stage: counts exact, Inf / NaN class exact
    dev = torch.device("cuda:0")
    e_sum, e_cnt = orc.group_aggregate("sum", e_out, e_valid, jobs, G)
    assert np.isinf(e_sum).any() and np.isnan(e_sum).any()
    d_ts, d_val = torch.from_numpy(ts).to(dev), torch.from_numpy(val).to(dev)
    d_off = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    d_gid = torch.from_numpy(jobs.astype(np.int32)).to(dev)
    ctx.use_own_stream()
    torch.cuda.synchronize()
    ix = ctx.group_index_create_dev(d_gid, S, G)
    try:
        gsum = torch.zeros(G * T, dtype=torch.float64, device=dev)
        gcnt = torch.zeros(G * T, dtype=torch.int32, device=dev)
        ctx.range_group_sum_indexed_dev(p, d_ts, d_val, d_off, ts.size, S, ix, 0, G, gsum, gcnt)
        ctx.sync()
    finally:
        ctx.group_index_destroy(ix)
    got, cnt = gsum.cpu().numpy().reshape(G, T), gcnt.cpu().numpy().view(np.uint32).reshape(G, T)
    assert (cnt == e_cnt).all()
    assert (np.isnan(got) == np.isnan(e_sum)).all()
    assert (got[np.isinf(e_sum)] == e_sum[np.isinf(e_sum)]).all() and (np.isinf(got) == np.isinf(e_sum)).all()
    fin = np.isfinite(e_sum) & (e_cnt > 0)
    assert (np.abs(got[fin] - e_sum[fin]) <= REL * np.abs(e_sum[fin])).all()


def test_histogram_fold_with_infinite_and_nan_bucket_rates(ctx):
    """Non-finite bucket counters take the previous bucket's value (histogram_fold.rs:1074-1092); rows without a
    +Inf bucket are the constant NaN.  Device fold == the row-literal fold, NaN bits included."""
    import torch
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(12)
    H, B, T = 12, 6, 40
    bounds = [0.1, 0.5, 1.0, 5.0, 10.0, np.inf]
    S = H * B
    rates = np.cumsum(rng.random((H, B, T)), axis=1).reshape(S, T)
    pick = rng.random((S, T))
    rates[pick < 0.05] = np.inf
    rates[(pick >= 0.05) & (pick < 0.08)] = -np.inf
    rates[(pick >= 0.08) & (pick < 0.11)] = POS_NAN
    rates[(pick >= 0.11) & (pick < 0.14)] = NEG_NAN
    Tw = (T + 31) // 32
    keep = rng.random((S, T)) > 0.05
    keep[np.arange(S) % B == B - 1] |= (np.arange(T) % 3 != 0)[None, :]
    pad = np.zeros((S, Tw * 32), bool)
    pad[:, :T] = keep
    valid = np.packbits(pad, axis=1, bitorder="little").view(np.uint32).copy()
    lit = []
    for h in range(H):
        for k in range(T):
            lit += [((h,), k, "+Inf" if np.isinf(bounds[b]) else repr(bounds[b]), rates[h * B + b, k])
                    for b in range(B) if keep[h * B + b, k]]
    exp = {(t[0], k): v for t, k, v in orc.histogram_fold_rows(lit, 0.9)}
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    hist_off = (np.arange(H + 1) * B).astype(np.int32)
    out = torch.zeros(H * T, dtype=torch.float64, device=dev)
    ov = torch.zeros(H * Tw, dtype=torch.int32, device=dev)
    ctx.use_own_stream()
    torch.cuda.synchronize()
    ctx.histogram_fold_dev(0.9, d(hist_off), d(np.arange(S, dtype=np.int32)), d(np.tile(bounds, H)), H, d(rates),
                           d(valid.astype(np.int32)), T, out, ov)
    ctx.sync()
    got, gv = out.cpu().numpy().reshape(H, T), ov.cpu().numpy().view(np.uint32).reshape(H, Tw)
    n_nan = 0
    for h in range(H):
        for k in range(T):
            has = bool((gv[h, k >> 5] >> (k & 31)) & 1)
            assert has == ((h, k) in exp), (h, k)
            if has:
                e, g = np.float64(exp[(h, k)]), got[h, k]
                n_nan += int(np.isnan(e))
                assert g.view(np.uint64) == e.view(np.uint64), (h, k, g, e)
    assert n_nan > 0


# ---------------------------------------------------------------------------------------------------
# 4. device twin of the sum(rate) table (tql/range.result, the config-3 query shape)
# ---------------------------------------------------------------------------------------------------
def _sum_rate_cases():
    import json
    with open(os.path.join(os.path.dirname(__file__), "golden", "reference_sum_rate_vectors.json")) as f:
        return json.load(f)


SUM_RATE = _sum_rate_cases()


@pytest.mark.parametrize("case", SUM_RATE["cases"], ids=lambda c: c["name"])
def test_sum_rate_reference_tables_on_the_device(ctx, case):
    """Every printed value of range.result, to the last digit, through the fused sum by and through the plan layer."""
    import pyarrow as pa
    import torch
    from greptimedb_b200 import make_params
    from greptimedb_b200.plan import PromRangeExec
    keep = [s for s in SUM_RATE["series"] if all(s[k] == v for k, v in case["filter"].items())]
    if not keep:
        assert case["expected"] == []
        return
    ts = np.concatenate([np.array(s["ts"], np.int64) for s in keep])
    val = np.concatenate([np.array(s["val"], np.float64) for s in keep])
    lens = [len(s["ts"]) for s in keep]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    keys = sorted({tuple(s[t] for t in case["by"]) for s in keep})
    gid = np.array([keys.index(tuple(s[t] for t in case["by"])) for s in keep], np.uint32)
    S, G = len(keep), len(keys)
    T = orc.num_steps(case["start"], case["end"], case["interval"])
    scale = case.get("scale", 1.0)
    p = make_params("rate", case["start"], case["end"], case["interval"], case["range"])
    dev = torch.device("cuda:0")
    ctx.use_own_stream()
    torch.cuda.synchronize()
    ix = ctx.group_index_create_dev(torch.from_numpy(gid.astype(np.int32)).to(dev), S, G)
    try:
        gsum = torch.zeros(G * T, dtype=torch.float64, device=dev)
        gcnt = torch.zeros(G * T, dtype=torch.int32, device=dev)
        ctx.range_group_sum_indexed_dev(p, torch.from_numpy(ts).to(dev), torch.from_numpy(val).to(dev),
                                        torch.from_numpy(offsets.astype(np.int64)).to(dev), ts.size, S, ix, 0, G, gsum, gcnt)
        ctx.sync()
    finally:
        ctx.group_index_destroy(ix)
    gs, gc = gsum.cpu().numpy().reshape(G, T), gcnt.cpu().numpy().view(np.uint32).reshape(G, T)
    fused = [[dict(zip(case["by"], keys[g])), case["start"] + k * case["interval"], float(gs[g, k]) * scale]
             for g in range(G) for k in range(T) if gc[g, k]]
    assert fused == case["expected"]
    # the plan layer: rows in scan order (sorted by the tag tuple), the sum by the case's labels
    tags = ["host", "service"]
    order = sorted(range(S), key=lambda s: tuple(keep[s][t] for t in tags))
    rows = np.concatenate([np.arange(int(offsets[s]), int(offsets[s + 1])) for s in order])
    cols = [pa.array(ts[rows], pa.timestamp("ms")), pa.array(val[rows])]
    cols += [pa.array(np.repeat([keep[s][t] for s in order], [lens[s] for s in order])) for t in tags]
    ex = PromRangeExec(ctx, "prom_rate", case["start"], case["end"], case["interval"], case["range"], "ts", "val", tags,
                       aggregate="sum", by_columns=case["by"])
    ex.push(pa.record_batch(cols, names=["ts", "val"] + tags))
    res = ex.execute()
    by_cols = [res.column(res.schema.get_field_index(t)).to_pylist() for t in case["by"]]
    t_col = [int(t.timestamp() * 1000) for t in res.column(res.schema.get_field_index("ts")).to_pylist()]
    v_col = res.column(res.num_columns - 1).to_pylist()
    plan = [[dict(zip(case["by"], [c[i] for c in by_cols])), t_col[i], v_col[i] * scale] for i in range(res.num_rows)]
    assert plan == case["expected"]
