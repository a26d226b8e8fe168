"""Multi-GPU plumbing for the by-label aggregate: series are hash-sharded across ranks (one process
per GPU), every rank reduces its shard into [n_groups x T] (sum f64, cnt u32) partials, and ONE
all-reduce per buffer merges them — the analogue of the reference's __sum_state (datanode) /
__sum_merge (frontend) split, src/query/src/dist_plan/commutativity.rs:85-113,158-176.
rate() alone needs no collective.  torch.distributed is plumbing only (NCCL over NVLink on GPUs,
gloo in the CPU tests); the arithmetic before and after the collective is in libb200promql.so.
"""
from __future__ import annotations

import numpy as np


def mix32(x: np.ndarray) -> np.ndarray:
    """murmur3 fmix32 — the series -> shard / series -> synthetic group hash."""
    x = np.asarray(x, dtype=np.uint32).copy()
    x ^= x >> np.uint32(16)
    x *= np.uint32(0x85EBCA6B)
    x ^= x >> np.uint32(13)
    x *= np.uint32(0xC2B2AE35)
    x ^= x >> np.uint32(16)
    return x


def shard_of_series(series_id: np.ndarray, world: int) -> np.ndarray:
    """Owner rank of every (dense, global) series id: hash(series key) mod n_gpu (SURVEY §8e)."""
    return (mix32(series_id) % np.uint32(world)).astype(np.int64)


def shard_rows(offsets: np.ndarray, world: int, rank: int):
    """Rows and local offsets of the series owned by `rank`.
    -> (series_idx[int64] global ids owned, row_index[int64] gather list, local_offsets[uint64])"""
    offsets = np.asarray(offsets, dtype=np.uint64)
    n_series = offsets.size - 1
    owned = np.flatnonzero(shard_of_series(np.arange(n_series, dtype=np.uint32), world) == rank)
    lens = (offsets[owned + 1] - offsets[owned]).astype(np.int64)
    local_offsets = np.zeros(owned.size + 1, np.uint64)
    np.cumsum(lens, out=local_offsets[1:].view(np.int64))
    rows = np.concatenate([np.arange(int(offsets[s]), int(offsets[s + 1]), dtype=np.int64) for s in owned]) \
        if owned.size else np.zeros(0, np.int64)
    return owned, rows, local_offsets


def allreduce_group_partials(sum_t, cnt_t, group=None):
    """In-place SUM all-reduce of the (sum, cnt) partial matrices (torch tensors, CPU/gloo or CUDA/NCCL).
    cnt is reduced as int64 on gloo-safe dtypes; on CUDA it stays int32."""
    import torch
    import torch.distributed as dist
    dist.all_reduce(sum_t, op=dist.ReduceOp.SUM, group=group)
    if cnt_t.dtype in (torch.int32, torch.int64):
        dist.all_reduce(cnt_t, op=dist.ReduceOp.SUM, group=group)
    else:
        tmp = cnt_t.to(torch.int64)
        dist.all_reduce(tmp, op=dist.ReduceOp.SUM, group=group)
        cnt_t.copy_(tmp.to(cnt_t.dtype))
    return sum_t, cnt_t


def finalize_host(agg: str, sum_a: np.ndarray, cnt_a: np.ndarray) -> np.ndarray:
    """Host mirror of b2p_group_finalize_dev (used by the gloo tests): avg = sum/cnt, count = cnt."""
    out = sum_a.copy()
    nz = cnt_a > 0
    if agg == "avg":
        out[nz] = sum_a[nz] / cnt_a[nz]
    elif agg == "count":
        out = cnt_a.astype(np.float64)
    out[~nz] = 0.0
    return out


def total_key(bits):
    """f64::total_cmp key of float64 values viewed as int64 (torch tensor): an int64 whose signed order is the total
    order of the floats (-NaN < -inf < ... < -0.0 < +0.0 < ... < +inf < +NaN).  The map is its own inverse."""
    return bits ^ ((bits >> 63) & 0x7FFFFFFFFFFFFFFF)


def merge_partials(agg: str, val_t, cnt_t, mean_t=None, group=None):
    """Host mirror of b2p_allreduce_partials_dev (same formulas, torch.distributed instead of the library's NCCL
    communicator; used by the gloo tests): in-place merge of every rank's by-label partials.
      sum / avg / count : val and cnt are added                       (commutativity.rs:85-113)
      min / max         : val is reduced as total-order keys (int64 min / max), so NaNs of either sign and signed
                          zeros merge like the single-rank by-label min / max (f64 min / max would depend on the
                          rank order there); groups absent on a rank (cnt == 0) hold the neutral key (INT64_MAX /
                          INT64_MIN), cnt is added, groups absent everywhere read 0.0 again
      stddev / stdvar   : per-rank (cnt, mean, M2 = val) states; global mean from an all-reduce of cnt * mean,
                          M2 = sum_r [M2_r + cnt_r (mean_r - mean)^2]  (commutativity.rs:158-191)"""
    import torch
    import torch.distributed as dist
    cnt64 = cnt_t.to(torch.int64)
    if agg in ("min", "max"):
        key = total_key(val_t.contiguous().view(torch.int64))
        key[cnt64 == 0] = torch.iinfo(torch.int64).max if agg == "min" else torch.iinfo(torch.int64).min
        dist.all_reduce(key, op=dist.ReduceOp.MIN if agg == "min" else dist.ReduceOp.MAX, group=group)
        dist.all_reduce(cnt64, op=dist.ReduceOp.SUM, group=group)
        val_t.copy_(total_key(key).view(torch.float64))
        val_t[cnt64 == 0] = 0.0
    elif agg in ("stddev", "stdvar"):
        cnt_r = cnt64.clone()
        wsum = cnt_r.to(torch.float64) * mean_t
        dist.all_reduce(wsum, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(cnt64, op=dist.ReduceOp.SUM, group=group)
        mg = torch.where(cnt64 > 0, wsum / cnt64.clamp_min(1).to(torch.float64), torch.zeros_like(wsum))
        d = mean_t - mg
        val_t.copy_(torch.where(cnt_r > 0, val_t + cnt_r.to(torch.float64) * d * d, torch.zeros_like(val_t)))
        mean_t.copy_(mg)
        dist.all_reduce(val_t, op=dist.ReduceOp.SUM, group=group)
    else:
        dist.all_reduce(val_t, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(cnt64, op=dist.ReduceOp.SUM, group=group)
    cnt_t.copy_(cnt64.to(cnt_t.dtype))
    return val_t, cnt_t


def partial_state_host(agg: str, vals: np.ndarray, valid: np.ndarray, gid: np.ndarray, n_groups: int):
    """Host mirror of b2p_group_aggregate_partial_dev for stddev / stdvar: (M2, cnt, mean) per (group, step), Welford in
    series order like the by-label kernel."""
    S, T = vals.shape
    Tw = valid.shape[1]
    m2 = np.zeros((n_groups, T))
    mean = np.zeros((n_groups, T))
    cnt = np.zeros((n_groups, T), np.int64)
    bits = ((valid[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(S, Tw * 32)[:, :T].astype(bool)
    for s in range(S):
        g = int(gid[s])
        if g >= n_groups:
            continue
        k = np.flatnonzero(bits[s])
        x = vals[s, k]
        n1 = cnt[g, k] + 1.0
        d1 = x - mean[g, k]
        nm = d1 / n1 + mean[g, k]
        m2[g, k] += d1 * (x - nm)
        mean[g, k] = nm
        cnt[g, k] += 1
    return m2, cnt, mean
