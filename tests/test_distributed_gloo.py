"""World-size-2 gloo test (CPU) of the N>1 host logic: hash-sharding of series, per-rank partial
(sum, cnt), one all-reduce, finalize == unsharded result.  The per-shard compute is the oracle here
(the CUDA kernels need a GPU; tests/test_gpu_parity.py covers them)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from greptimedb_b200 import distributed as D
    from oracle import oracle as orc
    S, N, G, T0 = 96, 200, 7, 1_700_000_000_000
    ts, val, sid = orc.synth_fill(0, S, N, T0, 15_000, 1000, 1, 0x5EED)
    offsets = np.arange(S + 1, dtype=np.uint64) * N
    gid = (D.mix32(np.arange(S, dtype=np.uint32)) % np.uint32(G)).astype(np.uint32)
    p = orc.make_params("rate", T0, T0 + (N - 1) * 15_000, 15_000, 300_000)
    owned, rows, loffs = D.shard_rows(offsets, world, rank)
    out, valid = orc.range_query(p, ts[rows], val[rows], None, loffs)
    psum, pcnt = orc.group_aggregate("sum", out, valid, gid[owned], G)
    st, ct = torch.from_numpy(psum), torch.from_numpy(pcnt.astype(np.int64))
    D.allreduce_group_partials(st, ct)
    res = D.finalize_host("avg", st.numpy(), ct.numpy())
    full_out, full_valid = orc.range_query(p, ts, val, sid, offsets)
    worst = 0.0
    ok_all = True
    # min / max: groups missing on one rank must not poison the extreme; stddev / stdvar: (cnt, mean, M2) states merge
    for agg in ("min", "max", "stddev", "stdvar"):
        e_val, e_cnt = orc.group_aggregate(agg, full_out, full_valid, gid, G)
        if agg in ("min", "max"):
            pv, pc = orc.group_aggregate(agg, out, valid, gid[owned], G)
            vt, ctt = torch.from_numpy(pv.copy()), torch.from_numpy(pc.astype(np.int64))
            D.merge_partials(agg, vt, ctt)
            got = vt.numpy()
        else:
            m2, pc, mean = D.partial_state_host(agg, out, valid, gid[owned], G)
            vt, ctt, mt = torch.from_numpy(m2), torch.from_numpy(pc), torch.from_numpy(mean)
            D.merge_partials(agg, vt, ctt, mt)
            n = np.maximum(ctt.numpy(), 1)
            got = vt.numpy() / n if agg == "stdvar" else np.sqrt(vt.numpy() / n)
            got[ctt.numpy() == 0] = 0.0
        ok_all = ok_all and bool((ctt.numpy() == e_cnt).all())
        m = e_cnt > 0
        rel_a = np.abs(got[m] - e_val[m]) / np.maximum(np.abs(e_val[m]), 1e-300)
        # variance of near-constant samples cancels: compare absolutely against the scale of the data there
        scale = np.abs(full_out).max()
        bad = (rel_a > 1e-9) & (np.abs(got[m] - e_val[m]) > 1e-9 * scale)
        ok_all = ok_all and not bool(bad.any())
        if agg in ("min", "max"):
            ok_all = ok_all and bool((got[m] == e_val[m]).all())   # extremes are exact
    if rank == 0:
        e_avg, e_cnt = orc.group_aggregate("avg", full_out, full_valid, gid, G)
        ok_cnt = bool((ct.numpy() == e_cnt).all()) and ok_all
        rel = np.abs(res - e_avg) / np.maximum(np.abs(e_avg), 1e-300)
        q.put((ok_cnt, float(rel[e_cnt > 0].max()), int(owned.size)))
    else:
        q.put((ok_all, 0.0, int(owned.size)))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_partials_allreduce_equals_unsharded():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(r[0] for r in results)
    assert max(r[1] for r in results) <= 1e-9          # summation order differs across shards: 1e-9 rel, like the reference
    assert sum(r[2] for r in results) == 96              # every series owned exactly once


def special_members():
    """Group members whose order only f64::total_cmp settles: both zeros, both infinities, NaNs of both signs and with a
    payload, a subnormal and values next to overflow."""
    bits = [0x0000000000000000, 0x8000000000000000, 0x7FF0000000000000, 0xFFF0000000000000, 0x7FF8000000000000,
            0xFFF8000000000000, 0x7FF0000000000002, 0x0000000000000001]
    return np.concatenate([np.array(bits, np.uint64).view(np.float64), [1e308, -1e308]])


def _minmax_worker(rank, world, port, q):
    """Every column is one placement of the members: digit m of the column index (base world + 1) is the rank that
    holds member m, or `world` when no rank has it.  Each rank reduces the members it holds, then the ranks merge."""
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from greptimedb_b200 import distributed as D
    from oracle import oracle as orc
    members = special_members()
    M = members.size
    C = (world + 1) ** M
    owner = (np.arange(C)[None, :] // (world + 1) ** np.arange(M)[:, None]) % (world + 1)   # [M x C]
    vals = np.repeat(members[:, None], C, axis=1)
    gid = np.zeros(M, np.uint32)

    def words(mask):
        pad = np.zeros((M, (C + 31) // 32 * 32), bool)
        pad[:, :C] = mask
        return np.packbits(pad, axis=1, bitorder="little").view(np.uint32)

    failures = []
    for agg in ("min", "max"):
        e_val, e_cnt = orc.group_aggregate(agg, vals, words(owner < world), gid, 1)
        pv, pc = orc.group_aggregate(agg, vals, words(owner == rank), gid, 1)
        vt, ct = torch.from_numpy(pv.copy()), torch.from_numpy(pc.astype(np.int64))
        D.merge_partials(agg, vt, ct)
        got = vt.numpy()
        bad = (got.view(np.uint64) != e_val.view(np.uint64)) | (ct.numpy() != e_cnt)
        if bad.any():
            c = int(np.flatnonzero(bad[0])[0])
            failures.append(f"{agg}: {int(bad.sum())} of {C} placements differ, first owners {owner[:, c].tolist()}: "
                            f"{got[0, c].view(np.uint64):#018x} vs {e_val[0, c].view(np.uint64):#018x}")
    q.put((rank, failures))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_minmax_merge_follows_the_total_order_for_every_placement(world):
    """min / max by (..) merged across ranks equals the single-rank by-label result bit for bit, wherever the special
    members sit: f64 min / max on the collective would depend on the rank order for NaNs and signed zeros."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_minmax_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert [f for _, fs in results for f in fs] == []


def test_total_key_orders_and_round_trips():
    from greptimedb_b200 import distributed as D
    members = special_members()
    extra = np.array([-5e-324, 2.2250738585072014e-308, -2.2250738585072009e-308, 1.0, -1.0])
    v = np.concatenate([members, extra])
    key = D.total_key(torch.from_numpy(v.copy()).view(torch.int64))
    assert (D.total_key(key).view(torch.float64).numpy().view(np.uint64) == v.view(np.uint64)).all()
    order = np.argsort(key.numpy(), kind="stable")
    s = v[order].view(np.uint64)
    expect = np.array([0xFFF8000000000000, 0xFFF0000000000000], np.uint64)
    assert (s[:2] == expect).all() and (s[-3:] == np.array([0x7FF0000000000000, 0x7FF0000000000002,
                                                             0x7FF8000000000000], np.uint64)).all()
    finite = v[order][2:-3]
    assert (np.diff(finite) >= 0).all()
    z = np.flatnonzero(finite == 0.0)
    assert np.signbit(finite[z[0]]) and not np.signbit(finite[z[1]])


def test_shard_function_is_a_partition():
    from greptimedb_b200 import distributed as D
    ids = np.arange(10_000, dtype=np.uint32)
    for world in (1, 2, 4, 8):
        own = D.shard_of_series(ids, world)
        assert own.min() >= 0 and own.max() < world
        counts = np.bincount(own, minlength=world)
        assert counts.sum() == ids.size and counts.min() > 0.8 * ids.size / world
