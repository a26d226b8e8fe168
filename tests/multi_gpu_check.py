"""Multi-rank check of the library's own collective path (run under torchrun, one rank per GPU; started by
tests/test_multi_gpu.py when at least two GPUs are visible):

  * sum by (..)(rate(..)) with series hash-sharded over the ranks, through b2p_range_group_sum_allreduce_dev (fused
    partials, tiles all-reduced on the library's NCCL communicator) == the oracle on the unsharded data;
  * b2p_allreduce_partials_dev for min / max (bit for bit, with NaNs of both signs, signed zeros and infinities among
    the members) and for the (count, mean, M2) states of stddev / stdvar == the oracle.
torch.distributed only carries the 128-byte communicator id and the final verdict."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from greptimedb_b200 import Context, make_params
    from greptimedb_b200 import distributed as D
    from oracle import oracle as orc
    ctx = Context(local)
    ctx.use_own_stream()
    box = [ctx.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    ctx.comm_init(box[0], world, rank)

    S, N, G, T0 = 2400, 500, 61, 1_700_000_000_000
    ts, val, sid = orc.synth_fill(0, S, N, T0, 15_000, 1000, 1, 0x5EED)
    val[77::4001] = np.nan
    offsets = np.arange(S + 1, dtype=np.uint64) * N
    gid = (D.mix32(np.arange(S, dtype=np.uint32)) % np.uint32(G)).astype(np.uint32)
    owned, rows, loffs = D.shard_rows(offsets, world, rank)
    T = N
    p = make_params("rate", T0, T0 + (N - 1) * 15_000, 15_000, 300_000)
    op = orc.make_params("rate", T0, T0 + (N - 1) * 15_000, 15_000, 300_000)
    full_out, full_valid = orc.range_query(op, ts, val, sid, offsets, threads=4)
    ok, worst = True, 0.0

    d_ts, d_val = torch.from_numpy(ts[rows]).to(dev), torch.from_numpy(val[rows]).to(dev)
    d_off = torch.from_numpy(loffs.astype(np.int64)).to(dev)
    d_gid = torch.from_numpy(gid[owned].astype(np.int32)).to(dev)
    torch.cuda.synchronize()
    ns = int(owned.size)
    ix = ctx.group_index_create_dev(d_gid, ns, G)
    e_sum, e_cnt = orc.group_aggregate("sum", full_out, full_valid, gid, G)
    for tiles in (1, 3):
        gsum = torch.zeros(G * T, dtype=torch.float64, device=dev)
        gcnt = torch.zeros(G * T, dtype=torch.int32, device=dev)
        ctx.range_group_sum_allreduce_dev(p, d_ts, d_val, d_off, rows.size, ns, ix, tiles, gsum, gcnt)
        ctx.sync()
        got, cnt = gsum.cpu().numpy().reshape(G, T), gcnt.cpu().numpy().view(np.uint32).reshape(G, T)
        ok = ok and bool((cnt == e_cnt).all())
        rel = np.abs(got - e_sum) / np.maximum(np.abs(e_sum), 1e-300)
        worst = max(worst, float(rel[e_cnt > 0].max()))
    ctx.group_index_destroy(ix)

    # min / max / stddev / stdvar: per-rank partial state from the by-label kernel, merged by the library
    out = torch.zeros(ns * T, dtype=torch.float64, device=dev)
    valid = torch.zeros(ns * ((T + 31) // 32), dtype=torch.int32, device=dev)
    ctx.range_eval_dev(p, d_ts, d_val, d_off, rows.size, ns, out, valid)
    ctx.sync()
    scale = float(np.abs(full_out).max())
    # min / max also merge NaNs of both signs, signed zeros and infinities: a quarter of the cells of every series hold
    # one of them, so most (group, step) cells see several on different ranks, where only the total order decides
    spec = np.concatenate([np.array([0x0, 0x8000000000000000, 0x7FF0000000000000, 0xFFF0000000000000,
                                     0x7FF8000000000000, 0xFFF8000000000000, 0x7FF0000000000002, 0x1],
                                    np.uint64).view(np.float64), [1e308, -1e308]])

    def specialize(a, series):
        a = a.copy()
        k = np.arange(T)[None, :] + series[:, None]
        hit = (k + 2 * series[:, None]) % 4 == 0
        a[hit] = spec[(k % spec.size)[hit]]
        return a

    full_mm = specialize(full_out, np.arange(S))
    out_mm = torch.from_numpy(specialize(out.cpu().numpy().reshape(ns, T), owned).reshape(-1)).to(dev)
    for agg in ("min", "max", "stddev", "stdvar", "avg"):
        mm = agg in ("min", "max")
        e_val, e_c = orc.group_aggregate(agg, full_mm if mm else full_out, full_valid, gid, G)
        pv = torch.zeros(G * T, dtype=torch.float64, device=dev)
        pc = torch.zeros(G * T, dtype=torch.int32, device=dev)
        pm = torch.zeros(G * T, dtype=torch.float64, device=dev)
        var = agg in ("stddev", "stdvar")
        ctx.group_aggregate_partial_dev(agg, out_mm if mm else out, valid, d_gid, ns, G, T, pv, pc, pm if var else None)
        ctx.allreduce_partials_dev(agg, pv, pc, pm if var else None, G * T)
        if agg in ("stddev", "stdvar", "avg"):
            ctx.group_finalize_dev(agg, pv, pc, G * T)
        ctx.sync()
        got, cnt = pv.cpu().numpy().reshape(G, T), pc.cpu().numpy().view(np.uint32).reshape(G, T)
        ok = ok and bool((cnt == e_c).all())
        m = e_c > 0
        if mm:
            ok = ok and bool((got.view(np.uint64)[m] == e_val.view(np.uint64)[m]).all())
        else:
            err = np.abs(got[m] - e_val[m])
            bad = (err > 1e-9 * np.maximum(np.abs(e_val[m]), 1e-300)) & (err > 1e-9 * scale)
            ok = ok and not bool(bad.any())
    ctx.comm_destroy()
    ctx.close()
    verdict = torch.tensor([1.0 if (ok and worst <= 1e-9) else 0.0], device=dev)
    dist.all_reduce(verdict, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"MULTI_GPU_CHECK world={world} ok={bool(verdict.item() == 1.0)} worst_rel={worst:.3e}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if verdict.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
