"""Checks of bench.py's contract pieces.  Without a GPU: the committed ncu traffic file carries the kernel variants the
JSON line's roofline.traffic is read from, the reference arm (--impl reference: the oracle port timed on the host cores)
prints one JSON line with the keys its readers use, and its --dump-outputs files hold the oracle's results.  On a GPU:
--steps sets the timed steps of every timed path and --dump-outputs holds what they computed, the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T0, SCRAPE, SEED = 1_700_000_000_000, 15_000, 0x5EED


def _bench(*args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def _load_dump(d):
    files = sorted(os.listdir(d))
    arrays = {f[:-4]: np.load(os.path.join(d, f)) for f in files}
    assert all(f.endswith(".npy") for f in files)
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(os.path.getsize(os.path.join(d, f)) for f in files) <= 64_000_000
    return arrays


def _oracle_rows(rows, jitter_ms):
    """rate(x[5m]) at a 15 s step of the bench's synthetic series `rows` (global ids, 1000 samples each)
    -> (out [rows x T], validity words, validity as 0/1)."""
    from oracle import oracle as orc
    n = 1000
    parts = [orc.synth_fill(int(r), 1, n, T0, SCRAPE, jitter_ms, 0, SEED) for r in rows]
    ts = np.concatenate([p[0] for p in parts])
    val = np.concatenate([p[1] for p in parts])
    offsets = np.arange(len(rows) + 1, dtype=np.uint64) * n
    p = orc.make_params("rate", T0, T0 + (n - 1) * SCRAPE, SCRAPE, 300_000)
    out, valid = orc.range_query(p, ts, val, None, offsets, mode="faithful", threads=2)
    return out, valid, orc.valid_to_bool(valid, n).astype(np.float32)


def _rows(a):
    r = a.astype(np.int64)
    assert (r == a).all() and (np.diff(r) > 0).all()
    return r


def test_committed_traffic_file_has_the_kernel_variants_the_bench_reads():
    sys.path.insert(0, ROOT)
    import bench
    for key in ("range_lean_kernel", "range_lean_kernel_uniform"):
        per_sample, src = bench.load_traffic(key)
        assert per_sample is not None and src, key
        # ts 8 + val 8 read, 8 B + 1 bit written per step (steps ~ samples in config 2): ~24 B per input sample
        assert 20.0 < per_sample < 30.0, (key, per_sample)


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"]


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs on the reference arm: a seeded sample of the rows of the last timed step's [S x T] rate() result,
    float files only, equal to the oracle recomputed on the same series."""
    d = _bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    a = _load_dump(tmp_path)
    assert set(a) == {"rate_rows", "rate_out", "rate_valid"}
    rows = _rows(a["rate_rows"])
    assert rows.size == min(2048, d["config"]["series_per_step"]) and rows[-1] < d["config"]["series_per_step"]
    out, _, valid = _oracle_rows(rows, 0)
    assert (a["rate_valid"] == valid).all()
    assert a["rate_out"].tobytes() == out.tobytes()


@pytest.mark.gpu
def test_gpu_dump_is_what_the_timed_paths_computed_and_steps_are_the_timed_steps(tmp_path):
    """Two runs of the GPU arm at a small size: --steps is the number of timed steps of every timed path, the dumps of
    the two runs agree (seeded inputs), and the sampled results equal the oracle on the same synthetic series."""
    S, Se, G, H, B, N = 3000, 700, 50, 40, 64, 128
    args = ["--gpus", "1", "--steps", "3", "--warmup", "1", "--series-per-gpu", str(S), "--e2e-series", str(Se),
            "--groups", str(G), "--hist-per-gpu", str(H), "--wide-rows-per-gpu", "200000", "--no-cpu-baseline"]
    runs = []
    for i in range(2):
        d = _bench(*args, "--dump-outputs", str(tmp_path / str(i)), timeout=900)
        assert d["steps"] == 3 and d["e2e"]["steps"] == 3 and d["jitter_variant"]
        for c in ("3", "4", "5"):
            assert "error" not in d["configs"][c] and d["configs"][c]["steps"] == 3, d["configs"][c]
        runs.append(_load_dump(tmp_path / str(i)))
    a, b = runs
    assert set(a) == set(b) == {f"{n}_{k}" for n in ("rate", "rate_jitter", "rate_e2e", "hist") for k in ("rows", "out", "valid")} | \
        {"sumby_rows", "sumby_out", "sumby_count", "wide_sum", "wide_count"}
    for k in a:
        if k.startswith(("sumby_out", "hist_out")):
            assert np.allclose(a[k], b[k], rtol=1e-12, atol=0, equal_nan=True), k
        else:
            assert a[k].tobytes() == b[k].tobytes(), k

    def close(got, exp, what):
        rel = np.abs(got - exp) / np.maximum(np.abs(exp), 1e-300)
        assert float(rel.max()) <= 1e-9, (what, float(rel.max()))

    for name, jitter in (("rate", 0), ("rate_jitter", 1000), ("rate_e2e", 0)):
        rows = _rows(a[f"{name}_rows"])
        assert rows.size == min(2048 if name == "rate" else 512, Se if name == "rate_e2e" else S)
        out, _, valid = _oracle_rows(rows, jitter)
        assert (a[f"{name}_valid"] == valid).all(), name
        close(a[f"{name}_out"], out, name)

    from greptimedb_b200 import distributed as D
    from oracle import oracle as orc
    out, words, _ = _oracle_rows(np.arange(S), 0)
    gid = (D.mix32(np.arange(S, dtype=np.uint32)) % np.uint32(G)).astype(np.uint32)
    gsum, gcnt = orc.group_aggregate("sum", out, words, gid, G)
    rows = _rows(a["sumby_rows"])
    assert rows.tolist() == list(range(G))
    assert (a["sumby_count"] == gcnt).all()
    close(a["sumby_out"], gsum, "sumby")

    ts, val, sid = orc.synth_fill(0, H * B, N, T0, SCRAPE, 0, 0, SEED)
    val = val.reshape(H, B, N).cumsum(axis=1).ravel()
    p = orc.make_params("rate", T0, T0 + (N - 1) * SCRAPE, SCRAPE, 300_000)
    rates, rvalid = orc.range_query(p, ts, val, sid, np.arange(H * B + 1, dtype=np.uint64) * N, threads=2)
    le = np.concatenate([0.001 * 1.25 ** np.arange(B - 1), [np.inf]])
    q, qv = orc.histogram_quantile(0.99, le, rates, rvalid)
    assert _rows(a["hist_rows"]).tolist() == list(range(H))
    assert (a["hist_valid"] == orc.valid_to_bool(qv, N)).all()
    assert np.isnan(a["hist_out"]).tolist() == np.isnan(q).tolist()
    ok = ~np.isnan(q)
    close(a["hist_out"][ok], q[ok], "hist")

    assert (a["wide_count"] == 200_000 - len(range(0, 200_000, 1009))).all()
    assert np.allclose(a["wide_sum"] / a["wide_count"], 0.5, atol=0.01)
