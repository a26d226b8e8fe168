#!/usr/bin/env python
"""bench.py — PromQL range-query throughput on B200 (BASELINE.json metric), all four GPU configs in one JSON line.

  python bench.py --gpus N --steps K --warmup W            # our CUDA path  (one JSON line on rank 0)
  python bench.py --impl reference --gpus N --steps K --warmup W   # reference CPU path (oracle port)

Headline (`value`, `roofline`, `e2e`, `cpu_baseline`): BASELINE config 2 — a "step" is one pass of the hot path (K0
series offsets + the fused normalize/range/rate stage: K2L first tier, K2 / its long-window instantiation / the slow
kernel over what is handed on) over one HBM-resident chunk of synthetic series: 1000 samples/series at a 15 s scrape
(on the schedule by default, --jitter-ms 0; the +<1 s jitter generator — round 1's headline — is measured in the same run
and reported as `jitter_variant`), rate(x[5m]) at a 15 s step => 1000 eval steps.  Config 2's 10 M series (200 GB of input) exceed one
GPU's HBM, so they are processed as 8 chunks of 1.25 M series; the default K = 8 timed steps are exactly one
10 M-series job.  `value` is input samples/s with inputs resident in HBM; `e2e` is the same metric through the
host-pointer C-ABI call (pinned host buffers, H2D + kernels + D2H inside the timed region).

`configs` carries one object per BASELINE config measured the same way (W warm-up steps, K timed steps bracketed by
barrier + synchronize, CUDA events on the launching stream, max over ranks), each with its own ms_per_step, dominant
kernel, roofline and — on rank 0 at N=1 — cpu_baseline:
  "3"  sum by(pod)(rate(x[5m])), 1.25 M series/GPU -> 100 k label groups: K0 + fused rate/by-label partials
       (no [S x T] intermediate) + for N>1 ONE all-reduce of the [G x T] (sum f64, cnt u32) partials INSIDE the
       timed region, issued tile by tile by the library on its NCCL communicator;
  "4"  histogram_quantile(0.99, rate(latency_bucket[5m])): 125 k histograms x 64 buckets x 128 samples per GPU
       (1 M histograms over 8 GPUs): K0 + rate + HistogramFold (K5); shards hold whole histograms, no collective;
  "5"  avg_over_time wide-events scan: 12.5 M rows x 32 f64 columns per GPU (100 M rows over 8 GPUs): K6 per-column
       (sum, count) + for N>1 the all-reduce of the 32 x 2 scalars.
Inputs are far larger than L2 (126 MB) in every config, so no explicit L2 flush is needed between steps.

--dump-outputs DIR writes, after the timed steps, what each timed path returned in its last timed step as DIR/<name>.npy
(a fixed, seeded sample of the rows of the larger results; see OutputDump).  Every input is generated from SEED, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

T0 = 1_700_000_000_000
N_SAMPLES = 1000
SCRAPE = 15_000
RANGE = int(os.environ.get("B2P_BENCH_RANGE_MS", "300000"))  # 5m lookback (override: tuning experiments only)
SEED = 0x5EED
METRIC = "rate() input samples/sec"
UNIT = "samples/s"


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(key="range_lean_kernel"):
    """dram__bytes_read.sum + dram__bytes_write.sum per input sample of the dominant kernel, from the committed ncu
    --set full capture of the shipped kernel (profiles/r2_traffic.json, written by profiles/summarize_ncu.py)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            d = json.load(f)
        return float(d[key]["dram_bytes_per_sample"]), f"profiles/r2_traffic.json[{key}] ({d[key].get('kernel', '')})"
    except Exception:
        return None, None


class OutputDump:
    """--dump-outputs DIR: the results of the last timed step of each timed path, as DIR/<name>.npy.

    A [rows x T] result is sampled: a fixed, seeded choice of rows (the same for every run with the same arguments),
    written as <name>_rows (row indices), <name>_out (f64 values, 0.0 where there is no value) and <name>_valid (f32
    0/1 per slot, unpacked from the validity bit words).  Counts are written as f64.  All files together stay below
    LIMIT bytes.  Only rank 0 writes (its own shard)."""
    LIMIT = 64_000_000

    def __init__(self, path, rank=0):
        self.path = path if rank == 0 else None
        self.bytes = 0
        if self.path:
            os.makedirs(self.path, exist_ok=True)

    @staticmethod
    def sample(n, k):
        import numpy as np
        if n <= k:
            return np.arange(n, dtype=np.int64)
        return np.sort(np.random.default_rng(SEED).choice(n, k, replace=False)).astype(np.int64)

    @staticmethod
    def _rows(a, idx, shape):
        """rows idx of `a` viewed as `shape` -> numpy; `a` is a numpy array or a torch tensor (device or host)."""
        if hasattr(a, "index_select"):
            import torch
            return a.reshape(shape).index_select(0, torch.from_numpy(idx).to(a.device)).cpu().numpy()
        return a.reshape(shape)[idx]

    def put(self, name, a):
        import numpy as np
        if not self.path:
            return
        a = np.ascontiguousarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        self.bytes += a.nbytes
        if self.bytes > self.LIMIT:
            raise RuntimeError(f"--dump-outputs: {name} takes the dump past {self.LIMIT} bytes")
        np.save(os.path.join(self.path, name + ".npy"), a)

    def result(self, name, out, valid, n_rows, T, k):
        """A sample of k rows of an [n_rows x T] f64 result and its [n_rows x ceil(T / 32)] u32 validity words."""
        import numpy as np
        if not self.path:
            return
        idx = self.sample(n_rows, k)
        words = self._rows(valid, idx, (n_rows, (T + 31) // 32)).view(np.uint32)
        self.put(name + "_rows", idx.astype(np.float64))
        self.put(name + "_out", self._rows(out, idx, (n_rows, T)).astype(np.float64))
        self.put(name + "_valid", np.unpackbits(words.view(np.uint8), axis=1, bitorder="little")[:, :T].astype(np.float32))

    def groups(self, name, vals, cnt, n_rows, T, k):
        """A sample of k rows of an [n_rows x T] (f64 value, u32 count) pair."""
        import numpy as np
        if not self.path:
            return
        idx = self.sample(n_rows, k)
        self.put(name + "_rows", idx.astype(np.float64))
        self.put(name + "_out", self._rows(vals, idx, (n_rows, T)).astype(np.float64))
        self.put(name + "_count", self._rows(cnt, idx, (n_rows, T)).view(np.uint32).astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.

    The sampler is started before the warm-up (nvidia-smi takes a few hundred ms to produce its first line) and
    every line carries a timestamp; stop(t0, t1) keeps the samples that fall inside the timed window [t0, t1]
    (wall clock), or — if the window was shorter than the sampling period — the samples nearest to it."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = []
        for seen, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                import datetime
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except Exception:
                ts = seen
            try:
                rows.append((ts, float(f[2]), float(f[3]), f[5:9]))
            except ValueError:
                continue
        inside = [r for r in rows if t0 is not None and t0 <= r[0] <= t1]
        where = "inside the timed region"
        if not inside and rows and t0 is not None:
            mid = 0.5 * (t0 + t1)
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
            where = "nearest to the timed region (region shorter than the sampling period)"
        if t0 is None:
            inside = rows
        sm = [r[1] for r in inside]
        mx = [r[2] for r in inside]
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": where}


def query_params(n_samples=N_SAMPLES):
    from greptimedb_b200 import make_params
    return make_params("rate", T0, T0 + (n_samples - 1) * SCRAPE, SCRAPE, RANGE)


# ---------------------------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference's CPU path; test infrastructure timed as the reported baseline)
# ---------------------------------------------------------------------------------------------------------------
JITTER_MS = 0  # set from --jitter-ms


def cpu_reference_pass(n_series: int, threads: int, faithful: bool = True, series_begin: int = 0, with_resets=0,
                       n_samples: int = N_SAMPLES):
    """One pass of the reference's CPU algorithm (oracle port, structure-faithful) -> (seconds, samples, out, valid)."""
    import numpy as np
    from oracle import oracle as orc
    ts, val, sid = orc.synth_fill(series_begin, n_series, n_samples, T0, SCRAPE, JITTER_MS, with_resets, SEED)
    offsets = np.arange(n_series + 1, dtype=np.uint64) * n_samples
    p = orc.make_params("rate", T0, T0 + (n_samples - 1) * SCRAPE, SCRAPE, RANGE)
    t = time.perf_counter()
    out, valid = orc.range_query(p, ts, val, sid, offsets, mode="faithful" if faithful else "flat", threads=threads)
    return time.perf_counter() - t, n_series * n_samples, out, valid


def cpu_baseline_config(cfg: str, cores: int):
    """Bounded CPU sample of one config -> cpu_baseline object (oracle port; a reported baseline, not the target)."""
    import numpy as np
    from oracle import oracle as orc
    if cfg == "3":
        S, G = min(max(cores * 512, 4096), 65_536), 5000
        dt, n, out, valid = cpu_reference_pass(S, cores)
        from greptimedb_b200 import distributed as D
        gid = (D.mix32(np.arange(S, dtype=np.uint32)) % np.uint32(G)).astype(np.uint32)
        t = time.perf_counter()
        orc.group_aggregate("sum", out, valid, gid, G)
        dt += time.perf_counter() - t
        return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{S} series x {N_SAMPLES} samples -> {G} groups; range stage on {cores} threads, by-label sum on 1"}
    if cfg == "4":
        H, B, N = min(max(cores * 16, 256), 2048), 64, 128
        dt, n, out, valid = cpu_reference_pass(H * B, cores, n_samples=N)
        le = np.concatenate([1.5 ** np.arange(B - 1), [np.inf]])
        t = time.perf_counter()
        orc.histogram_quantile(0.99, le, out, valid)
        dt += time.perf_counter() - t
        return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{H} histograms x {B} buckets x {N} samples; range stage on {cores} threads, fold on 1"}
    if cfg == "5":
        rows, cols = 2_000_000, 32
        rng = np.random.default_rng(5)
        a = rng.random((cols, rows))
        t = time.perf_counter()
        for c in range(cols):
            orc.arrow_sum(a[c])
        dt = time.perf_counter() - t
        return {"value": rows * cols / dt, "unit": "values/s", "cores": 1, "kind": "port",
                "sample": f"{rows} rows x {cols} columns, arrow-rs ordered sum per column (avg_over_time = sum/len), 1 thread"}
    raise ValueError(cfg)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The Rust/DataFusion build is
    impossible here (no rustc/cargo/network), so this times the oracle port — the C restatement of
    SeriesDivide -> SeriesNormalize -> RangeManipulate -> prom_rate -> Filter, structure-faithful
    (per-series batch materialisation, packed RangeArray keys, tag take, null filter) — on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = max(cores * 1024, 4096)
    per_step = min(per_step, 262_144)
    for _ in range(args.warmup):
        cpu_reference_pass(per_step, cores)
    t = 0.0
    samples = 0
    for _ in range(args.steps):
        dt, n, out, valid = cpu_reference_pass(per_step, cores)
        t += dt
        samples += n
    if args.dump_outputs:
        OutputDump(args.dump_outputs).result("rate", out, valid, per_step, N_SAMPLES, 2048)
    value = samples / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"rate(x[5m]) step 15s over {per_step} series x {N_SAMPLES} samples per step "
                               "(bounded sample of BASELINE config 2), CPU oracle port of the reference path",
                   "series_per_step": per_step, "samples_per_series": N_SAMPLES},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} x {per_step} series x {N_SAMPLES} samples, structure-faithful port, "
                                   "gcc -O3 -march=native"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def gpu_numa_cpus(local: int):
    """CPUs of the NUMA node the GPU hangs off (sysfs), or None.  Pinned staging buffers first-touched from these CPUs
    land in host memory next to the GPU's PCIe root: with eight ranks copying at once, remote-node traffic was what
    held 8-GPU end-to-end efficiency at 0.59 in round 1."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        return (node, cpus) if cpus else None
    except Exception:
        return None


class numa_local:
    """with numa_local(local): allocate + first-touch host buffers on the GPU's NUMA node, then restore the affinity."""

    def __init__(self, local):
        self.info = gpu_numa_cpus(local)
        self.saved = None

    def __enter__(self):
        if self.info:
            try:
                self.saved = os.sched_getaffinity(0)
                os.sched_setaffinity(0, self.info[1] & self.saved or self.info[1])
            except Exception:
                self.saved = None
        return self.info[0] if self.info else None

    def __exit__(self, *exc):
        if self.saved:
            try:
                os.sched_setaffinity(0, self.saved)
            except Exception:
                pass
        return False


class Harness:
    """Per-process state shared by the config benches: device, context, distributed plumbing, timing helper."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from greptimedb_b200 import Context
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (the product has no CPU fallback); "
                             "use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.dump = OutputDump(args.dump_outputs, self.rank) if args.dump_outputs else None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.ctx = Context(self.local)
        self.ctx.use_torch_stream()
        if self.world > 1:
            # the library's own communicator (the collective on the data path lives behind the C ABI); torch.distributed
            # only ships the 128-byte id and provides the barrier / max-over-ranks of the timing contract
            box = [self.ctx.comm_unique_id() if self.rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            self.ctx.comm_init(box[0], self.world, self.rank)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, step, steps, warmup, sampler=None):
        """W warm-up steps, then K timed steps bracketed by barrier + synchronize -> (ms per step [max over ranks],
        launches, wall window)."""
        torch = self.torch
        for _ in range(warmup):
            step()
        self.ctx.sync()
        self.barrier()
        launches0 = self.ctx.launch_count()
        wall0 = time.time()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            step()
        ev1.record()
        self.ctx.sync()
        self.barrier()
        wall1 = time.time()
        ms = self.max_over_ranks(ev0.elapsed_time(ev1)) / steps
        return ms, self.ctx.launch_count() - launches0, (wall0, wall1)

    def stage_ms(self, step, stages, reps=3):
        """Kernel-stage durations from the library's own CUDA events (untimed extra steps)."""
        acc = {s: [] for s in stages}
        for _ in range(reps):
            step()
            self.ctx.sync()
            self.torch.cuda.synchronize()
            for s in stages:
                acc[s].append(self.ctx.kernel_ms(s))
        return {s: (statistics.mean(v) if v and min(v) >= 0 else None) for s, v in acc.items()}

    def free(self):
        import gc
        gc.collect()
        self.torch.cuda.empty_cache()


def bench_config2(h: Harness, sampler):
    torch, args, ctx, dev = h.torch, h.args, h.ctx, h.dev
    S = args.series_per_gpu
    n_rows, T = S * N_SAMPLES, N_SAMPLES
    Tw = (T + 31) // 32
    p = query_params()
    ts = torch.empty(n_rows, dtype=torch.int64, device=dev)
    val = torch.empty(n_rows, dtype=torch.float64, device=dev)
    sid = torch.empty(n_rows, dtype=torch.int32, device=dev)
    offsets = torch.empty(S + 1, dtype=torch.int64, device=dev)
    out = torch.empty(S * T, dtype=torch.float64, device=dev)
    valid = torch.empty(S * Tw, dtype=torch.int32, device=dev)
    # series are hash-sharded across GPUs: rank r owns global series [r*S, (r+1)*S) of this step's chunk
    def step():
        ctx.series_offsets_dev(sid, n_rows, S, offsets)
        ctx.range_eval_dev(p, ts, val, offsets, n_rows, S, out, valid)

    # the scrape-jitter variant of the generator (BASELINE.md section 4: timestamps +< 1 s off the schedule; the
    # round-1 headline workload), measured the same way before the headline so that the resident data is the headline's
    jitter_variant = None
    if args.jitter_variant_ms > 0 and args.jitter_variant_ms != args.jitter_ms:
        ctx.synth_fill_dev(h.rank * S, S, N_SAMPLES, T0, SCRAPE, args.jitter_variant_ms, args.resets, SEED, ts, val, sid)
        ctx.sync()
        jms, _, _ = h.timed(step, args.steps, args.warmup)
        if h.dump:
            h.dump.result("rate_jitter", out, valid, S, T, 512)
        jitter_variant = {"jitter_ms": args.jitter_variant_ms, "ms_per_step": jms,
                          "value": n_rows * h.world / (jms * 1e-3), "unit": UNIT,
                          "warp_tier_series": ctx.last_warp_tier_series(), "slow_path_series": ctx.last_slow_series()}
    ctx.synth_fill_dev(h.rank * S, S, N_SAMPLES, T0, SCRAPE, args.jitter_ms, args.resets, SEED, ts, val, sid)
    ctx.sync()

    ms, launches, window = h.timed(step, args.steps, args.warmup)
    if h.dump:
        h.dump.result("rate", out, valid, S, T, 2048)
    slow_series, warp_tier_series = ctx.last_slow_series(), ctx.last_warp_tier_series()
    clocks = sampler.stop(*window) if sampler else None
    st = h.stage_ms(step, (0, 1), reps=min(args.steps, 5))
    res = {"S": S, "n_rows": n_rows, "T": T, "Tw": Tw, "ms": ms, "launches": launches, "clocks": clocks,
           "k0_ms": st[0], "k2_ms": st[1], "slow_series": slow_series, "warp_tier_series": warp_tier_series,
           "jitter_variant": jitter_variant}

    # ---- end to end through the host-pointer C ABI: pinned host buffers, H2D + kernels + D2H timed ----
    Se = args.e2e_series
    res["e2e"] = None
    if Se > 0:
        import ctypes as C
        with numa_local(h.local) as numa_node:   # pinned staging next to this GPU's PCIe root
            h_ts = torch.empty(Se * N_SAMPLES, dtype=torch.int64).pin_memory()
            h_val = torch.empty(Se * N_SAMPLES, dtype=torch.float64).pin_memory()
            h_sid = torch.empty(Se * N_SAMPLES, dtype=torch.int32).pin_memory()
            h_out = torch.empty(Se * T, dtype=torch.float64).pin_memory()
            h_valid = torch.empty(Se * Tw, dtype=torch.int32).pin_memory()
            h_out.zero_()
            h_valid.zero_()
            h_ts.copy_(ts[: Se * N_SAMPLES])
            h_val.copy_(val[: Se * N_SAMPLES])
            h_sid.copy_(sid[: Se * N_SAMPLES])
            h_off = (torch.arange(Se + 1, dtype=torch.int64) * N_SAMPLES).pin_memory()
        torch.cuda.synchronize()
        L = ctx._L

        def e2e_step(with_offsets=False):
            rc = L.b2p_range_eval(ctx._h, C.byref(p), C.c_void_p(h_ts.data_ptr()), C.c_void_p(h_val.data_ptr()),
                                  None if with_offsets else C.c_void_p(h_sid.data_ptr()),
                                  C.c_void_p(h_off.data_ptr()) if with_offsets else None, Se * N_SAMPLES, Se,
                                  C.c_void_p(h_out.data_ptr()), C.c_void_p(h_valid.data_ptr()), None)
            if rc != 0:
                raise RuntimeError(L.b2p_last_error().decode())

        for _ in range(max(1, min(args.warmup, 2))):
            e2e_step()
        h.barrier()
        n_e2e = args.steps          # the full --steps, like the device-resident leg
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()          # synchronous: returns after the D2H of the result
        torch.cuda.synchronize()
        dt = h.max_over_ranks(time.perf_counter() - t0)
        h2d_ids = ctx.last_h2d_bytes()   # counted by the library from the copies it issued for one call
        # the same call when the caller (SeriesDivide's boundaries are known to it) hands over series offsets instead of
        # the 4 B/row id column: 16 B/sample over PCIe and no K0
        h.barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step(True)
        torch.cuda.synchronize()
        dt_off = h.max_over_ranks(time.perf_counter() - t0)
        h2d_off = ctx.last_h2d_bytes()
        if h.dump:
            h.dump.result("rate_e2e", h_out, h_valid, Se, T, 512)
        res["e2e"] = {"value": Se * N_SAMPLES * h.world * n_e2e / dt, "unit": UNIT,
                      "h2d_bytes_per_step": h2d_ids, "d2h_bytes_per_step": Se * T * 8 + Se * Tw * 4,
                      "host_columns_bytes_per_step": Se * N_SAMPLES * 20,
                      "h2d_note": ("the call takes the i64 timestamp, f64 value and u32 id columns in pinned host memory; it scans "
                                   "them on the host (worker threads, ahead of the copies) and sends chunks of equally spaced "
                                   "series as values + (offsets, first timestamp, cadence) per series, every other chunk as it "
                                   "is (B2P_HOST_TS_SCAN=0: always as it is)"),
                      "series_per_step": Se, "steps": n_e2e, "pinned_numa_node": numa_node,
                      "with_series_offsets_instead_of_ids": {"value": Se * N_SAMPLES * h.world * n_e2e / dt_off,
                                                             "h2d_bytes_per_step": h2d_off}}
        del h_ts, h_val, h_sid, h_out, h_valid, h_off
    del ts, val, sid, offsets, out, valid
    h.free()
    return res


def bench_config3(h: Harness):
    """sum by(pod)(rate(x[5m])): K0 + fused rate / by-label partials + (N>1) the all-reduce inside the library call."""
    import numpy as np
    from greptimedb_b200 import distributed as D
    torch, args, ctx, dev = h.torch, h.args, h.ctx, h.dev
    S, G = args.series_per_gpu, args.groups
    n_rows, T = S * N_SAMPLES, N_SAMPLES
    p = query_params()
    ts = torch.empty(n_rows, dtype=torch.int64, device=dev)
    val = torch.empty(n_rows, dtype=torch.float64, device=dev)
    sid = torch.empty(n_rows, dtype=torch.int32, device=dev)
    offsets = torch.empty(S + 1, dtype=torch.int64, device=dev)
    ctx.synth_fill_dev(h.rank * S, S, N_SAMPLES, T0, SCRAPE, args.jitter_ms, args.resets, SEED, ts, val, sid)
    gid_np = (D.mix32(np.arange(h.rank * S, (h.rank + 1) * S, dtype=np.uint32)) % np.uint32(G)).astype(np.int32)
    gid = torch.from_numpy(gid_np).to(dev)
    gsum = torch.zeros(G * T, dtype=torch.float64, device=dev)
    gcnt = torch.zeros(G * T, dtype=torch.int32, device=dev)
    ctx.sync()
    torch.cuda.synchronize()
    ix = ctx.group_index_create_dev(gid, S, G)   # built once per label assignment, reused by every step
    fused = ctx.range_group_sum_fused(p, ix)
    tiles = args.allreduce_tiles if h.world > 1 else 1

    def step():
        gsum.zero_()
        gcnt.zero_()
        ctx.series_offsets_dev(sid, n_rows, S, offsets)
        ctx.range_group_sum_allreduce_dev(p, ts, val, offsets, n_rows, S, ix, tiles, gsum, gcnt)

    steps = args.steps
    ms, launches, _ = h.timed(step, steps, max(3, args.warmup))
    if h.dump:
        h.dump.groups("sumby", gsum, gcnt, G, T, 512)
    st = h.stage_ms(step, (0, 1, 4))
    # compute-only variant of the same step (no collective) on N>1, to name the collective's share
    ms_nocoll = None
    if h.world > 1:
        def step_nocoll():
            gsum.zero_()
            gcnt.zero_()
            ctx.series_offsets_dev(sid, n_rows, S, offsets)
            ctx.range_group_sum_indexed_dev(p, ts, val, offsets, n_rows, S, ix, 0, G, gsum, gcnt)
        ms_nocoll, _, _ = h.timed(step_nocoll, steps, 3)
    ctx.sync()
    ctx.group_index_destroy(ix)
    peak, _ = load_peaks()
    alg = 16.0 * n_rows + 12.0 * G * T + 8.0 * (S + 1) + 8.0 * S   # range stage: samples in, partial rows out, offsets, members+gid
    k = st[1]
    payload = 12.0 * G * T
    res = {
        "workload": f"sum by(pod)(rate(x[5m])) over {S} series x {N_SAMPLES} samples per GPU -> {G} label groups "
                    f"(hash of the global series id), partials [G x T] (sum f64, cnt u32)",
        "ms_per_step": ms, "steps": steps, "value": S * N_SAMPLES * h.world / (ms * 1e-3), "unit": UNIT,
        "fused": bool(fused), "gpu_launches": launches,
        "kernel": ("range_lean_kernel<rate, grouped> (first tier adds into the by-label partials group by group; no "
                   "[S x T] intermediate)" if fused else "range_lean_kernel<rate> + group_aggregate_kernel (two passes)"),
        "roofline": {"bound": "hbm", "achieved": alg / (k * 1e-3) / 1e9 if k else None, "peak": peak, "unit": "GB/s",
                     "frac": (alg / (k * 1e-3) / 1e9 / peak) if k else None, "algorithmic_bytes_per_launch": alg,
                     "kernel_ms": k, "k0_series_offsets_ms": st[0],
                     "hbm_read_frac_whole_step": 20.0 * n_rows / (ms * 1e-3) / 1e9 / peak},
        "collective": None if h.world == 1 else {
            "what": f"all-reduce of [G x T] partials, {payload / 1e9:.2f} GB per rank (sum f64 + cnt u32), NCCL behind the C "
                    f"ABI, {tiles} tile(s) overlapped with the next tile's compute",
            "ms_per_step_without_collective": ms_nocoll, "ms_exposed": ms - ms_nocoll if ms_nocoll else None,
            "share_of_step": (ms - ms_nocoll) / ms if ms_nocoll else None,
            "last_tile_allreduce_kernel_ms": st[4], "tiles": tiles},
    }
    del ts, val, sid, offsets, gid, gsum, gcnt
    h.free()
    return res


def bench_config4(h: Harness):
    """histogram_quantile(0.99, rate(latency_bucket[5m])): K0 + rate over H*B bucket series + HistogramFold (K5)."""
    import numpy as np
    torch, args, ctx, dev = h.torch, h.args, h.ctx, h.dev
    H, B, N = args.hist_per_gpu, 64, 128
    S, n_rows, T = H * B, H * B * N, N
    Tw = (T + 31) // 32
    p = query_params(N)
    ts = torch.empty(n_rows, dtype=torch.int64, device=dev)
    val = torch.empty(n_rows, dtype=torch.float64, device=dev)
    sid = torch.empty(n_rows, dtype=torch.int32, device=dev)
    ctx.synth_fill_dev(h.rank * S, S, N, T0, SCRAPE, args.jitter_ms, 0, SEED, ts, val, sid)
    ctx.sync()
    torch.cuda.synchronize()
    # cumulative histogram: bucket b counts everything below le[b] -> prefix sum over the bucket axis
    v3 = val.view(H, B, N)
    v3.copy_(torch.cumsum(v3, dim=1))
    le = torch.from_numpy(np.concatenate([0.001 * 1.25 ** np.arange(B - 1), [np.inf]])).to(dev)
    offsets = torch.empty(S + 1, dtype=torch.int64, device=dev)
    rates = torch.empty(S * T, dtype=torch.float64, device=dev)
    rvalid = torch.empty(S * Tw, dtype=torch.int32, device=dev)
    out = torch.empty(H * T, dtype=torch.float64, device=dev)
    ovalid = torch.empty(H * Tw, dtype=torch.int32, device=dev)

    def step():
        ctx.series_offsets_dev(sid, n_rows, S, offsets)
        ctx.range_eval_dev(p, ts, val, offsets, n_rows, S, rates, rvalid)
        ctx.histogram_quantile_dev(0.99, le, B, rates, rvalid, H, T, out, ovalid)

    steps = args.steps
    ms, launches, _ = h.timed(step, steps, max(3, args.warmup))
    if h.dump:
        h.dump.result("hist", out, ovalid, H, T, 4096)
    st = h.stage_ms(step, (0, 1, 3))
    peak, _ = load_peaks()
    alg_range = 16.0 * n_rows + 8.0 * S * T + 4.0 * S * Tw + 8.0 * (S + 1)
    alg_fold = 8.0 * S * T + 4.0 * S * Tw + 8.0 * H * T + 4.0 * H * Tw
    res = {
        "workload": f"histogram_quantile(0.99, rate(latency_bucket[5m])) over {H} histograms x {B} buckets x {N} samples "
                    f"per GPU ({H * h.world} histograms in the job), cumulative counters, le = 63 exponential bounds + Inf",
        "ms_per_step": ms, "steps": steps, "value": n_rows * h.world / (ms * 1e-3), "unit": UNIT,
        "gpu_launches": launches, "slow_path_series": ctx.last_slow_series(),
        "warp_tier_series": ctx.last_warp_tier_series(),
        "kernel": "range_lean_kernel<rate> (short series: 128 samples) + histogram_quantile_kernel (one pass, counters in shared memory)",
        "roofline": {"bound": "hbm", "achieved": alg_range / (st[1] * 1e-3) / 1e9 if st[1] else None, "peak": peak,
                     "unit": "GB/s", "frac": (alg_range / (st[1] * 1e-3) / 1e9 / peak) if st[1] else None,
                     "algorithmic_bytes_per_launch": alg_range, "kernel_ms": st[1], "k0_series_offsets_ms": st[0],
                     "fold": {"kernel_ms": st[3], "algorithmic_bytes_per_launch": alg_fold,
                              "achieved": alg_fold / (st[3] * 1e-3) / 1e9 if st[3] else None,
                              "frac": (alg_fold / (st[3] * 1e-3) / 1e9 / peak) if st[3] else None},
                     "hbm_read_frac_whole_step": 20.0 * n_rows / (ms * 1e-3) / 1e9 / peak},
        "collective": None if h.world == 1 else {"what": "none: shards hold whole histograms (hash of the labels without le)"},
    }
    del ts, val, sid, offsets, rates, rvalid, out, ovalid, le, v3
    h.free()
    return res


def bench_config5(h: Harness):
    """avg_over_time wide-events scan: per-column (sum, count) of 32 f64 columns + (N>1) the all-reduce of the scalars."""
    torch, args, ctx, dev = h.torch, h.args, h.ctx, h.dev
    rows, cols = args.wide_rows_per_gpu, 32
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED + h.rank)   # the same table on every run
    data = torch.rand((cols, rows), dtype=torch.float64, device=dev, generator=gen)
    data[:, ::1009] = float("nan")     # stale markers are skipped like SeriesNormalize's filter
    ptrs = torch.tensor([data[c].data_ptr() for c in range(cols)], dtype=torch.int64, device=dev)
    col_sum = torch.zeros(cols, dtype=torch.float64, device=dev)
    col_cnt = torch.zeros(cols, dtype=torch.int64, device=dev)

    def step():
        col_sum.zero_()
        col_cnt.zero_()
        ctx.column_reduce_dev(ptrs, cols, rows, col_sum, col_cnt)
        ctx.allreduce_columns_dev(col_sum, col_cnt, cols)

    steps = args.steps
    ms, launches, _ = h.timed(step, steps, max(3, args.warmup))
    if h.dump:
        h.dump.put("wide_sum", col_sum.cpu().numpy())
        h.dump.put("wide_count", col_cnt.cpu().numpy().astype("float64"))
    st = h.stage_ms(step, (3, 4))
    avg = (col_sum / col_cnt.to(torch.float64)).cpu()
    peak, _ = load_peaks()
    alg = 8.0 * rows * cols
    res = {
        "workload": f"avg_over_time over the whole range of a wide table: {rows} rows x {cols} f64 columns per GPU "
                    f"({rows * h.world} rows in the job), NaN rows skipped",
        "ms_per_step": ms, "steps": steps, "value": rows * cols * h.world / (ms * 1e-3), "unit": "values/s",
        "gpu_launches": launches, "kernel": "column_reduce_stage1 / stage2 (deterministic two-stage per-column sum, count)",
        "check": {"avg_col0": float(avg[0]), "expected": "~0.5 (uniform [0,1))"},
        "roofline": {"bound": "hbm", "achieved": alg / (st[3] * 1e-3) / 1e9 if st[3] else None, "peak": peak,
                     "unit": "GB/s", "frac": (alg / (st[3] * 1e-3) / 1e9 / peak) if st[3] else None,
                     "algorithmic_bytes_per_launch": alg, "kernel_ms": st[3]},
        "collective": None if h.world == 1 else {"what": "all-reduce of 32 x (sum f64, count u64), NCCL behind the C ABI",
                                                 "allreduce_kernel_ms": st[4]},
    }
    del data, ptrs, col_sum, col_cnt
    h.free()
    return res


def run_ours(args):
    h = Harness(args)
    sampler = ClockSampler(h.local) if h.rank == 0 else None
    if sampler:
        sampler.start()
    c2 = bench_config2(h, sampler)
    extra = {}
    want = {"all": ("3", "4", "5"), "rate": (), "sumby": ("3",), "hist": ("4",), "wide": ("5",)}[args.workload]
    for name, fn in (("3", bench_config3), ("4", bench_config4), ("5", bench_config5)):
        if name in want:
            try:
                extra[name] = fn(h)
            except Exception as e:  # a failing side config must not take the headline line down with it
                extra[name] = {"error": f"{type(e).__name__}: {e}"}
                h.free()
    if h.rank != 0:
        if h.world > 1:
            h.dist.destroy_process_group()
        return

    S, n_rows, T, Tw = c2["S"], c2["n_rows"], c2["T"], c2["Tw"]
    peak, peak_src = load_peaks()
    k2, k0, step_ms = c2["k2_ms"], c2["k0_ms"], c2["ms"]
    alg_k2 = 16.0 * n_rows + 8.0 * S * T + 4.0 * S * Tw + 8.0 * (S + 1)   # bytes per launch of the dominant kernel
    achieved = alg_k2 / (k2 * 1e-3) / 1e9
    lean_on = os.environ.get("B2P_DISABLE_LEAN_TIER", "0") != "1" and os.environ.get("B2P_ENABLE_THREAD_TIER", "0") != "1"
    if lean_on and c2["warp_tier_series"] * 2 > S:
        lean_on = False   # the first tier still declined most series in the timed steps: K2 did the work
        kernel_name = "range_fast_kernel<rate> (the lean first tier handed off most series)"
    elif lean_on and args.resets:
        kernel_name = ("range_lean_kernel<rate, bit words> (adaptive: the plain variant handed off every series during the "
                       "warm-up) + range_fast_kernel<rate> over the series it hands off")
    elif lean_on and args.jitter_ms == 0 and os.environ.get("B2P_UNIFORM", "") != "0":
        kernel_name = ("range_lean_kernel<rate, uniform cadence> (picked by cadence_probe_kernel: samples exactly one eval "
                       "interval apart) + range_fast_kernel<rate> over the series it hands off")
    else:
        kernel_name = ("range_lean_kernel<rate> (+ range_fast_kernel<rate> over the series it hands off)" if lean_on
                       else "range_fast_kernel<rate>")
    uniform = lean_on and not args.resets and args.jitter_ms == 0 and os.environ.get("B2P_UNIFORM", "") != "0"
    per_sample, traffic_src = load_traffic("range_lean_kernel_uniform" if uniform else "range_lean_kernel")
    value = S * N_SAMPLES * h.world / (step_ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": h.world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"rate(x[5m]) step 15s over {S} series x {N_SAMPLES} samples per GPU per step "
                               f"(BASELINE config 2 = 10M series processed as chunks of {S}); resets={args.resets}; "
                               + ("scrapes on the 15 s schedule (BASELINE.md section 4 main shape)" if args.jitter_ms == 0
                                  else f"scrape timestamps +<{args.jitter_ms} ms off the schedule (BASELINE.md section 4 variant)"),
                   "scrape_jitter_ms": args.jitter_ms,
                   "compare_with_round_1": ("jitter_variant (round 1 benchmarked the +<1 s jitter generator as its headline; "
                                            "this run's `value` is on scrapes exactly on the schedule)") if args.jitter_ms == 0
                   else "value (same generator as round 1's headline)",
                   "series_per_gpu_per_step": S, "samples_per_series": N_SAMPLES, "eval_steps": T,
                   "parallelism": f"series-sharded x{h.world}, no data-path collective in config 2 "
                                  "(configs.3 / configs.5 carry the collectives)",
                   "l2": "inputs (16-25 GB per step) >> 126 MB L2; no flush needed"},
        "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak,
                     # dram__bytes_read.sum + dram__bytes_write.sum per launch: bytes per sample of the committed ncu
                     # --set full capture of the shipped kernel (profiles/r2_traffic.json) x the samples of this launch
                     "traffic": per_sample * n_rows if (per_sample and lean_on) else None, "traffic_source": traffic_src,
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_k2, "kernel_ms": k2, "k0_series_offsets_ms": k0,
                     "hbm_read_frac_whole_step": 20.0 * n_rows / (step_ms * 1e-3) / 1e9 / peak},
        "gpu_launches": c2["launches"], "slow_path_series": c2["slow_series"], "warp_tier_series": c2["warp_tier_series"],
        "clocks": c2["clocks"],
    }
    if c2["jitter_variant"]:
        # the same step over the generator's jittered timestamps (round 1's headline workload): the general first tier
        jv = dict(c2["jitter_variant"])
        jv["hbm_read_frac_whole_step"] = 20.0 * n_rows / (jv["ms_per_step"] * 1e-3) / 1e9 / peak
        line["jitter_variant"] = jv
    if c2["e2e"]:
        line["e2e"] = c2["e2e"]
    cores = os.cpu_count() or 1
    if h.world == 1 and not args.no_cpu_baseline:
        n_cpu = min(max(cores * 2048, 8192), 262_144)
        dt, n, _, _ = cpu_reference_pass(n_cpu, cores, faithful=True)
        dt_flat, n_flat, _, _ = cpu_reference_pass(n_cpu, cores, faithful=False)
        line["cpu_baseline"] = {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{n_cpu} series x {N_SAMPLES} samples, structure-faithful oracle port "
                                          f"(gcc -O3 -march=native), {cores} threads", "algorithm_only_value": n_flat / dt_flat}
        for name in extra:
            if "error" not in extra[name]:
                try:
                    extra[name]["cpu_baseline"] = cpu_baseline_config(name, cores)
                except Exception as e:
                    extra[name]["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"}
    if extra:
        line["configs"] = extra
    print(json.dumps(line), flush=True)
    if h.world > 1:
        h.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--series-per-gpu", type=int, default=1_250_000)
    ap.add_argument("--e2e-series", type=int, default=131_072)
    ap.add_argument("--resets", type=int, default=0, help="1 = counter-reset variant of the value generator")
    ap.add_argument("--jitter-ms", type=int, default=0,
                    help="scrape jitter of the generator: 0 = timestamps on the schedule (BASELINE.md section 4, main shape), "
                         "1000 = the +<1 s variant (round 1's headline)")
    ap.add_argument("--jitter-variant-ms", type=int, default=1000,
                    help="config 2 is measured a second time with this jitter and reported as configs['2'].jitter_variant (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="all", choices=["all", "rate", "sumby", "hist", "wide"],
                    help="all = config 2 (headline) + configs 3, 4, 5 in `configs`; rate = config 2 only; "
                         "sumby / hist / wide = config 2 + that one")
    ap.add_argument("--groups", type=int, default=100_000)
    ap.add_argument("--allreduce-tiles", type=int, default=4,
                    help="config 3, N>1: group ranges the partials are computed and all-reduced in (overlap)")
    ap.add_argument("--hist-per-gpu", type=int, default=125_000)
    ap.add_argument("--wide-rows-per-gpu", type=int, default=12_500_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write what each timed path returned in its last step as DIR/<name>.npy "
                         f"(f32 / f64, a seeded sample of rows, at most {OutputDump.LIMIT} bytes in all)")
    args = ap.parse_args()
    global JITTER_MS
    JITTER_MS = args.jitter_ms
    # NCCL's banner ("NCCL version ...", printed to stdout at NCCL_DEBUG=VERSION) would precede the one JSON line
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
