#!/usr/bin/env python
"""bench.py - the measurement contract of this repo.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c3f32|c4|c5|c1] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input: the FULL stats_generator
(measures_of_counts / centralTendency / cardinality / dispersion / percentiles / shape) of a synthetic frame that is
already resident in HBM.  Default workload = BASELINE.json configs[2], the north-star configuration: 100 M rows x 200
mixed columns (150 float32 + 50 dictionary-coded string columns; `c3f32` is the all-float32 variant, `c2` =
configs[1], 10 M x 50).  Rank 0 prints ONE JSON line.  `value` = rows x cols / s over all ranks (weak scaling: every
rank owns `cols` columns - columns shard with no data-path collective, one NCCL all_gather of the per-column summaries
per step).  `e2e` = the same step through the public API from pinned HOST buffers (H2D inside the timed region, the
process bound to the GPU's NUMA node).  `roofline` describes the dominant C call of the step, `roofline_kernels` the
other calls, all timed with CUDA events inside the timed region; `fused_stats_hist_pass` = the north-star kernel (moments
+ histogram in one read) and drift statistics on the same frame; `parity` = the step's own results checked against the
oracle on the bit-identical NumPy twin of the generator (outside the timed region).  `--impl reference` times the CPU
oracle restatement on the host cores (Spark is not available on the box).
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "c2": dict(rows=10_000_000, cols=50, cat_every=0, desc="synthetic 10M rows x 50 float32 cols: full stats_generator"),
    # BASELINE.json configs[2] / north_star target: 75 % numeric / 25 % categorical (SURVEY.md 8d)
    "c3": dict(rows=100_000_000, cols=200, cat_every=4,
               desc="synthetic 100M rows x 200 mixed num/cat cols (150 float32 + 50 dictionary-coded string): "
                    "stats_generator + histogram binning"),
    "c3f32": dict(rows=100_000_000, cols=200, cat_every=0, desc="synthetic 100M rows x 200 float32 cols: full stats_generator"),
    "tiny": dict(rows=200_000, cols=8, cat_every=4, desc="smoke-size synthetic frame"),
    # BASELINE.json configs[0], the reference's own CPU-runnable plumbing check (SURVEY.md 8d: "always report C1")
    "c1": dict(rows=32_561, cols=17, c1=True, desc="income dataset (data/test_dataset, 32 561 x 17: 7 int + 1 double + 9 string): "
                                                   "measures_of_centralTendency"),
    # streamed workloads (BASELINE.json configs[3], [4]): the frames do not fit HBM, row chunks are (re)generated on the
    # device pass by pass; step = drift statistics(all methods) + counts/shape of both frames from the same passes
    "c4": dict(rows=100_000_000, cols=200, chunk=12_500_000, cat_every=4, stream=True,
               desc="synthetic source 100M + target 100M rows x 200 mixed num/cat cols: drift_statistics PSI/HD/JSD/KS, streamed"),
    "c5": dict(rows=1_000_000_000, cols=63, chunk=16_777_216, cat_every=0, stream=True,
               desc="synthetic source 1B + target 1B rows x 63 float32 cols per GPU (504 on 8): fused stats + drift, streamed"),
    "tiny_stream": dict(rows=300_000, cols=8, chunk=65_536, cat_every=4, stream=True, desc="smoke-size streamed drift"),
}
METRIC = "rows x cols / s, full stats_generator (+ HBM GB/s of the fused scan kernel)"
CPU_SAMPLE_ROWS = 1_000_000
# words of HBM traffic per sorted key the sort path needs BY DESIGN (DESIGN.md section 3): pack write 1, per 8-bit pass
# {tile histogram read 1, scatter read 1 + write 1} x 4, run summaries read 1
SORT_WORDS_PER_KEY = 1 + 4 * 3 + 1
SORT_DESIGN = ("batched 8-bit LSD radix sort + run summaries (anv_mode_distinct: pack, 4 x {sort_hist, sort_totals + sort_scan, "
               "sort_scatter}, run_tile, run_merge) - exact mode / distinct / percentiles")
# the partition + count path (anv_mode_distinct_partition, 32-bit columns): one read of the column, then every key that is not
# a splitter value (zeros and heavy hitters are only counted) is written once to its bucket and read once by the counting CTA
PARTITION_WORDS_PER_KEY = 2
PARTITION_DESIGN = ("partition + count (anv_mode_distinct_partition: sample, split, pc_partition_kernel, pc_cum_kernel, pc_count_kernel) - "
                    "exact mode / distinct / percentiles without sorting")



def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def settle_gc():
    """Collect once and move everything alive (the imported modules: ~10^6 objects) to the permanent generation, the way a
    long-running service does after start-up.  Otherwise ONE full collection lands inside the timed region every ~20 steps and
    stalls the host for ~40 ms while it walks the module objects (measured: 19 steps of 14.65 ms and one of 57 ms at c2).
    The collector stays enabled: what the steps allocate is still collected."""
    import gc
    gc.collect()
    gc.freeze()


class ClockSampler:
    """nvidia-smi polling the SM clock and the throttle reasons every 200 ms (the profiling recipe's line).  The process is started BEFORE the warm-up: its
    start-up (NVML init over every GPU of the box) takes about a second of driver work and used to land inside the timed
    region of short runs; begin() waits for its first sample and opens the window, stop() keeps the samples taken inside it."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, "/tmp/anv_clocks_%d.csv" % os.getpid()
        self.t_begin = None
        self.period_ms = int(os.environ.get("ANV_BENCH_CLOCK_PERIOD_MS", "200"))   # the profiling recipe's period; 0 = diagnostics only: no sampling
        self.disabled = self.period_ms <= 0

    def start(self):
        if self.disabled:
            return
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", str(self.period_ms), "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self._kill)      # a run that fails before stop() must not leave the sampler polling
        except Exception:
            self.proc = None

    def _kill(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.kill()
            self.proc.wait()

    def begin(self):
        """Open the sampling window (call right before the timed region; starts the sampler if start() was not called)."""
        if self.proc is None and not self.disabled:
            self.start()
        t0 = time.time()
        while self.proc is not None and time.time() - t0 < 5.0:      # the sampler is past its start-up once a line is out
            try:
                if os.path.getsize(self.path) > 0:
                    break
            except OSError:
                break
            time.sleep(0.02)
        self.t_begin = time.time()

    @staticmethod
    def _when(text):
        import datetime
        try:
            return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["not sampled (ANV_BENCH_CLOCK_PERIOD_MS=0)" if self.disabled else "nvidia-smi unavailable"]}
        t_end = time.time()
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                rows.append((self._when(parts[0]), float(parts[1]), float(parts[2]),
                             [nme for nme, v in zip(names, parts[5:9]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        try:
            os.remove(self.path)
        except OSError:
            pass
        if self.t_begin is not None:
            inside = [r for r in rows if r[0] is not None and self.t_begin - 0.1 <= r[0] <= t_end + 0.15]
            rows = inside or rows       # a timed region shorter than the polling period: keep what there is
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(r[1] for r in rows)
        reasons = sorted({x for r in rows for x in r[3]})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[2] for r in rows), "reasons": reasons, "samples": len(rows)}


# ---------------------------------------------------------------------------------------------
# the step
# ---------------------------------------------------------------------------------------------

def stats_step(frame, keep_cache=False):
    """Full stats_generator through the public API; returns the result frames (pandas), in STATS_FUNCTIONS order."""
    import anovos.data_analyzer.stats_generator as sg
    if not keep_cache:
        frame._cache = {k: v for k, v in frame._cache.items() if isinstance(k, tuple) and k and k[0] == "desc"}
    out = [sg.measures_of_counts(None, frame), sg.measures_of_centralTendency(None, frame),
           sg.measures_of_cardinality(None, frame), sg.measures_of_dispersion(None, frame),
           sg.measures_of_percentiles(None, frame), sg.measures_of_shape(None, frame)]
    return [o.toPandas() for o in out]


STATS_FUNCTIONS = ["measures_of_counts", "measures_of_centralTendency", "measures_of_cardinality", "measures_of_dispersion",
                   "measures_of_percentiles", "measures_of_shape"]


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, named_frames, limit_bytes=DUMP_LIMIT_BYTES):
    """Write the result tables of the last timed step as `path/<table>.<field>.npy`, float64, one value per row in the order the
    caller receives the rows.  Every value written is finite: where a field holds a cell that is null or not finite, that cell
    is 0 in `<table>.<field>.npy` and `<table>.<field>.nonfinite.npy` says what the caller gets there (0 = the value written,
    1 = null / NaN, 2 = +inf, 3 = -inf).  A text field (the attribute name, the mode) is written as the CRC-32 of its UTF-8
    text in `<table>.<field>.crc32.npy`, and also parsed as a number in `<table>.<field>.npy` when some cell holds one (the
    mode of a numeric column; text that is not a number counts as null there).  When the arrays would exceed `limit_bytes`,
    every table keeps the same share of its rows, picked by a generator with a fixed seed; the attribute CRCs name the rows
    kept."""
    import zlib
    import numpy as np
    import pandas as pd

    def number(v):
        try:
            return float(v)      # exact, unlike pandas' fast text parser
        except (TypeError, ValueError):
            return np.nan
    arrays = []

    def add(name, field, a):
        code = np.select([np.isnan(a), a == np.inf, a == -np.inf], [1.0, 2.0, 3.0], 0.0)
        if code.any():
            arrays.append((name, field + ".nonfinite", code))
            a = np.where(code == 0, a, 0.0)
        arrays.append((name, field, a))
    for name, df in named_frames:
        for field in df.columns:
            s = df[field]
            if pd.api.types.is_numeric_dtype(s) or pd.api.types.is_bool_dtype(s):
                add(name, field, s.to_numpy(dtype=np.float64, na_value=np.nan))
                continue
            num = np.array([np.nan if pd.isna(v) else number(v) for v in s.tolist()], dtype=np.float64)
            if not np.isnan(num).all():
                add(name, field, num)
            add(name, field + ".crc32", np.array([np.nan if pd.isna(v) else float(zlib.crc32(str(v).encode("utf-8")))
                                                  for v in s.tolist()], dtype=np.float64))
    total = sum(a.nbytes for _, _, a in arrays)
    keep = {}
    if total > limit_bytes:
        share = limit_bytes / total
        for name, df in named_frames:
            n = len(df)
            keep[name] = np.sort(np.random.default_rng(0).choice(n, int(n * share), replace=False))
    os.makedirs(path, exist_ok=True)
    for name, field, a in arrays:
        np.save(os.path.join(path, "%s.%s.npy" % (name, field)), a[keep[name]] if name in keep else a)


class StdoutGuard:
    """Route everything that libraries print on fd 1 (e.g. NCCL's version banner) to stderr, so
    that stdout carries exactly ONE JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, text):
        os.write(self.saved, (text + "\n").encode())

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def run_ours(args):
    with StdoutGuard() as out:
        _run_ours(args, out)


KERNEL_NAMES = {
    "anv_moments": "scan_kernel<MOM> (anv_moments: count/nonzero/min/max/mean/M2/M3/M4, FP64)",
    "anv_hll_registers": "hll_kernel (anv_hll_registers: XXH64 + HLL++ registers)",
    "anv_hist_codes": "code histogram (anv_hist_codes: groupBy(col).count() of dictionary codes)",
    "anv_hist": "scan_kernel<HIST> (anv_hist: binning + histogram)",
    "anv_moments_hist": "scan_kernel<MOM+HIST> (anv_moments_hist: moments + histogram in one read)",
}
# what limits each call (ncu evidence under profiles/): the roofline fraction is always quoted against HBM
BOUND = {"anv_mode_distinct": "issue", "anv_mode_distinct_partition": "l2 (per-key atomics and 4-byte stores)", "anv_hll_registers": "issue",
         "anv_moments_hist": "issue"}


def _run_ours(args, out):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from anovos_b200 import parallel
    numa = parallel.bind_numa(local)      # BEFORE any pinned allocation: host buffers land on the GPU's NUMA node
    import datetime
    import torch
    import torch.distributed as dist
    from anovos_b200 import engine, frame as framemod, synth

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(minutes=45))
    wl = WORKLOADS[args.workload]
    rows, cols = args.rows or wl["rows"], args.cols or wl["cols"]
    if wl.get("stream"):
        return _run_stream(args, out, wl, rows, cols, world, rank, local)
    if wl.get("c1"):
        return _run_c1(args, out, wl, world, rank, local)
    cat_every = wl.get("cat_every", 0)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident input: this rank's column shard (weak scaling: `cols` columns per GPU) -------
    src = synth.device_frame(rows, cols, seed=42, first_col=rank * cols, cat_every=cat_every)
    torch.cuda.synchronize()

    pending = []
    last = []

    def step():
        frames = stats_step(src)
        if world > 1:  # the only exchange of the path: per-column summaries (tiny, latency-bound, asynchronous)
            mat, _ = parallel.frames_to_matrix(frames)
            pending.append(parallel.gather_summaries_async(mat, cols, device="cuda"))
            if len(pending) > 1:
                pending.pop(0).result()   # consume the previous step's global table: ranks never stall inside a step
        last[:] = frames
        return frames

    def drain():
        while pending:
            pending.pop(0).result()

    if not args.no_extras:
        args.warmup = max(args.warmup, 3)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(args.warmup):
        step()
    drain()
    barrier()
    engine.timer = engine.KernelTimer()
    l0 = engine.launch_count
    if rank == 0:
        clocks.begin()
    settle_gc()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    walls = []
    for _ in range(args.steps):
        w0 = time.perf_counter()
        step()
        walls.append(round((time.perf_counter() - w0) * 1e3, 2))
    drain()   # every step's exchange has completed inside the timed region
    e1.record()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, list(zip(STATS_FUNCTIONS, last)))
    ms = e0.elapsed_time(e1)
    launches = engine.launch_count - l0
    kt = engine.timer.totals()
    engine.timer = None
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    ms_per_step = ms_max / args.steps
    value = rows * cols * world / (ms_per_step / 1e3)

    # ---- rooflines from the timed region: every C call of the step, the dominant one first ------------------
    # algorithmic bytes per call (DESIGN.md section 3, SURVEY.md 8d): ONE read of the call's input columns (values + bitmap;
    # recorded by the engine next to each call's CUDA events); the sort additionally moves SORT_WORDS_PER_KEY words per sorted key.
    num = [c for c in src.columns if src.column(c).kind == "num"]
    n_keys = int(sum(int(v) for v in engine.moments(src, num)["n_nonzero"])) if num else 0   # exact zeros are counted, not sorted
    peak, peak_src = peaks()
    traffic_tbl, traffic_src = {}, None
    for cand in sorted(os.listdir(os.path.join(ROOT, "profiles")), reverse=True):   # newest round first
        if not (cand.startswith("r") and "traffic" in cand and cand.endswith(".json")):
            continue
        try:  # dram__bytes_read+write per call from a committed ncu capture of the SAME workload
            tj = json.load(open(os.path.join(ROOT, "profiles", cand)))
            if tj.get("rows") == rows and tj.get("cols") == cols and tj.get("cat_every", 0) == cat_every:
                traffic_tbl, traffic_src = tj["dram_bytes_per_launch"], "profiles/" + cand
                break
        except Exception:
            pass

    def roof(call):
        v = kt[call]
        per_step = v["calls"] / args.steps                 # a step may batch the columns over several launches (c3 sort)
        ms_step = v["ms"] / args.steps                     # device time of this call per step
        alg = v["input_bytes"] / args.steps
        if call == "anv_mode_distinct":
            alg += n_keys * 4 * SORT_WORDS_PER_KEY
        elif call == "anv_mode_distinct_partition":
            alg += n_keys * 4 * PARTITION_WORDS_PER_KEY
        ach = alg / (ms_step * 1e-3) / 1e9 if (alg and ms_step > 0) else None
        traffic = traffic_tbl.get(call)
        more = {}
        if call == "anv_mode_distinct" and ms_step > 0:
            # context for an issue-bound kernel: keys sorted per second (pack, run summaries and HLL++ registers included in the
            # time) next to the CUDA toolkit's radix sort on the same GPU (recorded by scripts/yardstick/cub_sort.cu)
            more = {"sorted_keys_per_step": n_keys, "gkeys_per_s_incl_pack_and_summaries": n_keys / (ms_step * 1e-3) / 1e9,
                    "library_yardstick": library_yardstick(rows)}
        return {**more, "kernel": KERNEL_NAMES.get(call, {"anv_mode_distinct": SORT_DESIGN, "anv_mode_distinct_partition": PARTITION_DESIGN}.get(call, call)),
                "call": call,
                "bound": BOUND.get(call, "hbm"), "achieved": ach, "peak": peak,
                "peak_source": peak_src, "unit": "GB/s", "frac": ach / peak if ach else None,
                "traffic": traffic if traffic else None, "traffic_source": traffic_src if traffic else None,
                "algorithmic_bytes_per_launch": alg / per_step if alg else None,
                "ms_per_launch": ms_step / per_step, "launches_per_step": per_step,
                "share_of_step": v["ms"] / ms if ms > 0 else None}
    by_share = sorted(kt, key=lambda c: -kt[c]["ms"])
    roofline = roof(by_share[0]) if by_share else None
    if roofline is not None and roofline["bound"] != "hbm":
        roofline["note"] = ("bound by instruction issue, not by HBM (ncu: profiles/); frac is still achieved algorithmic GB/s over the "
                            "measured HBM peak - see roofline_kernels for the HBM-bound scan kernels the step also runs")
    roofline_kernels = [roof(c) for c in by_share[1:]]
    kernels = {k: {"ms_per_step": v["ms"] / args.steps, "calls_per_step": v["calls"] / args.steps,
                   "share_of_step": v["ms"] / ms} for k, v in sorted(kt.items())}
    kernel_ms = sum(v["ms"] for v in kt.values()) / args.steps

    rowslab = None
    if world > 1 and not args.no_extras:      # every rank takes part (collectives), outside the timed region
        try:
            rowslab = rowslab_check(rank, world, torch, dist)
        except Exception as ex:
            rowslab = {"error": repr(ex)}
    # N > 1: the end-to-end leg runs on EVERY rank at once (each GPU pulls its own columns over its own PCIe link) when the
    # host has room for all the pinned copies; otherwise rank 0 measures its share alone and says so
    e2e_all = False
    if world > 1 and not args.no_extras:
        e2e_all = all_ranks_have_host_room(rows, cols, world, torch, dist)
    line = None
    if rank != 0 and e2e_all:
        holder = [src]
        src = None
        try:
            e2e_numbers(args, rows, cols, holder, torch, framemod, engine, dist=dist, world=world)
        except Exception as ex:      # reported by rank 0 as a rank-0-only measurement; never take the job down
            print("rank %d: end-to-end leg failed: %r" % (rank, ex), file=sys.stderr)
    if rank == 0:
        extra, e2e, cpu, parity = {}, None, None, None
        if not args.no_extras:
            # ---- fused stats+histogram pass of a drift target (north-star kernel), timed alone ----------
            try:
                extra = fused_pass_numbers(src, rows, num, peak, torch, engine)
            except Exception as ex:  # never lose the main line
                extra = {"error": repr(ex)}
            drift_res = None
            try:
                extra["drift_statistics"], drift_res = drift_numbers(args, src, rows, cols, rank, cat_every, torch, engine, synth)
            except Exception as ex:
                extra["drift_statistics"] = {"error": repr(ex)}
            # ---- parity: the timed step's own results vs the oracle on the bit-identical NumPy twin ----
            if world == 1 or args.parity:
                try:
                    parity = parity_check(rows, cols, rank * cols, cat_every, src, last, drift_res)
                except Exception as ex:
                    parity = {"error": repr(ex)}
            else:
                parity = {"skipped": "N > 1 runs the identical per-rank path on other column ids: see the N = 1 line (or pass --parity)"}
            # ---- e2e: same step from pinned HOST buffers through the public API ---------------------
            holder = [src]
            src = None   # the leg frees the resident frame once it is copied: at c3 (80 GB) it would not fit twice
            try:
                e2e = e2e_numbers(args, rows, cols, holder, torch, framemod, engine, dist=dist if e2e_all else None, world=world)
                e2e["numa"] = numa
            except Exception as ex:
                e2e = {"error": repr(ex)}
            cpu = cpu_baseline(cols, cat_every=cat_every, first_col=rank * cols)
        line = {"metric": METRIC, "value": value, "unit": "rows*cols/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic (on-device Philox4x32-10, bit-identical NumPy twin: normal/lognormal/uniform/zero-inflated "
                        "float32, null rates 0 / 0.1 / 2 / 30 percent" +
                        (", every 4th column a Zipf(1.2) string column of cardinality 2/12/100/10000)" if cat_every else ")"),
                "config": {"workload": args.workload + ": " + wl["desc"], "rows": rows, "cols_per_gpu": cols,
                           "numeric_cols_per_gpu": len(num), "categorical_cols_per_gpu": cols - len(num),
                           "l2": "inputs (%.1f GB per GPU) are larger than L2" % (rows * cols * 4 / 1e9),
                           "sharding": "columns per rank, one NCCL all_gather of per-column summaries per step",
                           "kernel_ms_per_step": kernel_ms, "host_ms_per_step": ms_per_step - kernel_ms,
                           "wall_ms_each_step_rank0": walls},
                "gpu_launches": launches, "clocks": clk, "e2e": e2e, "roofline": roofline,
                "roofline_kernels": roofline_kernels, "cpu_baseline": cpu, "parity": parity, "kernels": kernels,
                "fused_stats_hist_pass": extra, "rowslab_nccl": rowslab}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        out.emit(json.dumps(line))


def library_yardstick(rows):
    """cub::DeviceRadixSort::SortKeys (bare sort of uniform 32-bit keys) as recorded under profiles/ for this row count."""
    for cand in sorted(os.listdir(os.path.join(ROOT, "profiles")), reverse=True):
        if "cub_yardstick" in cand and cand.endswith(".json"):
            try:
                for e in json.load(open(os.path.join(ROOT, "profiles", cand)))["library"]:
                    if e["key_bits"] == 32 and e["n_keys"] == rows:
                        return {"library": e["library"], "gkeys_per_s": e["gkeys_per_s"], "ms_per_column": e["ms_per_column"],
                                "what": "bare key sort, no pack / run summaries / HLL++", "source": "profiles/" + cand}
            except Exception:
                pass
    return None


def rowslab_check(rank, world, torch, dist):
    """N >= 2 only, outside the timed region, EVERY rank: the row-sharded variant of the path (SURVEY.md 8e) under NCCL.  Each
    rank holds a row slab of all columns of one frame; moments / histograms / HLL registers / radix-select histograms merge with
    all_gather + all_reduce, the exact mode needs the one real exchange of the path (row slabs -> column blocks, grouped
    point-to-point sends over NVLink).  Results must equal the single-frame results computed locally on every rank."""
    import tempfile
    import numpy as np
    import anovos.data_analyzer.stats_generator as sg
    import anovos.drift_stability.drift_detector as dd
    from anovos_b200 import engine, parallel, synth
    from anovos_b200.partitioned import PartitionedFrame, repartition_to_columns
    ROWS, COLS = 4_000_000, 16
    per = ROWS // world // 32 * 32
    r0 = rank * per
    r1 = ROWS if rank == world - 1 else r0 + per

    def mk(seed, a=0, b=ROWS):
        return synth.device_frame(b - a, COLS, seed=seed, cat_every=4, row0=a, shifted=seed != 42)
    whole, twhole = mk(42), mk(43)
    slab, tslab = mk(42, r0, r1), mk(43, r0, r1)
    parts = PartitionedFrame.from_frame(slab, 1 << 19, group=True)
    tparts = PartitionedFrame.from_frame(tslab, 1 << 19, group=True)
    ok = parts.count() == ROWS
    mw, mp = engine.moments(whole, whole.columns), engine.moments(parts, whole.columns)
    ok &= all(np.array_equal(mw[f], mp[f], equal_nan=True) for f in ("n_valid", "n_nonzero", "min", "max"))
    ok &= all(np.allclose(mw[f], mp[f], rtol=1e-9, atol=0) for f in ("mean", "m2", "m4"))
    for fn in ("measures_of_counts", "measures_of_percentiles", "measures_of_cardinality", "measures_of_centralTendency"):
        ok &= getattr(sg, fn)(None, whole).toPandas().equals(getattr(sg, fn)(None, parts).toPandas())
    kw = dict(method_type="all", use_sampling=False)
    a = dd.statistics(None, twhole, whole, source_path=tempfile.mkdtemp(), **kw).toPandas()
    b = dd.statistics(None, tparts, parts, source_path=tempfile.mkdtemp(), **kw).toPandas()
    ok &= all(np.allclose(a[m], b[m], rtol=1e-9, atol=0) for m in ("PSI", "HD", "JSD", "KS")) and list(a["flagged"]) == list(b["flagged"])
    repartition_to_columns(slab, True)      # first exchange: NCCL sets up the point-to-point connections (seconds at 8 ranks)
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    mine = repartition_to_columns(slab, True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    names = parallel.shard_columns(slab.columns, rank, world)
    ok &= mine.columns == names and mine.count() == ROWS
    for n in names:
        d, v = mine.column(n).device()
        dw, vw = whole.column(n).device()
        ok &= bool(torch.equal(d, dw)) and ((v is None and vw is None) or bool(torch.equal(v.view(torch.int32), vw.view(torch.int32))))
    t = torch.tensor([1.0 if ok else 0.0, ms], dtype=torch.float64, device="cuda")
    tmin = t.clone()
    dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    recv_bytes = sum(ROWS * 4 for _ in names) * (world - 1) / world
    return {"ok_on_every_rank": bool(tmin[0].item() == 1.0), "ranks": world, "rows": ROWS, "cols": COLS,
            "checked": "row-slab moments / counts / percentiles / HLL / exact mode / drift == single-frame results; "
                       "repartition_to_columns == the whole columns bit for bit",
            "exchange_ms_max_over_ranks": float(t[1].item()),
            "exchange_gbs_per_rank": recv_bytes / (float(t[1].item()) * 1e-3) / 1e9,
            "collectives": "all_gather(moment records) + all_reduce(sum: histograms, code counts, select histograms; max: HLL registers) "
                           "+ batched isend/irecv (row slabs -> column blocks) over NCCL"}


def parity_check(rows, cols, first_col, cat_every, src, frames, drift_res):
    """The results of the last timed step (and of the drift extra) against the ORACLE on the NumPy twin of the generator
    (bit-identical values, tests/test_gpu_parity_scale.py), for one numeric column of every family + one string column at
    the FULL row count; one process per column.  Outside the timed region; the oracle is the checker, never the product."""
    import pandas as pd
    from oracle import cpu_bench
    t0 = time.perf_counter()
    ids, fams = [], set()
    from anovos_b200 import synth
    for c in range(first_col, first_col + cols):
        if cat_every and c % cat_every == cat_every - 1:
            if "cat" not in fams:
                fams.add("cat")
                ids.append(c)
        else:
            f = synth.column_params(synth.numeric_ordinal(c, cat_every), 42)[0]
            if f not in fams:
                fams.add(f)
                ids.append(c)
    drift_ids = [c for c in ids if drift_res is not None and ("c%04d" % c) in set(drift_res["attribute"])]
    exp = cpu_bench.oracle_columns(lambda c, seed, shifted: synth.host_table(rows, 1, seed=seed, shifted=shifted, columns=[c],
                                                                           cat_every=cat_every), ids, drift_ids)
    names = ["c%04d" % c for c in ids]
    fn_names = ["measures_of_counts", "measures_of_centralTendency", "measures_of_cardinality", "measures_of_dispersion",
                "measures_of_percentiles", "measures_of_shape"]
    cells = bad = 0
    worst, examples = 0.0, []
    for fn, got in zip(fn_names, frames):
        g = got.set_index("attribute")
        for nme in names:
            e = exp[nme][fn]
            if e is None:
                continue
            for col, ev in e.items():
                gv = g.loc[nme, col] if nme in g.index else None
                cells += 1
                g_none, e_none = gv is None or (isinstance(gv, float) and gv != gv), ev is None or (isinstance(ev, float) and ev != ev)
                if g_none or e_none:
                    ok = g_none and e_none
                elif isinstance(ev, str) or isinstance(gv, str):
                    ok = str(gv) == str(ev)
                else:
                    d = abs(float(gv) - float(ev))
                    rel = d / max(abs(float(ev)), 1.0)
                    worst = max(worst, rel)
                    ok = d == 0 if col.endswith(("count", "rows", "values")) else d <= 1.0001e-4 * (1 + 2 * abs(float(ev)) ** 0.5)
                if not ok:
                    bad += 1
                    examples.append([nme, fn, col, repr(gv), repr(ev)])
    drift = None
    if drift_ids:
        d = drift_res.set_index("attribute")
        dworst = 0.0
        for c in drift_ids:
            nme = "c%04d" % c
            for m in ("PSI", "HD", "JSD", "KS"):
                gv, ev = float(d.loc[nme, m]), float(exp[nme]["drift"][m])
                cells += 1
                r = abs(gv - ev) / max(abs(ev), 1e-300)
                dworst = max(dworst, r if ev != 0 else abs(gv))
                if r > 1e-6 and abs(gv - ev) > 1e-12:
                    bad += 1
                    examples.append([nme, "statistics", m, repr(gv), repr(ev)])
        drift = {"columns": ["c%04d" % c for c in drift_ids], "max_rel_err": dworst, "tolerance": 1e-6}
    return {"checker": "oracle (NumPy restatement of the Spark semantics) on the bit-identical NumPy twin of the generator",
            "rows": rows, "columns": names, "functions": fn_names, "cells_checked": cells, "mismatches": bad,
            "max_rel_diff_of_rounded_outputs": worst, "drift": drift, "examples": examples[:5],
            "tolerance": "counts / modes / distinct / HLL++ / percentiles equal; round(x, 4) outputs within one rounding step; "
                         "PSI/HD/JSD/KS <= 1e-6 relative",
            "seconds": round(time.perf_counter() - t0, 1)}


def _same_cells(a, b):
    """Cell-wise equality of two result tables (null == null)."""
    import pandas as pd
    if list(a.columns) != list(b.columns) or len(a) != len(b):
        return False
    for c in a.columns:
        for x, y in zip(a[c].tolist(), b[c].tolist()):
            if not ((pd.isna(x) and pd.isna(y)) or x == y):
                return False
    return True


def income_table():
    """data/test_dataset of the reference = the two parquet parts committed under tests/golden/."""
    import pyarrow as pa
    import pyarrow.parquet as pq
    g = os.path.join(ROOT, "tests", "golden")
    return pa.concat_tables([pq.read_table(os.path.join(g, "income_part0.parquet")), pq.read_table(os.path.join(g, "income_part1.parquet"))])


def _run_c1(args, out, wl, world, rank, local):
    """configs[0]: measures_of_centralTendency on the income dataset.  A plumbing check, not a throughput claim: 32 561
    rows fit in L2, the step is launch- and host-bound.  `value` from the device-resident frame, `e2e` from the pyarrow
    table (conversion + H2D inside), `cpu_baseline` = the oracle in this process (1 core)."""
    import torch
    import anovos.data_analyzer.stats_generator as sg
    from anovos_b200 import engine, frame as framemod
    from oracle import api as O
    if rank != 0:
        return
    t = income_table()
    rows, cols = t.num_rows, t.num_columns
    fr = framemod.ColumnFrame.from_arrow(t)
    for c in fr.columns:
        if fr.column(c).kind != "other":
            fr.column(c).device()

    def step():
        fr._cache = {k: v for k, v in fr._cache.items() if isinstance(k, tuple) and k and k[0] == "desc"}
        return sg.measures_of_centralTendency(None, fr).toPandas()

    clocks = ClockSampler(local)
    clocks.start()
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    engine.timer = engine.KernelTimer()
    l0 = engine.launch_count
    clocks.begin()
    settle_gc()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = step()
    e1.record()
    torch.cuda.synchronize()
    clk = clocks.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [("measures_of_centralTendency", res)])
    ms = e0.elapsed_time(e1)
    kt = engine.timer.totals()
    engine.timer = None
    launches = engine.launch_count - l0
    h0, d0 = framemod.h2d_bytes, engine.d2h_bytes
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sg.measures_of_centralTendency(None, t).toPandas()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / args.steps
    e2e = {"value": rows * cols / dt, "unit": "rows*cols/s", "ms_per_step": dt * 1e3,
           "h2d_bytes_per_step": (framemod.h2d_bytes - h0) // args.steps, "d2h_bytes_per_step": (engine.d2h_bytes - d0) // args.steps,
           "note": "pyarrow table -> ColumnFrame (dictionary encoding on the host) -> H2D -> measures_of_centralTendency -> pandas"}
    t0 = time.perf_counter()
    exp = O.measures_of_centralTendency(t)
    tc = time.perf_counter() - t0
    by = sorted(kt, key=lambda c: -kt[c]["ms"])
    peak, peak_src = peaks()
    top = by[0] if by else None
    from anovos_b200 import _lib as L_
    nbytes = rows * sum(4 if fr.column(c).anv_dtype in (L_.ANV_F32, L_.ANV_I32) else 8 for c in fr.columns if fr.column(c).kind != "other")
    roofline = None
    if top:
        ms_step = kt[top]["ms"] / args.steps
        ach = nbytes / (ms_step * 1e-3) / 1e9
        roofline = {"kernel": top, "call": top, "bound": "hbm", "achieved": ach, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                    "frac": ach / peak, "traffic": None, "algorithmic_bytes_per_launch": nbytes, "ms_per_launch": ms_step /
                    max(kt[top]["calls"] / args.steps, 1), "share_of_step": kt[top]["ms"] / ms,
                    "note": "1.8 MB of input: latency-bound by construction, the fraction is not meaningful at this size"}
    line = {"metric": "rows x cols / s, measures_of_centralTendency on the income dataset (reference plumbing check)",
            "value": rows * cols / (ms / args.steps / 1e3), "unit": "rows*cols/s", "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "tests/golden/income_part{0,1}.parquet (= data/test_dataset of the reference)",
            "config": {"workload": args.workload + ": " + wl["desc"], "rows": rows, "cols_per_gpu": cols,
                       "l2": "input (1.8 MB) is SMALLER than L2: plumbing check only"},
            "gpu_launches": launches, "clocks": clk, "e2e": e2e, "roofline": roofline,
            "cpu_baseline": {"value": rows * cols / tc, "unit": "rows*cols/s", "cores": 1, "kind": "port",
                             "sample": "the whole dataset, oracle measures_of_centralTendency in this process, %.3f s" % tc},
            "kernels": {k: {"ms_per_step": v["ms"] / args.steps, "calls_per_step": v["calls"] / args.steps} for k, v in sorted(kt.items())},
            "matches_oracle": _same_cells(res, exp)}
    out.emit(json.dumps(line))


STREAM_METRIC = "rows x cols / s, streamed fused stats + drift_statistics (source + target, + HBM GB/s of the fused pass)"


def _run_stream(args, out, wl, rows, cols, world, rank, local):
    """BASELINE.json configs[3]/[4]: source and target frames larger than HBM, streamed in row chunks.
    Step = drift_detector.statistics(method_type="all", use_sampling=False) on two PartitionedFrames
    + measures_of_counts / measures_of_shape of both (served by the moments the drift passes leave
    behind): source numeric columns are read twice (K1 min/max -> cutoffs on the host -> K2), the
    target once (fused K1+K2), string columns once per frame.  rows*cols counts ONE frame, like the
    resident drift extra.  The chunks are generated on the device inside the timed region (there
    is nowhere to keep them): generation time is measured separately and reported."""
    import tempfile
    import torch
    import torch.distributed as dist
    import anovos.data_analyzer.stats_generator as sg
    import anovos.drift_stability.drift_detector as dd
    from anovos_b200 import engine, parallel, synth
    chunk, cat_every = args.chunk or wl["chunk"], wl["cat_every"]
    tmp = tempfile.mkdtemp()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def frames():
        kw = dict(first_col=rank * cols, cat_every=cat_every)
        return (synth.partitioned_frame(rows, cols, chunk, seed=42, **kw),
                synth.partitioned_frame(rows, cols, chunk, seed=43, shifted=True, **kw))

    def step():
        src, tgt = frames()
        r = [dd.statistics(None, tgt, src, method_type="all", use_sampling=False, source_path=tmp).toPandas()]
        for f in (src, tgt):
            r += [sg.measures_of_counts(None, f).toPandas(), sg.measures_of_shape(None, f).toPandas()]
        if world > 1:
            mat, _ = parallel.frames_to_matrix(r[:1])
            parallel.gather_summaries(mat, device="cuda")
        return r, src.passes + tgt.passes

    def generation_only():
        """The same chunk generation the step performs (every column of every pass), without kernels."""
        src, tgt = frames()
        num = [n for n in src.columns if src.column(n).kind == "num"]
        cat = [n for n in src.columns if src.column(n).kind == "cat"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for f, plan in ((src, [num, num, cat]), (tgt, [num, cat])):
            for names in plan:
                if not names:
                    continue
                for ch in f.chunks(names):
                    for n in names:
                        ch.column(n).device()
                    torch.cuda.current_stream().synchronize()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(max(args.warmup, 1) if rows > 50_000_000 else max(args.warmup, 3)):
        step()
    barrier()
    engine.timer = engine.KernelTimer()
    l0 = engine.launch_count
    if rank == 0:
        clocks.begin()
    settle_gc()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        res, passes = step()
    e1.record()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, list(zip(["drift_statistics", "source.measures_of_counts", "source.measures_of_shape",
                                                  "target.measures_of_counts", "target.measures_of_shape"], res)))
    ms = e0.elapsed_time(e1)
    launches = engine.launch_count - l0
    kt = engine.timer.totals()
    engine.timer = None
    gen_ms = generation_only()
    t = torch.tensor([ms, gen_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step, gen_ms = float(t[0].item()) / args.steps, float(t[1].item())
    value = rows * cols * world / (ms_per_step / 1e3)
    src, _ = frames()
    n_num = sum(1 for c in src.columns if src.column(c).kind == "num")
    n_null = sum(1 for c in src.columns if src.column(c).kind == "num" and src.column(c).has_validity)
    alg_bytes = rows * n_num * 4 + n_null * ((rows + 7) // 8)      # one read of the numeric columns of ONE frame
    peak, peak_src = peaks()
    kf = kt.get("anv_moments_hist", {"ms": 0.0, "calls": 0})
    fused_ms = kf["ms"] / args.steps                                  # all chunks of the target frame, per step
    achieved = alg_bytes / (fused_ms * 1e-3) / 1e9 if fused_ms > 0 else None
    n_chunks = -(-rows // (chunk // 32 * 32))
    roofline = {"kernel": "scan_kernel<MOM+HIST> (anv_moments_hist: target pass, moments + 10-bin histogram in one read)",
                "bound": "hbm", "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                "frac": achieved / peak if achieved else None, "traffic": None,
                "algorithmic_bytes_per_launch": alg_bytes // n_chunks, "ms_per_launch": fused_ms / n_chunks,
                "launches_per_step": n_chunks, "share_of_step": kf["ms"] / ms if ms > 0 else None}
    kernels = {k: {"ms_per_step": v["ms"] / args.steps, "calls_per_step": v["calls"] / args.steps,
                   "share_of_step": v["ms"] / ms} for k, v in sorted(kt.items())}
    kernel_ms = sum(v["ms"] for v in kt.values()) / args.steps
    line = None
    if rank == 0:
        e2e = cpu = None
        if not args.no_extras:
            e2e = stream_e2e(args, wl, min(rows, 20_000_000), cols, chunk, torch, tmp)
            cpu = cpu_stream_baseline(min(cols, 50))
        line = {"metric": STREAM_METRIC, "value": value, "unit": "rows*cols/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64",
                "data": "synthetic (on-device Philox, regenerated chunk by chunk inside the timed region on a side stream: the frames exceed HBM)",
                "config": {"workload": args.workload + ": " + wl["desc"], "rows": rows, "cols_per_gpu": cols,
                           "chunk_rows": chunk, "chunks_per_frame": n_chunks, "frame_passes_per_step": passes,
                           "l2": "every chunk (%.1f GB) is larger than L2" % (chunk * cols * 4 / 1e9),
                           "generation_ms_per_step_standalone": gen_ms, "kernel_ms_per_step": kernel_ms,
                           "generation": "the Philox generator of chunk i+1 runs on a side stream while chunk i is scanned (ALU-bound "
                                         "generator under HBM-bound scans); generation_ms_per_step_standalone = the generator alone, serialised",
                           "flagged_columns": int(res[0]["flagged"].sum()),
                           "sharding": "columns per rank; rows streamed per rank; one all_gather of the drift table per step"},
                "gpu_launches": launches, "clocks": clk, "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu,
                "kernels": kernels}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        out.emit(json.dumps(line))


def stream_e2e(args, wl, rows, cols, chunk, torch, tmp):
    """The streamed step from pinned HOST frames (bounded row sample): every pass uploads its chunks,
    chunk i+1 in flight on the copy stream while chunk i is scanned."""
    import anovos.data_analyzer.stats_generator as sg
    import anovos.drift_stability.drift_detector as dd
    from anovos_b200 import engine, frame as framemod, synth
    from anovos_b200.partitioned import PartitionedFrame
    chunk = min(chunk, max(32, rows // 4 // 32 * 32))
    hosts = []
    for seed, shifted in ((42, False), (43, True)):
        fr = synth.device_frame(rows, cols, seed=seed, shifted=shifted, cat_every=wl["cat_every"])
        hh = {}
        for n, v in host_copy(fr, torch).items():
            dic = fr.column(n).dictionary
            if dic is None:
                hh[n] = v
            else:
                hh[n] = (v[0], v[1], dic) if isinstance(v, tuple) else (v, None, dic)
        hosts.append(hh)
        del fr
    torch.cuda.empty_cache()

    def one():
        src = PartitionedFrame.from_frame(framemod.ColumnFrame.from_tensors(hosts[0], n_rows=rows), chunk)
        tgt = PartitionedFrame.from_frame(framemod.ColumnFrame.from_tensors(hosts[1], n_rows=rows), chunk)
        r = [dd.statistics(None, tgt, src, method_type="all", use_sampling=False, source_path=tmp).toPandas()]
        for f in (src, tgt):
            r += [sg.measures_of_counts(None, f).toPandas(), sg.measures_of_shape(None, f).toPandas()]
        return r

    for _ in range(2):     # memory pools of the copy stream settle after a couple of rounds
        one()
    torch.cuda.synchronize()
    steps = 2
    h0, d0 = framemod.h2d_bytes, engine.d2h_bytes
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    return {"value": rows * cols / dt, "unit": "rows*cols/s", "ms_per_step": dt * 1e3, "rows": rows,
            "h2d_bytes_per_step": (framemod.h2d_bytes - h0) // steps, "d2h_bytes_per_step": (engine.d2h_bytes - d0) // steps,
            "steps": steps, "note": "bounded sample (%d rows per frame) of the streamed step from pinned host columns: "
                                    "every pass re-uploads its chunks (source numeric columns twice), wall clock" % rows}


def fused_pass_numbers(src, rows, names, peak, torch, engine):
    """anv_hist (K2) and anv_moments_hist (K1+K2 fused: the drift target pass, moments + 10-bin histogram in one read) over
    the numeric columns of the resident frame, each timed alone with CUDA events on the launching stream."""
    mom = engine.moments(src, names)
    cuts, lohi = [], []
    for i in range(len(names)):
        mn, mx = float(mom["min"][i]), float(mom["max"][i])
        w = (mx - mn) / 10
        cuts.append([mn + j * w for j in range(1, 10)])
        lohi.append((mn, mx))
    model = engine.BinModel(src, names, cuts, lohi)
    out = {"columns": len(names), "rows": rows}
    for name, fn in (("hist", lambda: engine.histogram(src, model)), ("fused", lambda: engine.moments_histogram(src, model))):
        for _ in range(3):
            fn()
        engine.timer = engine.KernelTimer()
        for _ in range(5):
            fn()
        tot = engine.timer.totals()
        engine.timer = None
        key = "anv_hist" if name == "hist" else "anv_moments_hist"
        ms = tot[key]["ms"] / tot[key]["calls"]
        alg_bytes = tot[key]["input_bytes"] / tot[key]["calls"]
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        out[name] = {"ms_per_launch": ms, "algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": gbs, "frac_of_peak": gbs / peak,
                     "rows_cols_per_s": rows * len(names) / (ms * 1e-3)}
    out["fused"]["loop"] = ("8 x 128-bit loads per thread in registers (default); ANV_FUSED_STAGED=1: null-free columns through a "
                            "thread-private cp.async ring instead (A/B: profiles/r2b_fused_ab.md)")
    return out


def drift_numbers(args, src, rows, cols, rank, cat_every, torch, engine, synth):
    """drift_detector.statistics(target, source, method_type="all", use_sampling=False) through the public
    API on two device-resident frames: source K1 + K2, target fused K1+K2 in one read, K3 reduce.  When source + target
    do not fit HBM together (c3: 2 x 80 GB) the call covers the first columns whose target still fits."""
    import tempfile
    import anovos.drift_stability.drift_detector as dd
    free = torch.cuda.mem_get_info()[0]
    n = int(min(cols, max(0, (free - (24 << 30)) // (rows * 4 + rows // 8 + 1))))
    if n < 1:
        return {"skipped": "no room for a resident target frame next to the source"}, None
    n = n // 4 * 4 if (cat_every and n >= 4) else n
    names = src.columns[:n]
    s_sub = src.select(names)
    tgt = synth.device_frame(rows, n, seed=43, first_col=rank * cols, shifted=True, cat_every=cat_every)
    d = tempfile.mkdtemp()

    def run():
        for f in (s_sub, tgt):
            f._cache = {k: v for k, v in f._cache.items() if isinstance(k, tuple) and k and k[0] == "desc"}
        return dd.statistics(None, tgt, s_sub, method_type="all", use_sampling=False, source_path=d)

    for _ in range(2):
        r = run()
    torch.cuda.synchronize()
    engine.timer = engine.KernelTimer()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = max(1, min(args.steps, 3))
    e0.record()
    for _ in range(steps):
        r = run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    kt = engine.timer.totals()
    engine.timer = None
    res = r.toPandas()
    del tgt
    torch.cuda.empty_cache()
    return {"ms_per_call": ms, "columns": n, "rows_cols_per_s": rows * n / (ms * 1e-3), "flagged_columns": int(res["flagged"].sum()),
            "kernels_ms_per_call": {k: v["ms"] / steps for k, v in sorted(kt.items())},
            "note": "rows*cols counts ONE frame; the call reads source twice (K1, K2) and target once (fused); %d of %d columns "
                    "(source + target resident together)" % (n, cols)}, res


def host_copy(src, torch):
    """Pinned host copy of every column (+ validity words, + the dictionary of string columns) of a device frame.  Dictionary
    codes are kept the way ColumnFrame.from_arrow keeps them on the host: in the narrowest integer type that holds the
    dictionary (frame.narrow_code_dtype); the upload widens them on the device."""
    import numpy as np
    from anovos_b200.frame import narrow_code_dtype
    host = {}
    for name in src.columns:
        c = src.column(name)
        d, v = c.device()
        if c.dictionary is not None:
            d = d.to(getattr(torch, np.dtype(narrow_code_dtype(len(c.dictionary))).name))
        hd = torch.empty(d.shape, dtype=d.dtype, pin_memory=True)
        hd.copy_(d)
        hv = None
        if v is not None:
            hv = torch.empty(v.shape, dtype=v.dtype, pin_memory=True)
            hv.copy_(v)
        if c.dictionary is not None:
            host[name] = (hd, hv, c.dictionary)
        else:
            host[name] = (hd, hv) if hv is not None else hd
    torch.cuda.synchronize()
    return host


def all_ranks_have_host_room(rows, cols, world, torch, dist):
    """Collective: may every rank of this node pin its own host copy of the frame at the same time?"""
    try:
        import psutil
        need = rows * cols * 4 * 1.05
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
        avail = psutil.virtual_memory().available
        for path in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):   # a container limit counts too
            try:
                lim = open(path).read().strip()
                if lim.isdigit():
                    used = 0
                    for up in ("/sys/fs/cgroup/memory.current", "/sys/fs/cgroup/memory/memory.usage_in_bytes"):
                        if os.path.exists(up):
                            used = int(open(up).read().strip())
                            break
                    avail = min(avail, int(lim) - used)
            except OSError:
                pass
        ok = avail > need * local_world * 1.5 + 64e9
    except Exception:
        ok = False
    t = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(int(t.item()))


def dist_rank(torch):
    import torch.distributed as td
    return td.get_rank() if td.is_available() and td.is_initialized() else 0


def e2e_numbers(args, rows, cols, src_holder, torch, framemod, engine, dist=None, world=1):
    """Full step from pinned host buffers: H2D of every column + the result read-back inside
    the timed region, through ColumnFrame.from_tensors + the stats_generator API.  With `dist` every rank runs it at the same
    time on its own columns (barrier before each step, MAX over ranks of each step's wall time): the whole-job number."""
    steps = max(1, min(args.steps, 5 if rows * cols <= 2_000_000_000 else 3))

    from anovos_b200 import profile
    host = None

    def one():
        fr = framemod.ColumnFrame.from_tensors(host, n_rows=rows)
        profile.prefetch(fr)   # H2D of column group g+1 overlaps the passes over group g
        r = stats_step(fr, keep_cache=True)
        del fr
        return r

    failure = None
    try:
        host = host_copy(src_holder.pop(), torch)     # `src_holder` = [device frame]: released here, it would not fit twice
        torch.cuda.empty_cache()
        for _ in range(5):   # the copy-stream memory pool needs a few rounds to reach its steady size
            one()
        torch.cuda.synchronize()
    except Exception as ex:
        failure = ex
    if dist is not None:     # go on together only if EVERY rank got this far (a rank that could not pin its copy must not leave the others in a barrier)
        flag = torch.tensor([0 if failure is not None else 1], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if not int(flag.item()):
            dist = None
            if dist_rank(torch) != 0 and failure is None:
                return None
    if failure is not None:
        raise failure
    h0, d0 = framemod.h2d_bytes, engine.d2h_bytes
    settle_gc()
    times = []
    for _ in range(steps):
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        one()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    h2d, d2h = (framemod.h2d_bytes - h0) // steps, (engine.d2h_bytes - d0) // steps
    ranks = 1
    if dist is not None:
        tt = torch.tensor(times + [float(h2d), float(d2h)], dtype=torch.float64, device="cuda")
        mx = tt.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        times = mx[:steps].tolist()
        h2d, d2h = int(tt[steps].item()), int(tt[steps + 1].item())     # whole job: summed over the ranks
        ranks = world
    dt = sorted(times)[len(times) // 2]     # median: one step that collides with another tenant's PCIe / host traffic is listed, not averaged in
    return {"value": ranks * rows * cols / dt, "unit": "rows*cols/s", "ms_per_step": dt * 1e3,
            "ms_each_step": [round(t * 1e3, 2) for t in times],
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "h2d_gbs_lower_bound": h2d / dt / 1e9,   # the whole step's wall time charged to the copy: >= 50 per GPU means PCIe-bound
            "steps": steps, "ranks_measured": ranks,
            "scope": ("all %d ranks at once, each from its own pinned host copy over its own PCIe link; step time = MAX over ranks" % ranks) if ranks > 1
                     else ("this rank's columns only" + (" (N > 1: the host cannot pin every rank's copy at once - the other ranks idle)" if world > 1 else "")),
            "note": "pinned host columns (string columns: dictionary codes in the narrowest of uint8 / int16 / int32, widened on the device) -> pipelined H2D (profile.prefetch) -> 6 measures_of_* -> pandas, wall clock incl. host post-processing; MEDIAN of the steps (each listed: PCIe time varies with what else the host is doing)"}


# ---------------------------------------------------------------------------------------------
# CPU legs (oracle restatement on the host cores)
# ---------------------------------------------------------------------------------------------

def cpu_baseline(cols, with_drift=False, rows=CPU_SAMPLE_ROWS, workers=None, cat_every=0, first_col=0):
    from anovos_b200 import synth
    from oracle import cpu_bench
    workers = workers or min(cols, os.cpu_count() or 1)
    table = synth.host_table(rows, cols, first_col=first_col, cat_every=cat_every)
    target = synth.host_table(rows, cols, seed=43, shifted=True, first_col=first_col, cat_every=cat_every) if with_drift else None
    t_stats, t_drift, used = cpu_bench.time_stats_generator(table, workers, target)
    out = {"value": rows * cols / t_stats, "unit": "rows*cols/s", "cores": used, "kind": "port",
           "sample": "the first %d rows of the SAME %d columns (bit-identical NumPy twin of the device generator), oracle (NumPy "
                     "restatement of the Spark semantics, not Spark), one column per task over all host cores, %.2f s; rows*cols/s is "
                     "extrapolated linearly in rows (the sorts are n log n: this favours the CPU)" % (rows, cols, t_stats),
           "host_cores": os.cpu_count()}
    if t_drift is not None:
        out["drift_value"] = rows * cols / t_drift
    return out


def cpu_stream_baseline(cols, rows=CPU_SAMPLE_ROWS):
    from anovos_b200 import synth
    from oracle import cpu_bench
    workers = min(cols, os.cpu_count() or 1)
    t, used = cpu_bench.time_stream_step(synth.host_table(rows, cols), synth.host_table(rows, cols, seed=43, shifted=True), workers)
    return {"value": rows * cols / t, "unit": "rows*cols/s", "cores": used, "kind": "port", "host_cores": os.cpu_count(),
            "sample": "source + target of %d rows x %d float32 cols, oracle drift statistics(all) + counts + shape of both "
                      "frames (NumPy restatement of the Spark semantics, not Spark), one process per column, %.2f s"
                      % (rows, cols, t)}


def run_reference(args):
    """`--impl reference`: the reference's CPU path.  Spark/JVM are not installed on the box, so
    this is the oracle port on all host cores, on bounded samples of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    if wl.get("c1"):
        from oracle import api as O
        t = income_table()
        times = []
        for i in range(max(args.warmup, 1) + args.steps):
            t0 = time.perf_counter()
            O.measures_of_centralTendency(t)
            if i >= max(args.warmup, 1):
                times.append(time.perf_counter() - t0)
        dt = sum(times) / len(times)
        v = t.num_rows * t.num_columns / dt
        print(json.dumps({"impl": "reference", "metric": "rows x cols / s, measures_of_centralTendency on the income dataset "
                          "(reference plumbing check)", "value": v, "unit": "rows*cols/s", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": max(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f64", "data": "tests/golden/income_part{0,1}.parquet",
                          "config": {"workload": args.workload + ": " + wl["desc"], "rows": t.num_rows, "cols_per_gpu": t.num_columns},
                          "cpu_baseline": {"value": v, "unit": "rows*cols/s", "cores": 1, "kind": "port", "sample": "the whole dataset"},
                          "e2e": {"value": v, "unit": "rows*cols/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
        return
    cols = args.cols or wl["cols"]
    rows = min(args.rows or wl["rows"], CPU_SAMPLE_ROWS)
    cat_every = wl.get("cat_every", 0)
    from anovos_b200 import synth
    from oracle import cpu_bench
    workers = min(cols, os.cpu_count() or 1)
    table = synth.host_table(rows, cols, cat_every=cat_every)
    stream = bool(wl.get("stream"))
    target = synth.host_table(rows, cols, seed=43, shifted=True, cat_every=cat_every) if stream else None
    times = []
    for i in range(max(args.warmup, 1) + args.steps):
        if stream:
            t, used = cpu_bench.time_stream_step(table, target, workers)
        else:
            t, _, used = cpu_bench.time_stats_generator(table, workers)
        if i >= max(args.warmup, 1):
            times.append(t)
    dt = sum(times) / len(times)
    v = rows * cols / dt
    cpu = {"value": v, "unit": "rows*cols/s", "cores": used, "kind": "port",
           "sample": "the first %d rows of the SAME %d columns as %s per step (bit-identical NumPy twin of the device generator; "
                     "rows*cols/s extrapolates linearly in rows, which favours the CPU: its sorts are n log n)" % (rows, cols, args.workload)}
    print(json.dumps({"impl": "reference", "metric": STREAM_METRIC if stream else METRIC, "value": v, "unit": "rows*cols/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": dt * 1e3,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                      "data": "synthetic (bit-identical NumPy twin of the device generator)",
                      "config": {"workload": args.workload + ": " + wl["desc"], "rows": args.rows or wl["rows"], "cols_per_gpu": cols,
                                 "rows_sampled_per_step": rows},
                      "cpu_baseline": cpu,
                      "e2e": {"value": v, "unit": "rows*cols/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}),
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--parity", action="store_true", help="run the oracle parity check also when N > 1")
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--cols", type=int, default=0)
    ap.add_argument("--chunk", type=int, default=0, help="rows per chunk of the streamed workloads (c4, c5)")
    ap.add_argument("--no-extras", action="store_true", help="profiling runs: skip e2e / cpu_baseline / fused extras")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result tables of the last timed step to DIR/<table>.<field>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
