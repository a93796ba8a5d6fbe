#!/usr/bin/env python
"""bench.py -- createIndex rows/s on the synthetic table T of SURVEY.md section 8d (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W [--rows R] [--impl reference] [--workload createIndex|filter|join|refresh|snappy|files]

A "step" is one createIndex over the whole table: scan (Parquet decode) -> project -> hash-repartition into 200 buckets
-> sort within bucket -> Parquet encode, through the C ABI (hs_create_index).

* ``value``     rows/s with the source Parquet file images already resident in HBM and the index file images left in HBM.
* ``e2e``       the same work with HOST file images in and HOST file images out (pinned memory), every step's H2D and D2H
                inside the timed region, software-pipelined across steps through the public staging API
                (hs_stage_sources -> hs_create_index_async -> hs_pending_wait): the H2D copy of step i+1 and the D2H copy
                of step i-1 run beside the kernels of step i.  One call alone cannot overlap its own copies (every index
                file depends on every source file); its latency is reported as ``e2e.single_call_ms``.
* ``verified``  the output of the LAST timed e2e step is checked outside the timed region: on the GPU over all rows
                (bucket id of every row == bucket of its file, every file sorted, row count, order-independent row and column
                checksums == the generator's) and on the host for two whole buckets against the CPU oracle.  A mismatch
                fails the run (exit code 1).
* ``roofline``  achieved HBM GB/s of the dominant kernel from CUDA events recorded by the library around every launch on
                its stream, against the measured copy bandwidth in MEASURED_PEAKS.json.
* ``cpu_baseline``  the CPU oracle port (pyarrow decode/encode + pthreads C bucket/sort) timed on this host's cores on a
                bounded sample of the same table (rank 0, N=1 only).
* ``--impl reference``  the reference arm.  The reference itself (Scala on Spark) cannot run here (no JVM in this
                image), so this arm times the oracle port with all host threads, as the task statement prescribes.
* ``extra``     the read-side and refresh workloads of BASELINE.json configs[2..4] (C3 filter, C4 join, C5 incremental
                refresh + Hybrid Scan), each runnable alone with ``--workload``.
* ``--dump-outputs DIR``  after the timed steps, a seeded sample of the index files of the last timed step as
                DIR/<name>.npy (see dump_outputs), the same for the same arguments, to compare two builds output for output.
                That step's index files stay in HBM until the dump is written, so its release (hs_result_free, a stream
                synchronize) falls outside the timed region: compare timings of dump runs with dump runs only.

Every workload (and the reference arm) runs ``--warmup`` untimed and ``--steps`` timed repetitions, except that the
pipelined e2e path always warms up at least two steps and the ``cpu_baseline`` is a fixed best of 3 after one warm-up.

Multi-GPU (torchrun, one rank per GPU): the 256 source files are split across ranks, rows move to the owner of their
bucket inside the fused partition + NVLink peer-store kernel, the table size is fixed (strong scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

INDEXED = ["k"]
INCLUDED = ["v1", "v2", "v3", "v4"]
NUM_BUCKETS = int(os.environ.get("HS_BENCH_BUCKETS", "200"))  # (override: experiments only; the benchmark config is 200)
ROW_BYTES = 32  # decoded bytes per row of T
ALGO_BYTES_PER_ROW = 64  # 32 read + 32 written (SURVEY.md section 8d)

# Algorithmic HBM bytes per row and launch of the big kernels for table T with dictionary-encoded v1, v3, v4 (DESIGN.md 4);
# "rows" says which row count a launch processes: "in" = rows this rank decodes, "out" = rows this rank owns after the exchange
KERNEL_BYTES = {
    "k_sort_scatter": {"first": 20.0, "rest": 24.0, "rows": "out",
                       "note": "per launch: (8 B key + 4 B row index) read + written; a step's first launch reads the raw 8 B key only"},
    "k_onesweep": {"first": 20.0, "rest": 24.0, "rows": "out",
                   "note": "per launch: (8 B key + 4 B row index) read + written; a step's first launch reads the raw 8 B key only"},
    "k_partition_rows": {"first": 48.0, "rest": 48.0, "rows": "in",
                         "note": "2 B bucket id + 8 B k + 8 B v2 + 3 x 2 B codes read; 8 + 8 + 8 B (k, v2, code record) written"},
    "k_decode_pages": {"first": 41.65, "rest": 41.65, "rows": "in",
                       "note": "19.65 B encoded read; 8 + 8 B values + 3 x 2 B codes written"},
    "k_gather_encode": {"first": 14.0, "rest": 14.0, "rows": "out", "note": "per launch (one 8-byte column): 4 B row index + 8 B value gathered (sector-granular), 8 B written; the key column streams 8 + 8"},
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rows", type=int, default=1_000_000_000)
    ap.add_argument("--files", type=int, default=256)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="createIndex", choices=["createIndex", "filter", "join", "refresh", "snappy", "files"])
    ap.add_argument("--cpu-sample-rows", type=int, default=128_000_000)
    ap.add_argument("--cpu-sample-files", type=int, default=128)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C3/C4/C5 workloads attached under 'extra'")
    ap.add_argument("--plain", action="store_true", help="PLAIN-only source and index files (no dictionary encoding)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed, seeded sample of the index rows of the last timed createIndex step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "createIndex"):
        ap.error("--dump-outputs needs the createIndex workload on the GPU")
    return args


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    smax.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(smax), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU oracle arm
# ---------------------------------------------------------------------------------------------------------------------

def cpu_write_sources(sample_rows: int, n_files: int, nthreads: int, workdir: str):
    """Writes the sample of T as n_files Parquet files (outside any timed region).  Returns the paths."""
    import pyarrow as pa
    import pyarrow.parquet as pq
    from concurrent.futures import ThreadPoolExecutor

    from oracle import oracle as O

    src_dir = os.path.join(workdir, "src")
    os.makedirs(src_dir, exist_ok=True)
    per = sample_rows // n_files

    def write(f):
        p = os.path.join(src_dir, f"part-{f:05d}.parquet")
        if not os.path.exists(p):
            pq.write_table(pa.table(O.synthetic_table(f * per, per, 5)), p, compression="NONE", use_dictionary=["v1", "v3", "v4"])
        return p

    with ThreadPoolExecutor(max_workers=max(1, min(nthreads, n_files))) as ex:
        return list(ex.map(write, range(n_files)))


def cpu_create_index(paths, nthreads: int, workdir: str):
    """Times the oracle port (CPU restatement of the reference path) over the given source files.  Returns seconds."""
    import numpy as np
    import pyarrow as pa
    import pyarrow.parquet as pq
    from concurrent.futures import ThreadPoolExecutor

    from oracle import oracle as O

    pa.set_cpu_count(nthreads)
    out_dir = os.path.join(workdir, "idx")
    t0 = time.perf_counter()
    order = INDEXED + INCLUDED
    # one decode task per file over all cores (Spark: one scan task per file split); every task writes its rows straight
    # into the table-wide column arrays, so nothing is concatenated on one thread afterwards
    counts = [pq.ParquetFile(p).metadata.num_rows for p in paths]
    starts = np.concatenate([[0], np.cumsum(counts)])
    schema = pq.ParquetFile(paths[0]).schema_arrow
    cols = {name: np.empty(int(starts[-1]), dtype=schema.field(name).type.to_pandas_dtype()) for name in order}

    def decode(i):
        t = pq.read_table(paths[i], columns=order, use_threads=False)
        for name in order:
            cols[name][starts[i]:starts[i + 1]] = t.column(name).to_numpy()

    with ThreadPoolExecutor(max_workers=max(1, min(nthreads, len(paths)))) as ex:
        list(ex.map(decode, range(len(paths))))
    perm, offs, _ = O.index_rows(cols, INDEXED, INCLUDED, NUM_BUCKETS, nthreads=nthreads)
    os.makedirs(out_dir, exist_ok=True)

    def write_bucket(b):
        lo, hi = int(offs[b]), int(offs[b + 1])
        if hi == lo:
            return
        idx = perm[lo:hi]
        part = pa.table({name: cols[name][idx] for name in order})
        pq.write_table(part, os.path.join(out_dir, O.bucket_file_name(b, "cpu")), compression="NONE",
                       use_dictionary=["v1", "v3", "v4"])

    with ThreadPoolExecutor(max_workers=nthreads) as ex:
        list(ex.map(write_bucket, range(NUM_BUCKETS)))
    return time.perf_counter() - t0


def cpu_sample_text(rows, files, cores):
    return (f"{rows} rows of T in {files} Parquet files per step, one createIndex each: pyarrow decode (one task per file over "
            f"{cores} threads) + pthreads C Murmur3 bucket + per-bucket radix sort + pyarrow encode of 200 bucket files "
            "(oracle port; the reference is Scala on Spark and cannot run without a JVM)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O

    O.lib()  # built by __graft_entry__.build(); no staleness rebuild here, as the tree may be read-only
    cores = os.cpu_count() or 1
    rows, files = args.cpu_sample_rows, args.cpu_sample_files
    rows = rows // files * files
    with tempfile.TemporaryDirectory() as wd:
        paths = cpu_write_sources(rows, files, cores, wd)
        for _ in range(args.warmup):
            cpu_create_index(paths, cores, wd)
        times = [cpu_create_index(paths, cores, wd) for _ in range(args.steps)]
    sec = sum(times) / len(times)
    value = rows / sec
    line = {
        "impl": "reference", "metric": "createIndex rows/sec", "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "kind": "port", "sample": cpu_sample_text(rows, files, cores),
                         "step_s_min": min(times), "step_s_max": max(times), "spread": (max(times) - min(times)) / min(times)},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args):
    return {"workload": "createIndex: 1B rows x (k:int64 indexed; v1:int64, v2:float64, v3:int32, v4:float32 included), "
                        "200 buckets, 256 source Parquet files" if args.rows == 1_000_000_000 else
                        f"createIndex: {args.rows} rows x 5 columns of T, 200 buckets, {args.files} source Parquet files",
            "rows": args.rows, "source_files": args.files, "num_buckets": NUM_BUCKETS,
            "source_encoding": "PLAIN, UNCOMPRESSED" if args.plain else
            "PLAIN_DICTIONARY (v1, v3, v4) + PLAIN (k, v2), UNCOMPRESSED -- what parquet-mr / pyarrow write by default minus snappy",
            "index_encoding": "PLAIN, UNCOMPRESSED" if args.plain else "PLAIN_DICTIONARY (v1, v3, v4) + PLAIN (k, v2), UNCOMPRESSED",
            "l2": "inputs (>= 32 B/row x rows) far exceed the 126 MB L2; no flush needed",
            "cpu_sample_rows": args.cpu_sample_rows // args.cpu_sample_files * args.cpu_sample_files,
            "cpu_sample_files": args.cpu_sample_files}


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------

class Rig:
    """One rank's context + the torch.distributed plumbing around it."""

    def __init__(self, args):
        import torch

        from hyperspace_b200 import _native as N

        self.torch, self.N, self.args = torch, N, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (the engine has no CPU fallback); use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local_rank)
        # host threads and pinned file images next to this rank's GPU (matters once several ranks copy at the same time)
        from hyperspace_b200.distributed import bind_to_gpu_numa_node

        self.numa_node = bind_to_gpu_numa_node(self.local_rank) if self.world > 1 else None
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist_mod

            self.dist = dist_mod
            self.dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.stream = torch.cuda.current_stream()
        self.ctx = N.Context(self.local_rank, self.stream.cuda_stream)
        if self.world > 1:
            ids = [N.Context.comm_unique_id() if self.rank == 0 else None]
            self.dist.broadcast_object_list(ids, src=0)
            self.ctx.comm_init(self.rank, self.world, ids[0])

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms: float) -> float:
        if not self.dist:
            return ms
        t = self.torch.tensor([ms], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather_objects(self, obj):
        if not self.dist:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def timed(self, fn):
        """barrier; CUDA events around fn() on the library's stream; barrier; max over ranks (ms)."""
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record(self.stream)
        out = fn()
        e1.record(self.stream)
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)), out

    def close(self):
        self.ctx.close()
        if self.dist:
            self.dist.destroy_process_group()


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        try:
            return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def roofline_of(kernels, steps, rows_in, rows_out, value, world):
    """Roofline of the kernel with the largest share of the step, from the library's per-launch CUDA events."""
    peak, peak_src = hbm_peak()
    if not kernels:
        return None
    per_step = {k: v["ms"] / steps for k, v in sorted(kernels.items(), key=lambda kv: -kv[1]["ms"])}
    known = [k for k in per_step if k in KERNEL_BYTES]
    if not known:
        return {"bound": "hbm", "peak": peak, "peak_source": peak_src, "unit": "GB/s", "kernel_ms_per_step": per_step}
    name = known[0]
    kb, ks = KERNEL_BYTES[name], kernels[name]
    launches_per_step = max(1.0, ks["launches"] / steps)
    rows = rows_in if kb["rows"] == "in" else rows_out
    bytes_per_row = (kb["first"] + kb["rest"] * (launches_per_step - 1)) / launches_per_step
    avg_ms = ks["ms"] / max(1, ks["launches"])
    achieved = bytes_per_row * rows / (avg_ms / 1e3) / 1e9
    traffic, traffic_note = None, None
    for fn in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", fn)))[name]
            per_row = (tr["dram_bytes_read"] + tr["dram_bytes_write"]) / tr["rows_per_launch"]
            traffic = per_row * rows
            traffic_note = (f"dram__bytes_read+write.sum = {per_row:.2f} B/row measured by ncu --set full at "
                            f"{tr['rows_per_launch']} rows/launch (profiles/{fn}), scaled to this launch size")
            break
        except Exception:
            continue
    return {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
            "algorithmic_bytes_per_launch": bytes_per_row * rows,
            "algorithmic_bytes_note": f"{launches_per_step:.0f} launches per step; {kb['note']}",
            "avg_launch_ms": avg_ms, "launches_timed": ks["launches"],
            "whole_path": {"achieved": ALGO_BYTES_PER_ROW * value / world / 1e9, "unit": "GB/s",
                           "frac": ALGO_BYTES_PER_ROW * value / world / 1e9 / peak,
                           "note": "64 algorithmic B/row x rows/s per GPU vs HBM peak (SURVEY.md 8d yardstick)"},
            "kernel_ms_per_step": per_step}


def verify_output(rig, res, first_row, my_rows, total_rows, what):
    """Checks one createIndex result (host or device images) of this rank; returns the 'verified' object (rank 0) and ok."""
    import numpy as np

    N, ctx = rig.N, rig.ctx
    buckets = [f.bucket for f in res.files]
    t0 = time.perf_counter()
    rep = ctx.verify_index(res.as_sources(), buckets, INDEXED, INCLUDED, NUM_BUCKETS)
    gen = ctx.synth_checksum(first_row, my_rows, 5)
    mine = {"rep": rep, "gen": gen, "buckets": buckets, "file_rows": [f.rows for f in res.files]}
    allr = rig.gather_objects(mine)
    M = 1 << 64
    rows = sum(a["rep"]["rows"] for a in allr)
    all_buckets = [b for a in allr for b in a["buckets"]]
    ok = {
        "rows": rows == total_rows == sum(r for a in allr for r in a["file_rows"]),
        "bucket_ids": sum(a["rep"]["bucket_mismatches"] for a in allr) == 0,
        "sorted": sum(a["rep"]["order_violations"] for a in allr) == 0,
        "row_checksum": sum(a["rep"]["row_checksum"] for a in allr) % M == sum(a["gen"]["row_checksum"] for a in allr) % M,
        "column_checksums": all(sum(a["rep"]["column_checksum"][c] for a in allr) % M == sum(a["gen"]["column_checksum"][c] for a in allr) % M
                                for c in range(5)),
        "one_file_per_bucket": len(all_buckets) == len(set(all_buckets)) and all(b % rig.world == r for r, a in enumerate(allr) for b in a["buckets"]),
    }
    gpu_s = time.perf_counter() - t0
    # host side, rank 0: two whole buckets (its first and last file) decoded by pyarrow against the CPU oracle
    oracle_buckets, oracle_ok, oracle_s = [], None, 0.0
    if rig.rank == 0 and res.output == N.HS_OUT_HOST and res.files:
        import pyarrow as pa
        import pyarrow.parquet as pq

        from oracle import oracle as O

        O.lib()  # built by __graft_entry__.build(); no staleness rebuild here, as the tree may be read-only
        t1 = time.perf_counter()
        oracle_ok = True
        for i in sorted({0, len(res.files) - 1}):
            f = res.files[i]
            want = O.synthetic_bucket(0, total_rows, NUM_BUCKETS, f.bucket, 5, nthreads=os.cpu_count() or 1)
            got = pq.ParquetFile(pa.py_buffer(res.host_view(i))).read()
            same = got.num_rows == len(want["k"]) and all(
                np.array_equal(got.column(c).to_numpy().view(np.uint8), want[c].view(np.uint8)) for c in INDEXED + INCLUDED)
            oracle_ok = oracle_ok and bool(same)
            oracle_buckets.append(f.bucket)
        oracle_s = time.perf_counter() - t1
    flags = rig.gather_objects(oracle_ok)
    oracle_ok = flags[0]
    all_ok = all(ok.values()) and oracle_ok is not False
    verified = {"ok": bool(all_ok), "what": what, "rows_checked": rows, "files_checked": len(all_buckets), "checks": ok,
                "oracle_buckets": oracle_buckets, "oracle_buckets_equal": oracle_ok,
                "how": "GPU (hs_verify_index, every row of every index file of every rank): pmod(murmur3(k)) == bucket of the file, "
                       "adjacent keys ascending, row count, order-independent 64-bit row and column checksums == hs_synth_checksum "
                       "of the generator; host: whole bucket files read by pyarrow == oracle.synthetic_bucket (bit-exact, incl. order)",
                "seconds": {"gpu": gpu_s, "oracle": oracle_s}}
    return verified, all_ok


DUMP_SAMPLE_ROWS = 1 << 19  # index rows written by --dump-outputs over all buckets (~36 MB of .npy files)
DUMP_SEED = 20201017


def _float_columns(name, a):
    """A column as float arrays that hold it exactly: int64 as its high (signed) and low 32 bits, int32 and float64 as
    float64, float32 as is."""
    import numpy as np

    if a.dtype == np.int64:
        return {f"{name}_hi": (a >> 32).astype(np.float64), f"{name}_lo": (a & 0xFFFFFFFF).astype(np.float64)}
    if a.dtype == np.float32:
        return {name: a}
    return {name: a.astype(np.float64)}


def dump_outputs(rig, res, out_dir):
    """Writes what a caller of createIndex receives, for comparing two builds output for output: the row count of every
    bucket file, and for a seeded sample of positions inside every bucket file (the same positions whenever the bucket
    holds the same number of rows) the bucket, the position and every column of the rows found there.  `res` holds
    this rank's index files in HBM; rank 0 writes DIR/<name>.npy.  Returns what was written (rank 0)."""
    import types
    from concurrent.futures import ThreadPoolExecutor

    import numpy as np
    import pyarrow as pa
    import pyarrow.parquet as pq

    torch = rig.torch
    device = torch.device("cuda", rig.local_rank)
    per_bucket = max(1, DUMP_SAMPLE_ROWS // NUM_BUCKETS)

    def sample(f):
        # the engine's device allocation, wrapped by torch without a copy, then copied to the host
        cai = {"shape": (f.size,), "typestr": "|u1", "data": (f.ptr, False), "version": 3}
        # (worker threads start on device 0: name this rank's device, or the image would travel through GPU 0)
        image = torch.as_tensor(types.SimpleNamespace(__cuda_array_interface__=cai), device=device).cpu().numpy()
        t = pq.ParquetFile(pa.BufferReader(image)).read(columns=INDEXED + INCLUDED)
        rng = np.random.default_rng([DUMP_SEED, f.bucket])
        pos = np.sort(rng.choice(t.num_rows, size=min(per_bucket, t.num_rows), replace=False))
        rows = t.take(pa.array(pos))
        cols = {"bucket": np.full(len(pos), f.bucket, dtype=np.float64), "position": pos.astype(np.float64)}
        for c in INDEXED + INCLUDED:
            cols.update(_float_columns(c, rows.column(c).to_numpy()))
        return f.bucket, t.num_rows, cols

    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        mine = list(ex.map(sample, res.files))
    everything = sorted((s for part in rig.gather_objects(mine) for s in part), key=lambda s: s[0])
    if rig.rank != 0:
        return None
    bucket_rows = np.zeros(NUM_BUCKETS, dtype=np.float64)
    for b, n, _ in everything:
        bucket_rows[b] = n
    arrays = {"bucket_rows": bucket_rows}
    for name in everything[0][2] if everything else ():
        arrays[name] = np.concatenate([cols[name] for _, _, cols in everything])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return {"dir": out_dir, "arrays": sorted(arrays), "rows_sampled": int(len(arrays.get("bucket", ()))),
            "bytes": int(sum(a.nbytes for a in arrays.values())),
            "what": f"index files of the last timed step: rows of every bucket file, and at up to {per_bucket} seeded "
                    f"positions per bucket file (seed {DUMP_SEED}) the bucket, the position and every column; int64 "
                    "columns as <name>_hi / <name>_lo (high and low 32 bits)"}


def run_create_index(rig, args):
    N, ctx, torch = rig.N, rig.ctx, rig.torch
    world, rank = rig.world, rig.rank
    n_files = args.files
    rows_per_file = args.rows // n_files
    f0, f1 = rank * n_files // world, (rank + 1) * n_files // world
    my_files = f1 - f0
    my_rows = my_files * rows_per_file
    total_rows = rows_per_file * n_files
    first_row = f0 * rows_per_file
    kw = dict(job_uuid="bench", dictionary=not args.plain)

    # ---- inputs resident in HBM -----------------------------------------------------------------------------------
    src = ctx.synth_table(first_row, my_rows, 5, n_files=my_files, row_groups_per_file=4, output=N.HS_OUT_DEVICE,
                          dictionary=not args.plain)
    sources = src.as_sources()
    src_bytes = sum(f.size for f in src.files)

    kept = [None]  # index files of the last timed step, left in HBM for --dump-outputs

    def step_device(keep=False):
        res, st = ctx.create_index(sources, INDEXED, INCLUDED, NUM_BUCKETS, output=N.HS_OUT_DEVICE, **kw)
        if keep:
            kept[0] = res
        else:
            res.free()
        return st

    for _ in range(args.warmup):
        step_device()
    rig.barrier()
    ctx.profile_enable(True)
    sampler = ClockSampler(rig.local_rank)
    if rank == 0:
        sampler.start()
    launches = 0
    stage_ms = {}
    rows_out = [0]

    def timed_steps():
        nonlocal launches
        for i in range(args.steps):
            st = step_device(keep=bool(args.dump_outputs) and i == args.steps - 1)
            launches += int(st["gpu_launches"])
            rows_out[0] = int(st["rows_out"])
            for k, v in st.items():
                if k.startswith("ms_"):
                    stage_ms[k] = stage_ms.get(k, 0.0) + v / args.steps

    try:
        ms_total, _ = rig.timed(timed_steps)
    finally:
        clocks = sampler.stop() if rank == 0 else None  # never leave nvidia-smi running behind a failed step
    kernels = ctx.profile_report()
    ctx.profile_enable(False)
    dumped = None
    if args.dump_outputs:
        dumped = dump_outputs(rig, kept[0], args.dump_outputs)
        kept[0].free()
    ms_dev = ms_total / args.steps
    value = total_rows / (ms_dev / 1e3)
    roofline = roofline_of(kernels, args.steps, my_rows, rows_out[0] or total_rows / world, value, world)

    # ---- e2e: host images in, host images out, software-pipelined across steps ---------------------------------------
    e2e, verified, verified_ok = None, None, True
    last = [None]  # result of the last e2e step, kept for verification
    if not args.no_e2e:
        # "the caller's Parquet files in host memory": the same synthetic table, generated again straight into pinned
        # host memory (outside the timed region)
        src.free()
        ctx.trim()
        hsrc = ctx.synth_table(first_row, my_rows, 5, n_files=my_files, row_groups_per_file=4, output=N.HS_OUT_HOST,
                               dictionary=not args.plain)
        host_in = hsrc.as_sources()
        out_bytes = [0]

        def consume(pending, keep=False):
            res, st = pending.wait()
            out_bytes[0] = sum(f.size for f in res.files)
            chk = 0  # read the result on the host: first and last byte of every file image (complete Parquet files)
            for i in range(len(res.files)):
                v = res.host_view(i)
                chk += int(v[0]) + int(v[-1])
            if keep:
                last[0] = res
            else:
                res.free()
            return st

        copy_ms = {"h2d": [], "d2h": [], "build": []}

        def pipelined(steps, keep_last=False):
            """stage(i+1) | build(i) | drain(i-1): three calls in flight, each step's copies inside this function."""
            nxt = ctx.stage_sources(host_in)
            prev = None
            for i in range(steps):
                cur, nxt = nxt, (ctx.stage_sources(host_in) if i + 1 < steps else None)
                pend = ctx.create_index_async(cur.as_sources(), INDEXED, INCLUDED, NUM_BUCKETS, output=N.HS_OUT_HOST, **kw)
                copy_ms["h2d"].append(cur.wait())
                cur.free()
                if prev is not None:
                    st = consume(prev)
                    copy_ms["d2h"].append(st["ms_d2h"])
                    copy_ms["build"].append(st["ms_total"] - st["ms_d2h"])
                prev = pend
            consume(prev, keep=keep_last)

        def single_call():
            res, st = ctx.create_index(host_in, INDEXED, INCLUDED, NUM_BUCKETS, output=N.HS_OUT_HOST, **kw)
            v = res.host_view(0)
            _ = int(v[0]) + int(v[-1])
            res.free()
            return st

        # at least two steps: a one-step warm-up never has two calls in flight, and the timed steps then pay for that
        # set-up (e2e about 10x slower with --warmup 1 on a B200 at 1000 W)
        pipelined(max(2, args.warmup))
        for v in copy_ms.values():
            v.clear()
        ms_pipe, _ = rig.timed(lambda: pipelined(args.steps, keep_last=not args.no_verify))
        avg = lambda v: (sum(v) / len(v)) if v else None  # noqa: E731
        ms_e2e = ms_pipe / args.steps
        for _ in range(args.warmup):
            single_call()
        ms_single, st_single = rig.timed(lambda: [single_call() for _ in range(args.steps)][-1])
        ms_single /= args.steps
        e2e = {"value": total_rows / (ms_e2e / 1e3), "unit": "rows/s", "h2d_bytes_per_step": int(src_bytes),
               "d2h_bytes_per_step": int(out_bytes[0]), "ms_per_step": ms_e2e,
               "h2d_GBps_per_rank": src_bytes / (ms_e2e / 1e3) / 1e9, "d2h_GBps_per_rank": out_bytes[0] / (ms_e2e / 1e3) / 1e9,
               "calls_in_flight": 3, "single_call_ms": ms_single, "numa_node_bound": rig.numa_node,
               "pipelined_ms": {"h2d_copy": avg(copy_ms["h2d"]), "d2h_copy": avg(copy_ms["d2h"]), "build": avg(copy_ms["build"])},
               "single_call_copy_ms": {"h2d": st_single.get("ms_h2d"), "d2h": st_single.get("ms_d2h")},
               "note": "pinned HOST Parquet images in, HOST index images out, per-rank bytes; timed over K steps software-pipelined "
                       "through hs_stage_sources / hs_create_index_async / hs_pending_wait (H2D of step i+1 and D2H of step i-1 "
                       "beside the kernels of step i; every step's copies are inside the timed region, fill and drain included). "
                       "single_call_ms = one synchronous hs_create_index, averaged over K calls (H2D, build, D2H back to back: "
                       "a call cannot overlap its own copies because every index file depends on every source file)"}
        if not args.no_verify:
            verified, verified_ok = verify_output(rig, last[0], first_row, my_rows, total_rows,
                                                  "index files of the last timed e2e step (host images)")
            last[0].free()
        hsrc.free()
    elif not args.no_verify:
        res, _ = ctx.create_index(sources, INDEXED, INCLUDED, NUM_BUCKETS, output=N.HS_OUT_HOST, **kw)
        verified, verified_ok = verify_output(rig, res, first_row, my_rows, total_rows,
                                              "index files of one more createIndex over the resident sources (host images)")
        res.free()
        src.free()
    ctx.trim()

    line = {
        "metric": "createIndex rows/sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic", "config": workload_config(args),
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "verified": verified,
        "stage_ms_per_step": stage_ms,
    }
    if dumped:
        line["dump_outputs"] = dumped
    return line, verified_ok


def run_ours(args):
    rig = Rig(args)
    rank, world = rig.rank, rig.world
    ok = True
    if args.workload == "createIndex":
        line, ok = run_create_index(rig, args)
        if not args.no_extra:
            try:
                import bench_workloads as BW

                line["extra"] = BW.run_all(rig, args)
            except Exception as ex:  # the extra workloads must never take the headline number down with them
                line["extra"] = {"failed": f"{type(ex).__name__}: {ex}"}
    else:
        import bench_workloads as BW

        line = BW.run_one(rig, args)
    # ---- CPU baseline (rank 0, N=1 only) -----------------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.workload == "createIndex":
        try:
            from oracle import oracle as O

            O.lib()  # built by __graft_entry__.build(); no staleness rebuild here, as the tree may be read-only
            cores = os.cpu_count() or 1
            files = args.cpu_sample_files
            rows = args.cpu_sample_rows // files * files
            with tempfile.TemporaryDirectory() as wd:
                paths = cpu_write_sources(rows, files, cores, wd)
                cpu_create_index(paths, cores, wd)  # warm
                times = [cpu_create_index(paths, cores, wd) for _ in range(3)]
            cpu = {"value": rows / min(times), "unit": "rows/s", "cores": cores, "kind": "port",
                   "sample": cpu_sample_text(rows, files, cores) + f"; best of 3 ({min(times):.2f} s), spread "
                             f"{(max(times) - min(times)) / min(times):.1%}",
                   "step_s": times}
        except Exception as ex:  # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": "rows/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
    if rank == 0:
        if args.workload == "createIndex":
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
        sys.stdout.flush()
    rig.close()
    if not ok:
        if rank == 0:
            print("bench.py: verification of the benchmark output FAILED (see 'verified' in the line above)", file=sys.stderr)
        sys.exit(1)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
