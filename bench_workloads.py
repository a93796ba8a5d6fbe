"""bench_workloads.py -- the read-side and refresh workloads of BASELINE.json configs[2..4], driven by bench.py
(``--workload filter|join|refresh``, and attached under ``extra`` of the default createIndex line at every N).

Sizes follow SURVEY.md section 8d, scaled from ``--rows`` (1 B by default):

  C3  FilterIndexRule scan (index/covering/FilterIndexRule.scala:135-149): ``k BETWEEN lo AND hi`` covering 1 % of the int64
      key space over the rows-row / 200-bucket index, projecting k, v1, v2 (~rows/100 rows out), 20 distinct ranges.
      Buckets are owner-sharded (bucket b lives on GPU b mod N, where createIndex wrote it): every rank scans its own files,
      no collective.  A step is one pass over the 20 ranges; queries/s = 20 x steps / time (max over ranks).
  C4  JoinIndexRule bucket-aligned merge join (index/covering/JoinIndexRule.scala:653-687): L = rows/2 rows with
      k = splitmix64(42, i); R = rows/2 rows whose keys are those of the first rows/4 rows of T, each twice => rows/2 matches,
      half of L unmatched.  ``SELECT L.v1, R.v2``.  Bucket b of L and of R sit on the same GPU by construction: no collective.
  C5  (i) refreshIndex(incremental) (index/covering/CoveringIndexTrait.scala:57-106): createIndex over rows/10 appended rows
      in 26 files, append mode; rows/s on the delta.  (ii) Hybrid Scan before the refresh
      (index/covering/CoveringIndexRuleUtils.scala:146-288): filter = index scan + raw predicate scan of the appended files;
      join = appended rows bucketed on the fly + merge join over buckets that now hold two files.

Every number carries its algorithmic bytes (SURVEY.md 8d "read side") and the achieved fraction of the HBM peak.
Every timed loop runs ``--warmup`` untimed repetitions and then ``--steps`` timed ones.
Index files stay resident in HBM (the index of a running cluster is hot in the scan cache); results are produced both
into pinned host memory (D2H inside the timed region) and left on the device for the next GPU operator.
"""
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NB = 200
QUERIES = 20


def _peak():
    import bench

    return bench.hbm_peak()[0]


def _sum_over_ranks(rig, v: float) -> float:
    if not rig.dist:
        return v
    t = rig.torch.tensor([v], device="cuda", dtype=rig.torch.float64)
    rig.dist.all_reduce(t)
    return float(t.item())


def _my_share(rig, first_row, rows, n_files):
    """This rank's contiguous share of a table of `rows` rows in `n_files` equal files: (first_row, rows, files)."""
    per = rows // n_files
    f0, f1 = rig.rank * n_files // rig.world, (rig.rank + 1) * n_files // rig.world
    return first_row + f0 * per, (f1 - f0) * per, f1 - f0


def _build_index(rig, first_row, rows, n_files, included, repeat=1, dictionary=True):
    """createIndex over rows [first_row, first_row + rows) of T (every source file listed `repeat` times); the index files of
    the buckets this rank owns stay in HBM."""
    N, ctx = rig.N, rig.ctx
    fr, my_rows, my_files = _my_share(rig, first_row, rows, n_files)
    src = ctx.synth_table(fr, my_rows, 5, n_files=max(1, my_files), row_groups_per_file=4, output=N.HS_OUT_DEVICE,
                          dictionary=dictionary)
    idx, st = ctx.create_index(src.as_sources() * repeat, ["k"], included, NB, output=N.HS_OUT_DEVICE, job_uuid="w",
                               dictionary=dictionary)
    src.free()
    ctx.trim()
    return idx


def _ranges(nq):
    width = int(0.01 * 2 ** 64)
    return [(-(width // 2) + i * (width // 40), (width // 2) + i * (width // 40)) for i in range(nq)]


# ---------------------------------------------------------------------------------------------------------------------
# C3
# ---------------------------------------------------------------------------------------------------------------------

def run_filter(rig, args, idx=None, appended=None):
    """C3 (appended = device source files not covered by the index: the Hybrid Scan variant of C5)."""
    N, ctx = rig.N, rig.ctx
    own = idx is None
    if own:
        idx = _build_index(rig, 0, args.rows, args.files, ["v1", "v2"])
    files = idx.as_sources()
    proj = ["k", "v1", "v2"]
    out = {}
    for mode, output in (("host", N.HS_OUT_HOST), ("device", N.HS_OUT_DEVICE)):
        def one(lo, hi):
            n = 0
            b, st = ctx.filter_scan(files, "k", proj, lo=lo, hi=hi, output=output)
            n += b.num_rows
            b.free()
            if appended:
                b, _ = ctx.filter_scan(appended, "k", proj, lo=lo, hi=hi, sorted_on_key=False, output=output)
                n += b.num_rows
                b.free()
            return n, st

        rs = _ranges(QUERIES)
        for _ in range(args.warmup):
            for lo, hi in rs:
                one(lo, hi)
        rows_out = [0]
        last = [None]

        def timed():
            for _ in range(args.steps):
                for lo, hi in rs:
                    n, st = one(lo, hi)
                    rows_out[0] += n
                    last[0] = st

        ms, _ = rig.timed(timed)
        nq = QUERIES * args.steps
        total_out = _sum_over_ranks(rig, rows_out[0])
        sec = ms / 1e3
        per_q = total_out / nq
        algo = per_q * 48.0  # 24 B read + 24 B written per qualifying row (SURVEY.md 8d); the probes are negligible
        out[mode] = {"queries_per_s": nq / sec, "ms_per_query": ms / nq, "rows_out_per_query": per_q,
                     "rows_out_per_s": total_out / sec, "algorithmic_GB_per_query": algo / 1e9,
                     "achieved_GBps_per_gpu": algo / (ms / nq / 1e3) / 1e9 / rig.world,
                     "frac_of_hbm_peak": algo / (ms / nq / 1e3) / 1e9 / rig.world / _peak()}
    # cross-check of one query: the indexed answer has as many rows as a full predicate scan of the same files
    lo, hi = _ranges(1)[0]
    a, _ = ctx.filter_scan(files, "k", ["k"], lo=lo, hi=hi, output=N.HS_OUT_DEVICE)
    b, _ = ctx.filter_scan(files, "k", ["k"], lo=lo, hi=hi, sorted_on_key=False, output=N.HS_OUT_DEVICE)
    same = a.num_rows == b.num_rows
    a.free()
    b.free()
    if own:
        idx.free()
        ctx.trim()
    res = {"workload": f"C3: k BETWEEN lo AND hi (1% of the key space) over the {args.rows}-row {NB}-bucket index, project k,v1,v2; "
                       f"{QUERIES} ranges per step; buckets owner-sharded over {rig.world} GPU(s), no collective; index resident in HBM",
           "result_to_host": out["host"], "result_on_device": out["device"],
           "checked": {"indexed_rows == full_scan_rows": bool(same)}}
    if appended:
        res["workload"] += f"; Hybrid Scan: + raw predicate scan of {len(appended)} appended source files"
    return res


# ---------------------------------------------------------------------------------------------------------------------
# C4
# ---------------------------------------------------------------------------------------------------------------------

def run_join(rig, args):
    N, ctx = rig.N, rig.ctx
    jr = args.rows // 2
    files = max(rig.world, args.files // 2)
    L = _build_index(rig, 0, jr, files, ["v1"])
    R = _build_index(rig, 0, jr // 2, max(rig.world, files // 2), ["v2"], repeat=2)  # every key of the first jr/2 rows twice
    lb, rb = [f.bucket for f in L.files], [f.bucket for f in R.files]
    out = {}
    nout_total = 0
    for mode, output in (("host", N.HS_OUT_HOST), ("device", N.HS_OUT_DEVICE)):
        def one():
            b, st = ctx.bucket_join(L.as_sources(), lb, R.as_sources(), rb, NB, "k", "k", ["v1"], ["v2"], output=output)
            n = b.num_rows
            b.free()
            return n, st

        for _ in range(args.warmup):
            one()
        acc = [0, None]

        def timed():
            for _ in range(args.steps):
                acc[0], acc[1] = one()

        ms, _ = rig.timed(timed)
        ms /= args.steps
        nout_total = _sum_over_ranks(rig, acc[0])
        algo = 16.0 * jr + 16.0 * jr + 16.0 * nout_total  # (k + payload) of both sides read once, 16 B per output row written
        out[mode] = {"joins_per_s": 1e3 / ms, "ms_per_join": ms, "rows_out": nout_total, "rows_out_per_s": nout_total / (ms / 1e3),
                     "algorithmic_GB": algo / 1e9, "achieved_GBps_per_gpu": algo / (ms / 1e3) / 1e9 / rig.world,
                     "frac_of_hbm_peak": algo / (ms / 1e3) / 1e9 / rig.world / _peak(),
                     # hs_stats has no field of its own for the join kernels: hs_bucket_join reports count + scan + emit +
                     # compose under ms_sort (nothing is sorted when every bucket holds one file)
                     "stage_ms_last": {("ms_join_kernels" if k == "ms_sort" else k): round(v, 3) for k, v in acc[1].items()
                                       if k.startswith("ms_") and v}}
    L.free()
    R.free()
    ctx.trim()
    return {"workload": f"C4: L = {jr} rows (k = splitmix64(42, i)), R = {jr} rows (keys of the first {jr // 2} rows, each twice), both "
                        f"indexed on k with {NB} buckets; SELECT L.v1, R.v2 FROM L JOIN R ON L.k = R.k; bucket-aligned merge join, "
                        f"no exchange; {rig.world} GPU(s); indexes resident in HBM",
            "result_to_host": out["host"], "result_on_device": out["device"],
            "checked": {"matches == rows/2": bool(int(nout_total) == jr)}}


# ---------------------------------------------------------------------------------------------------------------------
# C5
# ---------------------------------------------------------------------------------------------------------------------

def run_refresh(rig, args):
    N, ctx = rig.N, rig.ctx
    rows = args.rows
    delta = rows // 10
    dfiles = max(rig.world, 26)
    idx = _build_index(rig, 0, rows, args.files, ["v1", "v2", "v3", "v4"])
    fr, my_rows, my_files = _my_share(rig, rows, delta // dfiles * dfiles, dfiles)
    app = ctx.synth_table(fr, my_rows, 5, n_files=max(1, my_files), row_groups_per_file=4, output=N.HS_OUT_DEVICE)
    app_files = app.as_sources()
    total_delta = delta // dfiles * dfiles
    # (i) incremental refresh: the write path over the appended files only, append mode (log entry: old files U new files)
    def refresh():
        res, st = ctx.create_index(app_files, ["k"], ["v1", "v2", "v3", "v4"], NB, output=N.HS_OUT_DEVICE, job_uuid="inc",
                                   save_mode=N.HS_SAVE_APPEND)
        return res, st

    for _ in range(args.warmup):
        r, _ = refresh()
        r.free()
    keep = [None]

    def timed():
        for i in range(args.steps):
            res, st = refresh()
            if i == args.steps - 1:
                keep[0] = (res, st)
            else:
                res.free()

    ms, _ = rig.timed(timed)
    ms /= args.steps
    inc, st = keep[0]
    rep = ctx.verify_index(inc.as_sources(), [f.bucket for f in inc.files], ["k"], ["v1", "v2", "v3", "v4"], NB)
    gen = ctx.synth_checksum(fr, my_rows, 5)
    allr = rig.gather_objects((rep, gen))
    ok = (sum(a[0]["bucket_mismatches"] + a[0]["order_violations"] for a in allr) == 0 and
          sum(a[0]["rows"] for a in allr) == total_delta and
          sum(a[0]["row_checksum"] for a in allr) % 2 ** 64 == sum(a[1]["row_checksum"] for a in allr) % 2 ** 64)
    refresh_res = {"rows_per_s": total_delta / (ms / 1e3), "ms": ms, "delta_rows": total_delta, "delta_files": dfiles,
                   "files_written": int(_sum_over_ranks(rig, len(inc.files))),
                   "algorithmic_GB": 64.0 * total_delta / 1e9,
                   "frac_of_hbm_peak": 64.0 * total_delta / (ms / 1e3) / 1e9 / rig.world / _peak(),
                   "verified": bool(ok)}
    # (ii) Hybrid Scan before the refresh: filter
    hyb_filter = run_filter(rig, args, idx=idx, appended=app_files)
    # Hybrid Scan join: index (rows) JOIN-side = index U appended rows bucketed on the fly, against an index over the delta's
    # keys (so that every appended row finds its match and the multi-file bucket path does real work)
    other = inc  # index over the appended rows: its keys match exactly the appended part of the hybrid side
    ob = [f.bucket for f in other.files]

    def hybrid_join(output):
        tmp, _ = ctx.create_index(app_files, ["k"], ["v1"], NB, output=N.HS_OUT_DEVICE, job_uuid="hs")  # appended rows, on the fly
        files = idx.as_sources() + tmp.as_sources()
        buckets = [f.bucket for f in idx.files] + [f.bucket for f in tmp.files]
        b, stj = ctx.bucket_join(files, buckets, other.as_sources(), ob, NB, "k", "k", ["v1"], ["v2"], output=output)
        n = b.num_rows
        b.free()
        tmp.free()
        return n, stj

    for _ in range(args.warmup):
        hybrid_join(N.HS_OUT_DEVICE)
    acc = [0]

    def timed_join():
        for _ in range(args.steps):
            acc[0], _ = hybrid_join(N.HS_OUT_DEVICE)

    msj, _ = rig.timed(timed_join)
    msj /= args.steps
    nout = _sum_over_ranks(rig, acc[0])
    hyb_join = {"ms": msj, "rows_out": nout, "checked": {"matches == delta_rows": bool(int(nout) == total_delta)},
                "what": f"({rows}-row index U {total_delta} appended rows bucketed on the fly) JOIN ({total_delta}-row index) ON k; "
                        "result left on the device"}
    inc.free()
    app.free()
    idx.free()
    ctx.trim()
    return {"workload": f"C5: +{total_delta} rows appended as {dfiles} files onto the {rows}-row index; {rig.world} GPU(s)",
            "refresh_incremental": refresh_res, "hybrid_scan_filter": hyb_filter, "hybrid_scan_join": hyb_join}


# ---------------------------------------------------------------------------------------------------------------------
# SNAPPY variants of the createIndex workload (SURVEY.md 8d: "two variants: UNCOMPRESSED and SNAPPY (Spark's default)")
# ---------------------------------------------------------------------------------------------------------------------

def run_snappy(rig, args):
    N, ctx = rig.N, rig.ctx
    fr, my_rows, my_files = _my_share(rig, 0, args.rows // args.files * args.files, args.files)
    total_rows = args.rows // args.files * args.files
    inc = ["v1", "v2", "v3", "v4"]
    out = {}

    def timed_builds(sources, **kw):
        def one():
            res, st = ctx.create_index(sources, ["k"], inc, NB, output=N.HS_OUT_DEVICE, job_uuid="z", **kw)
            nbytes = sum(f.size for f in res.files)
            res.free()
            return st, nbytes
        for _ in range(args.warmup):
            one()
        ctx.profile_enable(True)
        acc = [None, 0]

        def loop():
            for _ in range(args.steps):
                acc[0], acc[1] = one()
        ms, _ = rig.timed(loop)
        kernels = ctx.profile_report()
        ctx.profile_enable(False)
        return ms / args.steps, {k: v["ms"] / args.steps for k, v in kernels.items()}, acc[1]

    usrc = ctx.synth_table(fr, my_rows, 5, n_files=max(1, my_files), row_groups_per_file=4, output=N.HS_OUT_DEVICE)
    ms_u, k_u, bytes_u = timed_builds(usrc.as_sources())
    ms_o, k_o, bytes_o = timed_builds(usrc.as_sources(), compression=N.HS_CODEC_SNAPPY)
    src_bytes_u = sum(f.size for f in usrc.files)
    usrc.free()
    ctx.trim()
    ssrc = ctx.synth_table(fr, my_rows, 5, n_files=max(1, my_files), row_groups_per_file=4, output=N.HS_OUT_DEVICE,
                           compression=N.HS_CODEC_SNAPPY)
    src_bytes_s = sum(f.size for f in ssrc.files)
    ms_s, k_s, _ = timed_builds(ssrc.as_sources())
    ssrc.free()
    ctx.trim()
    dec_ms = k_s.get("k_snappy_index", 0.0) + k_s.get("k_snappy_blocks", 0.0)
    comp_ms = k_o.get("k_snappy_compress", 0.0)
    out = {
        "workload": f"createIndex over {total_rows} rows of T: UNCOMPRESSED source and index (reference point), SNAPPY index, SNAPPY source; "
                    f"{rig.world} GPU(s), images resident in HBM",
        "uncompressed": {"rows_per_s": total_rows / (ms_u / 1e3), "ms": ms_u},
        "snappy_index": {"rows_per_s": total_rows / (ms_o / 1e3), "ms": ms_o, "relative": ms_u / ms_o,
                         "index_bytes_per_rank": bytes_o, "uncompressed_index_bytes_per_rank": bytes_u,
                         "k_snappy_compress_ms": comp_ms,
                         "compress_GBps_per_gpu": (bytes_u / (comp_ms / 1e3) / 1e9) if comp_ms else None,
                         "compress_frac_of_hbm_peak": (2 * bytes_u / (comp_ms / 1e3) / 1e9 / _peak()) if comp_ms else None},
        "snappy_source": {"rows_per_s": total_rows / (ms_s / 1e3), "ms": ms_s, "relative": ms_u / ms_s,
                          "source_bytes_per_rank": src_bytes_s, "uncompressed_source_bytes_per_rank": src_bytes_u,
                          "k_snappy_decompress_ms": dec_ms, "k_snappy_index_ms": k_s.get("k_snappy_index", 0.0),
                          "k_snappy_blocks_ms": k_s.get("k_snappy_blocks", 0.0),
                          "decompress_GBps_per_gpu": (src_bytes_u / (dec_ms / 1e3) / 1e9) if dec_ms else None,
                          "decompress_frac_of_hbm_peak": ((src_bytes_s + src_bytes_u) / (dec_ms / 1e3) / 1e9 / _peak()) if dec_ms else None},
    }
    return out


def run_files(rig, args):
    """The reference's actual effect: Parquet files in, bucket files out (index/DataFrameWriterExtensions.scala:50-68 writes
    them under <index>/v__=N).  createIndex with path sources and HS_OUT_FILES: file reads (a few host threads into pinned
    memory), H2D, build, D2H, file writes (a few host threads) -- one blocking call, nothing pipelined; the best of --steps
    calls after --warmup untimed ones.  tmpfs and, where a writable disk with room exists, the local file system; a quarter
    of --rows to keep the run short."""
    import shutil
    import tempfile
    import time

    N, ctx = rig.N, rig.ctx
    if rig.world > 1:
        return {"skipped": "measured on one GPU (the ranks of a multi-GPU build write disjoint bucket files the same way)"}
    rows = max(1 << 20, (args.rows // 4) // 64 * 64)
    n_files = 64
    src = ctx.synth_table(0, rows, 5, n_files=n_files, row_groups_per_file=4, output=N.HS_OUT_HOST)
    src_bytes = sum(f.size for f in src.files)
    out = {"workload": f"createIndex over {rows} rows of T from {n_files} Parquet files on a file system to {NB} index files on "
                       f"the same file system (hs_create_index, HS_OUT_FILES), one blocking call", "source_bytes": src_bytes}
    for label, base in (("tmpfs", "/dev/shm"), ("local_fs", tempfile.gettempdir())):
        try:
            if not os.path.isdir(base) or shutil.disk_usage(base).free < 3 * src_bytes + (1 << 30):
                out[label] = {"skipped": f"no room under {base}"}
                continue
            root = tempfile.mkdtemp(prefix="hs_bench_", dir=base)
        except Exception as ex:
            out[label] = {"skipped": f"{type(ex).__name__}: {ex}"}
            continue
        try:
            paths = []
            for i, f in enumerate(src.files):
                p = os.path.join(root, f"src-{i:03d}.parquet")
                with open(p, "wb") as fh:
                    fh.write(src.host_bytes(i))
                paths.append(p)
            files = [N.FileImage(path=p, file_id=i) for i, p in enumerate(paths)]
            best, stats, out_dir = None, None, None
            for rep in range(args.warmup + args.steps):
                if out_dir:
                    shutil.rmtree(out_dir)  # keep one call's output at a time: the room needed does not grow with --steps
                out_dir = os.path.join(root, f"v__={rep}")
                t0 = time.perf_counter()
                res, st = ctx.create_index(files, ["k"], ["v1", "v2", "v3", "v4"], NB, out_dir=out_dir, output=N.HS_OUT_FILES,
                                           job_uuid="f")
                dt = time.perf_counter() - t0
                n_out = len(res.files)
                res.free()
                if rep >= args.warmup and (best is None or dt < best):
                    best, stats = dt, st
            idx_bytes = sum(os.path.getsize(os.path.join(out_dir, n)) for n in os.listdir(out_dir) if n.endswith(".parquet"))
            out[label] = {"rows_per_s": rows / best, "ms": best * 1e3, "index_files": n_out, "index_bytes": idx_bytes,
                          "GBps_in_plus_out": (src_bytes + idx_bytes) / best / 1e9,
                          "stage_ms": {k: round(v, 2) for k, v in stats.items() if k.startswith("ms_")},
                          "note": f"wall clock of the call, best of {args.steps} after {args.warmup} warm-up call(s); files come from / "
                                  "go to the page cache"}
        except Exception as ex:
            out[label] = {"failed": f"{type(ex).__name__}: {ex}"}
        finally:
            shutil.rmtree(root, ignore_errors=True)
    src.free()
    ctx.trim()
    return out


# ---------------------------------------------------------------------------------------------------------------------

def run_all(rig, args):
    out = {}
    for name, fn in (("filter_C3", run_filter), ("join_C4", run_join), ("refresh_C5", run_refresh), ("snappy_variants", run_snappy),
                     ("files_in_files_out", run_files)):
        try:
            out[name] = fn(rig, args)
        except Exception as ex:
            out[name] = {"failed": f"{type(ex).__name__}: {ex}"}
            try:
                rig.ctx.trim()
            except Exception:
                pass
    return out


def run_one(rig, args):
    import bench

    fn = {"filter": run_filter, "join": run_join, "refresh": run_refresh, "snappy": run_snappy, "files": run_files}[args.workload]
    res = fn(rig, args)
    if args.workload == "files":
        best = max((v.get("rows_per_s", 0.0) for v in res.values() if isinstance(v, dict)), default=0.0)
        metric, value, unit = "createIndex rows/sec, files in -> files out", best, "rows/s"
    elif args.workload == "snappy":
        metric, value, unit = "createIndex rows/sec over a SNAPPY source", res["snappy_source"]["rows_per_s"], "rows/s"
    elif args.workload == "filter":
        metric, value, unit = "filter queries/sec", res["result_to_host"]["queries_per_s"], "queries/s"
    elif args.workload == "join":
        metric, value, unit = "join queries/sec", res["result_to_host"]["joins_per_s"], "joins/s"
    else:
        metric, value, unit = "refreshIndex(incremental) rows/sec", res["refresh_incremental"]["rows_per_s"], "rows/s"
    return {"metric": metric, "value": value, "unit": unit, "n_gpus": rig.world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": res["workload"], "rows": args.rows, "num_buckets": NB}, "detail": res}
