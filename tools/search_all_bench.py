"""--usearch_global with candidate lists longer than the ranker's 1 024-entry shared-memory list, on configs[1]-shaped
inputs (bench.py's usearch workload: a 100 000 x 1 500-nt random database, 250-nt windows mutated 5 %, --id 0.9,
wordlength 8, no masking).  Three configurations of the same queries:

  (a) defaults: --maxaccepts 1 --maxrejects 32 (control; the shared-memory ranker)
  (b) --maxaccepts 0 --maxrejects 32 --maxhits 10 (LULU-style match lists)
  (c) --maxaccepts 0 --maxrejects 0 (exhaustive)

For each: queries/s (host clock around one vsg_search_batch call, which ends in a device synchronise), candidates per
query (mean, p50, p99, from vsg_rank on a sample), the reference-counted pairs and DP cells (work[0..1]) and GCUPS over
them, ranking kernel time (pass A + pass B + sort; or the one ranking pass of (a)) against forward + traceback kernel
time (cudaEvents; summed over the driver's worker streams, so they overlap), and the number of sub-batch pieces beyond
the first (candidate-volume splits, from VSG_TRACE).  For (b) and (c) it also times the reference's search_batch
(oracle/_ref) on this box's host cores on a sample of the queries and checks the first hit per query against the
device, as bench.py's parity gate does.  Prints the GPU's name, power limit and max SM clock.  Measurement only.

    python tools/search_all_bench.py [--queries N] [--ref-sample S] [--out DIR]
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ["VSG_TRACE"] = "1"       # read by libvsg; the driver reports its pieces per sub-batch

import numpy as np  # noqa: E402

from vsearch_b200 import lib as vlib, synth  # noqa: E402

N_DB, DB_LEN, Q_LEN, DIV, SEED = 100_000, 1500, 250, 0.05, 2024
IDENT, K = 0.9, 8
CONFIGS = [("a_defaults", 1, 32, 0), ("b_maxaccepts0_maxrejects32_maxhits10", 0, 32, 10), ("c_maxaccepts0_maxrejects0", 0, 0, 0)]


def gpu_info():
    try:
        p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return p.stdout.strip().splitlines()[0] if p.returncode == 0 and p.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run_traced(fn, log):
    """fn() with the process's stderr (where libvsg writes its trace) sent to `log`"""
    sys.stderr.flush()
    saved = os.dup(2)
    with open(log, "wb") as f:
        os.dup2(f.fileno(), 2)
        try:
            return fn()
        finally:
            os.dup2(saved, 2); os.close(saved)


def clamp(v):
    return N_DB if v == 0 or v > N_DB else v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=20000)
    ap.add_argument("--ref-sample", type=int, default=200)
    ap.add_argument("--rank-sample", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    out = {"gpu": gpu_info(), "host_cores": os.cpu_count(), "queries": args.queries,
           "workload": f"configs[1] shape: {N_DB} x {DB_LEN} nt database, {Q_LEN}-nt queries, div {DIV}, id {IDENT}, k {K}"}
    print(json.dumps({"gpu": out["gpu"]}), flush=True)
    dbm = synth.config2_db(N_DB, DB_LEN, SEED)
    dbs = synth.SeqSet.from_matrix(dbm)
    qss, _ = synth.config2_query_batch(dbm, args.queries, Q_LEN, DIV, SEED, batch=0)
    ctx = vlib.Context(0)
    db = ctx.seqset(dbs); ix = ctx.index(db, K, 0); qs = ctx.seqset(qss)
    ns = min(args.rank_sample, args.queries)
    results = {}
    tmp = tempfile.mkdtemp()
    for name, ma, mr, maxhits in CONFIGS:
        o = vlib.default_search_opts(); o.id = IDENT; o.maxaccepts = ma; o.maxrejects = mr; o.wordlength = K
        max_results = maxhits if maxhits > 0 else 16
        ctx.search(ix, db, qs, 0, min(512, args.queries), o, max_results)          # warm-up (modules, allocations)
        ctx.profile_reset()
        log = os.path.join(tmp, name + ".log")
        t0 = time.perf_counter()
        res, counts, work = run_traced(lambda: ctx.search(ix, db, qs, 0, args.queries, o, max_results), log)
        dt = time.perf_counter() - t0
        prof = ctx.profile()
        trace = open(log).read()
        pieces = [int(x) for x in re.findall(r"searched in (\d+) pieces", trace)]
        tophits = min(clamp(ma) + clamp(mr) + 8, N_DB)
        _, _, nc = ctx.rank(ix, qs, 0, ns, 12, tophits)
        first = np.array([res[i * max_results].target if counts[i] > 0 else -1 for i in range(args.queries)], dtype=np.int32)
        r = {"queries_per_s": args.queries / dt, "seconds": dt, "tophits": tophits,
             "candidates_per_query": {"sample": ns, "mean": float(nc.mean()), "p50": float(np.percentile(nc, 50)),
                                      "p99": float(np.percentile(nc, 99)), "max": int(nc.max())},
             "pairs": int(work[0]), "dp_cells": int(work[1]), "gcups": float(work[1]) / dt / 1e9,
             "aligned_pairs": int(work[2]), "aligned_cells": int(work[3]),
             "rank_kernel_ms": prof.rank_ms, "align_kernel_ms": prof.fwd_ms + prof.traceback_ms,
             "sub_batches": len(pieces), "splits": int(sum(p - 1 for p in pieces)),
             "queries_with_hits": int((counts > 0).sum())}
        results[name] = (r, first)
        print(json.dumps({name: r}), flush=True)
    # the reference's search_batch on the host cores, first hit per query against the device
    import checkers
    lib = checkers.ref()
    ref = {}
    if lib is None:
        ref = {"unavailable": "oracle/_ref/libvsref.so not built"}
    else:
        cores = os.cpu_count() or 1
        sample = min(args.ref_sample, args.queries)
        sq = synth.SeqSet([qss.seq(i) for i in range(sample)])
        for name, ma, mr, _ in CONFIGS[1:]:
            rdb = checkers.RefDb(dbs, k=K, id=IDENT, maxaccepts=clamp(ma), maxrejects=clamp(mr))
            ft = np.zeros(sample, dtype=np.int32)
            lib.vsref_work_reset()
            t0 = time.perf_counter()
            lib.vsref_db_search_batch(C.c_void_p(rdb.h), C.c_int(sample), checkers._p(sq.cat, C.c_char),
                                      checkers._p(sq.offs, C.c_int64), checkers._p(sq.lens, C.c_int), C.c_int(cores),
                                      checkers._p(ft, C.c_int))
            dt = time.perf_counter() - t0
            p = C.c_longlong(); c = C.c_longlong(); k = C.c_longlong()
            lib.vsref_work_get(C.byref(p), C.byref(c), C.byref(k))
            rdb.close()
            dev_first = results[name][1][:sample]
            ref[name] = {"queries": sample, "threads": cores, "queries_per_s": sample / dt, "pairs": p.value,
                         "dp_cells": c.value, "gcups": c.value / dt / 1e9,
                         "parity_checked": sample, "parity_mismatches": int((dev_first != ft).sum())}
            print(json.dumps({"reference_" + name: ref[name]}), flush=True)
    out["device"] = {k: v[0] for k, v in results.items()}
    out["reference"] = ref
    out["gpu_after"] = gpu_info()
    qs.close(); ix.close(); db.close(); ctx.close()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        open(os.path.join(args.out, "search_all_bench.json"), "w").write(text)


if __name__ == "__main__":
    main()
