"""--cluster_fast with --strand both against plus only on the device, on configs[2]-shaped reads (300 nt, 1 % divergence,
Zipf-ish root choice) of which about 40 % are reverse-complemented.  For each mode: reads/s (host clock around upload,
DUST, clustering and results, ending in a device synchronise), kernel launches per round, aligned pairs and DP cells,
and the VSG_TRACE phase split of the timed runs.  With oracle/_ref/vsearch present it also runs
`vsearch --cluster_fast --strand both` at the same round size (--threads) and checks that the cluster count is equal.
Prints the GPU's name and power limit with the numbers.  Measurement only; not part of the product.

    python tools/cluster_strand_bench.py [--reads N] [--round T] [--steps K] [--out DIR]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["VSG_TRACE"] = "1"       # read once by libvsg; one line per vsg_cluster_fast call

import numpy as np  # noqa: E402

from vsearch_b200 import lib as vlib, synth  # noqa: E402

_COMP = bytes.maketrans(b"ACGT", b"TGCA")


def reads_of(n, flip, seed=3):
    rng = np.random.default_rng(seed)
    nroots = max(50, n // 200)
    roots = synth.random_seqs(rng, nroots, 300)
    w = 1.0 / np.arange(1, nroots + 1); w /= w.sum()
    m = synth.mutate_batch(rng, roots[rng.choice(nroots, size=n, p=w)], 0.01)
    rev = rng.random(n) < flip
    return [m.seq(i).translate(_COMP)[::-1] if rev[i] else m.seq(i) for i in range(n)], int(rev.sum())


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
    with open(log, "ab") as f:
        os.dup2(f.fileno(), 2)
        try:
            return fn()
        finally:
            os.dup2(saved, 2); os.close(saved)


PHASES = ("rank", "candidate groups", "speculative extras", "serial pass", "index append")


def phase_sum(log):
    tot = dict.fromkeys(PHASES, 0.0)
    for line in open(log):
        for ph in PHASES:
            m = re.search(re.escape(ph) + r" (\d+) ms", line)
            if m:
                tot[ph] += float(m.group(1))
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=100_000)
    ap.add_argument("--round", type=int, default=0, help="round size = the reference's --threads (0 = host cores)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--flip", type=float, default=0.4, help="share of reads reverse-complemented")
    ap.add_argument("--no-reference", action="store_true")
    ap.add_argument("--out", default=None, help="directory for the trace logs (default: a temporary one)")
    a = ap.parse_args()
    T = a.round if a.round > 0 else (os.cpu_count() or 1)
    n = a.reads
    reads, nrev = reads_of(n, a.flip)
    labels = [f"a{i:08d}" for i in range(n)]
    order = sorted(range(n), key=lambda i: (-len(reads[i]), labels[i]))    # Database::sortbylength
    host = synth.SeqSet([reads[i] for i in order])
    out = a.out or tempfile.mkdtemp(prefix="cluster_strand_bench_")
    os.makedirs(out, exist_ok=True)
    card = gpu_info()
    rounds = (n + T - 1) // T
    ctx = vlib.Context(0)
    results = {}
    for mode in ("plus", "both"):
        o = vlib.default_search_opts(); o.id = 0.97; o.mask_lower = 1; o.maxrejects = 8
        o.strand_both = 1 if mode == "both" else 0
        log = os.path.join(out, f"trace_{mode}.log")

        def one():
            ss = ctx.seqset(host)
            ss.dust()
            r = vlib.cluster_fast(ctx, ss, o, T)
            ctx.sync()
            ss.close()
            return r
        one()                                                   # warm-up (module load, scratch growth)
        open(log, "wb").close()
        l0 = vlib.launch_count()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            res, ncl, work = run_traced(one, log)
        dt = (time.perf_counter() - t0) / a.steps
        launches = (vlib.launch_count() - l0) / a.steps
        ph = {k: v / a.steps for k, v in phase_sum(log).items()}
        results[mode] = {"mode": mode, "reads": n, "reversed_reads": nrev, "round_size": T, "reads_per_s": n / dt,
                         "ms_per_run": 1e3 * dt, "clusters": int(ncl), "minus_members": int(((res["centroid"] >= 0) & (res["strand"] == 1)).sum()),
                         "launches_per_round": launches / rounds, "pairs": int(work[0]), "dp_cells": int(work[1]),
                         "phase_ms": ph, "gpu": card}
        print(json.dumps(results[mode]), flush=True)
    ctx.close()
    stock = os.path.join(ROOT, "oracle", "_ref", "vsearch")
    if not a.no_reference and os.path.exists(stock):
        fa = os.path.join(out, "reads.fasta"); uc = os.path.join(out, "ref.uc")
        with open(fa, "wb") as f:
            for i in range(n):
                f.write(b">" + labels[i].encode() + b"\n" + reads[i] + b"\n")
        t0 = time.perf_counter()
        p = subprocess.run([stock, "--cluster_fast", fa, "--id", "0.97", "--strand", "both", "--threads", str(T), "--uc", uc, "--quiet"],
                           capture_output=True, text=True)
        dt = time.perf_counter() - t0
        assert p.returncode == 0, p.stderr[-1000:]
        ncl = sum(1 for l in open(uc) if l.startswith("S"))
        r = {"mode": "reference --strand both", "reads": n, "round_size": T, "reads_per_s": n / dt, "clusters": ncl,
             "cpu_cores": os.cpu_count(), "equal_cluster_count": ncl == results["both"]["clusters"]}
        print(json.dumps(r), flush=True)
        assert r["equal_cluster_count"], (ncl, results["both"]["clusters"])
    print(f"# GPU: {card}; {n} reads ({nrev} reverse-complemented), round size {T}")
    print("# mode   reads/s   launches/round   pairs   DP cells   " + "   ".join(f"{k} ms" for k in PHASES))
    for m, r in results.items():
        print(f"# {m:5s} {r['reads_per_s']:9.0f} {r['launches_per_round']:10.2f} {r['pairs']:10d} {r['dp_cells']:14d}   "
              + "   ".join(f"{r['phase_ms'][k]:.0f}" for k in PHASES))


if __name__ == "__main__":
    main()
