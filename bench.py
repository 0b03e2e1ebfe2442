#!/usr/bin/env python
"""bench.py — the hot path on BASELINE.json's headline configuration.

Workload (configs[1]): --usearch_global, 250-nt queries (5 % mutated windows of database
sequences) against a 100 000 x 1 500 nt iid database, --id 0.9, default scoring, k = 8,
maxaccepts 1 / maxrejects 32, masking none.  One STEP = one pass of the whole hot path (k-mer
ranking -> batched 16-bit global alignment -> traceback -> accept/reject replay) over one batch of
`--batch` queries of that stream per GPU; per-GPU work is fixed as N grows (weak scaling), the
database is broadcast from rank 0 over NCCL and every rank builds its index from it on device.

metric = GCUPS as SURVEY.md §8(d) defines it: sum over the pairs the reference's driver hands to
search16 of qlen*dlen, divided by time.  Our driver aligns exactly that set of pairs
(tests/test_search_gpu.py checks the counts against the reference), so numerator and unit are the
same for both arms.

  value   inputs (database, index, query batches) already resident in HBM when the timed region starts
  e2e     the same steps through the C ABI with HOST buffers: each step uploads its query batch from
          pinned host memory (vsg_seqset_create) and gets its hit table back in host memory
  --impl reference   the UNMODIFIED reference (oracle/_ref/libvsref.so: its own search_batch on all
          host threads, workload counted by a link-time wrapper around search16) on a bounded sample
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_DB, DB_LEN, Q_LEN, DIV, SEED = 100_000, 1500, 250, 0.05, 2024
IDENT, MAXACC, MAXREJ, K = 0.9, 1, 32, 8
WORKLOADS = {
    # configs[1]: the headline
    "usearch": dict(n_db=100_000, db_len=1500, q_len=250, div=0.05, seed=2024, ident=0.9,
                    name="usearch_global 250nt queries vs 100k x 1500nt DB, id 0.9 (configs[1])"),
    # configs[3] shape: 31 index shards, 2.4 GB of postings
    "c4": dict(n_db=1_000_000, db_len=1200, q_len=150, div=0.10, seed=4, ident=0.85,
               name="usearch_global 150nt queries vs 1M x 1200nt DB, id 0.85 (configs[3] shape)"),
}


def set_workload(name):
    global N_DB, DB_LEN, Q_LEN, DIV, SEED, IDENT, WL_NAME
    w = WORKLOADS[name]
    N_DB, DB_LEN, Q_LEN, DIV, SEED, IDENT = w["n_db"], w["db_len"], w["q_len"], w["div"], w["seed"], w["ident"]
    WL_NAME = w["name"]


WL_NAME = WORKLOADS["usearch"]["name"]


def host_info():
    """what the CPU arm ran on: the same "128 cores" gave 9.5 and 69 GCUPS on two boxes of the pool in round 1"""
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    try:
        la = [round(x, 2) for x in os.getloadavg()]
    except Exception:
        la = None
    return {"nproc": os.cpu_count(), "cpu_model": model, "loadavg_1_5_15": la}


def gpu_first_targets(qs, dust=False):
    """first hit per query through the product path (C ABI), for the parity gate; None without a GPU"""
    try:
        from vsearch_b200 import lib as vlib, synth
        ctx = vlib.Context(int(os.environ.get("LOCAL_RANK", "0")))
    except Exception:
        return None
    from vsearch_b200 import synth
    dbm = synth.config2_db(N_DB, DB_LEN, SEED)
    db = ctx.seqset(synth.SeqSet.from_matrix(dbm))
    if dust:
        db.dust()
    ix = ctx.index(db, K, 1 if dust else 0)
    h = ctx.seqset(qs)
    if dust:
        h.dust()
    o = vlib.default_search_opts()
    o.id = IDENT; o.maxaccepts = MAXACC; o.maxrejects = MAXREJ; o.wordlength = K; o.mask_lower = 1 if dust else 0
    res, counts, _ = ctx.search(ix, db, h, 0, len(qs), o, 1)
    out = np.array([res[i].target if counts[i] > 0 else -1 for i in range(len(qs))], dtype=np.int32)
    h.close(); ix.close(); db.close(); ctx.close()
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nme in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def pinned_seqset(ss):
    """copy a SeqSet's arrays into pinned host memory (torch allocator)"""
    import torch
    from vsearch_b200 import synth
    out = synth.SeqSet.__new__(synth.SeqSet)
    for name in ("cat", "offs", "lens"):
        a = getattr(ss, name)
        t = torch.empty(a.shape, dtype=getattr(torch, str(a.dtype)), pin_memory=True)
        v = t.numpy()
        v[...] = a
        setattr(out, name, v)
        setattr(out, "_keep_" + name, t)
    return out


def reference_arm(args, rank):
    """Times the unmodified reference on this box's host cores (rank 0 only).  Outside the timed region the
    same queries also go through the product path (if a GPU is present) and the first hit per query must agree."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import checkers
    from vsearch_b200 import synth
    cores = os.cpu_count() or 1
    if checkers.ref() is None:
        emit(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libvsref.so not built"}))
        return
    lib = checkers.ref()
    dust = 1 if args.masking == "dust" else 0
    dbm = synth.config2_db(N_DB, DB_LEN, SEED)
    dbs = synth.SeqSet.from_matrix(dbm)
    t0 = time.time()
    r = checkers.RefDb(dbs, k=K, id=IDENT, maxaccepts=MAXACC, maxrejects=MAXREJ, dust=dust)
    build_s = time.time() - t0
    sample = args.ref_sample
    times, cells_l, pairs_l = [], [], []
    last_qs, last_ft = None, None
    for step in range(args.warmup + args.steps):
        qs, _ = synth.config2_query_batch(dbm, sample, Q_LEN, DIV, SEED, batch=step)
        ft = np.zeros(sample, dtype=np.int32)
        lib.vsref_work_reset()
        t0 = time.perf_counter()
        lib.vsref_db_search_batch(C.c_void_p(r.h), C.c_int(sample), checkers._p(qs.cat, C.c_char),
                                  checkers._p(qs.offs, C.c_int64), checkers._p(qs.lens, C.c_int),
                                  C.c_int(cores), checkers._p(ft, C.c_int))
        dt = time.perf_counter() - t0
        p = C.c_longlong(); c = C.c_longlong(); k = C.c_longlong()
        lib.vsref_work_get(C.byref(p), C.byref(c), C.byref(k))
        if step >= args.warmup:
            times.append(dt); cells_l.append(c.value); pairs_l.append(p.value)
        last_qs, last_ft = qs, ft
    r.close()
    # parity gate (not timed): the last step's queries through the product path
    parity = {"parity_checked": 0, "parity_mismatches": 0}
    got = gpu_first_targets(last_qs, dust=bool(dust)) if not args.no_parity else None
    if got is not None:
        parity = {"parity_checked": int(sample), "parity_mismatches": int((got != last_ft).sum())}
    tot = sum(times)
    gcups = sum(cells_l) / tot / 1e9
    line = {"impl": "reference", "metric": "usearch_global_gcups", "value": gcups, "unit": "GCUPS",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * tot / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int16", "data": "synthetic",
            "config": {"workload": WL_NAME, "queries_per_step": sample, "masking": args.masking,
                       "wordlength": K, "maxaccepts": MAXACC, "maxrejects": MAXREJ,
                       "reference_index_build_s": round(build_s, 1)},
            "queries_per_s": sample * args.steps / tot, "pairs_per_s": sum(pairs_l) / tot,
            "host": host_info(),
            "cpu_baseline": {"value": gcups, "unit": "GCUPS", "cores": cores, "kind": "reference",
                             "sample": f"{sample} queries per step of the same stream, reference search_batch "
                                       f"--threads {cores}"},
            "e2e": {"value": gcups, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    line.update(parity)
    emit(json.dumps(line))
    if parity["parity_mismatches"]:
        raise SystemExit(3)


def allpairs_workload(args, rank, world, local):
    """configs[4] shape: --allpairs_global on 200 000 reads x 400 nt (2 000 roots, 15 % divergence),
    --id 0.7.  One step = `rows` query rows per GPU against all later reads (the full run would be
    3.2e15 cells; SURVEY.md §8d prescribes a stated prefix).  Rows shard across GPUs, no collective."""
    from vsearch_b200 import synth
    N_READS, L, ROOTS, DIVA, SEEDA, IDA = 200_000, 400, 2000, 0.15, 5, 0.7
    rng = np.random.default_rng(SEEDA)
    roots = synth.random_seqs(rng, ROOTS, L)
    reads = synth.mutate_batch(rng, roots[rng.integers(0, ROOTS, size=N_READS)], DIVA)
    nsteps = args.warmup + args.steps
    cfg = {"workload": "allpairs_global 200k x 400nt reads, id 0.7 (configs[4]), prefix of query rows",
           "masking": "none", "l2": "direction blocks of one step (> 100 GB streamed) exceed the 126 MB L2"}
    if args.impl == "reference":
        if rank != 0:
            return
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import checkers
        cores = os.cpu_count() or 1
        if checkers.ref() is None:
            emit(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libvsref.so not built"}))
            return
        lib = checkers.ref(); lib.vsref_allpairs_rows.restype = C.c_longlong
        if args.ref_rows <= 0:
            args.ref_rows = max(1, cores // 8)   # ~10-15 s of CPU work per step
        r = checkers.RefDb(reads, id=IDA, dust=0)
        tot_t = 0.0; tot_c = 0; tot_p = 0
        for step in range(nsteps):
            lib.vsref_work_reset()
            t0 = time.perf_counter()
            lib.vsref_allpairs_rows(C.c_void_p(r.h), C.c_int(step * args.ref_rows), C.c_int(args.ref_rows), C.c_int(cores))
            dt = time.perf_counter() - t0
            p = C.c_longlong(); c = C.c_longlong(); k = C.c_longlong()
            lib.vsref_work_get(C.byref(p), C.byref(c), C.byref(k))
            if step >= args.warmup:
                tot_t += dt; tot_c += c.value; tot_p += p.value
        r.close()
        g = tot_c / tot_t / 1e9
        cfg["rows_per_step"] = args.ref_rows
        emit(json.dumps({"impl": "reference", "metric": "allpairs_global_gcups", "value": g, "unit": "GCUPS",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "int16", "data": "synthetic", "config": cfg,
                          "pairs_per_s": tot_p / tot_t,
                          "cpu_baseline": {"value": g, "unit": "GCUPS", "cores": cores, "kind": "reference",
                                           "sample": f"{args.ref_rows} query rows per step, search16 on {cores} threads"},
                          "e2e": {"value": g, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch
    import torch.distributed as dist
    from vsearch_b200 import lib as vlib
    torch.cuda.set_device(local)
    pg_init(world, local)
    ctx = vlib.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream_ptr(), device=torch.device("cuda", local))
    if world > 1:   # rank 0's packed reads go to every GPU over NCCL
        d_cat = torch.empty(reads.cat.shape[0], dtype=torch.uint8, device="cuda")
        d_off = torch.empty(N_READS, dtype=torch.int64, device="cuda")
        d_len = torch.empty(N_READS, dtype=torch.int32, device="cuda")
        if rank == 0:
            d_cat.copy_(torch.from_numpy(reads.cat)); d_off.copy_(torch.from_numpy(reads.offs)); d_len.copy_(torch.from_numpy(reads.lens))
        for t in (d_cat, d_off, d_len):
            dist.broadcast(t, 0)
        torch.cuda.synchronize()
        ss = ctx.seqset_from_device(d_cat.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), N_READS)
    else:
        ss = ctx.seqset(reads)
    o = vlib.default_search_opts(); o.id = IDA
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    work = np.zeros(2, dtype=np.int64); nh = 0; sampler = None; l0 = 0
    for step in range(nsteps):
        if step == args.warmup:
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            sampler = ClockSampler(local); sampler.start(); ctx.profile_reset(); l0 = vlib.launch_count()
            ev0.record(stream)
        row0 = (step * world + rank) * args.rows
        hits, w = vlib.allpairs(ctx, ss, row0, args.rows, o, args.rows * N_READS)
        if step >= args.warmup:
            work += w; nh += len(hits)
    ev1.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.summary(); prof = ctx.profile(); launches = vlib.launch_count() - l0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
        wt = torch.tensor(work, dtype=torch.int64, device="cuda"); dist.all_reduce(wt, op=dist.ReduceOp.SUM); work = wt.cpu().numpy()
    if rank == 0:
        g = work[1] / (ms * 1e-3) / 1e9
        peak_ops = ctx.int_peak()
        cfg.update({"rows_per_step_per_gpu": args.rows, "parallelism": f"query rows sharded x{world}, reads NCCL-broadcast"})
        emit(json.dumps({"metric": "allpairs_global_gcups", "value": g, "unit": "GCUPS", "n_gpus": world,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16",
                          "data": "synthetic", "config": cfg, "pairs_per_s": float(work[0]) / (ms * 1e-3),
                          "hits_per_step": nh / args.steps,
                          "e2e": {"value": g, "unit": "GCUPS", "h2d_bytes_per_step": 16,
                                  "d2h_bytes_per_step": int(48 * nh / max(1, args.steps)),
                                  "note": "reads resident; per step only the row range goes up and the hit table comes back (included)"},
                          "gpu_launches": int(launches), "clocks": clocks,
                          "roofline": {"bound": "int_alu", "kernel": "nw_fast_kernel<13,false>",
                                       "achieved_in_step_overlapping_streams": prof.cells / max(1e-9, prof.fwd_ms * 1e-3) / 1e9,
                                       "peak": 2.0 * peak_ops / 15.0 / 1e9, "unit": "GCUPS", "frac": g / (2.0 * peak_ops / 15.0 / 1e9),
                                       "note": "frac uses whole-step throughput (forward + traceback + host) against the forward-kernel peak"}}))
    ss.close(); ctx.close()
    pg_done(world)


def cluster_workload(args, rank, world, local):
    """configs[2] shape: --cluster_fast on 300-nt amplicon reads (1 % divergence, Zipf-ish root choice), --id 0.97.
    One step = clustering a stated PREFIX of the read stream from scratch (SURVEY.md §8d: the full 10 M reads are
    hours on the CPU), round size = the host's core count on both arms (the reference's results depend on --threads).
    cluster_fast is a sequential greedy: N GPUs run N independent replicas (SURVEY.md §8e)."""
    from vsearch_b200 import synth
    N = args.cluster_reads
    cores = os.cpu_count() or 1
    T = args.cluster_round if args.cluster_round > 0 else cores
    rng = np.random.default_rng([3, rank if args.impl != "reference" else 0])
    nroots = max(50, N // 200)
    roots = synth.random_seqs(rng, nroots, 300)
    w = 1.0 / np.arange(1, nroots + 1); w /= w.sum()
    reads = synth.mutate_batch(rng, roots[rng.choice(nroots, size=N, p=w)], 0.01)
    labels = [f"a{i:08d}" for i in range(N)]
    order = np.lexsort((np.arange(N), -reads.lens.astype(np.int64)))     # Database::sortbylength (labels ascend with i)
    cfg = {"workload": f"cluster_fast first {N} reads of the 300nt amplicon stream (configs[2] shape), id 0.97",
           "reads_per_step": N, "round_size": T, "masking": "dust", "parallelism": f"{world} independent replica(s)"}
    nsteps = args.warmup + args.steps
    if args.impl == "reference":
        if rank != 0:
            return
        stock = os.path.join(ROOT, "oracle", "_ref", "vsearch")
        if not os.path.exists(stock):
            emit(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/vsearch not built"}))
            return
        fa = "/tmp/bench_cluster.fasta"
        with open(fa, "wb") as f:
            for i in range(N):
                f.write(b">" + labels[i].encode() + b"\n" + reads.seq(i) + b"\n")
        times = []
        for step in range(max(1, min(nsteps, 2))):      # the CPU run is long: one warm-up, one timed
            t0 = time.perf_counter()
            p = subprocess.run([stock, "--cluster_fast", fa, "--id", "0.97", "--threads", str(T), "--uc", "/tmp/bench_cluster.uc", "--quiet"],
                               capture_output=True, text=True)
            times.append(time.perf_counter() - t0)
            assert p.returncode == 0, p.stderr[-500:]
        dt = times[-1]
        ncl = sum(1 for l in open("/tmp/bench_cluster.uc") if l.startswith("S"))
        emit(json.dumps({"impl": "reference", "metric": "cluster_fast_reads_per_s", "value": N / dt, "unit": "reads/s", "n_gpus": args.gpus,
                          "steps": 1, "warmup": len(times) - 1, "ms_per_step": 1e3 * dt, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "int16", "data": "synthetic", "config": cfg, "clusters": ncl, "host": host_info(),
                          "cpu_baseline": {"value": N / dt, "unit": "reads/s", "cores": cores, "kind": "reference",
                                           "sample": f"vsearch --cluster_fast --threads {T} on the same {N} reads, wall time of the CLI (FASTA read and uc write included)"},
                          "e2e": {"value": N / dt, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch
    from vsearch_b200 import lib as vlib
    torch.cuda.set_device(local)
    import torch.distributed as dist
    pg_init(world, local)
    ctx = vlib.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream_ptr(), device=torch.device("cuda", local))
    sorted_host = pinned_seqset(synth.SeqSet([reads.seq(int(i)) for i in order]))
    o = vlib.default_search_opts(); o.id = 0.97; o.mask_lower = 1; o.maxrejects = 8   # --cluster_fast default (cli.cc:4163-4172)
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    sampler = None; l0 = 0; work = np.zeros(2, dtype=np.int64); ncl = 0
    for step in range(nsteps):
        if step == args.warmup:
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            sampler = ClockSampler(local); sampler.start(); l0 = vlib.launch_count()
            ev0.record(stream)
        ss = ctx.seqset(sorted_host)     # upload + DUST + clustering + results: all inside the timed region
        ss.dust()
        res, ncl, w = vlib.cluster_fast(ctx, ss, o, T)
        ss.close()
        if step >= args.warmup:
            work += w
    ev1.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.summary(); launches = vlib.launch_count() - l0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    if rank == 0:
        rps = N * world * args.steps / (ms * 1e-3)
        emit(json.dumps({"metric": "cluster_fast_reads_per_s", "value": rps, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "int16", "data": "synthetic", "config": cfg, "clusters": int(ncl),
                          "aligned_pairs_per_step": int(work[0] // max(1, args.steps)), "gcups": float(work[1]) / (ms * 1e-3) / 1e9,
                          "e2e": {"value": rps, "unit": "reads/s", "h2d_bytes_per_step": int(sorted_host.cat.nbytes + sorted_host.offs.nbytes + sorted_host.lens.nbytes),
                                  "d2h_bytes_per_step": int(N * 40), "note": "value IS end to end: upload, DUST, clustering and the result table are inside the timed region"},
                          "gpu_launches": int(launches), "clocks": clocks}))
    ctx.close()
    pg_done(world)


_RESULT_FD = None
_SINK = None      # when a list: emit() collects result lines (legs of the default run) instead of printing them


def pg_init(world, local):
    """NCCL process group, once per process (the legs of the default run share it)"""
    if world <= 1:
        return
    import torch
    import torch.distributed as dist
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))


def pg_done(world):
    if world <= 1 or _SINK is not None:
        return
    import torch.distributed as dist
    if dist.is_initialized():
        dist.destroy_process_group()


def emit(text):
    """the result line: the only thing this program writes to its original stdout"""
    if _SINK is not None:
        _SINK.append(json.loads(text))
        return
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, (text + "\n").encode())


def quiet_stdout():
    """Libraries print banners to stdout (NCCL's version line under torchrun): keep the real stdout
    for the one JSON line and point fd 1 at stderr for everything else."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = sys.stderr


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vsg", choices=["vsg", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="queries per step per GPU")
    ap.add_argument("--ref-sample", type=int, default=16384, help="queries per step of the reference arm")
    ap.add_argument("--masking", default="none", choices=["none", "dust"],
                    help="none (headline, as round 1) or dust = the reference's default --qmask/--dbmask, DUST on the device")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity gate against the reference")
    ap.add_argument("--cpu-sample", type=int, default=4096, help="queries of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="usearch", choices=["usearch", "c4", "allpairs", "cluster"],
                    help="usearch = configs[1] (default, the headline); c4 = configs[3] shape (1M x 1200 DB, 150-nt queries, "
                         "id 0.85); allpairs = configs[4] shape (dense N^2 DP)")
    ap.add_argument("--rows", type=int, default=32, help="allpairs: query rows per step per GPU")
    ap.add_argument("--cluster-reads", type=int, default=200_000, help="cluster: reads per step (prefix of the configs[2] stream)")
    ap.add_argument("--cluster-round", type=int, default=0, help="cluster: round size = the reference's --threads (0 = host cores)")
    ap.add_argument("--ref-rows", type=int, default=0,
                    help="allpairs: query rows per step of the reference arm (0 = one per host thread)")
    ap.add_argument("--no-job", dest="no_job", action="store_true", help="skip the whole-job (1M queries incl. set-up) leg")
    ap.add_argument("--no-legs", action="store_true",
                    help="default run only: skip the short configs[2] / configs[3] / configs[4] legs appended to the headline line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="usearch / c4: write the hit table of the last timed step (device-resident path) as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "vsg" or args.workload not in ("usearch", "c4")):
        ap.error("--dump-outputs: the usearch and c4 workloads of --impl vsg only")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.workload == "allpairs":
        allpairs_workload(args, rank, world, local)
        return
    if args.workload == "cluster":
        cluster_workload(args, rank, world, local)
        return
    set_workload(args.workload)
    if args.impl == "reference":
        reference_arm(args, rank)
        return
    if args.workload == "usearch" and not args.no_legs:
        # the default run: headline (configs[1]) plus short legs of the other configurations, ONE JSON line
        global _SINK
        _SINK = []
        rc = 0
        try:
            usearch_workload(args, rank, world, local)
        except SystemExit as e:
            rc = e.code if isinstance(e.code, int) else 1
        line = _SINK[0] if _SINK else None
        legs = {}
        import copy
        for name, fn, over in (
                ("configs3_c4", usearch_workload, dict(workload="c4", steps=2, warmup=3, batch=32768, no_cpu_baseline=True, no_parity=True)),
                ("configs4_allpairs", allpairs_workload, dict(workload="allpairs", steps=2, warmup=3, rows=24)),
                ("configs2_cluster", cluster_workload, dict(workload="cluster", steps=1, warmup=3, cluster_reads=100_000))):
            a2 = copy.copy(args)
            for k_, v_ in over.items():
                setattr(a2, k_, v_)
            a2.leg = True
            del _SINK[:]
            if a2.workload == "c4":
                set_workload("c4")
            try:
                fn(a2, rank, world, local)
                if _SINK:
                    d = _SINK[0]
                    legs[name] = {k_: d[k_] for k_ in ("metric", "value", "unit", "ms_per_step", "steps", "config", "e2e", "gpu_launches",
                                                         "queries_per_s", "pairs_per_s", "clusters", "gcups", "hits_per_step") if k_ in d}
            except BaseException as e:   # a leg must never take the headline down
                legs[name] = {"error": repr(e)[:300]}
            set_workload("usearch")
        _SINK = None
        pg_done(world)
        if rank == 0 and line is not None:
            line["legs"] = legs
            emit(json.dumps(line))
        if rc:
            raise SystemExit(rc)
        return
    usearch_workload(args, rank, world, local)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, res, counts, work, max_results):
    """What vsg_search_batch handed back in the last timed step: one float64 array per SearchResult field (query-major,
    max_results slots per query; slots past counts[q] are as the library left them), counts and the work counters.
    Above 64 MB in all, a fixed seeded sample of queries is kept and query_index.npy says which."""
    os.makedirs(out_dir, exist_ok=True)
    rows = np.ctypeslib.as_array(res).reshape(len(counts), max_results)
    nq = len(counts)
    per_query = 8 * (max_results * len(rows.dtype.names) + 1)
    if nq * per_query > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(nq, size=DUMP_LIMIT_BYTES // per_query - 1, replace=False))
        np.save(os.path.join(out_dir, "query_index.npy"), keep.astype(np.float64))
        rows, counts = rows[keep], counts[keep]
    for name in rows.dtype.names:
        np.save(os.path.join(out_dir, name + ".npy"), rows[name].astype(np.float64))
    np.save(os.path.join(out_dir, "counts.npy"), counts.astype(np.float64))
    np.save(os.path.join(out_dir, "work.npy"), np.asarray(work, dtype=np.float64))


def usearch_workload(args, rank, world, local):
    """configs[1] (headline) / configs[3] shape: --usearch_global through vsg_search_batch"""
    leg = getattr(args, "leg", False)
    import torch
    import torch.distributed as dist
    from vsearch_b200 import lib as vlib, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference "
                         "for the reference's CPU arm)")
    torch.cuda.set_device(local)
    pg_init(world, local)

    ctx = vlib.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream_ptr(), device=torch.device("cuda", local))

    # ---- database: rank 0 makes it; the packed bytes go to every GPU over NCCL/NVLink -------------
    dbm = synth.config2_db(N_DB, DB_LEN, SEED)  # every rank needs the matrix to draw its queries
    if world > 1:
        n = N_DB
        d_cat = torch.empty(n * DB_LEN, dtype=torch.uint8, device="cuda")
        d_off = torch.empty(n, dtype=torch.int64, device="cuda")
        d_len = torch.empty(n, dtype=torch.int32, device="cuda")
        if rank == 0:
            d_cat.copy_(torch.from_numpy(dbm.reshape(-1)))
            d_off.copy_(torch.arange(n, dtype=torch.int64) * DB_LEN)
            d_len.fill_(DB_LEN)
        dist.broadcast(d_cat, 0); dist.broadcast(d_off, 0); dist.broadcast(d_len, 0)
        torch.cuda.synchronize()
        db = ctx.seqset_from_device(d_cat.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), n)
    else:
        db = ctx.seqset(synth.SeqSet.from_matrix(dbm))
    dust = args.masking == "dust"
    t_ix = time.perf_counter()
    if dust:
        db.dust()          # --dbmask dust on the device (core/mask.cpp:79-188)
    ix = ctx.index(db, K, 1 if dust else 0)
    ctx.sync()
    index_build_ms = 1e3 * (time.perf_counter() - t_ix)

    opts = vlib.default_search_opts()
    opts.id = IDENT; opts.maxaccepts = MAXACC; opts.maxrejects = MAXREJ; opts.wordlength = K
    opts.mask_lower = 1 if dust else 0
    max_results = 1

    nsteps = args.warmup + args.steps
    batches = []
    for step in range(nsteps):
        qs, _ = synth.config2_query_batch(dbm, args.batch, Q_LEN, DIV, SEED, batch=step * world + rank)
        batches.append(pinned_seqset(qs))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def run_steps(e2e: bool, lazy: bool = False, mask=None):
        """returns (device ms for the K timed steps, work, launches, profile, clocks).  mask = (db, index): the
        DUST leg — queries are masked on the device inside the timed region, database and index are the masked ones"""
        opts.lazy = 1 if lazy else 0
        use_db, use_ix = (db, ix) if mask is None else mask
        qdust = dust or mask is not None
        opts.mask_lower = 1 if qdust else 0
        handles = None
        if not e2e:
            handles = [ctx.seqset(b) for b in batches]
            if qdust:
                for hh in handles:
                    hh.dust()
        work_tot = np.zeros(4, dtype=np.int64)
        ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
        sampler = None
        launches0 = 0
        for step in range(nsteps):
            if step == args.warmup:
                barrier()
                sampler = ClockSampler(local); sampler.start()
                ctx.profile_reset()
                launches0 = vlib.launch_count()
                ev0.record(stream)
            h = ctx.seqset(batches[step]) if e2e else handles[step]
            if e2e and qdust:
                h.dust()       # --qmask dust (commands/usearch_global.cpp:386-389), inside the timed region
            res, counts, work = ctx.search(use_ix, use_db, h, 0, args.batch, opts, max_results)
            if e2e:
                h.close()
            if step >= args.warmup:
                work_tot += work
        ev1.record(stream)
        barrier()
        last.update(res=res, counts=counts, work=work)
        ms = ev0.elapsed_time(ev1)
        clocks = sampler.summary() if sampler else {}
        prof = ctx.profile()
        launches = vlib.launch_count() - launches0
        hits = int((counts > 0).sum())
        if handles:
            for hh in handles:
                hh.close()
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            w = torch.tensor(work_tot, dtype=torch.int64, device="cuda")
            dist.all_reduce(w, op=dist.ReduceOp.SUM)
            work_tot = w.cpu().numpy()
        return ms, work_tot, launches, prof, clocks, hits

    if leg:     # a leg of the default run: the end-to-end number only
        ms_e2e, work_e2e, launches, prof, clocks, hits = run_steps(e2e=True)
        if rank == 0:
            emit(json.dumps({"metric": "usearch_global_gcups", "value": float(work_e2e[1]) / (ms_e2e * 1e-3) / 1e9, "unit": "GCUPS",
                              "steps": args.steps, "ms_per_step": ms_e2e / args.steps,
                              "config": {"workload": WL_NAME, "queries_per_step_per_gpu": args.batch, "index_build_ms_per_gpu": round(index_build_ms, 1),
                                         "masking": args.masking},
                              "queries_per_s": args.batch * world * args.steps / (ms_e2e * 1e-3), "pairs_per_s": float(work_e2e[0]) / (ms_e2e * 1e-3),
                              "gpu_launches": int(launches),
                              "e2e": {"value": float(work_e2e[1]) / (ms_e2e * 1e-3) / 1e9, "unit": "GCUPS",
                                      "note": "value IS end to end: query upload and hit table download inside the timed region"}}))
        ix.close(); db.close(); ctx.close()
        return
    ms_dev, work_dev, launches, prof, clocks, hits = run_steps(e2e=False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["res"], last["counts"], last["work"], max_results)
    ms_e2e, work_e2e, _, _, _, _ = run_steps(e2e=True)
    # optional mode, reported separately and NOT the headline: candidates are aligned only when the
    # accept/reject replay is about to examine them (same hit tables, tests/test_search_gpu.py); the
    # job is the same, the DP cells actually computed are fewer, so its "GCUPS" is job-equivalent only
    ms_lazy, work_lazy, _, _, _, _ = run_steps(e2e=True, lazy=True)
    opts.lazy = 0
    # the reference's DEFAULT masking (DUST on queries and database) as an extra leg when the headline runs unmasked
    dust_leg = None
    if not dust and args.workload == "usearch":
        db2 = ctx.seqset(synth.SeqSet.from_matrix(dbm)); db2.dust()
        ix2 = ctx.index(db2, K, 1)
        ms_d, work_d, _, _, _, _ = run_steps(e2e=True, mask=(db2, ix2))
        dust_leg = {"note": "--qmask dust --dbmask dust (the reference's defaults): DUST of every query batch on the device "
                            "inside the timed e2e region, database masked before indexing",
                    "ms_per_step": ms_d / args.steps, "e2e_gcups": float(work_d[1]) / (ms_d * 1e-3) / 1e9,
                    "queries_per_s": args.batch * world * args.steps / (ms_d * 1e-3)}
        ix2.close(); db2.close()
    opts.mask_lower = 1 if dust else 0
    # 2 % of the queries carry an ambiguous base: those pairs run on the GENERAL (16x16 score table) kernel classes
    iupac_leg = None
    if args.workload == "usearch":
        rng_n = np.random.default_rng(SEED + 17)
        saved = []
        for b in batches:
            nq_b = len(b.lens)
            who = rng_n.choice(nq_b, size=max(1, nq_b // 50), replace=False)
            pos = b.offs[who] + rng_n.integers(0, np.maximum(b.lens[who], 1))
            saved.append((pos, b.cat[pos].copy()))
            b.cat[pos] = ord("N")
        ms_n, work_n, _, _, _, hits_n = run_steps(e2e=True)
        for b, (pos, old) in zip(batches, saved):
            b.cat[pos] = old
        iupac_leg = {"note": "one N in 2 % of the queries: their k-mers over the N are skipped (unique.cpp:155-353), their pairs "
                             "go through the GENERAL aligner classes (16x16 scores, align_simd.cpp:1718-1733); e2e path",
                     "ms_per_step": ms_n / args.steps, "e2e_gcups": float(work_n[1]) / (ms_n * 1e-3) / 1e9,
                     "hit_fraction_last_step": hits_n / float(args.batch)}
    # the WHOLE job of configs[1]: 1M queries from nothing — context, database upload (and NCCL broadcast at N > 1),
    # index build, every batch end to end.  Strong scaling: the 1M queries are divided over the ranks.
    job_leg = None
    if args.workload == "usearch" and not getattr(args, "no_job", False):
        total_q = 1_048_576
        per_rank = total_q // world
        nb = max(1, per_rank // args.batch)
        jb = [pinned_seqset(synth.config2_query_batch(dbm, args.batch, Q_LEN, DIV, SEED, batch=1000 + r_ * world + rank)[0]) for r_ in range(nb)]
        barrier()
        t_job = time.perf_counter()
        ctx_j = vlib.Context(local)
        if world > 1:
            j_cat = torch.empty(N_DB * DB_LEN, dtype=torch.uint8, device="cuda")
            j_off = torch.empty(N_DB, dtype=torch.int64, device="cuda")
            j_len = torch.empty(N_DB, dtype=torch.int32, device="cuda")
            if rank == 0:
                j_cat.copy_(torch.from_numpy(dbm.reshape(-1)))
                j_off.copy_(torch.arange(N_DB, dtype=torch.int64) * DB_LEN)
                j_len.fill_(DB_LEN)
            dist.broadcast(j_cat, 0); dist.broadcast(j_off, 0); dist.broadcast(j_len, 0)
            torch.cuda.synchronize()
            db_j = ctx_j.seqset_from_device(j_cat.data_ptr(), j_off.data_ptr(), j_len.data_ptr(), N_DB)
        else:
            db_j = ctx_j.seqset(synth.SeqSet.from_matrix(dbm))
        ix_j = ctx_j.index(db_j, K, 0)
        ctx_j.sync()
        t_setup = time.perf_counter()
        opts.lazy = 0; opts.mask_lower = 0
        nhit = 0
        for b in jb:
            h = ctx_j.seqset(b)
            res_j, counts_j, _ = ctx_j.search(ix_j, db_j, h, 0, args.batch, opts, max_results)
            nhit += int((counts_j > 0).sum())
            h.close()
        barrier()
        t_end = time.perf_counter()
        wall = t_end - t_job
        if world > 1:
            tw = torch.tensor([wall, t_setup - t_job], dtype=torch.float64, device="cuda")
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
            wall, setup_s = float(tw[0].item()), float(tw[1].item())
        else:
            setup_s = t_setup - t_job
        job_leg = {"note": "whole job, wall clock, max over ranks: context + database upload (+ NCCL broadcast) + index build + "
                           "every query batch end to end; queries already parsed in pinned host memory",
                   "queries": nb * args.batch * world, "wall_s": wall, "setup_s": setup_s,
                   "queries_per_s": nb * args.batch * world / wall, "scaling": "strong", "hit_fraction_rank0": nhit / float(nb * args.batch)}
        ix_j.close(); db_j.close(); ctx_j.close()
        opts.mask_lower = 1 if dust else 0

    value = work_dev[1] / (ms_dev * 1e-3) / 1e9
    e2e_value = work_e2e[1] / (ms_e2e * 1e-3) / 1e9

    # ---- roofline of the dominant kernel (forward DP), timed ALONE on the library's stream --------
    # (inside the steps above four host threads keep several streams busy, so per-kernel event times
    #  overlap; here the same pairs of one batch go through a single stream, cudaEvents around the
    #  forward launches: vsg_profile.fwd_ms)
    nq_r = min(args.batch, 32768)
    hq = ctx.seqset(batches[args.warmup])
    seqno, count, nc = ctx.rank(ix, hq, 0, nq_r, 12, min(MAXACC + MAXREJ + 8, N_DB))
    qi = np.repeat(np.arange(nq_r, dtype=np.uint32), 8)
    ti = np.ascontiguousarray(seqno[:, :8].reshape(-1), dtype=np.uint32)
    res_r = None
    for _ in range(3):
        res_r = ctx.align_pairs(hq, db, qi, ti)
    prof_r = ctx.profile()
    ctx.profile_reset()
    ctx.rank(ix, hq, 0, nq_r, 12, min(MAXACC + MAXREJ + 8, N_DB))
    rank_ms_alone = ctx.profile().rank_ms
    hq.close()
    peak_ops = ctx.int_peak()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    fwd_gcups = res_r.cells / (res_r.fwd_ms * 1e-3) / 1e9 if res_r.fwd_ms > 0 else 0.0
    # algorithmic bytes: 8 B of row checkpoints per lane-step + 8 B x R of column checkpoints per lane and 32 steps, for the
    # 2 x R cells of a lane-step, with the wavefront's (D + 31) / D and the row padding's 256 / Q overheads (DESIGN.md 4.1)
    ck_bytes_per_cell = (8.0 + 8.0 * 8 / 32.0) / 16.0 * (DB_LEN + 31) / DB_LEN * 256 / Q_LEN
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None
    ncu_facts = {}
    try:   # dram bytes and instruction counts of one launch from the committed ncu --set full summary, scaled to this launch's cells
        tj = json.load(open(os.path.join(ROOT, "profiles", "nw_ckpt_r02_traffic.json")))
        per_cell = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) / tj["cells_per_launch_nominal"]
        traffic = {"bytes_per_launch": per_cell * res_r.cells / max(1, prof_r.fwd_launches), "bytes_per_cell": per_cell,
                   "source": "profiles/nw_ckpt_r02_traffic.json (ncu --set full)"}
        ncu_facts = {"issue_active_pct": tj["issue_active_pct"], "thread_instructions_per_cell": tj["thread_instructions_per_cell"],
                     "pipe_alu_pct": tj["pipe_alu_pct"], "pipe_fma_pct": tj["pipe_fma_pct"],
                     "lsu_data_pipe_wavefronts_pct": tj["lsu_data_pipe_wavefronts_pct"], "source": "profiles/nw_ckpt_r02_traffic.json"}
    except Exception:
        pass
    # Peak: this kernel's own floor is 3 thread-instructions per cell (6 per packed pair of cells: 3 DPX on the ALU pipe +
    # 3 IMAD.IADD on the FMA pipe; DESIGN.md 4.1) at the issue rate the SM sustains for an even mix of exactly those
    # three-operand instructions, measured live (vsg_measure_int_peak, about 0.62 warp-instructions/clk/SMSP).  Everything
    # the kernel issues beyond 3 per cell (shuffles, profile loads, ring moves, stores, the edge path) lowers frac.
    own_peak = peak_ops / 3.0 / 1e9
    issue_ceiling = 148 * 4 * 32 * 1.965e9      # 1 warp-instruction / clk / SMSP at the 1965 MHz boost clock
    roofline = {"bound": "int_alu", "kernel": "nw_ckpt_kernel<8,CK_PROF>",
                "achieved": fwd_gcups, "peak": own_peak, "unit": "GCUPS", "frac": fwd_gcups / own_peak,
                "peak_source": "vsg_measure_int_peak (even mix of VIADDMNMX.U16x2 and IMAD, thread-instructions/s, measured live, "
                               "burst) / 3 thread-instructions per cell (the kernel's 6-instruction recurrence per packed cell pair)",
                "packed_lane_ops_per_s": peak_ops,
                "model_2p15": {"note": "round 1's model, kept for comparison: 15 SSE ops per cell of the reference's onestep "
                                       "(align_simd.cpp:765-780) at 1 warp-instruction/clk/SMSP; this kernel computes no "
                                       "direction bits and needs 3, so this fraction is not a hardware bound for it",
                               "peak": 2.0 * issue_ceiling / 15.0 / 1e9,
                               "frac": fwd_gcups / (2.0 * issue_ceiling / 15.0 / 1e9)},
                "ncu": ncu_facts,
                "avg_launch_ms": res_r.fwd_ms / max(1, prof_r.fwd_launches), "launches": int(prof_r.fwd_launches),
                "cells_per_launch": res_r.cells / max(1, prof_r.fwd_launches),
                "hbm": {"achieved_gbs": fwd_gcups * ck_bytes_per_cell, "peak_gbs": hbm_peak,
                        "frac": fwd_gcups * ck_bytes_per_cell / hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6.65 TB/s",
                        "algorithmic_bytes_per_cell": ck_bytes_per_cell},
                "traffic": traffic,
                "alone_ms": {"forward": res_r.fwd_ms, "traceback": res_r.tb_ms, "rank": rank_ms_alone,
                             "queries": nq_r, "pairs": int(qi.shape[0])},
                "in_step_kernel_ms_overlapping_streams": {"forward": prof.fwd_ms, "traceback": prof.traceback_ms,
                                                          "rank": prof.rank_ms}}

    # ---- cpu_baseline: the unmodified reference on this box's cores, bounded sample ---------------
    cpu_baseline = None
    parity = {"parity_checked": 0, "parity_mismatches": 0}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import checkers
        cores = os.cpu_count() or 1
        sample = args.cpu_sample
        qs, _ = synth.config2_query_batch(dbm, sample, Q_LEN, DIV, SEED, batch=0)
        if checkers.ref() is not None:
            rlib = checkers.ref()
            r = checkers.RefDb(synth.SeqSet.from_matrix(dbm), k=K, id=IDENT, maxaccepts=MAXACC, maxrejects=MAXREJ,
                               dust=1 if dust else 0)
            ft = np.zeros(sample, dtype=np.int32)
            rlib.vsref_work_reset()
            t0 = time.perf_counter()
            rlib.vsref_db_search_batch(C.c_void_p(r.h), C.c_int(sample), checkers._p(qs.cat, C.c_char),
                                       checkers._p(qs.offs, C.c_int64), checkers._p(qs.lens, C.c_int),
                                       C.c_int(cores), checkers._p(ft, C.c_int))
            dt = time.perf_counter() - t0
            p = C.c_longlong(); c = C.c_longlong(); k = C.c_longlong()
            rlib.vsref_work_get(C.byref(p), C.byref(c), C.byref(k))
            r.close()
            cpu_baseline = {"value": c.value / dt / 1e9, "unit": "GCUPS", "cores": cores, "kind": "reference",
                            "sample": f"first {sample} queries of batch 0, reference search_batch --threads {cores}, "
                                      f"{dt:.1f} s", "queries_per_s": sample / dt, "host": host_info()}
            if not args.no_parity:
                # PARITY GATE: the product path's first hit for the same queries must equal the reference's
                hq = ctx.seqset(qs)
                if dust:
                    hq.dust()
                opts.lazy = 0
                resp, cntp, _ = ctx.search(ix, db, hq, 0, sample, opts, 1)
                gotp = np.array([resp[i].target if cntp[i] > 0 else -1 for i in range(sample)], dtype=np.int32)
                hq.close()
                parity = {"parity_checked": int(sample), "parity_mismatches": int((gotp != ft).sum())}
        else:
            od = checkers.OracleDb(synth.SeqSet.from_matrix(dbm))
            oo = checkers.search_opts(N_DB, id=IDENT, maxaccepts=MAXACC, maxrejects=MAXREJ)
            nsm = min(sample, 64)
            t0 = time.perf_counter(); cells = 0
            for i in range(nsm):
                _, _, cl = od.search(qs.seq(i), oo); cells += cl
            dt = time.perf_counter() - t0
            cpu_baseline = {"value": cells / dt / 1e9, "unit": "GCUPS", "cores": 1, "kind": "port",
                            "sample": f"first {nsm} queries of batch 0, scalar oracle"}

    if rank == 0:
        qbytes = int(np.mean([b.cat.nbytes + b.offs.nbytes + b.lens.nbytes for b in batches]))
        rbytes = args.batch * (max_results * 48 + 4) + 16
        line = {"metric": "usearch_global_gcups", "value": value, "unit": "GCUPS", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16",
                "data": "synthetic",
                "config": {"workload": WL_NAME,
                           "queries_per_step_per_gpu": args.batch, "global_queries_per_step": args.batch * world,
                           "masking": args.masking, "wordlength": K, "maxaccepts": MAXACC, "maxrejects": MAXREJ,
                           "index_build_ms_per_gpu": round(index_build_ms, 1),
                           "parallelism": f"query-sharded x{world}, DB NCCL-broadcast",
                           "l2": "per-step working set (index 300 MB + checkpoints > 10 GB) exceeds the 126 MB L2",
                           "traceback": ("every pair's forward DP is computed; the walk back of a group's other candidates is skipped "
                                         "when its first candidate is accepted and ends the query's search (never examined by "
                                         "align_delayed, searchcore.cpp:780-880); identical hit tables; VSG_TB_GATE=0 walks all"
                                         if os.environ.get("VSG_TB_GATE", "1") != "0" else "every pair walked back (VSG_TB_GATE=0)")},
                "queries_per_s": args.batch * world * args.steps / (ms_dev * 1e-3),
                "pairs_per_s": float(work_dev[0]) / (ms_dev * 1e-3),
                "walks_skipped_fraction": (float(prof.tb_skipped) / float(work_dev[0])) if work_dev[0] > 0 else 0.0,
                "hit_fraction_last_step": hits / args.batch,
                "e2e": {"value": e2e_value, "unit": "GCUPS", "h2d_bytes_per_step": qbytes,
                        "d2h_bytes_per_step": rbytes, "ms_per_step": ms_e2e / args.steps,
                        "queries_per_s": args.batch * world * args.steps / (ms_e2e * 1e-3)},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
                "lazy_mode": {"note": "opts.lazy=1, e2e path; identical hit tables, alignments on demand; job-equivalent "
                                      "GCUPS = the reference's search16 cells for these queries / time (NOT cells computed)",
                              "ms_per_step": ms_lazy / args.steps,
                              "queries_per_s": args.batch * world * args.steps / (ms_lazy * 1e-3),
                              "job_equivalent_gcups": float(work_lazy[1]) / (ms_lazy * 1e-3) / 1e9,
                              "cells_computed_gcups": float(work_lazy[3]) / (ms_lazy * 1e-3) / 1e9,
                              "pairs_aligned_fraction": float(work_lazy[2]) / max(1.0, float(work_lazy[0]))}}
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if dust_leg is not None:
            line["dust_mode"] = dust_leg
        if iupac_leg is not None:
            line["iupac_mode"] = iupac_leg
        if job_leg is not None:
            line["job_mode"] = job_leg
        line.update(parity)
        emit(json.dumps(line))
    ix.close(); db.close(); ctx.close()
    pg_done(world)
    if parity["parity_mismatches"]:
        raise SystemExit(3)


if __name__ == "__main__":
    main()
