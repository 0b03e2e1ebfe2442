"""Parity at BENCHMARK scale (VERDICT r1 item 1): the shapes bench.py and BASELINE.json's configs quote, not
miniatures.  The compiled, unmodified reference (oracle/_ref) runs on the host cores of the GPU box; every
result record must be equal.

  C2  8 192 queries x 250 nt against the real 100 000 x 1 500 nt database, --id 0.9  (configs[1])
  C4  4 096 queries x 150 nt (10 % mutated) against 230 000 x 1 200 nt = 8 index shards, --id 0.85  (configs[3] shape)
  C5  400-nt reads at 15 % divergence, --id 0.7: vsg_allpairs rows vs the reference CLI, and the seam-1 CLI with
      CIGARs (configs[4] shape; R = 13 rows per lane, the lane-replicated score table)
"""
import os
import subprocess

import numpy as np
import pytest

import checkers
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STOCK = os.path.join(ROOT, "oracle", "_ref", "vsearch")
GPU = os.path.join(ROOT, "oracle", "_ref", "vsearch_gpu")
needs_ref = pytest.mark.skipif(not checkers.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")


@pytest.fixture(scope="module")
def ctx():
    c = vlib.Context(0)
    yield c
    c.close()


def _rows_digest(res, counts, max_results, nq):
    return checkers.rows_digest([[(r.target, r.id, r.matches, r.mismatches, r.gaps, r.alignment_length, r.accepted, r.strand)
                                  for r in (res[q * max_results + j] for j in range(int(counts[q])))] for q in range(nq)])


@needs_ref
def test_c2_full_database_rows_equal_reference(ctx):
    n_db, db_len, nq = 100_000, 1500, 8192
    dbm = synth.config2_db(n_db, db_len, 2024)
    qs, src = synth.config2_query_batch(dbm, nq, 250, 0.05, 2024, batch=3)
    dbs = synth.SeqSet.from_matrix(dbm)
    r = checkers.RefDb(dbs, id=0.9, maxaccepts=1, maxrejects=32)
    max_results = 4
    want = r.search_rows_digest(qs, max_results=max_results)
    r.close()
    db = ctx.seqset(dbs); q = ctx.seqset(qs)
    ix = ctx.index(db, 8, 0)
    o = vlib.default_search_opts(); o.id = 0.9; o.maxaccepts = 1; o.maxrejects = 32
    for lazy in (0, 1):
        o.lazy = lazy
        res, counts, work = ctx.search(ix, db, q, 0, nq, o, max_results)
        assert _rows_digest(res, counts, max_results, nq) == want, lazy
    assert int((counts > 0).sum()) > 0.95 * nq
    hit = sum(1 for i in range(nq) if counts[i] > 0 and res[i * max_results].target == int(src[i]))
    assert hit > 0.95 * nq
    ix.close(); db.close(); q.close()


@needs_ref
def test_c4_shape_eight_shards_rows_equal_reference(ctx):
    n_db, db_len, nq = 230_000, 1200, 4096
    rng = np.random.default_rng(4)
    dbm = synth.random_seqs(rng, n_db, db_len)
    qs, src = synth.config2_query_batch(dbm, nq, 150, 0.10, 4, batch=0)
    dbs = synth.SeqSet.from_matrix(dbm)
    r = checkers.RefDb(dbs, id=0.85, maxaccepts=1, maxrejects=32)
    max_results = 4
    want = r.search_rows_digest(qs, max_results=max_results)
    r.close()
    db = ctx.seqset(dbs); q = ctx.seqset(qs)
    ix = ctx.index(db, 8, 0)
    o = vlib.default_search_opts(); o.id = 0.85; o.maxaccepts = 1; o.maxrejects = 32
    res, counts, work = ctx.search(ix, db, q, 0, nq, o, max_results)
    assert _rows_digest(res, counts, max_results, nq) == want
    assert int((counts > 0).sum()) > 0.5 * nq
    ix.close(); db.close(); q.close()


def _run(binary, args, threads):
    p = subprocess.run([binary] + args + ["--threads", str(threads), "--quiet"], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-2000:]


def _sorted(path):
    with open(path) as f:
        return sorted(f.readlines())


@pytest.mark.skipif(not checkers.have_reference_cli(), reason="neither oracle/_ref nor tests/golden/reference")
def test_c5_shape_allpairs_rows_equal_reference_cli(ctx, tmp_path):
    reads = synth.config5_allpairs(n_reads=1600, n_roots=16, length=400, div=0.15, seed=5)
    fa = str(tmp_path / "c5.fasta")
    synth.write_fasta(fa, reads, "r")
    uo = str(tmp_path / "cpu.userout")
    want = checkers.reference_cli(["--allpairs_global", fa, "--id", "0.7", "--qmask", "none", "--userout", uo,
                                   "--userfields", "query+target+id+alnlen+mism+raw+ids", "--quiet"],
                                  lambda: {"lines": len(_sorted(uo)), "sha256": checkers.digest("".join(_sorted(uo)))},
                                  threads=os.cpu_count())
    ss = ctx.seqset(reads)
    o = vlib.default_search_opts(); o.id = 0.7
    n = len(reads)
    bounds = np.zeros(4, dtype=np.int64)
    import ctypes as C
    assert vlib.load().vsg_allpairs_partition(reads.lens.ctypes.data_as(C.POINTER(C.c_int32)), C.c_int64(n), C.c_int(3),
                                              bounds.ctypes.data_as(C.POINTER(C.c_int64))) == 0
    hits = []
    pairs = 0
    for p in range(3):     # three row ranges of equal DP work, as three GPUs would take them
        h, w = vlib.allpairs(ctx, ss, int(bounds[p]), int(bounds[p + 1] - bounds[p]), o, 2_000_000)
        hits += list(h); pairs += int(w[0])
    got = sorted(f"r{h['query']}\tr{h['target']}\t{h['id']:.1f}\t{h['internal_alignment_length']}\t{h['mismatches']}\t"
                 f"{h['nwscore']}\t{h['matches']}\n" for h in hits)
    assert pairs == n * (n - 1) // 2
    assert want["lines"] > 20000 and {"lines": len(got), "sha256": checkers.digest("".join(got))} == want
    ss.close()


@pytest.mark.skipif(not (os.path.exists(STOCK) and os.path.exists(GPU)), reason="oracle/_ref/vsearch{,_gpu} not built")
def test_c5_shape_cli_with_cigars(tmp_path):
    reads = synth.config5_allpairs(n_reads=300, n_roots=6, length=400, div=0.15, seed=55)
    fa = str(tmp_path / "c5s.fasta")
    synth.write_fasta(fa, reads, "r")
    fields = "query+target+id+alnlen+mism+opens+raw+caln+qilo+qihi+tilo+tihi+id0+id1+id2+id3+id4+ids+gaps"
    outs = {}
    for name, binary, thr in (("cpu", STOCK, os.cpu_count()), ("gpu", GPU, 4)):
        uo = str(tmp_path / f"{name}.userout")
        _run(binary, ["--allpairs_global", fa, "--id", "0.7", "--userout", uo, "--userfields", fields], thr)
        outs[name] = _sorted(uo)
    assert len(outs["cpu"]) > 3000 and outs["cpu"] == outs["gpu"]
