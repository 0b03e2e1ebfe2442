"""Seam 1 end to end: the UNMODIFIED reference CLI versus the same CLI linked against
shim/align_simd_vsg.cpp + libvsg.so instead of its own core/align_simd.cpp (oracle/Makefile builds
both into oracle/_ref/).  Hit tables must be byte-identical after sorting (thread completion order
is the only legitimate difference, SURVEY.md §3.1)."""
import os
import subprocess
import time

import numpy as np
import pytest

import checkers
from vsearch_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STOCK = os.path.join(ROOT, "oracle", "_ref", "vsearch")
GPU = os.path.join(ROOT, "oracle", "_ref", "vsearch_gpu")
FIELDS = "query+target+id+alnlen+mism+opens+raw+caln+qilo+qihi+tilo+tihi+id0+id1+id2+id3+id4+ids+gaps"

needs_bins = pytest.mark.skipif(not (os.path.exists(STOCK) and os.path.exists(GPU)),
                                reason="oracle/_ref/vsearch{,_gpu} not built")


def _lines_digest(lines):
    return {"lines": len(lines), "sha256": checkers.digest("".join(lines))}


def run(binary, args, threads):
    t0 = time.time()
    p = subprocess.run([binary] + args + ["--threads", str(threads), "--quiet"], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-2000:]
    return time.time() - t0


def sorted_lines(path):
    with open(path) as f:
        return sorted(f.readlines())


@needs_bins
def test_allpairs_global_config1_full_size(tmp_path):
    """BASELINE configs[0]: 1 000 reads x ~200 nt, --id 0.8 — all 499 500 pairs, scores + CIGARs"""
    reads = synth.config1_allpairs()
    fa = str(tmp_path / "c1.fasta")
    synth.write_fasta(fa, reads, "r")
    outs = {}
    for name, binary, thr in (("cpu", STOCK, os.cpu_count()), ("gpu", GPU, 4)):
        uo = str(tmp_path / f"{name}.userout"); uc = str(tmp_path / f"{name}.uc")
        dt = run(binary, ["--allpairs_global", fa, "--id", "0.8", "--userout", uo, "--userfields", FIELDS, "--uc", uc], thr)
        outs[name] = (sorted_lines(uo), sorted_lines(uc), dt)
    assert len(outs["cpu"][0]) > 10000
    assert outs["cpu"][0] == outs["gpu"][0]
    assert outs["cpu"][1] == outs["gpu"][1]
    print(f"allpairs C1: cpu {outs['cpu'][2]:.2f}s ({os.cpu_count()} threads)  gpu-shim {outs['gpu'][2]:.2f}s")


@needs_bins
def test_usearch_global_and_cluster_fast(tmp_path):
    dbs, qss, _ = synth.config2_search(n_db=3000, db_len=1500, n_q=4000, q_len=250, div=0.05, seed=5)
    dbf = str(tmp_path / "db.fasta"); qf = str(tmp_path / "q.fasta")
    synth.write_fasta(dbf, dbs, "d"); synth.write_fasta(qf, qss, "q")
    res = {}
    for name, binary, thr in (("cpu", STOCK, os.cpu_count()), ("gpu", GPU, 4)):
        uo = str(tmp_path / f"{name}.u.userout"); b6 = str(tmp_path / f"{name}.b6")
        run(binary, ["--usearch_global", qf, "--db", dbf, "--id", "0.9", "--userout", uo, "--userfields", FIELDS,
                     "--blast6out", b6, "--strand", "both", "--maxaccepts", "2", "--maxrejects", "8"], thr)
        res[name] = (sorted_lines(uo), sorted_lines(b6))
    assert len(res["cpu"][0]) >= 3900 and res["cpu"] == res["gpu"]
    # cluster_fast: greedy and order dependent -> same thread count on both sides
    rng = np.random.default_rng(8)
    roots = synth.random_seqs(rng, 60, 300)
    reads = synth.SeqSet([synth.mutate(rng, roots[int(rng.integers(0, 60))], 0.01) for _ in range(3000)])
    cf = str(tmp_path / "c.fasta"); synth.write_fasta(cf, reads, "a")
    ucs = {}
    for name, binary in (("cpu", STOCK), ("gpu", GPU)):
        uc = str(tmp_path / f"{name}.c.uc")
        run(binary, ["--cluster_fast", cf, "--id", "0.97", "--uc", uc], 2)
        ucs[name] = sorted_lines(uc)
    assert len(ucs["cpu"]) > 3000 and ucs["cpu"] == ucs["gpu"]


@pytest.mark.skipif(not checkers.have_reference_cli(), reason="neither oracle/_ref nor tests/golden/reference")
def test_allpairs_api_vs_reference_cli(tmp_path):
    """vsg_allpairs (rows sharded in two halves, as two GPUs would) against the stock CLI on configs[0]"""
    from vsearch_b200 import lib as vlib
    reads = synth.config1_allpairs()
    fa = str(tmp_path / "c1.fasta")
    synth.write_fasta(fa, reads, "r")
    uo = str(tmp_path / "cpu.userout")
    want = checkers.reference_cli(["--allpairs_global", fa, "--id", "0.8", "--qmask", "none", "--userout", uo,
                                   "--userfields", "query+target+id+alnlen+mism+raw+ids", "--quiet"],
                                  lambda: _lines_digest(sorted_lines(uo)), threads=os.cpu_count())
    ctx = vlib.Context(0)
    ss = ctx.seqset(reads)
    o = vlib.default_search_opts(); o.id = 0.8
    n = len(reads)
    h1, w1 = vlib.allpairs(ctx, ss, 0, 300, o, 200000)
    h2, w2 = vlib.allpairs(ctx, ss, 300, n - 300, o, 200000)
    # userout's alnlen is the alignment length without terminal gaps (results.cpp / userfields)
    got = sorted(f"r{h['query']}\tr{h['target']}\t{h['id']:.1f}\t{h['internal_alignment_length']}\t{h['mismatches']}\t"
                 f"{h['nwscore']}\t{h['matches']}\n" for h in list(h1) + list(h2))
    assert want["lines"] > 10000 and _lines_digest(got) == want
    assert int(w1[0] + w2[0]) == n * (n - 1) // 2
    # per query: id descending, then target ascending (allpairs_hit_compare)
    q = h1["query"]; same = q[1:] == q[:-1]
    assert np.all((h1["id"][1:] <= h1["id"][:-1]) | ~same)
    ss.close(); ctx.close()
