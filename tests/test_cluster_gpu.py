"""vsg_cluster_fast (device ranker + aligner behind the reference's greedy round structure) against the unmodified
reference CLI: `vsearch --cluster_fast --threads T` must give the same S/H records — cluster numbers, centroids,
identities and CIGARs — for the same round size T, including T = 1 (cluster_core_serial) and rounds in which several
new centroids meet (evaluate_extra_hits)."""

import numpy as np
import pytest

import checkers
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

pytestmark = pytest.mark.gpu


def _reads(n, nroots, seed, divs=(0.01, 0.01, 0.02, 0.035, 0.05)):
    rng = np.random.default_rng(seed)
    roots = synth.random_seqs(rng, nroots, 300)
    w = 1.0 / np.arange(1, nroots + 1); w /= w.sum()      # Zipf-ish root choice: a few roots own most reads
    pick = rng.choice(nroots, size=n, p=w)
    seqs = []
    for i in range(n):
        r = roots[int(pick[i])]
        m = synth.mutate(rng, r, float(divs[int(rng.integers(0, len(divs)))]))
        a = int(rng.integers(0, 6)); b = int(rng.integers(0, 6))
        s = m[a: m.shape[0] - b].tobytes()
        if i % 97 == 5:
            s = s[:100] + b"AT" * 30 + s[100:]      # DUST bait
        seqs.append(s)
    return seqs


def _uc_records(path):
    rec = {}
    for line in open(path):
        f = line.rstrip("\n").split("\t")
        if f[0] == "S":
            rec[f[8]] = ("S", int(f[1]), "*", "*", "*")
        elif f[0] == "H":
            rec[f[8]] = ("H", int(f[1]), f[3], f[9], f[7])
    return rec


def _records_digest(rec):
    """the S/H records of every read, as the number of clusters and a digest of the records in label order"""
    text = "".join(f"{k}\t" + "\t".join(map(str, rec[k])) + "\n" for k in sorted(rec))
    return {"reads": len(rec), "clusters": sum(1 for v in rec.values() if v[0] == "S"), "sha256": checkers.digest(text)}


@pytest.mark.skipif(not checkers.have_reference_cli(), reason="neither oracle/_ref nor tests/golden/reference")
@pytest.mark.parametrize("threads,n,nroots,ident", [(1, 1500, 40, 0.97), (2, 1500, 40, 0.97), (8, 4000, 120, 0.97),
                                                     (64, 6000, 400, 0.97), (16, 3000, 60, 0.90), (128, 30000, 150, 0.97)])
def test_cluster_fast_equals_reference_cli(tmp_path, threads, n, nroots, ident):
    seqs = _reads(n, nroots, seed=100 + threads)
    labels = [f"a{i:07d}" for i in range(n)]
    fa = str(tmp_path / "reads.fasta")
    with open(fa, "wb") as f:
        for l, s in zip(labels, seqs):
            f.write(b">" + l.encode() + b"\n" + s + b"\n")
    uc = str(tmp_path / "ref.uc")
    want = checkers.reference_cli(["--cluster_fast", fa, "--id", str(ident), "--threads", str(threads), "--uc", uc, "--quiet"],
                                  lambda: _records_digest(_uc_records(uc)))
    # Database::sortbylength (core/db.cpp:433-449): length descending, abundance descending, label ascending, input order
    order = sorted(range(n), key=lambda i: (-len(seqs[i]), labels[i]))
    ss_host = synth.SeqSet([seqs[i] for i in order])
    ctx = vlib.Context(0)
    ss = ctx.seqset(ss_host)
    ss.dust()                                   # --qmask dust, the default (dust_all before clustering)
    o = vlib.default_search_opts(); o.id = ident; o.mask_lower = 1
    o.maxrejects = 8                            # the reference's default for --cluster_fast (cli.cc:4163-4172); 32 elsewhere
    res, ncl, work = vlib.cluster_fast(ctx, ss, o, threads)
    assert ncl == want["clusters"]
    hq = [k for k in range(n) if res["centroid"][k] >= 0]
    al = ctx.align_pairs(ss, ss, np.array(hq, dtype=np.uint32), res["centroid"][hq].astype(np.uint32), cigar=True)
    cig = dict(zip(hq, al.cigars))
    got = {}
    for k in range(n):
        lab = labels[order[k]]
        if res["centroid"][k] < 0:
            got[lab] = ("S", int(res["cluster"][k]), "*", "*", "*")
        else:
            c = cig[k]
            got[lab] = ("H", int(res["cluster"][k]), f"{res['id'][k]:.1f}", labels[order[int(res['centroid'][k])]],
                        "=" if res["id"][k] == 100.0 else c)   # '=' = identical ignoring terminal gaps (core/results.cpp:84-90)
    assert _records_digest(got) == want
    assert work[0] > 0 and work[1] > 0
    ss.close(); ctx.close()
