"""vsg_cluster_fast and the clustering session with --strand both against the unmodified reference CLI:
`vsearch --cluster_fast --strand both --threads T` must give the same S/H records — cluster numbers, centroids,
identities, the strand column and CIGARs (those of the reverse complement for '-' records) — for reads of mixed
orientation, including deferred pairs resolved by the linear-memory aligner on the reverse complement."""

import os
import re
import subprocess

import numpy as np
import pytest

import checkers
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

pytestmark = pytest.mark.gpu

needs_cli = pytest.mark.skipif(not checkers.have_reference_cli(), reason="neither oracle/_ref nor tests/golden/reference")

_COMP = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")


def _rc(s: bytes) -> bytes:
    return s.translate(_COMP)[::-1]


def _reads(n, nroots, seed, flip=0.4, divs=(0.01, 0.01, 0.02, 0.035, 0.05)):
    """the reads of test_cluster_gpu.py, about 40 % of them reverse-complemented"""
    rng = np.random.default_rng(seed)
    roots = synth.random_seqs(rng, nroots, 300)
    w = 1.0 / np.arange(1, nroots + 1); w /= w.sum()
    pick = rng.choice(nroots, size=n, p=w)
    seqs = []
    for i in range(n):
        m = synth.mutate(rng, roots[int(pick[i])], float(divs[int(rng.integers(0, len(divs)))]))
        a = int(rng.integers(0, 6)); b = int(rng.integers(0, 6))
        s = m[a: m.shape[0] - b].tobytes()
        if i % 97 == 5:
            s = s[:100] + b"AT" * 30 + s[100:]      # DUST bait
        if rng.random() < flip:
            s = _rc(s)
        seqs.append(s)
    return seqs


def _write(tmp_path, labels, seqs):
    fa = str(tmp_path / "reads.fasta")
    with open(fa, "wb") as f:
        for l, s in zip(labels, seqs):
            f.write(b">" + l.encode() + b"\n" + s + b"\n")
    return fa


def _uc_records(path):
    rec = {}
    for line in open(path):
        f = line.rstrip("\n").split("\t")
        if f[0] == "S":
            rec[f[8]] = ("S", int(f[1]), "*", "*", "*", "*")
        elif f[0] == "H":
            rec[f[8]] = ("H", int(f[1]), f[3], f[9], f[4], f[7])
    return rec


def _records_digest(rec):
    text = "".join(f"{k}\t" + "\t".join(map(str, rec[k])) + "\n" for k in sorted(rec))
    return {"reads": len(rec), "clusters": sum(1 for v in rec.values() if v[0] == "S"),
            "minus": sum(1 for v in rec.values() if v[0] == "H" and v[4] == "-"), "sha256": checkers.digest(text)}


def _cli(tmp_path, fa, ident, threads, strand_both=True, qmask="dust"):
    uc = str(tmp_path / "ref.uc")
    args = ["--cluster_fast", fa, "--id", str(ident), "--threads", str(threads), "--uc", uc, "--quiet"]
    if strand_both:
        args += ["--strand", "both"]
    if qmask != "dust":
        args += ["--qmask", qmask]
    return checkers.reference_cli(args, lambda: _records_digest(_uc_records(uc)))


def _opts(ident, mask_lower=1, strand_both=1):
    o = vlib.default_search_opts(); o.id = ident; o.mask_lower = mask_lower
    o.maxrejects = 8                            # the reference's default for --cluster_fast (cli.cc:4163-4172)
    o.strand_both = strand_both
    return o


def _order(seqs, labels):
    # Database::sortbylength (core/db.cpp:433-449): length descending, label ascending
    return sorted(range(len(seqs)), key=lambda i: (-len(seqs[i]), labels[i]))


def _records(ctx, ss, rc, res, labels, order, lma_cigar=None):
    """uc-style records from vsg_cluster_fast's results; CIGARs from one vsg_align_pairs call per strand"""
    n = res.shape[0]
    cig = {}
    for st, qs in ((0, ss), (1, rc)):
        hq = [k for k in range(n) if res["centroid"][k] >= 0 and res["strand"][k] == st]
        if hq:
            al = ctx.align_pairs(qs, ss, np.array(hq, dtype=np.uint32), res["centroid"][hq].astype(np.uint32), cigar=True)
            for j, k in enumerate(hq):
                cig[k] = lma_cigar(k, st, int(res["centroid"][k])) if int(al.score[j]) == 32767 else al.cigars[j]
    got = {}
    for k in range(n):
        lab = labels[order[k]]
        if res["centroid"][k] < 0:
            got[lab] = ("S", int(res["cluster"][k]), "*", "*", "*", "*")
        else:
            got[lab] = ("H", int(res["cluster"][k]), f"{res['id'][k]:.1f}", labels[order[int(res['centroid'][k])]],
                        "-" if res["strand"][k] else "+", "=" if res["id"][k] == 100.0 else cig[k])
    return got


@needs_cli
@pytest.mark.parametrize("threads,n,nroots,ident,qmask", [
    (1, 1500, 40, 0.97, "dust"), (2, 1500, 40, 0.97, "dust"), (8, 4000, 120, 0.97, "dust"),
    (64, 6000, 400, 0.97, "dust"), (128, 30000, 150, 0.97, "dust"),
    (16, 3000, 60, 0.90, "dust"),               # a lower --id: more candidates per strand
    (8, 3000, 60, 0.97, "none"),                # --qmask none
])
def test_cluster_fast_strand_both_equals_reference_cli(tmp_path, threads, n, nroots, ident, qmask):
    seqs = _reads(n, nroots, seed=300 + threads)
    labels = [f"a{i:07d}" for i in range(n)]
    fa = _write(tmp_path, labels, seqs)
    want = _cli(tmp_path, fa, ident, threads, qmask=qmask)
    order = _order(seqs, labels)
    ctx = vlib.Context(0)
    ss = ctx.seqset(synth.SeqSet([seqs[i] for i in order]))
    if qmask == "dust":
        ss.dust()                               # dust_all before clustering; the minus strand is not masked again
    res, ncl, work = vlib.cluster_fast(ctx, ss, _opts(ident, 1 if qmask == "dust" else 0), threads)
    assert ncl == want["clusters"]
    rc = ctx.revcomp(ss)
    got = _records(ctx, ss, rc, res, labels, order)
    assert _records_digest(got) == want
    nh = int((res["centroid"] >= 0).sum())
    assert want["minus"] >= 0.2 * nh > 0       # a substantial share of the members match on the minus strand
    assert work[0] > 0 and work[1] > 0
    if threads >= 8:
        # a read that joins, on the minus strand, a centroid founded earlier in its own round: the minus strand of
        # evaluate_extra_hits ran
        k = np.arange(n)
        same_round = (res["centroid"] >= 0) & (res["strand"] == 1) & (res["centroid"] // threads == k // threads)
        assert same_round.any()
    rc.close(); ss.close(); ctx.close()


def test_session_ranges_equal_cluster_fast_strand_both():
    """ranges that do not line up with the rounds give vsg_cluster_fast's results"""
    n, threads = 3000, 16
    seqs = _reads(n, 60, seed=401)
    ctx = vlib.Context(0)
    ss = ctx.seqset(synth.SeqSet(sorted(seqs, key=len, reverse=True)))
    ss.dust()
    o = _opts(0.97)
    whole, ncl, _ = vlib.cluster_fast(ctx, ss, o, threads)
    sess = vlib.ClusterSession(ctx, ss, o)
    parts = [sess.assign(s, min(257, n - s), threads) for s in range(0, n, 257)]
    assert np.array_equal(np.concatenate(parts), whole)
    assert sess.clusters == ncl
    assert (whole["strand"] == 1).sum() > 0
    sess.close(); ss.close(); ctx.close()


@needs_cli
def test_strand_plus_unchanged_and_both_strands_do_more_work(tmp_path):
    """the same mixed-orientation reads with strand plus equal the CLI without --strand both"""
    n, threads = 4000, 8
    seqs = _reads(n, 120, seed=402)
    labels = [f"a{i:07d}" for i in range(n)]
    fa = _write(tmp_path, labels, seqs)
    want = _cli(tmp_path, fa, 0.97, threads, strand_both=False)
    order = _order(seqs, labels)
    ctx = vlib.Context(0)
    ss = ctx.seqset(synth.SeqSet([seqs[i] for i in order]))
    ss.dust()
    res, ncl, work_plus = vlib.cluster_fast(ctx, ss, _opts(0.97, strand_both=0), threads)
    assert ncl == want["clusters"] and want["minus"] == 0
    assert (res["strand"] == 0).all()
    assert _records_digest(_records(ctx, ss, ss, res, labels, order)) == want
    res2, ncl2, work_both = vlib.cluster_fast(ctx, ss, _opts(0.97, strand_both=1), threads)
    assert ncl2 < ncl
    assert work_both[0] > work_plus[0] and work_both[1] > work_plus[1]
    ss.close(); ctx.close()


@needs_cli
def test_deferred_pairs_on_both_strands_go_through_the_fallback(tmp_path):
    """pairs of long reads (q*d > 25e6) are deferred to the linear-memory aligner, on the reverse complement for
    strand 1, and the records still equal the CLI's"""
    rng = np.random.default_rng(43)
    roots = synth.random_seqs(rng, 3, 5300)
    seqs = []
    for r in range(3):
        for j in range(3):
            s = synth.mutate(rng, roots[r], 0.02).tobytes()
            seqs.append(_rc(s) if (r + j) % 2 == 1 else s)
    seqs += [s.tobytes() for s in synth.random_seqs(rng, 4, 400)]   # ordinary reads, one cluster each
    n = len(seqs)
    labels = [f"L{i:03d}" for i in range(n)]
    fa = _write(tmp_path, labels, seqs)
    threads = 4
    want = _cli(tmp_path, fa, 0.9, threads, qmask="none")
    order = _order(seqs, labels)
    sorted_seqs = [seqs[i] for i in order]
    ref = checkers.RefDb(synth.SeqSet(sorted_seqs), id=0.9, maxaccepts=1, maxrejects=8)
    # which pairs the device defers is known only after it ran: ask the reference for every pair of long reads in
    # both orientations first, so that the answers exist without oracle/_ref
    lma = {}
    for a in range(n):
        for b in range(n):
            if a != b and len(sorted_seqs[a]) > 5000 and len(sorted_seqs[b]) > 5000:
                for st in (0, 1):
                    q = _rc(sorted_seqs[a]) if st else sorted_seqs[a]
                    lma[(a, st, b)] = ref.lma(q, sorted_seqs[b])

    def fallback(q, strand, t):
        out, cigar = lma[(q, strand, t)]
        ops = re.findall(r"(\d*)([MID])", cigar)
        f, l = ops[0], ops[-1]
        fr = int(f[0]) if f[0] else 1; lr = int(l[0]) if l[0] else 1
        return [out[0], out[1], out[2], out[3], out[4], fr if f[1] == "D" else 0, fr if f[1] == "I" else 0,
                lr if l[1] == "D" else 0, lr if l[1] == "I" else 0]

    ctx = vlib.Context(0)
    ss = ctx.seqset(synth.SeqSet(sorted_seqs))
    o = _opts(0.9, mask_lower=0)
    with pytest.raises(vlib.VsgError, match="linear-memory aligner"):
        vlib.cluster_fast(ctx, ss, o, threads)
    ctx.set_fallback(fallback)
    res, ncl, _ = vlib.cluster_fast(ctx, ss, o, threads)
    assert ncl == want["clusters"] == 3 + 4
    rc = ctx.revcomp(ss)
    got = _records(ctx, ss, rc, res, labels, order, lma_cigar=lambda k, st, t: lma[(k, st, t)][1])
    assert _records_digest(got) == want
    assert (res["strand"][res["centroid"] >= 0] == 1).sum() >= 2
    vlib.load().vsg_ctx_set_fallback(ctx.h, None, None)
    ref.close(); rc.close(); ss.close(); ctx.close()


def test_strand_both_keeps_the_wordlength_limit():
    ctx = vlib.Context(0)
    ss = ctx.seqset(synth.SeqSet([b"ACGTACGTACGTAAACCCGGGTTT" * 4, b"ACGTACGTACGTAAACCCGGGTTA" * 4]))
    o = _opts(0.97); o.wordlength = 11
    with pytest.raises(vlib.VsgError, match="wordlength 3..10"):
        vlib.cluster_fast(ctx, ss, o, 2)
    ss.close(); ctx.close()


# ---- seam 2: shim/cluster_session_vsg.cpp against the reference's clustering session, on both strands ----
REF = os.path.join(checkers.ROOT, "oracle", "_ref")
needs_strand_driver = pytest.mark.skipif(not os.path.exists(os.path.join(REF, "seam2_cluster_driver_strand_gpu")),
                                         reason="oracle/_ref (compiled reference + cluster shim) not present")


def _seam2_reads(tmp_path):
    """1 500 amplicon reads (sizes, DUST bait, IUPAC symbols), about 40 % reversed, and two families of three 5 300-nt
    reads, some reversed, whose pairs the 16-bit aligner defers to the linear-memory aligner"""
    rng = np.random.default_rng(78)
    recs = []
    big = synth.random_seqs(rng, 2, 5300)
    for r in range(2):
        for j in range(3):
            s = synth.mutate(rng, big[r], 0.01).tobytes()
            recs.append((f"L{r}{j};size={int(rng.integers(1, 200))}", _rc(s) if (r + j) % 2 else s))
    roots = synth.random_seqs(rng, 40, 320)
    for i in range(1500):
        m = synth.mutate(rng, roots[int(rng.integers(0, 40))], float(rng.uniform(0.0, 0.06))).tobytes()
        a, b = int(rng.integers(0, 25)), int(rng.integers(0, 25))
        s = m[a: len(m) - b]
        if i % 41 == 7:
            s = s[:100] + b"ACACACACACACACACACACACACACACACACACAC" + s[100:]
        if i % 97 == 11:
            s = s[:50] + b"NRY" + s[53:]
        if rng.random() < 0.4:
            s = _rc(s)
        recs.append((f"r{i};size={int(rng.integers(1, 200))}", s))
    path = str(tmp_path / "reads.fasta")
    with open(path, "wb") as f:
        for h, s in recs:
            f.write(b">" + h.encode() + b"\n" + s + b"\n")
    return path


@needs_strand_driver
@pytest.mark.parametrize("case", [
    ["strand=both", "id=0.97", "threads=1", "chunk=-1"],        # cluster_assign_single, one by one
    ["strand=both", "id=0.97", "threads=8", "chunk=0"],         # one cluster_assign_batch over everything
    ["strand=both", "id=0.95", "threads=16", "chunk=300"],      # ranges that do not line up with the rounds
    ["strand=both", "id=0.9", "threads=8", "chunk=0", "maxaccepts=4", "maxrejects=16", "sizeorder=1"],
    ["strand=plus", "id=0.97", "threads=8", "chunk=300"],
], ids=lambda c: " ".join(c))
def test_cluster_session_shim_strand_equals_the_reference(tmp_path, case):
    """seam2_cluster_driver linked against the untouched reference and against the shim prints identical records
    (cluster numbers, centroids, identities to ten digits, CIGARs of the reverse complement for minus-strand members)"""
    reads = _seam2_reads(tmp_path)
    env = dict(os.environ, SEAM2_STRAND=case[0].split("=", 1)[1])
    outs = []
    for exe in ("seam2_cluster_driver_strand_ref", "seam2_cluster_driver_strand_gpu"):
        r = subprocess.run([os.path.join(REF, exe), reads] + case[1:], capture_output=True, text=True, timeout=900, env=env)
        assert r.returncode == 0, (exe, r.stdout[-2000:], r.stderr[-2000:])
        outs.append(r.stdout.splitlines())
    assert len(outs[0]) == 1506
    assert outs[0] == outs[1], [x for x in zip(outs[0], outs[1]) if x[0] != x[1]][:5]
    long_centroids = sum(1 for l in outs[0] if l.split("\t")[1].startswith("L") and l.split("\t")[2] == "1")
    # each family of long reads is one cluster on both strands, two (one per orientation) on the plus strand alone:
    # the reversed reads join through the minus strand and the linear-memory aligner
    assert long_centroids == (2 if case[0] == "strand=both" else 4)
