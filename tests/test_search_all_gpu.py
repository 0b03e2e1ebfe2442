"""Searches whose candidate lists are longer than the shared-memory ranker's 1 024 entries: --maxaccepts 0,
--maxrejects 0 and large limits (tophits = min(maxaccepts + maxrejects + 8, database size) > 1024).  The ranker's
two-pass mode (vsg_rank), the whole search (vsg_search_batch), its split of a sub-batch by candidate volume, the
streaming driver and the drop-in search_batch() are compared with the oracle and the unmodified reference."""
import os
import re
import subprocess

import numpy as np
import pytest

import checkers
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")
COMP = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")

needs_reference = pytest.mark.skipif(not checkers.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")
needs_cli = pytest.mark.skipif(not checkers.have_reference_cli(), reason="neither oracle/_ref nor tests/golden/reference")


@pytest.fixture(scope="module")
def ctx():
    c = vlib.Context(0)
    yield c
    c.close()


def rows_of(res, counts, q, max_results):
    out = []
    for j in range(int(counts[q])):
        r = res[q * max_results + j]
        out.append([r.target, r.id, r.matches, r.mismatches, r.gaps, r.alignment_length, r.accepted, r.strand])
    return out


def gpu_opts(id, maxaccepts, maxrejects, strand_both=0, mask_lower=0, k=8):
    o = vlib.default_search_opts()
    o.id = id; o.maxaccepts = maxaccepts; o.maxrejects = maxrejects; o.strand_both = strand_both
    o.mask_lower = mask_lower; o.wordlength = k
    return o


def clamp(v, n):
    """the command line's fix-up of a limit (usearch_global.cpp:598-614): 0 or more than the database means all"""
    return n if v == 0 or v > n else v


# ---- the ranker -----------------------------------------------------------------------------------------------------
def _rank_db(mask=False):
    """70 050 targets in three shards: 6 000 near-copies of one root (thousands tie on the k-mer count; length, then the
    target number decide among them), 64 000 unrelated ones, 50 distant relatives"""
    rng = np.random.default_rng(8101)
    root = synth.random_seqs(rng, 1, 150)[0]
    seqs = []
    for i in range(6000):
        s = root.copy()
        if i % 3 == 1:
            s[int(rng.integers(0, 150))] = synth.ACGT[int(rng.integers(0, 4))]
        seqs.append(s[: 150 - (i % 5)].tobytes())
    other = synth.random_seqs(rng, 64000, 90)
    seqs += [other[i].tobytes() for i in range(64000)]
    seqs += [synth.mutate(rng, root, 0.1).tobytes() for _ in range(50)]
    if mask:
        seqs = [s[:40].lower() + s[40:] if i % 4 == 0 else s for i, s in enumerate(seqs)]
    long_q = b"".join([root.tobytes()] + [synth.random_seqs(rng, 1, 400)[0].tobytes() for _ in range(6)])   # 2 550 nt
    queries = [root.tobytes(), synth.mutate(rng, root, 0.04).tobytes(), root[:60].tobytes(), other[5].tobytes(),
               synth.random_seqs(rng, 1, 120)[0].tobytes(), long_q, long_q[:2200] + root.tobytes()]
    if mask:
        queries = [q[:30].lower() + q[30:] for q in queries]
    return synth.SeqSet(seqs), synth.SeqSet(queries)


@pytest.mark.parametrize("k,mask", [(8, 0), (12, 0), (8, 1)], ids=["k8", "k12_sparse", "k8_mask_lower"])
def test_rank_long_lists_vs_oracle(ctx, k, mask):
    dbs, qss = _rank_db(mask=bool(mask))
    n = len(dbs)
    assert n > 2 * 32766 and max(qss.lens) - k + 1 > 2048
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, k, mask)
    od = checkers.OracleDb(dbs, k=k, mask_lower=mask)
    opts = checkers.search_opts(n, k=k, mask_lower=mask)
    longest = 0
    for th in (1025, 4096, n):
        opts.tophits = th
        seqno, count, nc = ctx.rank(ix, qs, 0, len(qss), opts.minwordmatches, th, mask)
        for i in range(len(qss)):
            s, c = od.topscores(qss.seq(i), opts)
            assert nc[i] == len(s), (th, i, nc[i], len(s))
            assert seqno[i, :nc[i]].tolist() == s.tolist() and count[i, :nc[i]].tolist() == c.tolist(), (th, i)
            longest = max(longest, int(nc[i]))
    assert longest > 6000     # the family and more
    od.close(); ix.close(); db.close(); qs.close()


@needs_reference
def test_rank_long_lists_vs_reference(ctx):
    dbs, qss = _rank_db()
    r = checkers.RefDb(dbs, id=0.9, maxaccepts=1, maxrejects=4087)
    assert r.tophits == 4096
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    seqno, count, nc = ctx.rank(ix, qs, 0, len(qss), 12, 4096)
    for i in range(len(qss)):
        s, c = r.topscores(qss.seq(i))
        assert seqno[i, :nc[i]].tolist() == s.tolist() and count[i, :nc[i]].tolist() == c.tolist(), i
    assert int(nc[0]) == 4096
    r.close(); ix.close(); db.close(); qs.close()


# ---- the whole search -----------------------------------------------------------------------------------------------
def _family_db(n_fam=1300, n_random=400, seed=8201):
    """two families of n_fam mutated copies of a 300-nt root (every query of a family has > 1 024 candidates) and
    n_random unrelated targets; queries: 250-nt windows of the roots, mutated, some reverse-complemented, two unrelated"""
    rng = np.random.default_rng(seed)
    roots = synth.random_seqs(rng, 2, 300)
    seqs = []
    for i in range(2 * n_fam):
        m = synth.mutate(rng, roots[i % 2], float(rng.uniform(0.01, 0.12)))
        a, b = int(rng.integers(0, 15)), int(rng.integers(0, 15))
        seqs.append(m[a: m.shape[0] - b].tobytes())
    seqs += [s.tobytes() for s in synth.random_seqs(rng, n_random, 300)]
    queries = []
    for i in range(22):
        a = int(rng.integers(0, 50))
        q = synth.mutate(rng, roots[i % 2][a: a + 250], 0.03).tobytes()
        queries.append(q[::-1].translate(COMP) if i % 5 == 3 else q)
    queries += [s.tobytes() for s in synth.random_seqs(rng, 2, 250)]
    return synth.SeqSet(seqs), synth.SeqSet(queries)


SEARCH_CASES = [(0, 0), (0, 32), (40, 2000)]


def _reference_rows(dbs, qss, maxaccepts, maxrejects, id=0.9):
    n = len(dbs)
    r = checkers.RefDb(dbs, id=id, maxaccepts=clamp(maxaccepts, n), maxrejects=clamp(maxrejects, n), strand_both=1)
    want = r.search(qss, max_results=2 * n)
    r.close()
    return [[list(t) for t in rows] for rows in want]


@needs_reference
@pytest.mark.parametrize("maxaccepts,maxrejects", SEARCH_CASES, ids=[f"maxaccepts{a}_maxrejects{b}" for a, b in SEARCH_CASES])
def test_search_long_lists_vs_reference(ctx, maxaccepts, maxrejects):
    dbs, qss = _family_db()
    n = len(dbs)
    want = _reference_rows(dbs, qss, maxaccepts, maxrejects)
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    mr = 2 * n
    res, counts, work = ctx.search(ix, db, qs, 0, len(qss), gpu_opts(0.9, maxaccepts, maxrejects, strand_both=1), mr)
    nrows = 0
    for i in range(len(qss)):
        got = rows_of(res, counts, i, mr)
        assert got == want[i], (i, len(got), len(want[i]))
        nrows += len(got)
    assert nrows > 200 and (maxaccepts > 0 or max(int(c) for c in counts) > 100)
    assert any(r[7] == 1 for rows in want for r in rows)      # minus-strand hits
    if maxaccepts == maxrejects == 0:
        # no limit can stop a list early: every list is aligned in the first round; in groups of eight without the tail
        os.environ["VSG_TAIL_PAIRS"] = "0"
        try:
            res2, counts2, work2 = ctx.search(ix, db, qs, 0, len(qss), gpu_opts(0.9, 0, 0, strand_both=1), mr)
        finally:
            del os.environ["VSG_TAIL_PAIRS"]
        for i in range(len(qss)):
            assert rows_of(res2, counts2, i, mr) == want[i], i
        assert (int(work2[0]), int(work2[1])) == (int(work[0]), int(work[1]))
    # the reference's pairs and DP cells (work[0..1]) for a sample of queries, plus strand, against the oracle
    od = checkers.OracleDb(dbs)
    oo = checkers.search_opts(n, id=0.9, maxaccepts=clamp(maxaccepts, n), maxrejects=clamp(maxrejects, n))
    sample = [0, 1, 6, 22]
    pairs = cells = 0
    for i in sample:
        _, p, c = od.search(qss.seq(i), oo)
        pairs += p; cells += c
    sq = ctx.seqset(synth.SeqSet([qss.seq(i) for i in sample]))
    _, _, w = ctx.search(ix, db, sq, 0, len(sample), gpu_opts(0.9, maxaccepts, maxrejects), mr)
    assert (int(w[0]), int(w[1])) == (pairs, cells) and pairs > (1024 if maxaccepts == maxrejects == 0 else 0)
    od.close(); sq.close(); ix.close(); db.close(); qs.close()


@needs_reference
def test_search_splits_a_sub_batch_by_candidate_volume(ctx, capfd):
    """a candidate budget far below one sub-batch's volume: the call runs in many pieces and still equals the
    reference (the stored answer of the exhaustive case above)"""
    dbs, qss = _family_db()
    want = _reference_rows(dbs, qss, 0, 0)
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    mr = 2 * len(dbs)
    os.environ["VSG_CAND_BUDGET"] = "3000"
    os.environ["VSG_TRACE"] = "1"
    try:
        capfd.readouterr()
        res, counts, _ = ctx.search(ix, db, qs, 0, len(qss), gpu_opts(0.9, 0, 0, strand_both=1), mr)
        err = capfd.readouterr().err
    finally:
        del os.environ["VSG_CAND_BUDGET"], os.environ["VSG_TRACE"]
    pieces = [int(m) for m in re.findall(r"searched in (\d+) pieces", err)]
    assert pieces and max(pieces) > 4, err[-2000:]
    for i in range(len(qss)):
        assert rows_of(res, counts, i, mr) == want[i], i
    ix.close(); db.close(); qs.close()


@needs_reference
def test_long_lists_with_deferred_pairs_through_the_fallback_callback(ctx):
    """pairs the 16-bit aligner cannot take (q*d > 25e6) in an exhaustive search, resolved by the reference's own
    LinearMemoryAligner through vsg_ctx_set_fallback"""
    rng = np.random.default_rng(8301)
    big = synth.random_seqs(rng, 3, 5200)
    small = synth.random_seqs(rng, 30, 400)
    filler = synth.random_seqs(rng, 1100, 200)
    dbs = synth.SeqSet([big[i].tobytes() for i in range(3)] + [small[i].tobytes() for i in range(30)] +
                       [filler[i].tobytes() for i in range(1100)])
    n = len(dbs)
    queries = [synth.mutate(rng, big[0], 0.03).tobytes(), synth.mutate(rng, big[1][:5100], 0.05).tobytes(),
               synth.mutate(rng, small[3], 0.05).tobytes(), synth.mutate(rng, small[7], 0.02).tobytes()]
    qss = synth.SeqSet(queries)
    r = checkers.RefDb(dbs, id=0.8, maxaccepts=2, maxrejects=n)
    want = r.search(qss, max_results=64)

    def fallback(q, strand, t):
        out, cigar = r.lma(queries[q], dbs.seq(t))
        ops = re.findall(r"(\d*)([MID])", cigar)
        f, l = ops[0], ops[-1]
        fr = int(f[0]) if f[0] else 1; lr = int(l[0]) if l[0] else 1
        return [out[0], out[1], out[2], out[3], out[4], fr if f[1] == "D" else 0, fr if f[1] == "I" else 0,
                lr if l[1] == "D" else 0, lr if l[1] == "I" else 0]

    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    ctx.set_fallback(fallback)
    try:
        res, counts, _ = ctx.search(ix, db, qs, 0, len(queries), gpu_opts(0.8, 2, 0), 64)
    finally:
        vlib.load().vsg_ctx_set_fallback(ctx.h, None, None)
    for i in range(len(queries)):
        assert rows_of(res, counts, i, 64) == [list(t) for t in want[i]], i
    assert counts[0] >= 1 and rows_of(res, counts, 0, 64)[0][0] == 0
    r.close(); ix.close(); db.close(); qs.close()


# ---- the streaming driver against the reference CLI -----------------------------------------------------------------
def _file_digest(path):
    data = open(path, "rb").read()
    return {"size": len(data), "sha256": checkers.digest(data)}


def _write(path, seqs, prefix):
    with open(path, "w") as f:
        for i, s in enumerate(seqs):
            f.write(f">{prefix}{i}\n{s.decode()}\n")


STREAM_CASES = {
    "exhaustive": (["--maxaccepts", "0", "--maxrejects", "0"], dict(maxaccepts=0, maxrejects=0), {}),
    "lulu_without_self": (["--maxaccepts", "0", "--maxhits", "10"], dict(maxaccepts=0), dict(maxhits=10)),
    "both_strands_maxrejects0": (["--strand", "both", "--maxrejects", "0"], dict(strand_both=1, maxrejects=0), {}),
    "idprefix_selfid": (["--maxaccepts", "0", "--maxrejects", "0", "--idprefix", "6", "--selfid"],
                        dict(maxaccepts=0, maxrejects=0, idprefix=6, selfid=1), {}),
    "small_db_all_accepted": (["--maxaccepts", "0"], dict(maxaccepts=0), {}),
}


@needs_cli
@pytest.mark.parametrize("case", list(STREAM_CASES))
def test_stream_long_lists_equal_the_reference_cli(tmp_path, case):
    args_extra, opt, kw = STREAM_CASES[case]
    if case == "small_db_all_accepted":
        # 800 targets: the ranker's ordinary mode (tophits <= 1024), but more than 1 + maxrejects = 33 rows per query
        rng = np.random.default_rng(8401)
        roots = synth.random_seqs(rng, 8, 300)
        dbs = synth.SeqSet([synth.mutate(rng, roots[i % 8], float(rng.uniform(0.0, 0.06))).tobytes() for i in range(800)])
        qss = synth.SeqSet([synth.mutate(rng, roots[i % 8], 0.02).tobytes() for i in range(24)])
    else:
        dbs, qss = _family_db()
        if case == "idprefix_selfid":
            qss = synth.SeqSet([qss.seq(i) for i in range(len(qss))] + [dbs.seq(5), dbs.seq(8)])
    dbf = str(tmp_path / "db.fasta"); qf = str(tmp_path / "q.fasta")
    _write(dbf, [dbs.seq(i) for i in range(len(dbs))], "d")
    _write(qf, [qss.seq(i) for i in range(len(qss))], "q")
    ref_out = str(tmp_path / "ref.b6"); got_out = str(tmp_path / "got.b6")
    args = ["--usearch_global", qf, "--db", dbf, "--id", "0.9", "--blast6out", ref_out, "--threads", "1", "--quiet",
            "--qmask", "none", "--dbmask", "none"] + args_extra
    want = checkers.reference_cli(args, lambda: _file_digest(ref_out), timeout=900)
    o = vlib.default_search_opts(); o.id = 0.9
    for k, v in opt.items():
        setattr(o, k, v)
    g = vlib.Group([0], dbs, wordlength=8)
    st = g.stream([f"d{i}" for i in range(len(dbs))], qf, o, got_out, batch_queries=7, **kw)
    g.close()
    assert st["queries"] == len(qss)
    assert _file_digest(got_out) == want
    rows = open(got_out).read().splitlines()
    per_query = {}
    for row in rows:
        per_query[row.split("\t")[0]] = per_query.get(row.split("\t")[0], 0) + 1
    if case == "lulu_without_self":
        assert max(per_query.values()) == 10
    elif case in ("exhaustive", "small_db_all_accepted"):
        assert max(per_query.values()) > 33
    elif case == "both_strands_maxrejects0":
        assert len(per_query) > 20     # --maxaccepts 1: one row per query, after a search through every candidate


# ---- seam 2: the drop-in search_batch() ------------------------------------------------------------------------------
needs_seam2 = pytest.mark.skipif(not os.path.exists(os.path.join(REF, "seam2_driver_gpu")),
                                 reason="oracle/_ref (compiled reference + shims) not present")


@needs_seam2
def test_search_batch_shim_with_long_lists_equals_reference(tmp_path):
    rng = np.random.default_rng(8501)
    roots = synth.random_seqs(rng, 6, 380)
    db = []
    for i in range(2160):
        m = synth.mutate(rng, roots[i % 6], float(rng.uniform(0.0, 0.12))).tobytes()
        a, b = int(rng.integers(0, 30)), int(rng.integers(0, 30))
        db.append((f"t{i};size={int(rng.integers(1, 60))}", m[a: len(m) - b].decode()))
    queries = []
    for i in range(30):
        m = synth.mutate(rng, roots[i % 6], 0.04).tobytes()[int(rng.integers(0, 30)):]
        if i % 4 == 1:
            m = m[::-1].translate(COMP)
        queries.append((f"q{i};size={int(rng.integers(1, 60))}", m.decode()))
    dbf, qf = str(tmp_path / "db.fasta"), str(tmp_path / "q.fasta")
    for path, recs in ((dbf, db), (qf, queries)):
        with open(path, "w") as f:
            for head, seq in recs:
                f.write(f">{head}\n{seq}\n")
    case = ["id=0.8", "maxaccepts=40", "maxrejects=2000", "strand=1", "max_results=2100"]
    outs = []
    for exe in ("seam2_driver_ref", "seam2_driver_gpu"):
        r = subprocess.run([os.path.join(REF, exe), dbf, qf] + case, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (exe, r.stdout[-2000:], r.stderr[-2000:])
        outs.append(r.stdout.splitlines())
    assert outs[0] == outs[1], (len(outs[0]), len(outs[1]), [x for x in zip(outs[0], outs[1]) if x[0] != x[1]][:5])
    assert len(outs[0]) > 30 * 20
