"""GPU parity of the k-mer ranker (vsg_rank) and the whole search path (vsg_search_batch) against
the golden fixtures, the oracle and — when oracle/_ref travelled along — the unmodified reference."""
import json
import contextlib
import os

import numpy as np
import pytest

import checkers
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return json.load(open(os.path.join(G, name)))


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


@contextlib.contextmanager
def no_tail():
    """VSG_TAIL_PAIRS=0: never prefetch the remaining candidates of the last few active queries"""
    os.environ["VSG_TAIL_PAIRS"] = "0"
    try:
        yield
    finally:
        del os.environ["VSG_TAIL_PAIRS"]


def test_rank_and_search_golden(ctx):
    g = load("rank_search_vectors.json")
    dbs = synth.SeqSet([d.encode() for d in g["db"]])
    qss = synth.SeqSet([q.encode() for q in g["queries"]])
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    nq = len(qss)
    for case in g["cases"]:
        th = case["tophits"]
        seqno, count, nc = ctx.rank(ix, qs, 0, nq, 12, th)
        for i in range(nq):
            assert [seqno[i, :nc[i]].tolist(), count[i, :nc[i]].tolist()] == case["topscores"][i], (case["id"], i)
        o = gpu_opts(case["id"], case["maxaccepts"], case["maxrejects"], case["strand_both"])
        res, counts, work = ctx.search(ix, db, qs, 0, nq, o, th)
        for i in range(nq):
            got = rows_of(res, counts, i, th)
            want = case["rows"][i]
            if case["strand_both"]:
                assert sorted(map(tuple, got)) == sorted(map(tuple, want)), (case["id"], i)
                assert [r[1] for r in got] == sorted([r[1] for r in got], reverse=True)
            else:
                assert got == want, (case["id"], i, got, want)
        assert work[0] > 0 and work[1] > 0
        # the default run above took the "tail" shortcut at once (few queries: all remaining candidates
        # in one device call); without it the driver aligns exactly the reference's pairs
        with no_tail():
            res1, counts1, work1 = ctx.search(ix, db, qs, 0, nq, o, th)
        assert counts1.tolist() == counts.tolist()
        for i in range(nq):
            assert rows_of(res1, counts1, i, th) == rows_of(res, counts, i, th), (case["id"], i)
        assert (int(work1[0]), int(work1[1])) == (int(work[0]), int(work[1]))
        assert (int(work1[2]), int(work1[3])) == (int(work[0]), int(work[1]))
        assert work[2] >= work[0] and work[3] >= work[1]
        # lazy alignment: same hit tables and the same reference-equivalent workload, fewer cells aligned
        o.lazy = 1
        for tail in (True, False):
            if tail:
                res2, counts2, work2 = ctx.search(ix, db, qs, 0, nq, o, th)
            else:
                with no_tail():
                    res2, counts2, work2 = ctx.search(ix, db, qs, 0, nq, o, th)
            assert counts2.tolist() == counts.tolist()
            for i in range(nq):
                assert rows_of(res2, counts2, i, th) == rows_of(res, counts, i, th), (case["id"], i, tail)
            assert (int(work2[0]), int(work2[1])) == (int(work[0]), int(work[1]))
            if not tail:
                assert 0 < work2[2] <= work[0] and 0 < work2[3] <= work[1]
    ix.close(); db.close(); qs.close()


def test_reference_api_example_golden(ctx):
    g = load("search_api_example.json")
    p = g["params"]
    db = ctx.seqset(synth.SeqSet([s.encode() for s in g["ref_seqs"]]))
    qs = ctx.seqset(synth.SeqSet([s.encode() for s in g["query_seqs"]]))
    ix = ctx.index(db, p["wordlength"], 1)
    o = gpu_opts(p["id"], p["maxaccepts"], p["maxrejects"], mask_lower=1, k=p["wordlength"])
    res, counts, _ = ctx.search(ix, db, qs, 0, len(g["query_seqs"]), o, p["max_results"])
    got = []
    for i, ql in enumerate(g["query_labels"]):
        for r in rows_of(res, counts, i, p["max_results"]):
            got.append([ql, g["ref_labels"][r[0]], f"{r[1]:.1f}"])
    assert sorted(got) == sorted(g["expected_rows"])
    # and the full-precision rows the reference library returned when the fixture was made
    for i in range(len(g["query_labels"])):
        assert rows_of(res, counts, i, p["max_results"]) == g["full_rows"][i]
    ix.close(); db.close(); qs.close()


def test_multi_shard_database_vs_oracle(ctx):
    """> 32768 targets: several index shards, candidate-list overflow handling, ties on count"""
    rng = np.random.default_rng(31)
    roots = synth.random_seqs(rng, 40, 120)
    n = 70000
    pick = rng.integers(0, 40, size=n)
    seqs = []
    for i in range(n):
        s = roots[pick[i]].copy()
        pos = rng.integers(0, 120, size=3)
        s[pos] = synth.ACGT[rng.integers(0, 4, size=3)]
        seqs.append(s[: int(rng.integers(90, 121))].tobytes())
    dbs = synth.SeqSet(seqs)
    queries = [synth.mutate(rng, roots[i % 40], 0.03).tobytes() for i in range(24)]
    queries += [synth.random_seqs(rng, 1, 100)[0].tobytes(), b"ACGTACG"]   # no hit / shorter than k
    qss = synth.SeqSet(queries)
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    od = checkers.OracleDb(dbs)
    opts = checkers.search_opts(n, id=0.95, maxaccepts=2, maxrejects=8)
    seqno, count, nc = ctx.rank(ix, qs, 0, len(queries), opts.minwordmatches, opts.tophits)
    for i, q in enumerate(queries):
        s, c = od.topscores(q, opts)
        assert seqno[i, :nc[i]].tolist() == s.tolist() and count[i, :nc[i]].tolist() == c.tolist(), i
    o = gpu_opts(0.95, 2, 8)
    res, counts, work = ctx.search(ix, db, qs, 0, len(queries), o, opts.tophits)
    pairs = cells = 0
    for i, q in enumerate(queries):
        hits, p, cl = od.search(q, opts)
        pairs += p; cells += cl
        want = [[h.target, h.id, h.matches, h.mismatches, h.nwgaps, h.nwalignmentlength, h.accepted, h.strand]
                for h in hits]
        assert rows_of(res, counts, i, opts.tophits) == want, i
    assert (int(work[0]), int(work[1])) == (pairs, cells)   # same search16 workload as the reference's driver
    od.close(); ix.close(); db.close(); qs.close()


def test_ranker_ties_and_thresholds_vs_oracle(ctx):
    """the ranker's running threshold: thousands of targets tied on the k-mer count (more than its key
    buffer holds), few candidates (< tophits), tophits from 1 to 1024, in one and in several shards"""
    rng = np.random.default_rng(53)
    root = synth.random_seqs(rng, 1, 150)[0]
    seqs = []
    for i in range(6000):                      # 6000 near-copies: same k-mer count for thousands of them
        s = root.copy()
        if i % 3 == 1:
            s[int(rng.integers(0, 150))] = synth.ACGT[int(rng.integers(0, 4))]
        seqs.append(s[: 150 - (i % 5)].tobytes())          # length decides among equal counts, then seqno
    other = synth.random_seqs(rng, 34000, 90)
    seqs += [other[i].tobytes() for i in range(34000)]   # second shard: unrelated
    seqs += [synth.mutate(rng, root, 0.1).tobytes() for _ in range(50)]
    dbs = synth.SeqSet(seqs)
    queries = [root.tobytes(), synth.mutate(rng, root, 0.04).tobytes(), root[:60].tobytes(),
               other[5].tobytes(), synth.random_seqs(rng, 1, 120)[0].tobytes()]
    qss = synth.SeqSet(queries)
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    od = checkers.OracleDb(dbs)
    for maxaccepts, maxrejects in ((1, 0), (1, 32), (8, 100), (500, 516)):
        opts = checkers.search_opts(len(seqs), id=0.9, maxaccepts=maxaccepts, maxrejects=maxrejects)
        seqno, count, nc = ctx.rank(ix, qs, 0, len(queries), opts.minwordmatches, opts.tophits)
        for i, q in enumerate(queries):
            s_, c_ = od.topscores(q, opts)
            assert nc[i] == len(s_), (opts.tophits, i, nc[i], len(s_))
            assert seqno[i, :nc[i]].tolist() == s_.tolist() and count[i, :nc[i]].tolist() == c_.tolist(), (opts.tophits, i)
    od.close(); ix.close(); db.close(); qs.close()


@pytest.mark.skipif(not checkers.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")
def test_search_vs_compiled_reference(ctx):
    """config-2 shape in miniature: 250-nt windows of a random 1500-nt database, 5 % mutated"""
    dbs, qss, src = synth.config2_search(n_db=400, db_len=1500, n_q=120, q_len=250, div=0.05, seed=77)
    r = checkers.RefDb(dbs, id=0.9, maxaccepts=1, maxrejects=32)
    want = r.search(qss, max_results=r.tophits)
    th = r.tophits
    r.close()
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    res, counts, _ = ctx.search(ix, db, qs, 0, len(qss), gpu_opts(0.9, 1, 32), th)
    hit = 0
    for i in range(len(qss)):
        got = rows_of(res, counts, i, th)
        assert got == [list(t) for t in want[i]], i
        hit += bool(got) and got[0][0] == int(src[i])
    assert hit > 100
    ol = gpu_opts(0.9, 1, 32); ol.lazy = 1
    with no_tail():
        res2, counts2, work2 = ctx.search(ix, db, qs, 0, len(qss), ol, th)
    for i in range(len(qss)):
        assert rows_of(res2, counts2, i, th) == [list(t) for t in want[i]], i
    assert work2[2] * 4 < work2[0]     # the first candidate is almost always accepted: ~1 of 8 pairs aligned
    # the tail shortcut entered after ordinary rounds (threshold below the first round's size), and at once
    for tail_pairs in ("16", "100000"):
        os.environ["VSG_TAIL_PAIRS"] = tail_pairs
        try:
            for o in (gpu_opts(0.9, 1, 32), ol):
                res3, counts3, work3 = ctx.search(ix, db, qs, 0, len(qss), o, th)
                for i in range(len(qss)):
                    assert rows_of(res3, counts3, i, th) == [list(t) for t in want[i]], (tail_pairs, o.lazy, i)
                assert (int(work3[0]), int(work3[1])) == (int(work2[0]), int(work2[1]))
        finally:
            del os.environ["VSG_TAIL_PAIRS"]
    ix.close(); db.close(); qs.close()


@pytest.mark.skipif(not checkers.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")
@pytest.mark.parametrize("maxaccepts,ident", [(1, 0.9), (1, 0.97), (3, 0.9)])
def test_traceback_on_demand_does_not_change_the_hit_tables(ctx, maxaccepts, ident):
    """the followers of a group are walked back only when the leader is not accepted (align_ckpt.cuh, TbGate): same rows
    with the shortcut off, on, and with a device verdict that is always "accepted" (every needed follower re-aligned by
    the replay).  id 0.97 puts many leaders below the threshold (5 % mutated queries)."""
    dbs, qss, src = synth.config2_search(n_db=600, db_len=1500, n_q=400, q_len=250, div=0.05, seed=91)
    r = checkers.RefDb(dbs, id=ident, maxaccepts=maxaccepts, maxrejects=16)
    want = r.search(qss, max_results=r.tophits)
    th = r.tophits
    r.close()
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    os.environ["VSG_CKPT_MIN_PAIRS"] = "0"     # the checkpoint kernels at this call size too
    try:
        for env in ({"VSG_TB_GATE": "0"}, {}, {"VSG_TB_GATE_FORCE": "1"}):
            os.environ.update(env)
            try:
                with no_tail():
                    res, counts, work = ctx.search(ix, db, qs, 0, len(qss), gpu_opts(ident, maxaccepts, 16), th)
            finally:
                for k in env:
                    del os.environ[k]
            for i in range(len(qss)):
                assert rows_of(res, counts, i, th) == [list(t) for t in want[i]], (env, i)
    finally:
        del os.environ["VSG_CKPT_MIN_PAIRS"]
    ix.close(); db.close(); qs.close()


@pytest.mark.skipif(not checkers.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")
def test_deferred_pairs_go_through_the_fallback_callback(ctx):
    """pairs the 16-bit aligner cannot take (q*d > 25e6) are resolved by the host application's
    linear-memory aligner through vsg_ctx_set_fallback — here the reference's own LinearMemoryAligner —
    and the hit table still equals the reference's"""
    import re
    rng = np.random.default_rng(41)
    big = synth.random_seqs(rng, 3, 5200)
    small = synth.random_seqs(rng, 30, 400)
    dbs = synth.SeqSet([big[i].tobytes() for i in range(3)] + [small[i].tobytes() for i in range(30)])
    queries = [synth.mutate(rng, big[0], 0.03).tobytes(),            # 5200 x 5200 > 25e6 -> deferred
               synth.mutate(rng, big[1][:5100], 0.05).tobytes(),
               synth.mutate(rng, small[3], 0.05).tobytes(),          # ordinary
               synth.mutate(rng, small[7], 0.02).tobytes()]
    qss = synth.SeqSet(queries)
    r = checkers.RefDb(dbs, id=0.8, maxaccepts=2, maxrejects=8)
    want = r.search(qss, max_results=r.tophits)
    th = r.tophits

    def fallback(q, strand, t):
        assert strand == 0
        out, cigar = r.lma(queries[q], dbs.seq(t))
        ops = re.findall(r"(\d*)([MID])", cigar)
        f, l = ops[0], ops[-1]
        fr = int(f[0]) if f[0] else 1; lr = int(l[0]) if l[0] else 1
        return [out[0], out[1], out[2], out[3], out[4], fr if f[1] == "D" else 0, fr if f[1] == "I" else 0,
                lr if l[1] == "D" else 0, lr if l[1] == "I" else 0]

    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    o = gpu_opts(0.8, 2, 8)
    with pytest.raises(vlib.VsgError, match="linear-memory aligner"):
        ctx.search(ix, db, qs, 0, len(queries), o, th)
    ctx.set_fallback(fallback)
    res, counts, _ = ctx.search(ix, db, qs, 0, len(queries), o, th)
    for i in range(len(queries)):
        assert rows_of(res, counts, i, th) == [list(t) for t in want[i]], i
    assert counts[0] >= 1 and rows_of(res, counts, 0, th)[0][0] == 0
    load = vlib.load(); load.vsg_ctx_set_fallback(ctx.h, None, None)
    r.close(); ix.close(); db.close(); qs.close()


def test_long_queries_rank_vs_oracle(ctx):
    """queries with more than 2048 k-mer windows take the HBM de-duplication path of the ranker"""
    rng = np.random.default_rng(43)
    roots = synth.random_seqs(rng, 30, 700)
    dbs = synth.SeqSet([synth.mutate(rng, roots[i % 30], 0.05).tobytes() for i in range(400)])
    queries = [b"".join(roots[j].tobytes() for j in range(4)),                 # 2800 nt
               (roots[5].tobytes() + roots[6].tobytes()) * 4,                   # 5600 nt, every k-mer 4 times
               synth.random_seqs(rng, 1, 2056)[0].tobytes(),                    # just past the shared-memory capacity
               synth.random_seqs(rng, 1, 2055)[0].tobytes(),                    # exactly at it
               roots[9].tobytes()]
    qss = synth.SeqSet(queries)
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    od = checkers.OracleDb(dbs)
    opts = checkers.search_opts(len(dbs), id=0.9, maxaccepts=4, maxrejects=16)
    seqno, count, nc = ctx.rank(ix, qs, 0, len(queries), opts.minwordmatches, opts.tophits)
    for i, q in enumerate(queries):
        s, c = od.topscores(q, opts)
        assert seqno[i, :nc[i]].tolist() == s.tolist() and count[i, :nc[i]].tolist() == c.tolist(), i
    od.close(); ix.close(); db.close(); qs.close()


@pytest.mark.skipif(not checkers.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")
def test_optional_filters_vs_compiled_reference(ctx):
    """--minqt/--maxqt/--minsl/--maxsl (pre-alignment rejects consume the reject budget) and
    --maxsubs/--maxgaps/--mincols/--maxdiffs/--leftjust/--rightjust/--query_cov/--target_cov/--maxid/--mid"""
    rng = np.random.default_rng(47)
    roots = synth.random_seqs(rng, 8, 320)
    seqs = []
    for r in range(8):
        for _ in range(10):
            m = synth.mutate(rng, roots[r], float(rng.uniform(0.0, 0.15)))
            a = int(rng.integers(0, 60)); b = int(rng.integers(0, 60))
            seqs.append(m[a: m.shape[0] - b].tobytes())       # ragged ends: terminal gaps, length ratios
    dbs = synth.SeqSet(seqs)
    queries = [synth.mutate(rng, roots[i % 8], 0.05)[int(rng.integers(0, 40)):].tobytes() for i in range(32)]
    qss = synth.SeqSet(queries)
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, 8, 0)
    big = 2147483647.0
    cases = [
        dict(minqt=0.9, maxqt=1.1),
        dict(minsl=0.92, maxsl=0.99),
        dict(maxsubs=12, maxgaps=2, mincols=250),
        dict(maxdiffs=20, leftjust=1),
        dict(rightjust=1, query_cov=0.9, target_cov=0.9),
        dict(maxid=0.97, mid=93.0),
    ]
    for case in cases:
        v = dict(minqt=0.0, maxqt=1.7976931348623157e308, minsl=0.0, maxsl=1.7976931348623157e308, maxid=1.0, mid=0.0,
                 query_cov=0.0, target_cov=0.0, maxsubs=big, maxgaps=big, mincols=0.0, maxdiffs=big, leftjust=0.0, rightjust=0.0)
        v.update(case)
        order = ["minqt", "maxqt", "minsl", "maxsl", "maxid", "mid", "query_cov", "target_cov", "maxsubs", "maxgaps",
                 "mincols", "maxdiffs", "leftjust", "rightjust"]
        r = checkers.RefDb(dbs, id=0.85, maxaccepts=3, maxrejects=6)
        r.set_filters([v[k] for k in order])
        want = r.search(qss, max_results=r.tophits)
        th = r.tophits
        r.close()
        o = gpu_opts(0.85, 3, 6)
        for k in order:
            setattr(o, k, type(getattr(o, k))(v[k]))
        res, counts, _ = ctx.search(ix, db, qs, 0, len(queries), o, th)
        nrows = 0
        for i in range(len(queries)):
            got = rows_of(res, counts, i, th)
            assert got == [list(t) for t in want[i]], (case, i)
            nrows += len(got)
        assert nrows > 0, case
    ix.close(); db.close(); qs.close()
