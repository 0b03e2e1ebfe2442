"""Pins the oracle (oracle/*.c) against the UNMODIFIED reference compiled into
oracle/_ref/libvsref.so.  CPU only.  Without oracle/_ref the reference's answers are the ones stored
under tests/golden/reference (checkers.reference_result)."""
import numpy as np
import pytest

import checkers as _libs
from vsearch_b200 import synth

pytestmark = pytest.mark.skipif(not _libs.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")

IUPAC = b"ACGTUacgtuNnRYSWKMBDHVryswkmbdhvXx-*."


def rand_seq(rng, n, alphabet=b"ACGT"):
    a = np.frombuffer(alphabet, dtype=np.uint8)
    return a[rng.integers(0, a.shape[0], size=n)].tobytes()


def check_pairs(q, targets, pen=None, n_mismatch=0):
    got_ref = _libs.ref_search16(q, targets, pen, n_mismatch)
    for t, r in zip(targets, got_ref):
        o = _libs.oracle_nw16(q, t, pen, n_mismatch)
        assert o == r, (q, t, o, r)


def test_nw16_random_acgt_related():
    rng = np.random.default_rng(1)
    for _ in range(60):
        L = int(rng.integers(1, 260))
        root = np.frombuffer(rand_seq(rng, L), dtype=np.uint8)
        q = synth.mutate(rng, root, 0.1).tobytes()
        targets = [synth.mutate(rng, root, float(rng.uniform(0, 0.4))).tobytes() for _ in range(11)]
        targets += [rand_seq(rng, int(rng.integers(1, 300))) for _ in range(5)]
        check_pairs(q, targets)


def test_nw16_iupac_case_n_and_odd_bytes():
    rng = np.random.default_rng(2)
    for nm in (0, 1):
        for _ in range(40):
            q = rand_seq(rng, int(rng.integers(1, 120)), IUPAC)
            targets = [rand_seq(rng, int(rng.integers(1, 120)), IUPAC) for _ in range(9)]
            check_pairs(q, targets, n_mismatch=nm)


def test_nw16_all_byte_values_map():
    # every byte 1..255 appears in a sequence; the aligner sees them through map_4bit
    q = bytes(range(1, 256))
    t = bytes(reversed(range(1, 256)))
    check_pairs(q, [t, q, b"ACGT"])


def test_nw16_edge_lengths_and_empty():
    rng = np.random.default_rng(3)
    q = rand_seq(rng, 37)
    targets = [b"", b"A", b"AC", b"ACG", b"ACGT", b"ACGTA", rand_seq(rng, 1), rand_seq(rng, 500), b""]
    check_pairs(q, targets)
    check_pairs(b"", [b"", b"A", rand_seq(rng, 77)])
    check_pairs(b"G", [b"G", b"A", b"", rand_seq(rng, 9)])
    # homopolymers / repeats (tie-breaking stress)
    check_pairs(b"A" * 50, [b"A" * 40, b"A" * 60, b"AT" * 25, b"T" * 50])
    check_pairs(b"ACAC" * 20, [b"CACA" * 20, b"AC" * 33, b"ACC" * 20])


def test_nw16_non_default_penalties():
    rng = np.random.default_rng(4)
    for _ in range(30):
        pen = np.array([int(rng.integers(1, 6)), -int(rng.integers(1, 8))]
                       + [int(rng.integers(0, 25)) for _ in range(6)]
                       + [int(rng.integers(0, 5)) for _ in range(6)], dtype=np.int64)
        L = int(rng.integers(5, 150))
        root = np.frombuffer(rand_seq(rng, L), dtype=np.uint8)
        q = synth.mutate(rng, root, 0.15).tobytes()
        targets = [synth.mutate(rng, root, 0.25).tobytes() for _ in range(8)]
        targets.append(rand_seq(rng, int(rng.integers(1, 200))))
        check_pairs(q, targets, pen)


def test_nw16_overflow_and_limits():
    rng = np.random.default_rng(5)
    # big penalties so that 16-bit saturation / the h_min flag fire on short sequences
    pen = np.array([2, -4, 3000, 3000, 5000, 5000, 3000, 3000, 600, 600, 900, 900, 600, 600], dtype=np.int64)
    for L in (10, 30, 60, 120):
        q = rand_seq(rng, L)
        targets = [rand_seq(rng, int(rng.integers(1, 2 * L))) for _ in range(8)]
        check_pairs(q, targets, pen)
    # match score so large that h_max saturates
    pen2 = np.array([3000, -3000, 1, 1, 18, 18, 1, 1, 1, 1, 2, 2, 1, 1], dtype=np.int64)
    q = rand_seq(rng, 40)
    check_pairs(q, [q, q[:20], rand_seq(rng, 40), q + q], pen2)
    # values that do not fit a cell -> every pair deferred (force_scalar_fallback)
    pen3 = pen2.copy(); pen3[4] = 2 ** 31 - 1
    check_pairs(q, [q, b"A"], pen3)
    # long pair under default penalties: top row runs far negative but stays in range
    q = rand_seq(rng, 300)
    check_pairs(q, [rand_seq(rng, 6000), rand_seq(rng, 11)])
    # product limit (q*d > 25e6) and sum limit -> sentinel
    q = rand_seq(rng, 5001)
    check_pairs(q, [rand_seq(rng, 5000), rand_seq(rng, 4999)])
    # saturating boundary row: d long enough that -(go+(j+1)ge) passes -32768 with ge=6 (limit 6553)
    pen4 = np.array([2, -4, 1, 1, 18, 18, 1, 1, 6, 6, 2, 2, 6, 6], dtype=np.int64)
    q = rand_seq(rng, 50)
    check_pairs(q, [rand_seq(rng, 6000), rand_seq(rng, 5400), rand_seq(rng, 5461), rand_seq(rng, 5463)], pen4)


def test_unique_kmers():
    rng = np.random.default_rng(6)
    for k in (3, 8, 9, 10, 12):
        for ml in (0, 1):
            for _ in range(20):
                s = rand_seq(rng, int(rng.integers(0, 400)), b"ACGTACGTACGTacgtNnRU")
                a = _libs.oracle_unique_kmers(s, k, ml)
                assert _libs.kmers_digest(a) == _libs.ref_unique_kmers_digest(s, k, ml)


def _family_db(rng, n_roots=12, per=8, L=300):
    roots = synth.random_seqs(rng, n_roots, L)
    seqs = []
    for r in range(n_roots):
        for _ in range(per):
            seqs.append(synth.mutate(rng, roots[r], float(rng.uniform(0.0, 0.2))).tobytes())
    # some junk: short, ambiguous, duplicates
    seqs += [b"ACGT", b"N" * 50, seqs[0], seqs[1][:100], b"ACGTNNNNACGT" * 10]
    return synth.SeqSet(seqs), roots


def test_topscores_and_search_match_reference():
    rng = np.random.default_rng(7)
    db, roots = _family_db(rng)
    for (idv, ma, mr) in ((0.9, 1, 32), (0.5, 3, 16), (0.97, 2, 4), (0.8, 100, 100)):
        r = _libs.RefDb(db, id=idv, maxaccepts=ma, maxrejects=mr)
        o = _libs.OracleDb(db)
        opts = _libs.search_opts(len(db), id=idv, maxaccepts=ma, maxrejects=mr)
        assert opts.tophits == r.tophits
        qs = [synth.mutate(rng, roots[i % roots.shape[0]], 0.08).tobytes()[: int(rng.integers(60, 300))]
              for i in range(40)]
        qs += [b"ACGTACGTAC", synth.random_seqs(rng, 1, 200)[0].tobytes()]
        qset = synth.SeqSet(qs)
        ref_rows = r.search(qset, max_results=opts.tophits)
        for i, q in enumerate(qs):
            s1, c1 = r.topscores(q)
            s2, c2 = o.topscores(q, opts)
            assert np.array_equal(s1, s2) and np.array_equal(c1, c2)
            hits, _, _ = o.search(q, opts)
            got = [(h.target, h.id, h.matches, h.mismatches, h.nwgaps, h.nwalignmentlength,
                    h.accepted, h.strand) for h in hits]
            assert got == ref_rows[i], (i, got, ref_rows[i])
        o.close()
        r.close()


@pytest.mark.parametrize("k", [10, 11, 13, 14])
def test_large_wordlengths_match_reference(k):
    """k >= 10 is the reference's hash variant of unique_count (unique.cpp:243-334); from 13 on the oracle keeps its
    index as sorted (k-mer, target) pairs instead of 4^k list heads: candidate lists and whole searches still equal
    the reference's, soft-masked and IUPAC symbols included"""
    rng = np.random.default_rng(100 + k)
    db, roots = _family_db(rng)
    r = _libs.RefDb(db, k=k, id=0.9, maxaccepts=2, maxrejects=16)
    o = _libs.OracleDb(db, k=k)
    opts = _libs.search_opts(len(db), id=0.9, maxaccepts=2, maxrejects=16, k=k)
    assert opts.tophits == r.tophits
    qs = [synth.mutate(rng, roots[i % roots.shape[0]], 0.05).tobytes()[: int(rng.integers(60, 300))] for i in range(30)]
    qs += [b"ACGTACGTAC", synth.random_seqs(rng, 1, 200)[0].tobytes(), roots[0].tobytes()[:120] + b"NNRY" + roots[0].tobytes()[124:200]]
    ref_rows = r.search(synth.SeqSet(qs), max_results=opts.tophits)
    nonempty = 0
    for i, q in enumerate(qs):
        for m in (0, 1):
            assert _libs.kmers_digest(_libs.oracle_unique_kmers(q, k, m)) == _libs.ref_unique_kmers_digest(q, k, m), (k, i, m)
        s1, c1 = r.topscores(q)
        s2, c2 = o.topscores(q, opts)
        assert np.array_equal(s1, s2) and np.array_equal(c1, c2), (k, i)
        nonempty += len(s1) > 0
        hits, _, _ = o.search(q, opts)
        got = [(h.target, h.id, h.matches, h.mismatches, h.nwgaps, h.nwalignmentlength, h.accepted, h.strand) for h in hits]
        assert got == ref_rows[i], (k, i)
    assert nonempty >= 25
    o.close(); r.close()
