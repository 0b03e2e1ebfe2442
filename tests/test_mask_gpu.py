"""Device DUST masking (vsg_seqset_dust) against the reference's dust() (core/mask.cpp) and, end to
end, the default-masking search (--qmask dust --dbmask dust) against the compiled reference."""
import numpy as np
import pytest

import checkers
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not checkers.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")]


def low_complexity(rng, n):
    """sequences with homopolymers, short tandem repeats and ordinary stretches mixed"""
    parts = []
    while sum(map(len, parts)) < n:
        kind = int(rng.integers(0, 4))
        if kind == 0:
            parts.append(bytes([b"ACGT"[int(rng.integers(0, 4))]]) * int(rng.integers(5, 80)))
        elif kind == 1:
            unit = bytes(rng.choice(list(b"ACGT"), size=int(rng.integers(2, 5))).tolist())
            parts.append(unit * int(rng.integers(3, 30)))
        else:
            parts.append(bytes(rng.choice(list(b"ACGTacgtNn"), size=int(rng.integers(10, 120))).tolist()))
    return b"".join(parts)[:n]


def test_dust_matches_reference():
    rng = np.random.default_rng(51)
    seqs = [low_complexity(rng, int(rng.integers(1, 400))) for _ in range(300)]
    seqs += [b"A" * 7, b"A" * 8, b"A" * 9, b"ACGT" * 16, b"A" * 64, b"A" * 65, b"AC" * 100, b"", b"ACG",
             synth.random_seqs(rng, 1, 300)[0].tobytes(), b"acgt" * 40, b"N" * 100]
    ss = synth.SeqSet(seqs)
    ctx = vlib.Context(0)
    h = ctx.seqset(ss)
    h.dust()
    sym = h.symbols(int(ss.lens.sum()))
    masked_total = 0
    for i, s in enumerate(seqs):
        want = checkers.ref_dust(s)
        o = int(ss.offs[i])
        got_lower = (sym[o:o + len(s)] & 16) != 0
        want_lower = np.array([97 <= c <= 122 for c in want], dtype=bool)
        assert np.array_equal(got_lower, want_lower), (i, s, want)
        masked_total += int(want_lower.sum())
    assert masked_total > 1000
    h.close(); ctx.close()


def test_default_masking_search_vs_reference():
    rng = np.random.default_rng(52)
    roots = [low_complexity(rng, 350) for _ in range(10)]
    dbl = []
    for r in roots:
        ra = np.frombuffer(r.upper(), dtype=np.uint8)
        for _ in range(8):
            dbl.append(synth.mutate(rng, ra, float(rng.uniform(0, 0.1))).tobytes())
    dbs = synth.SeqSet(dbl)
    queries = [synth.mutate(rng, np.frombuffer(roots[i % 10].upper(), dtype=np.uint8), 0.05).tobytes()[:300] for i in range(30)]
    qss = synth.SeqSet(queries)
    r = checkers.RefDb(dbs, id=0.8, maxaccepts=2, maxrejects=8, dust=1)   # the reference dusts db and queries itself
    want = r.search(qss, max_results=r.tophits)
    th = r.tophits
    r.close()
    ctx = vlib.Context(0)
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    db.dust(); qs.dust()
    ix = ctx.index(db, 8, 1)
    o = vlib.default_search_opts(); o.id = 0.8; o.maxaccepts = 2; o.maxrejects = 8; o.mask_lower = 1
    res, counts, _ = ctx.search(ix, db, qs, 0, len(queries), o, th)
    nrows = 0
    for i in range(len(queries)):
        got = [[x.target, x.id, x.matches, x.mismatches, x.gaps, x.alignment_length, x.accepted, x.strand]
               for x in (res[i * th + j] for j in range(int(counts[i])))]
        assert got == [list(t) for t in want[i]], i
        nrows += len(got)
    assert nrows > 20
    ix.close(); db.close(); qs.close(); ctx.close()
