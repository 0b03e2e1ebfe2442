"""UDB databases on the device (vsg_udb_load / vsg_group_create_udb; SURVEY.md §8 f3) and --wordlength 11..15 (the
sparse index; §8 a10) against the UNMODIFIED reference."""
import os
import subprocess

import numpy as np
import pytest

import checkers
from test_udb_cpu import STOCK, make_db, makeudb, needs_stock
from test_search_gpu import gpu_opts, rows_of
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = vlib.Context(0)
    yield c
    c.close()


@needs_stock
@pytest.mark.parametrize("dbmask", ["dust", "none"])
def test_usearch_global_on_a_udb_file_equals_the_reference_cli(tmp_path, ctx, dbmask):
    """`vsearch --usearch_global q --db x.udb` (stored index, stored masking) vs the streaming driver on the database
    loaded from the same file; the masking convention of the stored index is detected from its word counts"""
    fasta, seqs = make_db(tmp_path, n=600, seed=8)
    udb = str(tmp_path / "db.udb")
    makeudb(fasta, udb, "--dbmask", dbmask)
    rng = np.random.default_rng(3)
    qf = str(tmp_path / "q.fasta")
    with open(qf, "w") as f:
        for i in range(1500):
            s = seqs[int(rng.integers(0, len(seqs)))].upper()
            a = int(rng.integers(0, max(1, len(s) - 120)))
            q = synth.mutate(rng, np.frombuffer(s[a:a + 200], dtype=np.uint8), 0.04).tobytes()
            f.write(f">q{i}\n{q.decode()}\n")
    ref_out = str(tmp_path / "ref.b6"); got_out = str(tmp_path / "got.b6")
    r = subprocess.run([STOCK, "--usearch_global", qf, "--db", udb, "--id", "0.9", "--blast6out", ref_out, "--threads", "1", "--quiet",
                        "--qmask", "none", "--maxaccepts", "2", "--maxrejects", "16"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    u = vlib.Udb(udb)
    db, ix, ml = ctx.udb_load(u)
    # DUST lower-cases what it masks, so the stored index of the "dust" file excludes lower case; a file made with
    # --dbmask none holds upper case only (makeudb_usearch upper-cases its input) and both conventions agree
    assert ml == 1
    ix.close(); db.close()
    if dbmask == "none":
        # lower-case a run of the stored sequences behind the index's back: the stored counts now only match an index
        # that lets lower-case symbols seed words (what --usearch_global --dbmask none builds from FASTA)
        data = bytearray(open(udb, "rb").read())
        tail = int(u.info.nucleotides)
        data[len(data) - tail + 100: len(data) - tail + 400] = bytes(data[len(data) - tail + 100: len(data) - tail + 400]).lower()
        udb2 = str(tmp_path / "db_lower.udb")
        open(udb2, "wb").write(bytes(data))
        u2 = vlib.Udb(udb2)
        db2, ix2, ml2 = ctx.udb_load(u2)
        assert ml2 == 0
        ix2.close(); db2.close(); u2.close()
    g = vlib.Group.from_udb([0], u)
    labels = [u.header(i) for i in range(u.n)]
    o = vlib.default_search_opts(); o.id = 0.9; o.maxaccepts = 2; o.maxrejects = 16
    st = g.stream(labels, qf, o, got_out, batch_queries=512)
    g.close(); u.close()
    want = open(ref_out, "rb").read(); got = open(got_out, "rb").read()
    assert st["queries"] == 1500 and len(want) > 20000
    assert got == want


def test_a_udb_whose_index_is_not_its_sequences_is_rejected(tmp_path, ctx):
    if not checkers.have_reference_cli():
        pytest.skip("neither oracle/_ref nor tests/golden/reference")
    fasta, _ = make_db(tmp_path, n=50)
    udb = str(tmp_path / "db.udb")
    makeudb(fasta, udb)
    data = bytearray(open(udb, "rb").read())
    # move one occurrence from one word to another: sizes stay consistent, the counts no longer match the sequences
    kc = np.frombuffer(bytes(data[200: 200 + 4 * 65536]), dtype=np.uint32).copy()
    a = int(np.flatnonzero(kc > 0)[0]); b = int(np.flatnonzero(kc > 0)[-1])
    kc[a] -= 1; kc[b] += 1
    data[200: 200 + 4 * 65536] = kc.tobytes()
    bad = str(tmp_path / "bad.udb")
    open(bad, "wb").write(bytes(data))
    u = vlib.Udb(bad)          # structurally valid
    with pytest.raises(vlib.VsgError, match="does not belong to its sequences"):
        ctx.udb_load(u)
    u.close()


@pytest.mark.skipif(not checkers.have_reference(), reason="neither oracle/_ref nor tests/golden/reference")
@pytest.mark.parametrize("k", [11, 12, 13])
def test_wordlength_above_10_vs_compiled_reference(ctx, k):
    """candidate lists (search_topscores) and whole searches with --wordlength 11..13: two shards' worth of targets
    would need 70 000 sequences, so the shard logic is covered by test_sparse_index_multi_shard_vs_oracle below"""
    dbs, qss, src = synth.config2_search(n_db=500, db_len=1200, n_q=100, q_len=250, div=0.04, seed=70 + k)
    r = checkers.RefDb(dbs, k=k, id=0.9, maxaccepts=2, maxrejects=16)
    want = r.search(qss, max_results=r.tophits)
    th = r.tophits
    tops = [r.topscores(qss.seq(i)) for i in range(len(qss))]
    r.close()
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    ix = ctx.index(db, k, 0)
    seqno, count, nc = ctx.rank(ix, qs, 0, len(qss), checkers.MINWORDMATCHES[k], th)
    for i in range(len(qss)):
        s_, c_ = tops[i]
        assert seqno[i, :nc[i]].tolist() == s_.tolist() and count[i, :nc[i]].tolist() == c_.tolist(), (k, i)
    o = gpu_opts(0.9, 2, 16); o.wordlength = k
    res, counts, _ = ctx.search(ix, db, qs, 0, len(qss), o, th)
    hit = 0
    for i in range(len(qss)):
        got = rows_of(res, counts, i, th)
        assert got == [list(t) for t in want[i]], (k, i)
        hit += bool(got) and got[0][0] == int(src[i])
    assert hit > 80
    ix.close(); db.close(); qs.close()


@pytest.mark.parametrize("k", [11, 15])
def test_sparse_index_multi_shard_masked_and_long_queries_vs_oracle(ctx, k):
    """three shards (70 000 short targets), soft-masked and IUPAC symbols, an empty and a too-short target, queries on
    the shared-memory path and on the HBM hash path (more than 2048 windows)"""
    rng = np.random.default_rng(100 + k)
    roots = synth.random_seqs(rng, 40, 300)
    seqs = []
    for i in range(70_000):
        r = roots[i % 40]
        a = int(rng.integers(0, 200))
        s = bytearray(synth.mutate(rng, r[a:a + 100], 0.03).tobytes())
        if i % 17 == 0:
            s[10:40] = bytes(s[10:40]).lower()
        if i % 29 == 0:
            s[50] = ord("N")
        seqs.append(bytes(s))
    seqs[5] = b""
    seqs[6] = b"ACGTACG"
    dbs = synth.SeqSet(seqs)
    queries = [roots[3].tobytes(), synth.mutate(rng, roots[7], 0.02).tobytes(),
               b"".join(roots[j].tobytes() for j in range(8)),              # 2400 nt: HBM de-duplication
               (roots[1].tobytes() + roots[2].tobytes().lower()) * 5,         # 3000 nt, repeats, half of it masked
               synth.random_seqs(rng, 1, 400)[0].tobytes(),                   # unrelated
               b"ACGTACGTAC"]                                                 # shorter than a word (k = 11, 15)
    qss = synth.SeqSet(queries)
    db = ctx.seqset(dbs); qs = ctx.seqset(qss)
    for mask_lower in (1, 0):
        ix = ctx.index(db, k, mask_lower)
        od = checkers.OracleDb(dbs, k=k, mask_lower=mask_lower)
        opts = checkers.search_opts(len(dbs), id=0.9, maxaccepts=4, maxrejects=32, k=k, mask_lower=mask_lower)
        seqno, count, nc = ctx.rank(ix, qs, 0, len(queries), opts.minwordmatches, opts.tophits, mask_lower)
        for i, q in enumerate(queries):
            s_, c_ = od.topscores(q, opts)
            assert nc[i] == len(s_), (k, mask_lower, i, nc[i], len(s_))
            assert seqno[i, :nc[i]].tolist() == s_.tolist() and count[i, :nc[i]].tolist() == c_.tolist(), (k, mask_lower, i)
        assert nc[0] > 0 and nc[2] > 0
        od.close(); ix.close()
    db.close(); qs.close()
