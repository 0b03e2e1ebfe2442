"""UDB reader (vsg_udb_open and its accessors; host code, no GPU): files written by the UNMODIFIED reference CLI
(`vsearch --makeudb_usearch`, oracle/_ref/vsearch) are parsed and compared with the FASTA they were made from, with the
reference's own --udb2fasta, and — the stored word index — with the oracle's index of the same sequences."""
import os
import subprocess

import numpy as np
import pytest

import checkers
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STOCK = os.path.join(ROOT, "oracle", "_ref", "vsearch")
needs_stock = pytest.mark.skipif(not os.path.exists(STOCK), reason="oracle/_ref/vsearch not built")
# the small files below are stored under tests/golden/reference as the reference wrote them (checkers.reference_cli)
needs_stock_or_stored = pytest.mark.skipif(not checkers.have_reference_cli(), reason="neither oracle/_ref nor tests/golden/reference")


def make_db(tmp_path, n=300, seed=5):
    """random sequences of ragged length; some with a low-complexity stretch (DUST masks it), some with lower-case
    runs in the input (soft masking), some with IUPAC codes; headers with descriptions"""
    rng = np.random.default_rng(seed)
    seqs = []
    for i in range(n):
        s = bytearray(synth.random_seqs(rng, 1, int(rng.integers(60, 900)))[0].tobytes())
        if i % 7 == 0:
            a = int(rng.integers(0, max(1, len(s) - 80)))
            s[a:a + 60] = b"ACACACACACACACACACACACACACACACACACACACACACACACACACACACACACAC"[: len(s[a:a + 60])]
        if i % 11 == 0:
            a = int(rng.integers(0, max(1, len(s) - 40)))
            s[a:a + 30] = bytes(s[a:a + 30]).lower()
        if i % 13 == 0:
            s[int(rng.integers(0, len(s)))] = ord("N")
            s[int(rng.integers(0, len(s)))] = ord("R")
        seqs.append(bytes(s))
    path = str(tmp_path / "db.fasta")
    with open(path, "w") as f:
        for i, s in enumerate(seqs):
            f.write(f">seq{i};size={i % 9 + 1} some description {i}\n")
            t = s.decode()
            for a in range(0, len(t), 70):
                f.write(t[a:a + 70] + "\n")
    return path, seqs


def makeudb(fasta, out, *extra):
    import base64
    import gzip
    data = checkers.reference_cli(["--makeudb_usearch", fasta, "--output", out, "--quiet", *extra],
                                  lambda: base64.b64encode(gzip.compress(open(out, "rb").read(), 9, mtime=0)).decode(), timeout=600)
    if not os.path.exists(STOCK):
        open(out, "wb").write(gzip.decompress(base64.b64decode(data)))


@needs_stock
@pytest.mark.parametrize("mode", [("dust", 8), ("none", 8), ("soft", 6), ("dust", 11)])
def test_udb_file_vs_fasta_and_oracle_index(tmp_path, mode):
    dbmask, k = mode
    fasta, seqs = make_db(tmp_path)
    udb = str(tmp_path / "db.udb")
    makeudb(fasta, udb, "--dbmask", dbmask, "--wordlength", str(k))
    assert vlib.udb_detect(udb) and not vlib.udb_detect(fasta)
    u = vlib.Udb(udb)
    assert u.info.wordlength == k and u.n == len(seqs)
    cat, off, ln = u.sequences()
    assert int(u.info.nucleotides) == sum(len(s) for s in seqs) == int(ln.sum())
    assert u.info.shortest == min(len(s) for s in seqs) and u.info.longest == max(len(s) for s in seqs)
    got = [cat[off[i]: off[i] + ln[i]].tobytes() for i in range(u.n)]
    # same letters; the case is the masking the file was made with
    assert [g.upper() for g in got] == [s.upper() for s in seqs]
    if dbmask == "dust":
        assert any(g != g.upper() for g in got)  # DUST-masked regions are lower case
    else:
        # makeudb_usearch reads its input upper-cased (makeudb_usearch.cpp:120, db.read(..., upcase = 1)): the case of
        # the input, and with it --dbmask soft, leaves no trace in the file
        assert got == [s.upper() for s in seqs]
    # headers: truncated at the first blank by the reference's FASTA parser
    assert [u.header(i) for i in range(u.n)] == [f"seq{i};size={i % 9 + 1}" for i in range(u.n)]
    # the reference's own dump of the file agrees with what we parsed
    dump = str(tmp_path / "dump.fasta")
    r = subprocess.run([STOCK, "--udb2fasta", udb, "--output", dump, "--quiet", "--fasta_width", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = open(dump).read().split("\n")
    assert [l[1:] for l in lines[0::2] if l] == [u.header(i) for i in range(u.n)]
    assert [l.encode() for l in lines[1::2] if l] == got
    # the stored index == the oracle's index of the parsed sequences (masked symbols excluded unless --dbmask none)
    kc, ki = u.words()
    ss = synth.SeqSet(got)
    od = checkers.OracleDb(ss, k=k, mask_lower=0 if dbmask == "none" else 1)
    o = checkers.oracle()
    import ctypes as C
    n_k = 1 << (2 * k)
    start = np.zeros(n_k + 1, dtype=np.uint64)
    o.oracle_index_starts(C.c_void_p(od.h), start.ctypes.data_as(C.POINTER(C.c_uint64)))
    post = np.zeros(int(start[-1]) + 1, dtype=np.uint32)
    o.oracle_index_postings(C.c_void_p(od.h), post.ctypes.data_as(C.POINTER(C.c_uint32)))
    assert np.array_equal(np.diff(start).astype(np.uint32), kc)
    assert np.array_equal(post[: int(start[-1])], ki)
    od.close()
    u.close()


@needs_stock_or_stored
def test_invalid_udb_files_are_rejected(tmp_path):
    fasta, _ = make_db(tmp_path, n=40)
    udb = str(tmp_path / "db.udb")
    makeudb(fasta, udb)
    data = bytearray(open(udb, "rb").read())

    def rejected(mutated: bytes, pattern: str):
        p = str(tmp_path / "bad.udb")
        open(p, "wb").write(mutated)
        with pytest.raises(vlib.VsgError, match=pattern):
            vlib.Udb(p)

    rejected(bytes(data[:-1]), "Invalid UDB file|Incorrect UDB file size")          # truncated
    rejected(bytes(data) + b"\0", "Incorrect UDB file size")                         # trailing byte
    bad = bytearray(data); bad[16] = 2                                               # wordlength 2
    rejected(bytes(bad), "Invalid UDB file")
    bad = bytearray(data); bad[4 * 49] ^= 1                                          # closing signature of the header
    rejected(bytes(bad), "Invalid UDB file")
    bad = bytearray(data)
    first_index_word = 4 * 50 + 4 * (1 << 16) + 4
    bad[first_index_word: first_index_word + 4] = (1000).to_bytes(4, "little")      # sequence number >= seqcount
    rejected(bytes(bad), "Invalid UDB file")
    assert vlib.udb_detect(str(tmp_path / "bad.udb"))                               # the signature alone says UDB
    with pytest.raises(vlib.VsgError):
        vlib.Udb(str(tmp_path / "missing.udb"))


@needs_stock_or_stored
def test_c_example_builds_and_parses_a_udb_file(tmp_path):
    """examples/usearch_udb.c (plain C against include/vsg.h) compiles with gcc, links libvsg.so, reads a UDB file made by
    the reference and — in a container without a GPU — stops at the first device call with the library's error message
    instead of falling back to anything"""
    fasta, seqs = make_db(tmp_path, n=30)
    udb = str(tmp_path / "db.udb")
    makeudb(fasta, udb)
    exe = str(tmp_path / "usearch_udb")
    csrc = os.path.join(ROOT, "vsearch_b200", "csrc")
    r = subprocess.run(["gcc", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "usearch_udb.c"), "-L", csrc, "-lvsg", f"-Wl,-rpath,{csrc}", "-o", exe],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe, udb, fasta, str(tmp_path / "out.b6"), "0.9"], capture_output=True, text=True, timeout=300)
    assert f"{len(seqs)} sequences" in r.stderr and "word length 8" in r.stderr
    import torch
    if not torch.cuda.is_available():
        assert r.returncode == 1 and "vsg_group_create_udb" in r.stderr
    else:
        assert r.returncode == 0, r.stderr
