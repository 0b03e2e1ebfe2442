"""The streaming --usearch_global driver (vsg_usearch_stream: FASTA in, --blast6out out; SURVEY.md §8 f1) against the
UNMODIFIED reference CLI on the same files: the output files must be byte-identical (the reference with --threads 1
writes in input order, as the driver does)."""

import numpy as np
import pytest

import checkers
from vsearch_b200 import lib as vlib
from vsearch_b200 import synth

pytestmark = pytest.mark.gpu

needs_stock = pytest.mark.skipif(not checkers.have_reference_cli(), reason="neither oracle/_ref nor tests/golden/reference")


def _file_digest(path):
    data = open(path, "rb").read()
    return {"size": len(data), "sha256": checkers.digest(data)}


def _files(tmp_path, n_db=4000, n_q=9000):
    dbs, qss, _ = synth.config2_search(n_db=n_db, db_len=1200, n_q=n_q, q_len=220, div=0.06, seed=21)
    rng = np.random.default_rng(9)
    # ragged queries, a few unrelated ones (no hit), descriptions after a blank, long lines folded
    qs = []
    for i in range(len(qss)):
        s = qss.seq(i)[: int(rng.integers(80, 220))]
        if i % 53 == 0:
            s = synth.random_seqs(rng, 1, 150)[0].tobytes()
        qs.append(s)
    dbf = str(tmp_path / "db.fasta"); qf = str(tmp_path / "q.fasta")
    synth.write_fasta(dbf, dbs, "d")
    with open(qf, "w") as f:
        for i, s in enumerate(qs):
            f.write(f">q{i} sample={i % 7}\tx\n")
            t = s.decode()
            for a in range(0, len(t), 80):
                f.write(t[a:a + 80] + ("\r\n" if i % 5 == 0 else "\n"))
    labels = [f"d{i}" for i in range(len(dbs))]
    return dbs, dbf, qf, labels


@needs_stock
@pytest.mark.parametrize("mode", ["plain", "both_strands_no_hits", "dust_maxhits"])
def test_stream_blast6out_equals_the_reference_cli(tmp_path, mode):
    dbs, dbf, qf, labels = _files(tmp_path)
    ref_out = str(tmp_path / "ref.b6"); got_out = str(tmp_path / "got.b6")
    args = ["--usearch_global", qf, "--db", dbf, "--id", "0.9", "--blast6out", ref_out, "--threads", "1", "--quiet"]
    o = vlib.default_search_opts(); o.id = 0.9
    kw = {}
    dust = 0
    if mode == "plain":
        args += ["--qmask", "none", "--dbmask", "none"]
    elif mode == "both_strands_no_hits":
        args += ["--qmask", "none", "--dbmask", "none", "--strand", "both", "--output_no_hits", "--maxaccepts", "3", "--maxrejects", "16"]
        o.strand_both = 1; o.maxaccepts = 3; o.maxrejects = 16
        kw = dict(output_no_hits=1)
    else:
        args += ["--maxaccepts", "4", "--maxhits", "2"]      # default masking: --qmask dust --dbmask dust
        o.maxaccepts = 4; o.mask_lower = 1; o.qmask_dust = 1
        dust = 1
        kw = dict(maxhits=2, qmask_dust=1)
    want = checkers.reference_cli(args, lambda: _file_digest(ref_out), timeout=900)
    g = vlib.Group([0], dbs, wordlength=8, mask_lower=dust, dust_db=dust)
    st = g.stream(labels, qf, o, got_out, batch_queries=2048, **kw)
    g.close()
    assert st["queries"] == 9000 and st["batches"] == 5
    assert want["size"] > 100000
    assert _file_digest(got_out) == want
