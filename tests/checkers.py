"""ctypes loaders for the CHECKERS (oracle/liboracle.so and oracle/_ref/libvsref.so).

Test infrastructure only — the product never imports this module.
"""
from __future__ import annotations

import ctypes as C
import gzip
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
STOCK = os.path.join(ORACLE_DIR, "_ref", "vsearch")

DEFAULT_PEN = np.array([2, -4, 1, 1, 18, 18, 1, 1, 1, 1, 2, 2, 1, 1], dtype=np.int64)


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class Scoring(C.Structure):
    _fields_ = [("v", C.c_int64 * 14), ("n_mismatch", C.c_int)]


def make_scoring(pen=None, n_mismatch=0):
    s = Scoring()
    pen = DEFAULT_PEN if pen is None else pen
    for i in range(14):
        s.v[i] = int(pen[i])
    s.n_mismatch = int(n_mismatch)
    return s


_oracle = None


def oracle():
    global _oracle
    if _oracle is None:
        path = os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)
        _oracle = C.CDLL(path)
        _oracle.oracle_unique_kmers.restype = C.c_uint
        _oracle.oracle_index_build.restype = C.c_void_p
        _oracle.oracle_map_4bit.restype = C.c_ubyte
    return _oracle


_ref = None


def ref():
    """The unmodified reference behind a C ABI, or None when oracle/_ref was not built."""
    global _ref
    if _ref is None:
        path = os.path.join(ORACLE_DIR, "_ref", "libvsref.so")
        if not os.path.exists(path):
            return None
        _ref = C.CDLL(path)
        _ref.vsref_db_create.restype = C.c_void_p
    return _ref


# ---- recorded reference results ------------------------------------------------------------------------------------
# Every call of the reference below goes through reference_result().  With oracle/_ref built the reference computes the
# answer; with VSG_RECORD_REFERENCE=<dir> set as well, the answers are also written to <dir>/<test module>.json.gz at
# exit.  Without oracle/_ref the answers come from tests/golden/reference/<test module>.json.gz, stored from such a run,
# so a plain checkout still compares against the reference.  Keys hash the call's complete inputs: a test whose inputs
# change finds no stored answer and fails until the store is re-recorded.
GOLDEN_REF_DIR = os.path.join(ROOT, "tests", "golden", "reference")
_stores = {}
_recorded = {}


def _test_module():
    cur = os.environ.get("PYTEST_CURRENT_TEST", "")
    return os.path.basename(cur.split("::")[0])[:-3] if cur else "misc"


def _digest(h, x):
    if isinstance(x, (bytes, bytearray)):
        h.update(b"b%d:" % len(x)); h.update(bytes(x))
    elif isinstance(x, np.ndarray):
        h.update(f"a{x.dtype.str}{x.shape}:".encode()); h.update(np.ascontiguousarray(x).tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(b"l%d:" % len(x))
        for y in x:
            _digest(h, y)
    elif hasattr(x, "cat") and hasattr(x, "offs") and hasattr(x, "lens"):     # synth.SeqSet
        for y in (x.cat, x.offs, x.lens):
            _digest(h, y)
    else:
        h.update(repr(x).encode())


def have_reference():
    """the reference itself (oracle/_ref) or its stored answers (tests/golden/reference)"""
    return ref() is not None or os.path.isdir(GOLDEN_REF_DIR)


def have_reference_cli():
    return os.path.exists(STOCK) or os.path.isdir(GOLDEN_REF_DIR)


def digest(data) -> str:
    import hashlib
    return hashlib.sha256(data.encode() if isinstance(data, str) else bytes(data)).hexdigest()


def reference_cli(args, summarize, threads=None, timeout=None):
    """Runs the reference CLI (oracle/_ref/vsearch) with args and returns summarize(), a JSON-serialisable account of the
    files it wrote (large outputs as a digest and a size), or the stored account for the same arguments and input files.
    Input files are keyed by content, output paths by name; `threads` is passed on but left out of the key, for runs
    whose output does not depend on it."""
    key = [("file", digest(open(a, "rb").read())) if os.path.isfile(a) else
           os.path.basename(a) if os.sep in a else a for a in args]

    def compute():
        p = subprocess.run([STOCK] + list(args) + (["--threads", str(threads)] if threads else []),
                           capture_output=True, text=True, timeout=timeout)
        assert p.returncode == 0, p.stderr[-2000:]
        return summarize()
    return reference_result("cli", key, compute, live=os.path.exists(STOCK))


def reference_result(name, inputs, compute, live=None):
    """compute() (a JSON-serialisable value) from the reference, or its stored answer for the same inputs"""
    import hashlib
    h = hashlib.sha256(name.encode())
    _digest(h, inputs)
    key = f"{name}:{h.hexdigest()[:32]}"
    mod = _test_module()
    if live is None:
        live = ref() is not None
    if live:
        val = compute()
        if os.environ.get("VSG_RECORD_REFERENCE"):
            if not _recorded:
                import atexit
                atexit.register(_write_recorded, os.environ["VSG_RECORD_REFERENCE"])
            _recorded.setdefault(mod, {})[key] = json.loads(json.dumps(val))
        return val
    if mod not in _stores:
        path = os.path.join(GOLDEN_REF_DIR, mod + ".json.gz")
        _stores[mod] = json.loads(gzip.open(path, "rt").read()) if os.path.exists(path) else {}
    if key not in _stores[mod]:
        raise AssertionError(f"no stored reference answer for {key} in tests/golden/reference/{mod}.json.gz: the inputs "
                             "changed; build oracle/_ref and re-record with VSG_RECORD_REFERENCE")
    return _stores[mod][key]


def _write_recorded(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    for mod, vals in _recorded.items():
        path = os.path.join(out_dir, mod + ".json.gz")
        old = json.loads(gzip.open(path, "rt").read()) if os.path.exists(path) else {}
        old.update(vals)
        with open(path, "wb") as f, gzip.GzipFile(fileobj=f, mode="wb", mtime=0) as g:
            g.write(json.dumps(old, sort_keys=True, separators=(",", ":")).encode())


def rows_digest(rows):
    """hit tables too large to store: per query the list of its rows (target, id, matches, mismatches, gaps, alignment
    length, accepted, strand) as the number of queries and rows and a digest of every row"""
    text = "".join(f"{q}\t" + "\t".join(repr(v) for v in row) + "\n" for q, rs in enumerate(rows) for row in rs)
    return {"queries": len(rows), "rows": sum(len(rs) for rs in rows), "sha256": digest(text)}


def oracle_nw16(q: bytes, d: bytes, pen=None, n_mismatch=0):
    lib = oracle()
    sc = make_scoring(pen, n_mismatch)
    score = C.c_int16(); al = C.c_uint16(); ma = C.c_uint16(); mi = C.c_uint16(); ga = C.c_uint16()
    cap = len(q) + len(d) + 64
    buf = C.create_string_buffer(cap)
    rc = lib.oracle_nw16(C.byref(sc), q, C.c_int64(len(q)), d, C.c_int64(len(d)),
                         C.byref(score), C.byref(al), C.byref(ma), C.byref(mi), C.byref(ga),
                         buf, C.c_size_t(cap))
    assert rc == 0
    return score.value, al.value, ma.value, mi.value, ga.value, buf.value.decode()


def ref_search16(q: bytes, targets, pen=None, n_mismatch=0):
    pen = np.ascontiguousarray(DEFAULT_PEN if pen is None else pen, dtype=np.int64)
    rows = reference_result("search16", (q, list(targets), pen, n_mismatch),
                            lambda: _ref_search16(q, targets, pen, n_mismatch))
    return [tuple(r) for r in rows]


def _ref_search16(q, targets, pen, n_mismatch):
    lib = ref()
    n = len(targets)
    lens = np.array([len(t) for t in targets], dtype=np.int32)
    offs = np.zeros(n, dtype=np.int64)
    if n:
        np.cumsum(lens[:-1], out=offs[1:])
    cat = b"".join(targets) + b"\0"
    scores = np.zeros(n, dtype=np.int16)
    al = np.zeros(n, dtype=np.uint16); ma = np.zeros(n, dtype=np.uint16)
    mi = np.zeros(n, dtype=np.uint16); ga = np.zeros(n, dtype=np.uint16)
    stride = len(q) + (int(lens.max()) if n else 0) + 64
    cig = C.create_string_buffer(stride * max(n, 1))
    rc = lib.vsref_search16(_p(pen, C.c_int64), C.c_int(n_mismatch), q, C.c_int(len(q)),
                            C.c_int(n), cat, _p(offs, C.c_int64), _p(lens, C.c_int),
                            _p(scores, C.c_int16), _p(al, C.c_uint16), _p(ma, C.c_uint16),
                            _p(mi, C.c_uint16), _p(ga, C.c_uint16), cig, C.c_int64(stride))
    assert rc == 0
    out = []
    raw = cig.raw
    for i in range(n):
        c = raw[i * stride:(i + 1) * stride].split(b"\0", 1)[0].decode()
        out.append((int(scores[i]), int(al[i]), int(ma[i]), int(mi[i]), int(ga[i]), c))
    return out


def oracle_unique_kmers(seq: bytes, k=8, mask_lower=0):
    out = np.zeros(max(len(seq), 1), dtype=np.uint32)
    n = oracle().oracle_unique_kmers(C.c_int(k), seq, C.c_int64(len(seq)), C.c_int(mask_lower),
                                     _p(out, C.c_uint32))
    return out[:n].copy()


def kmers_digest(kmers):
    """a list of k-mers (uint32 codes, in order) as its length and a digest: stored k-mer lists barely compress"""
    kmers = np.ascontiguousarray(kmers, dtype=np.uint32)
    return {"n": int(kmers.shape[0]), "sha256": digest(kmers.tobytes())}


def ref_unique_kmers_digest(seq: bytes, k=8, mask_lower=0):
    """kmers_digest() of the reference's unique_count() for seq"""
    def compute():
        out = np.zeros(max(len(seq), 1), dtype=np.uint32)
        n = ref().vsref_unique_count(C.c_int(k), seq, C.c_int(len(seq)), C.c_int(mask_lower),
                                     _p(out, C.c_uint32), C.c_int(out.shape[0]))
        return kmers_digest(out[:n])
    return reference_result("unique_count", (seq, k, mask_lower), compute)


def ref_dust(seq: bytes) -> bytes:
    """the reference's dust() (core/mask.cpp): masked symbols come back lower case"""
    def compute():
        b = C.create_string_buffer(seq)
        ref().vsref_dust(b, C.c_int(len(seq)))
        return b.value.decode("latin-1")
    return reference_result("dust", seq, compute).encode("latin-1")


class OracleHit(C.Structure):
    _fields_ = [("target", C.c_int), ("strand", C.c_int), ("count", C.c_uint),
                ("accepted", C.c_int), ("rejected", C.c_int), ("aligned", C.c_int), ("weak", C.c_int),
                ("nwscore", C.c_int), ("nwdiff", C.c_int), ("nwgaps", C.c_int), ("nwindels", C.c_int),
                ("nwalignmentlength", C.c_int), ("matches", C.c_int), ("mismatches", C.c_int),
                ("internal_alignmentlength", C.c_int), ("internal_gaps", C.c_int),
                ("internal_indels", C.c_int),
                ("trim_q_left", C.c_int), ("trim_q_right", C.c_int), ("trim_t_left", C.c_int),
                ("trim_t_right", C.c_int),
                ("id", C.c_double), ("id0", C.c_double), ("id1", C.c_double), ("id2", C.c_double),
                ("id3", C.c_double), ("id4", C.c_double), ("shortest", C.c_int), ("longest", C.c_int)]


class SearchOpts(C.Structure):
    _fields_ = [("id", C.c_double), ("weak_id", C.c_double), ("maxaccepts", C.c_int),
                ("maxrejects", C.c_int), ("minwordmatches", C.c_int), ("tophits", C.c_int),
                ("iddef", C.c_int), ("mask_lower", C.c_int)]


MINWORDMATCHES = [-1, -1, -1, 18, 17, 16, 15, 14, 12, 11, 10, 9, 8, 7, 5, 3]


def search_opts(n_db, id=0.9, maxaccepts=1, maxrejects=32, k=8, minwordmatches=-1, iddef=2,
                weak_id=10.0, mask_lower=0):
    """Effective options after the reference's fix-ups (vsearch.cc:186-276,
    usearch_global.cpp:598-614)."""
    o = SearchOpts()
    o.id = id
    o.weak_id = min(weak_id, id)
    o.maxaccepts = min(maxaccepts, n_db)
    o.maxrejects = min(maxrejects, n_db)
    o.minwordmatches = MINWORDMATCHES[k] if minwordmatches < 0 else minwordmatches
    o.tophits = min(o.maxaccepts + o.maxrejects + 8, n_db)
    o.iddef = iddef
    o.mask_lower = mask_lower
    return o


class OracleDb:
    def __init__(self, ss, k=8, mask_lower=0):
        self.ss = ss
        self.k = k
        self.h = oracle().oracle_index_build(C.c_int(k), C.c_int(len(ss)), _p(ss.cat, C.c_char),
                                             _p(ss.offs, C.c_int64), _p(ss.lens, C.c_int),
                                             C.c_int(mask_lower))

    def close(self):
        if self.h:
            oracle().oracle_index_free(C.c_void_p(self.h))
            self.h = None

    def topscores(self, q: bytes, opts):
        kmers = oracle_unique_kmers(q, self.k, opts.mask_lower)
        seqno = np.zeros(opts.tophits + 1, dtype=np.uint32)
        count = np.zeros(opts.tophits + 1, dtype=np.uint32)
        n = oracle().oracle_topscores(C.c_void_p(self.h), _p(self.ss.lens, C.c_int),
                                      _p(kmers, C.c_uint32), C.c_uint(kmers.shape[0]),
                                      C.c_int(opts.minwordmatches), C.c_int(opts.tophits),
                                      _p(seqno, C.c_uint32), _p(count, C.c_uint32))
        return seqno[:n].copy(), count[:n].copy()

    def search(self, q: bytes, opts, pen=None, strand=0):
        sc = make_scoring(pen)
        hits = (OracleHit * (opts.tophits + 1))()
        pairs = C.c_int64(); cells = C.c_int64()
        n = oracle().oracle_search_onequery(C.c_void_p(self.h), C.byref(sc), C.byref(opts),
                                            C.c_int(len(self.ss)), _p(self.ss.cat, C.c_char),
                                            _p(self.ss.offs, C.c_int64), _p(self.ss.lens, C.c_int),
                                            q, C.c_int(len(q)), C.c_int(strand),
                                            hits, C.c_int(opts.tophits + 1),
                                            C.byref(pairs), C.byref(cells))
        return [hits[i] for i in range(n)], pairs.value, cells.value


class RefDb:
    """Reference Database+Dbindex+session (one at a time per process); its answers go through reference_result(), so
    without oracle/_ref they are the stored ones (self.h is then None)."""

    def __init__(self, ss, k=8, id=0.9, maxaccepts=1, maxrejects=32, minwordmatches=-1,
                 dust=0, strand_both=0, iddef=2):
        self.ss = ss
        self.h = None
        self.key = [ss, k, id, maxaccepts, maxrejects, minwordmatches, dust, strand_both, iddef]
        if ref() is not None:
            self.h = ref().vsref_db_create(C.c_int(len(ss)), _p(ss.cat, C.c_char),
                                           _p(ss.offs, C.c_int64), _p(ss.lens, C.c_int),
                                           C.c_int(k), C.c_double(id), C.c_int(maxaccepts),
                                           C.c_int(maxrejects), C.c_int(minwordmatches), C.c_int(dust),
                                           C.c_int(strand_both), C.c_int(iddef))
        self.tophits = reference_result("db_tophits", self.key, lambda: int(ref().vsref_db_tophits(C.c_void_p(self.h))))

    def close(self):
        if self.h:
            ref().vsref_db_free(C.c_void_p(self.h))
            self.h = None

    def set_filters(self, values):
        """vsref_db_set_filters: the 14 optional filters in the shim's order (minqt ... rightjust)"""
        values = [float(v) for v in values]
        self.key = self.key + [values]
        if self.h:
            ref().vsref_db_set_filters(C.c_void_p(self.h), (C.c_double * 14)(*values))

    def lma(self, q: bytes, t: bytes):
        """the reference's LinearMemoryAligner on one pair: (five counters, CIGAR)"""
        def compute():
            out = (C.c_longlong * 5)()
            buf = C.create_string_buffer(len(q) + len(t) + 8)
            assert ref().vsref_lma(C.c_void_p(self.h), q, C.c_int(len(q)), t, C.c_int(len(t)), out, buf, C.c_int(len(buf))) == 0
            return [list(out), buf.value.decode()]
        return reference_result("lma", (self.key, q, t), compute)

    def topscores(self, q: bytes):
        def compute():
            seqno = np.zeros(self.tophits + 1, dtype=np.uint32)
            count = np.zeros(self.tophits + 1, dtype=np.uint32)
            length = np.zeros(self.tophits + 1, dtype=np.uint32)
            n = ref().vsref_db_topscores(C.c_void_p(self.h), q, C.c_int(len(q)),
                                         _p(seqno, C.c_uint32), _p(count, C.c_uint32),
                                         _p(length, C.c_uint32))
            return [seqno[:n].tolist(), count[:n].tolist()]
        s, c = reference_result("db_topscores", (self.key, q), compute)
        return np.array(s, dtype=np.uint32), np.array(c, dtype=np.uint32)

    def search_rows_digest(self, qs, max_results=8, threads=None):
        """rows_digest() of the reference's own multi-threaded search_batch, every record kept"""
        nq = len(qs)

        def compute():
            nthreads = threads or (os.cpu_count() or 1)
            counts = np.zeros(nq, dtype=np.int32)
            m = nq * max_results
            a = {k: np.zeros(m, dtype=np.int32) for k in ("target", "matches", "mismatches", "gaps", "alnlen", "accepted", "strand")}
            a["id"] = np.zeros(m, dtype=np.float64)
            ref().vsref_db_search_batch_rows(C.c_void_p(self.h), C.c_int(nq), _p(qs.cat, C.c_char), _p(qs.offs, C.c_int64),
                                             _p(qs.lens, C.c_int), C.c_int(nthreads), C.c_int(max_results), _p(counts, C.c_int),
                                             _p(a["target"], C.c_int), _p(a["id"], C.c_double), _p(a["matches"], C.c_int),
                                             _p(a["mismatches"], C.c_int), _p(a["gaps"], C.c_int), _p(a["alnlen"], C.c_int),
                                             _p(a["accepted"], C.c_int), _p(a["strand"], C.c_int))
            fields = ("target", "id", "matches", "mismatches", "gaps", "alnlen", "accepted", "strand")
            return rows_digest([[tuple(a[k][q * max_results + j].item() for k in fields) for j in range(counts[q])]
                                for q in range(nq)])

        # the result does not depend on the thread count, so the key leaves it out
        return reference_result("db_search_rows", (self.key, qs, max_results), compute)

    def search(self, qs, max_results=8):
        nq = len(qs)

        def compute():
            counts = np.zeros(nq, dtype=np.int32)
            m = nq * max_results
            target = np.zeros(m, dtype=np.int32); idv = np.zeros(m, dtype=np.float64)
            ma = np.zeros(m, dtype=np.int32); mi = np.zeros(m, dtype=np.int32)
            ga = np.zeros(m, dtype=np.int32); al = np.zeros(m, dtype=np.int32)
            acc = np.zeros(m, dtype=np.int32); st = np.zeros(m, dtype=np.int32)
            ref().vsref_db_search(C.c_void_p(self.h), C.c_int(nq), _p(qs.cat, C.c_char),
                                  _p(qs.offs, C.c_int64), _p(qs.lens, C.c_int), C.c_int(max_results),
                                  _p(counts, C.c_int), _p(target, C.c_int), _p(idv, C.c_double),
                                  _p(ma, C.c_int), _p(mi, C.c_int), _p(ga, C.c_int), _p(al, C.c_int),
                                  _p(acc, C.c_int), _p(st, C.c_int))
            out = []
            for q in range(nq):
                rows = []
                for j in range(counts[q]):
                    o = q * max_results + j
                    rows.append((int(target[o]), float(idv[o]), int(ma[o]), int(mi[o]), int(ga[o]),
                                 int(al[o]), int(acc[o]), int(st[o])))
                out.append(rows)
            return out
        return [[tuple(r) for r in rows] for rows in reference_result("db_search", (self.key, qs, max_results), compute)]
