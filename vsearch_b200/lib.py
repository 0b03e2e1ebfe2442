"""ctypes loader for the product library ``vsearch_b200/csrc/libvsg.so`` (C ABI: include/vsg.h).

This is host-side plumbing for tests and bench.py only.  There is no CPU implementation behind it:
if the library or a CUDA device is missing every call fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("VSG_LIB") or os.path.join(ROOT, "vsearch_b200", "csrc", "libvsg.so")   # VSG_LIB: an experimental build (A/B runs)
HEADER = os.path.join(ROOT, "include", "vsg.h")

DEFAULT_PEN = (2, -4, 1, 1, 18, 18, 1, 1, 1, 1, 2, 2, 1, 1)
STAT_WORDS = 8

_lib = None


class VsgError(RuntimeError):
    pass


class Scoring(C.Structure):
    _fields_ = [("v", C.c_int64 * 14), ("n_mismatch", C.c_int32)]


class SearchOpts(C.Structure):
    _fields_ = [("id", C.c_double), ("weak_id", C.c_double), ("maxaccepts", C.c_int32),
                ("maxrejects", C.c_int32), ("wordlength", C.c_int32), ("minwordmatches", C.c_int32),
                ("iddef", C.c_int32), ("strand_both", C.c_int32), ("mask_lower", C.c_int32),
                ("lazy", C.c_int32),
                ("minqt", C.c_double), ("maxqt", C.c_double), ("minsl", C.c_double), ("maxsl", C.c_double),
                ("maxid", C.c_double), ("mid", C.c_double), ("query_cov", C.c_double), ("target_cov", C.c_double),
                ("maxsubs", C.c_int64), ("maxgaps", C.c_int64), ("mincols", C.c_int64), ("maxdiffs", C.c_int64),
                ("leftjust", C.c_int32), ("rightjust", C.c_int32),
                ("maxqsize", C.c_int64), ("mintsize", C.c_int64), ("minsizeratio", C.c_double),
                ("maxsizeratio", C.c_double), ("idprefix", C.c_int32), ("idsuffix", C.c_int32),
                ("self", C.c_int32), ("selfid", C.c_int32), ("qmask_dust", C.c_int32), ("unoise", C.c_int32),
                ("query_sizes", C.POINTER(C.c_int64)), ("target_sizes", C.POINTER(C.c_int64)),
                ("query_labels", C.POINTER(C.c_int64)), ("target_labels", C.POINTER(C.c_int64)),
                ("unoise_alpha", C.c_double), ("sizeorder", C.c_int32), ("reserved1", C.c_int32)]


class Profile(C.Structure):
    _fields_ = [("cells", C.c_int64), ("fast_pairs", C.c_int64), ("exact_pairs", C.c_int64),
                ("fwd_launches", C.c_int64), ("fwd_ms", C.c_float), ("traceback_ms", C.c_float),
                ("rank_ms", C.c_float), ("reserved", C.c_float), ("tb_skipped", C.c_int64)]


class SearchResult(C.Structure):
    _fields_ = [("target", C.c_int32), ("matches", C.c_int32), ("mismatches", C.c_int32),
                ("gaps", C.c_int32), ("alignment_length", C.c_int32), ("query_length", C.c_int32),
                ("target_length", C.c_int32), ("accepted", C.c_int32), ("strand", C.c_int32),
                ("nwscore", C.c_int32), ("id", C.c_double),
                ("internal_alignment_length", C.c_int32), ("internal_gaps", C.c_int32)]


class PairHit(C.Structure):
    _fields_ = [("query", C.c_int32), ("target", C.c_int32), ("matches", C.c_int32), ("mismatches", C.c_int32),
                ("gaps", C.c_int32), ("alignment_length", C.c_int32), ("nwscore", C.c_int32),
                ("internal_alignment_length", C.c_int32), ("id", C.c_double)]


def declared_symbols() -> List[str]:
    """Every function name include/vsg.h declares."""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vsg_[a-z0-9_]+)\s*\(", text)))


def load():
    """dlopen libvsg.so and check that it exports everything the header declares."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VsgError(f"{LIB_PATH} not built: run `python __graft_entry__.py` (nvcc, sm_100a). "
                       "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    if missing:
        raise VsgError(f"libvsg.so does not export: {missing}")
    lib.vsg_last_error.restype = C.c_char_p
    lib.vsg_version.restype = C.c_char_p
    lib.vsg_launch_count.restype = C.c_int64
    lib.vsg_ctx_stream.restype = C.c_void_p
    lib.vsg_seqset_count.restype = C.c_int64
    lib.vsg_group_ctx.restype = C.c_void_p
    lib.vsg_group_db.restype = C.c_void_p
    lib.vsg_group_index.restype = C.c_void_p
    lib.vsg_udb_header.restype = C.c_char_p
    _lib = lib
    return lib


def launch_count() -> int:
    return int(load().vsg_launch_count())


def _check(rc: int, what: str):
    if rc != 0:
        raise VsgError(f"{what} failed ({rc}): {load().vsg_last_error().decode()}")


def _ptr(a: Optional[np.ndarray], t):
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(t))


@dataclass
class AlignResult:
    score: np.ndarray
    aligned: np.ndarray
    matches: np.ndarray
    mismatches: np.ndarray
    gaps: np.ndarray
    trims: np.ndarray
    cigars: Optional[List[str]]
    cells: int = 0
    fwd_ms: float = 0.0
    tb_ms: float = 0.0
    fast_pairs: int = 0
    exact_pairs: int = 0


class SeqSetHandle:
    def __init__(self, ctx: "Context", h, n: int, lens: np.ndarray):
        self.ctx, self.h, self.n, self.lens = ctx, h, n, lens

    def close(self):
        if self.h:
            load().vsg_seqset_destroy(self.h)
            self.h = None

    def dust(self):
        """DUST soft-masking in place on the device (vsg_seqset_dust)"""
        _check(load().vsg_seqset_dust(self.ctx.h, self.h), "vsg_seqset_dust")

    def symbols(self, total: int) -> np.ndarray:
        out = np.zeros(total, dtype=np.uint8)
        _check(load().vsg_seqset_symbols(self.ctx.h, self.h, _ptr(out, C.c_uint8), C.c_int64(total)),
               "vsg_seqset_symbols")
        return out


class IndexHandle:
    def __init__(self, h):
        self.h = h

    def close(self):
        if self.h:
            load().vsg_index_destroy(self.h)
            self.h = None


class Context:
    """vsg_ctx: one CUDA stream + scratch; mirrors the reference's per-thread s16info_s."""

    def __init__(self, device: int = 0, pen=DEFAULT_PEN, n_mismatch: int = 0):
        lib = load()
        sc = Scoring()
        for i in range(14):
            sc.v[i] = int(pen[i])
        sc.n_mismatch = int(n_mismatch)
        self.h = C.c_void_p()
        _check(lib.vsg_ctx_create(C.c_int(device), C.byref(sc), C.byref(self.h)), "vsg_ctx_create")

    def close(self):
        if self.h:
            load().vsg_ctx_destroy(self.h)
            self.h = None

    def set_fallback(self, fn):
        """fn(query_index, strand, target_index) -> 9 or 10 ints (score, alnlen, matches, mismatches, gaps,
        trim_q_left, trim_t_left, trim_q_right, trim_t_right[, forbidden]); see vsg_ctx_set_fallback."""
        proto = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.POINTER(C.c_int64))

        def tramp(_user, q, strand, t, out):
            try:
                vals = fn(int(q), int(strand), int(t))
                for i in range(len(vals)):
                    out[i] = int(vals[i])
                return 0
            except Exception:
                return 1
        self._fallback_keep = proto(tramp)
        _check(load().vsg_ctx_set_fallback(self.h, self._fallback_keep, None), "vsg_ctx_set_fallback")

    def profile_reset(self):
        _check(load().vsg_profile_reset(self.h), "vsg_profile_reset")

    def profile(self) -> Profile:
        p = Profile()
        _check(load().vsg_profile_get(self.h, C.byref(p)), "vsg_profile_get")
        return p

    def int_peak(self) -> float:
        v = C.c_double()
        _check(load().vsg_measure_int_peak(self.h, C.byref(v)), "vsg_measure_int_peak")
        return v.value

    def stream_ptr(self) -> int:
        return int(load().vsg_ctx_stream(self.h))

    def sync(self):
        _check(load().vsg_ctx_sync(self.h), "vsg_ctx_sync")

    def seqset(self, ss) -> SeqSetHandle:
        """Upload a synth.SeqSet-like object (cat uint8, offs int64, lens int32) into HBM."""
        h = C.c_void_p()
        cat = np.ascontiguousarray(ss.cat, dtype=np.uint8)
        offs = np.ascontiguousarray(ss.offs, dtype=np.int64)
        lens = np.ascontiguousarray(ss.lens, dtype=np.int32)
        _check(load().vsg_seqset_create(self.h, _ptr(cat, C.c_char), _ptr(offs, C.c_int64),
                                        _ptr(lens, C.c_int32), C.c_int64(lens.shape[0]), C.c_int(1),
                                        C.byref(h)), "vsg_seqset_create")
        return SeqSetHandle(self, h, int(lens.shape[0]), lens)

    def seqset_from_device(self, d_cat: int, d_off: int, d_len: int, n: int) -> SeqSetHandle:
        """Adopt ASCII/offset/length arrays that already live in this device's HBM (raw pointers)."""
        h = C.c_void_p()
        _check(load().vsg_seqset_create(self.h, C.cast(C.c_void_p(d_cat), C.POINTER(C.c_char)),
                                        C.cast(C.c_void_p(d_off), C.POINTER(C.c_int64)),
                                        C.cast(C.c_void_p(d_len), C.POINTER(C.c_int32)),
                                        C.c_int64(n), C.c_int(0), C.byref(h)), "vsg_seqset_create")
        return SeqSetHandle(self, h, n, None)

    def revcomp(self, ss: SeqSetHandle, q0: int = 0, n: Optional[int] = None) -> SeqSetHandle:
        """vsg_seqset_revcomp: the reverse complements of sequences [q0, q0 + n) of ss as a new set (case kept)"""
        n = ss.n - q0 if n is None else n
        h = C.c_void_p()
        _check(load().vsg_seqset_revcomp(self.h, ss.h, C.c_int64(q0), C.c_int64(n), C.byref(h)), "vsg_seqset_revcomp")
        lens = None if ss.lens is None else np.ascontiguousarray(ss.lens[q0:q0 + n])
        return SeqSetHandle(self, h, n, lens)

    def align_pairs(self, qs: SeqSetHandle, ts: SeqSetHandle, qidx: np.ndarray, tidx: np.ndarray,
                    cigar: bool = False) -> AlignResult:
        lib = load()
        qidx = np.ascontiguousarray(qidx, dtype=np.uint32)
        tidx = np.ascontiguousarray(tidx, dtype=np.uint32)
        n = int(qidx.shape[0])
        score = np.zeros(n, dtype=np.int16)
        al = np.zeros(n, dtype=np.uint16); ma = np.zeros(n, dtype=np.uint16)
        mi = np.zeros(n, dtype=np.uint16); ga = np.zeros(n, dtype=np.uint16)
        trims = np.zeros((n, 4), dtype=np.int32)
        cbuf = coff = None
        cap = 0
        if cigar:
            cap = int((qs.lens[qidx].astype(np.int64) + ts.lens[tidx].astype(np.int64) + 2).sum()) + 16
            cbuf = np.zeros(cap, dtype=np.uint8)
            coff = np.zeros(n + 1, dtype=np.int64)
        self.profile_reset()
        _check(lib.vsg_align_pairs(self.h, qs.h, ts.h, C.c_int64(n), _ptr(qidx, C.c_uint32),
                                   _ptr(tidx, C.c_uint32), _ptr(score, C.c_int16), _ptr(al, C.c_uint16),
                                   _ptr(ma, C.c_uint16), _ptr(mi, C.c_uint16), _ptr(ga, C.c_uint16),
                                   _ptr(trims, C.c_int32), _ptr(cbuf, C.c_char), C.c_int64(cap),
                                   _ptr(coff, C.c_int64)), "vsg_align_pairs")
        cigs = None
        if cigar:
            raw = cbuf.tobytes()
            cigs = [raw[int(coff[i]):int(coff[i + 1]) - 1].decode() for i in range(n)]
        pr = self.profile()
        return AlignResult(score, al, ma, mi, ga, trims, cigs, pr.cells, pr.fwd_ms, pr.traceback_ms,
                           pr.fast_pairs, pr.exact_pairs)

    def index(self, db: SeqSetHandle, wordlength: int = 8, mask_lower: int = 0) -> IndexHandle:
        h = C.c_void_p()
        _check(load().vsg_index_create(self.h, db.h, C.c_int(wordlength), C.c_int(mask_lower),
                                       C.byref(h)), "vsg_index_create")
        return IndexHandle(h)

    def udb_load(self, udb: "Udb"):
        """vsg_udb_load: (SeqSetHandle, IndexHandle, mask_lower) of a parsed UDB file"""
        sh = C.c_void_p(); ih = C.c_void_p(); ml = C.c_int(-1)
        _check(load().vsg_udb_load(self.h, udb.h, C.byref(sh), C.byref(ih), C.byref(ml)), "vsg_udb_load")
        _, _, lens = udb.sequences()
        return SeqSetHandle(self, sh, udb.n, lens), IndexHandle(ih), int(ml.value)

    def rank(self, ix: IndexHandle, qs: SeqSetHandle, q0: int, nq: int, minwordmatches: int,
             tophits: int, mask_lower: int = 0):
        seqno = np.zeros((nq, tophits), dtype=np.uint32)
        count = np.zeros((nq, tophits), dtype=np.uint32)
        nc = np.zeros(nq, dtype=np.int32)
        _check(load().vsg_rank(self.h, ix.h, qs.h, C.c_int64(q0), C.c_int64(nq), C.c_int(minwordmatches),
                               C.c_int(tophits), C.c_int(mask_lower), _ptr(seqno, C.c_uint32),
                               _ptr(count, C.c_uint32), _ptr(nc, C.c_int32)), "vsg_rank")
        return seqno, count, nc

    def search(self, ix: IndexHandle, db: SeqSetHandle, qs: SeqSetHandle, q0: int, nq: int,
               opts: SearchOpts, max_results: int):
        res = (SearchResult * (nq * max_results))()
        counts = np.zeros(nq, dtype=np.int32)
        work = np.zeros(4, dtype=np.int64)
        _check(load().vsg_search_batch(self.h, ix.h, db.h, qs.h, C.c_int64(q0), C.c_int64(nq),
                                       C.byref(opts), res, C.c_int(max_results), _ptr(counts, C.c_int32),
                                       _ptr(work, C.c_int64)), "vsg_search_batch")
        return res, counts, work


def allpairs(ctx: "Context", ss: SeqSetHandle, row0: int, nrows: int, opts: SearchOpts, cap: int):
    """vsg_allpairs -> (numpy structured array of hits, work[2])"""
    dt = np.dtype([("query", np.int32), ("target", np.int32), ("matches", np.int32), ("mismatches", np.int32),
                   ("gaps", np.int32), ("alignment_length", np.int32), ("nwscore", np.int32),
                   ("internal_alignment_length", np.int32), ("id", np.float64)])
    assert dt.itemsize == C.sizeof(PairHit)
    hits = np.zeros(cap, dtype=dt)
    n = C.c_int64()
    work = np.zeros(2, dtype=np.int64)
    _check(load().vsg_allpairs(ctx.h, ss.h, C.c_int64(row0), C.c_int64(nrows), C.byref(opts),
                               hits.ctypes.data_as(C.POINTER(PairHit)), C.c_int64(cap), C.byref(n),
                               _ptr(work, C.c_int64)), "vsg_allpairs")
    return hits[: n.value], work


class ClusterResult(C.Structure):
    _fields_ = [("cluster", C.c_int32), ("centroid", C.c_int32), ("matches", C.c_int32), ("mismatches", C.c_int32),
                ("gaps", C.c_int32), ("alignment_length", C.c_int32), ("nwscore", C.c_int32), ("strand", C.c_int32),
                ("id", C.c_double)]


def cluster_fast(ctx: "Context", ss: SeqSetHandle, opts: SearchOpts, round_size: int):
    """vsg_cluster_fast -> (numpy structured array of per-sequence results, number of clusters, work[2])"""
    dt = np.dtype([("cluster", np.int32), ("centroid", np.int32), ("matches", np.int32), ("mismatches", np.int32),
                   ("gaps", np.int32), ("alignment_length", np.int32), ("nwscore", np.int32), ("strand", np.int32),
                   ("id", np.float64)])
    assert dt.itemsize == C.sizeof(ClusterResult)
    res = np.zeros(ss.n, dtype=dt)
    ncl = C.c_int64()
    work = np.zeros(2, dtype=np.int64)
    _check(load().vsg_cluster_fast(ctx.h, ss.h, C.byref(opts), C.c_int(round_size), res.ctypes.data_as(C.POINTER(ClusterResult)),
                                   C.byref(ncl), _ptr(work, C.c_int64)), "vsg_cluster_fast")
    return res, int(ncl.value), work


_CLUSTER_DT = np.dtype([("cluster", np.int32), ("centroid", np.int32), ("matches", np.int32), ("mismatches", np.int32),
                        ("gaps", np.int32), ("alignment_length", np.int32), ("nwscore", np.int32), ("strand", np.int32),
                        ("id", np.float64)])


class ClusterSession:
    """vsg_cluster_session: the clustering fed range by range (cluster_assign_batch / cluster_assign_single)"""

    def __init__(self, ctx: "Context", ss: SeqSetHandle, opts: SearchOpts):
        self._keep = (ctx, ss, opts)
        self.h = C.c_void_p()
        lib = load()
        lib.vsg_cluster_session_clusters.restype = C.c_int64
        _check(lib.vsg_cluster_session_create(ctx.h, ss.h, C.byref(opts), C.byref(self.h)), "vsg_cluster_session_create")

    def assign(self, start: int, count: int, round_size: int):
        res = np.zeros(count, dtype=_CLUSTER_DT)
        _check(load().vsg_cluster_session_assign(self.h, C.c_int64(start), C.c_int64(count), C.c_int(round_size),
                                                 res.ctypes.data_as(C.POINTER(ClusterResult))), "vsg_cluster_session_assign")
        return res

    @property
    def clusters(self) -> int:
        return int(load().vsg_cluster_session_clusters(self.h))

    def close(self):
        if self.h:
            load().vsg_cluster_session_destroy(self.h)
            self.h = C.c_void_p()


class Group:
    """vsg_group: one process, several GPUs (database copied device to device, queries / rows sharded)"""

    def __init__(self, devices, ss, wordlength=8, mask_lower=0, dust_db=0, pen=DEFAULT_PEN, n_mismatch=0):
        lib = load()
        sc = Scoring()
        for i in range(14):
            sc.v[i] = int(pen[i])
        sc.n_mismatch = int(n_mismatch)
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        cat = np.ascontiguousarray(ss.cat, dtype=np.uint8)
        offs = np.ascontiguousarray(ss.offs, dtype=np.int64)
        lens = np.ascontiguousarray(ss.lens, dtype=np.int32)
        self.h = C.c_void_p()
        self.n = int(lens.shape[0])
        _check(lib.vsg_group_create(_ptr(dev, C.c_int), C.c_int(dev.shape[0]), C.byref(sc), _ptr(cat, C.c_char),
                                    _ptr(offs, C.c_int64), _ptr(lens, C.c_int32), C.c_int64(self.n), C.c_int(wordlength),
                                    C.c_int(mask_lower), C.c_int(dust_db), C.byref(self.h)), "vsg_group_create")

    @classmethod
    def from_udb(cls, devices, udb: "Udb", pen=DEFAULT_PEN, n_mismatch=0):
        """vsg_group_create_udb: the database of a parsed UDB file on every device"""
        self = cls.__new__(cls)
        sc = Scoring()
        for i in range(14):
            sc.v[i] = int(pen[i])
        sc.n_mismatch = int(n_mismatch)
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        self.h = C.c_void_p()
        self.n = udb.n
        _check(load().vsg_group_create_udb(_ptr(dev, C.c_int), C.c_int(dev.shape[0]), C.byref(sc), udb.h, C.byref(self.h)),
               "vsg_group_create_udb")
        return self

    def close(self):
        if self.h:
            load().vsg_group_destroy(self.h)
            self.h = None

    def stats(self):
        ms = np.zeros(3, dtype=np.float64)
        b = C.c_int64()
        _check(load().vsg_group_stats(self.h, _ptr(ms, C.c_double), C.byref(b)), "vsg_group_stats")
        return {"upload_ms": float(ms[0]), "broadcast_ms": float(ms[1]), "index_ms": float(ms[2]), "broadcast_bytes": int(b.value)}

    def search(self, qs, opts: SearchOpts, max_results: int, dust_queries: int = 0):
        nq = len(qs)
        res = (SearchResult * (nq * max_results))()
        counts = np.zeros(nq, dtype=np.int32)
        work = np.zeros(4, dtype=np.int64)
        cat = np.ascontiguousarray(qs.cat, dtype=np.uint8)
        offs = np.ascontiguousarray(qs.offs, dtype=np.int64)
        lens = np.ascontiguousarray(qs.lens, dtype=np.int32)
        _check(load().vsg_group_search(self.h, _ptr(cat, C.c_char), _ptr(offs, C.c_int64), _ptr(lens, C.c_int32),
                                       C.c_int64(nq), C.c_int(dust_queries), C.byref(opts), res, C.c_int(max_results),
                                       _ptr(counts, C.c_int32), _ptr(work, C.c_int64)), "vsg_group_search")
        return res, counts, work

    def allpairs(self, opts: SearchOpts, cap: int):
        dt = np.dtype([("query", np.int32), ("target", np.int32), ("matches", np.int32), ("mismatches", np.int32),
                       ("gaps", np.int32), ("alignment_length", np.int32), ("nwscore", np.int32),
                       ("internal_alignment_length", np.int32), ("id", np.float64)])
        hits = np.zeros(cap, dtype=dt)
        n = C.c_int64()
        work = np.zeros(2, dtype=np.int64)
        _check(load().vsg_group_allpairs(self.h, C.byref(opts), hits.ctypes.data_as(C.POINTER(PairHit)), C.c_int64(cap),
                                         C.byref(n), _ptr(work, C.c_int64)), "vsg_group_allpairs")
        return hits[: n.value], work

    def stream(self, target_labels, query_fasta: str, opts: SearchOpts, blast6out: str, qmask_dust: int = 0, notrunclabels: int = 0,
               batch_queries: int = 65536, maxhits: int = 0, output_no_hits: int = 0):
        """vsg_usearch_stream: FASTA file in, --blast6out file out; returns the statistics record as a dict"""
        labs = (C.c_char_p * len(target_labels))(*[l if isinstance(l, bytes) else l.encode() for l in target_labels])
        st = StreamStats()
        _check(load().vsg_usearch_stream(self.h, labs, query_fasta.encode(), C.byref(opts), C.c_int(qmask_dust), C.c_int(notrunclabels),
                                         C.c_int(batch_queries), C.c_int64(maxhits), C.c_int(output_no_hits), blast6out.encode(),
                                         C.byref(st)), "vsg_usearch_stream")
        return {k: getattr(st, k) for k, _ in StreamStats._fields_}


class UdbInfo(C.Structure):
    _fields_ = [("sequences", C.c_int64), ("nucleotides", C.c_int64), ("header_chars", C.c_int64), ("index_entries", C.c_int64),
                ("longest_header", C.c_int64), ("wordlength", C.c_int32), ("dbaccel", C.c_int32), ("shortest", C.c_int32),
                ("longest", C.c_int32)]


def udb_detect(path: str) -> bool:
    rc = load().vsg_udb_detect(path.encode())
    if rc < 0:
        _check(rc, "vsg_udb_detect")
    return rc == 1


class Udb:
    """A parsed UDB file (host side; no GPU needed): vsg_udb_open and its accessors."""

    def __init__(self, path: str):
        self.h = C.c_void_p()
        _check(load().vsg_udb_open(path.encode(), C.byref(self.h)), "vsg_udb_open")
        self.info = UdbInfo()
        _check(load().vsg_udb_info_get(self.h, C.byref(self.info)), "vsg_udb_info_get")
        self.n = int(self.info.sequences)

    def close(self):
        if self.h:
            load().vsg_udb_close(self.h)
            self.h = C.c_void_p()

    def sequences(self):
        """(cat bytes, offsets, lengths) as numpy copies"""
        cat = C.c_char_p(); off = C.POINTER(C.c_int64)(); ln = C.POINTER(C.c_int32)()
        cat_p = C.c_void_p()
        _check(load().vsg_udb_sequences(self.h, C.byref(cat_p), C.byref(off), C.byref(ln)), "vsg_udb_sequences")
        total = int(self.info.nucleotides)
        catb = np.frombuffer(C.string_at(cat_p.value, total), dtype=np.uint8).copy()
        return catb, np.ctypeslib.as_array(off, shape=(self.n,)).copy(), np.ctypeslib.as_array(ln, shape=(self.n,)).copy()

    def header(self, i: int) -> str:
        return load().vsg_udb_header(self.h, C.c_int64(i)).decode()

    def words(self):
        """the stored index: (kmercount[4^k], kmerindex[index_entries]) as numpy copies"""
        kc = C.POINTER(C.c_uint32)(); ki = C.POINTER(C.c_uint32)()
        _check(load().vsg_udb_words(self.h, C.byref(kc), C.byref(ki)), "vsg_udb_words")
        nk = 1 << (2 * int(self.info.wordlength))
        ne = int(self.info.index_entries)
        return (np.ctypeslib.as_array(kc, shape=(nk,)).copy(),
                np.ctypeslib.as_array(ki, shape=(ne,)).copy() if ne > 0 else np.zeros(0, dtype=np.uint32))


class StreamStats(C.Structure):
    _fields_ = [("queries", C.c_int64), ("matched", C.c_int64), ("rows", C.c_int64), ("batches", C.c_int64), ("nucleotides", C.c_int64),
                ("parse_s", C.c_double), ("search_s", C.c_double), ("write_s", C.c_double), ("wall_s", C.c_double)]


def default_search_opts() -> SearchOpts:
    o = SearchOpts()
    load().vsg_search_opts_default(C.byref(o))
    return o
