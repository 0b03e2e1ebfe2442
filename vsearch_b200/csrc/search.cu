// search.cu — the per-query accept/reject driver on top of the device ranker and aligner.
//
// Replaces search_batch (reference core/search.hpp:135-145, core/search.cpp:397-593), i.e. for every
// query: search_onequery (core/searchcore.cpp:884-957) -> align_delayed (:740-881) -> align_trim
// (:343-464) -> search_acceptable_aligned (:664-737) -> search_joinhits (:1028-1052).
//
// The reference walks one query at a time and aligns its candidates in groups of MAXDELAYED = 8
// (searchcore.hpp:71).  Here every query of a batch advances in lock step: each ROUND gathers, for
// all still-active queries, exactly the group of <= 8 candidates the reference would hand to search16
// next, aligns all groups of the round in one batched device call, and then replays the reference's
// sequential accept/reject bookkeeping on the results.  The set of pairs aligned, the order in which
// hits are examined and every counter are those of the reference, so the hit tables are identical.
#include "vsg_internal.h"
#include "hit_logic.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <climits>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <chrono>
#include <cstdio>

namespace vsg {
int rank_enqueue(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq,
                 int minwordmatches, int tophits, int mask_lower, uint32_t ** d_seqno, uint32_t ** d_count,
                 int32_t ** d_n, int32_t ** d_status);
int rank_all_count(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq,
                   int minwordmatches, int tophits, int mask_lower, uint32_t * h_T, int32_t * h_K);
int rank_all_emit(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq,
                  int minwordmatches, int tophits, int mask_lower, const uint32_t * h_T, const int32_t * h_K,
                  uint32_t ** d_seqno, uint32_t ** d_count, const int32_t ** d_coff);
int seqset_revcomp(vsg_ctx * c, const vsg_seqset * src, int64_t q0, int64_t nq, vsg_seqset ** out);
void rank_collect_time(vsg_ctx * c);
const vsg_seqset * index_db(const vsg_index * ix);
int index_wordlength(const vsg_index * ix);
}  // namespace vsg

using namespace vsg;

namespace {

struct QState {
  int ncand = 0, next = 0;
  const uint32_t * cs = nullptr;
  const uint32_t * cc = nullptr;
  const uint8_t * cf = nullptr;  // per-candidate device verdicts of the sequence-content filters (0 = pass)
  int64_t hit_base = 0;  // index of this state's first Hit in the batch-wide hit array
  int hit_count = 0, accepts = 0, rejects = 0, finalized = 0, delayed = 0;
  int gpos = -1;  // lazy mode: next hit of the open group to examine (-1: no group open)
  int gend = 0, greq = 0;  // lazy mode: end of the requested hit range, number of pairs requested
  int cache_first = -1, cache_off = 0;  // tail mode: results of hits >= cache_first sit at tail cache[cache_off + x - cache_first]
  bool done = false, waiting = false;
};

struct SearchScratch {  // per host thread, see vsg_ctx::search_scratch
  std::vector<uint32_t> h_seqno, h_count;
  std::vector<uint8_t> h_flags;
  std::vector<int32_t> h_n;
  std::vector<size_t> cand_at;          // where each state's candidates start in h_seqno / h_count / h_flags
  std::vector<uint32_t> all_T;          // candidate lists longer than 1 024: pass A's threshold and count per (strand, query)
  std::vector<int32_t> all_K;
  std::vector<QState> st;
  Hit * hits = nullptr;
  size_t hits_cap = 0;
  std::vector<uint32_t> pq, pt, lq, lt;
  std::vector<int> pstate, px, lstate;
  std::vector<int32_t> plead, lead_tmp;   // traceback on demand: each pair's group leader (index into the round's pair list) or -1
  std::vector<int64_t> ldest;
  std::vector<int16_t> a_score, l_score, t_score;
  std::vector<uint16_t> a_al, a_ma, a_mi, a_ga, l_al, l_ma, l_mi, l_ga, t_al, t_ma, t_mi, t_ga;
  std::vector<int32_t> a_tr, l_tr, t_tr;
  std::vector<Hit> joined;
  SearchScratch() = default;
  SearchScratch(const SearchScratch &) = delete;
  SearchScratch & operator=(const SearchScratch &) = delete;
  ~SearchScratch() { std::free(hits); }
};

// idprefix / idsuffix / selfid of search_acceptable_unaligned (searchcore.cpp:588-607) for every candidate
// of every query of a ranked batch: one warp per (query, candidate) compares 4-bit codes as seqcmp does
// (utils/seqcmp.cpp:72-92).  flags: 1 = idprefix fails, 2 = idsuffix fails, 4 = selfid fails.
// CSR = false: candidate j of query qi at [qi * tophits + j], ncand[qi] of them.  CSR = true (lists longer than 1 024):
// the candidates of query qi at [ncand[qi], ncand[qi + 1]).
template <bool CSR>
__global__ void prefilter_kernel(DevSeqs qs, int64_t q0, int nq, DevSeqs db, const uint32_t * __restrict__ cand,
                                 const int32_t * __restrict__ ncand, int tophits, int idprefix, int idsuffix, int selfid,
                                 uint8_t * __restrict__ flags)
{
  int64_t const w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  int const lane = threadIdx.x & 31;
  int qi;
  if constexpr (CSR) {
    if (w >= ncand[nq]) { return; }
    int lo = 0, hi = nq - 1;   // the last query whose list starts at or before w
    while (lo < hi) {
      int const mid = (lo + hi + 1) >> 1;
      if (ncand[mid] <= w) { lo = mid; } else { hi = mid - 1; }
    }
    qi = lo;
  } else {
    if (w >= static_cast<int64_t>(nq) * tophits) { return; }
    qi = static_cast<int>(w / tophits);
    int const j = static_cast<int>(w % tophits);
    if (j >= ncand[qi]) { return; }
  }
  uint32_t const t = cand[w];
  const uint8_t * __restrict__ q = qs.sym + qs.off[q0 + qi];
  const uint8_t * __restrict__ d = db.sym + db.off[t];
  int const ql = qs.len[q0 + qi], dl = db.len[t];
  auto differ = [&](const uint8_t * a, const uint8_t * b, int n) -> bool {
    int bad = 0;
    for (int i = lane; i < n; i += 32) { bad |= ((a[i] ^ b[i]) & 15) != 0; }
    return __any_sync(0xffffffffu, bad) != 0;
  };
  unsigned f = 0;
  if (idprefix > 0 && (ql < idprefix || dl < idprefix || differ(q, d, idprefix))) { f |= 1u; }
  if (idsuffix > 0 && (ql < idsuffix || dl < idsuffix || differ(q + ql - idsuffix, d + dl - idsuffix, idsuffix))) { f |= 2u; }
  if (selfid != 0 && ql == dl && !differ(q, d, ql)) { f |= 4u; }
  if (lane == 0) { flags[w] = static_cast<uint8_t>(f); }
}

}  // namespace

extern "C" void vsg_search_opts_default(vsg_search_opts * o)
{
  if (o == nullptr) { return; }
  o->id = 0.0; o->weak_id = 10.0; o->maxaccepts = 1; o->maxrejects = 32; o->wordlength = 8;
  o->minwordmatches = -1; o->iddef = 2; o->strand_both = 0; o->mask_lower = 0; o->lazy = 0;
  o->minqt = 0.0; o->maxqt = 1.7976931348623157e308; o->minsl = 0.0; o->maxsl = 1.7976931348623157e308;
  o->maxid = 1.0; o->mid = 0.0; o->query_cov = 0.0; o->target_cov = 0.0;
  o->maxsubs = 2147483647; o->maxgaps = 2147483647; o->mincols = 0; o->maxdiffs = 2147483647;
  o->leftjust = 0; o->rightjust = 0;
  o->maxqsize = INT64_MAX; o->mintsize = 0; o->minsizeratio = 0.0; o->maxsizeratio = 1.7976931348623157e308;
  o->idprefix = 0; o->idsuffix = 0; o->self = 0; o->selfid = 0; o->qmask_dust = 0; o->unoise = 0; o->unoise_alpha = 2.0; o->sizeorder = 0; o->reserved1 = 0;
  o->query_sizes = nullptr; o->target_sizes = nullptr; o->query_labels = nullptr; o->target_labels = nullptr;
}

// vsg_search_batch; the rows of query q go to results[q * max_results ...] or, with rows != nullptr, to rows[q]
static int search_batch(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * db, const vsg_seqset * queries, int64_t q0,
                        int64_t nq, const vsg_search_opts * opts, vsg_search_result * results, int64_t max_results,
                        std::vector<vsg_search_result> * rows, int32_t * counts, int64_t * work)
{
  if (c == nullptr || ix == nullptr || db == nullptr || queries == nullptr || opts == nullptr || counts == nullptr) {
    Error::set("vsg_search_batch: bad argument");
    return VSG_EINVAL;
  }
  if (index_db(ix) != db) { Error::set("vsg_search_batch: index was built for another sequence set"); return VSG_EINVAL; }
  if (q0 < 0 || nq < 0 || q0 + nq > queries->d.n) { Error::set("vsg_search_batch: query range out of bounds"); return VSG_EINVAL; }
  if (opts->wordlength != index_wordlength(ix)) { Error::set("vsg_search_batch: wordlength differs from the index"); return VSG_EINVAL; }
  if (opts->iddef < 0 || opts->iddef > 4) { Error::set("vsg_search_batch: iddef must be 0..4"); return VSG_EINVAL; }

  // option fix-ups: vsearch_apply_defaults_fixups (vsearch.cc:186-276) and the seqcount clamps of
  // search_prep / search_session_init (commands/usearch_global.cpp:598-614)
  int64_t const seqcount = db->d.n;
  int64_t maxaccepts = opts->maxaccepts, maxrejects = opts->maxrejects < 0 ? 32 : opts->maxrejects;
  if (maxaccepts < 0) { Error::set("vsg_search_batch: maxaccepts must not be negative"); return VSG_EINVAL; }
  if (maxaccepts > seqcount || maxaccepts == 0) { maxaccepts = seqcount; }
  if (maxrejects > seqcount || maxrejects == 0) { maxrejects = seqcount; }
  int64_t tophits64 = maxaccepts + maxrejects + MAXDELAYED;
  if (tophits64 > seqcount) { tophits64 = seqcount; }
  int const minwordmatches = opts->minwordmatches < 0 ? minwordmatches_defaults[opts->wordlength] : opts->minwordmatches;
  double const opt_id = opts->id;
  double const opt_weak_id = (opts->id >= 0.0 && opts->weak_id > opts->id) ? opts->id : opts->weak_id;
  int64_t total_pairs = 0, total_cells = 0, aligned_pairs = 0, aligned_cells = 0;
  bool const lazy = opts->lazy != 0;
  // Traceback on demand (align_ckpt.cuh, TbGate) needs the device's verdict on a group's first candidate to be the
  // host's: that holds when search_acceptable_aligned reduces to its identity test, i.e. every optional
  // post-alignment filter is at its default and no pair can be diverted to the caller's aligner.  VSG_TB_GATE=0 turns
  // it off (A/B runs; the results do not depend on it).
  // VSG_TB_GATE_FORCE=1 (tests): the device takes EVERY leader for accepted, so every follower the replay needs goes
  // through the re-alignment below
  bool const tb_force = [] { const char * e = std::getenv("VSG_TB_GATE_FORCE"); return e != nullptr && e[0] == '1'; }();
  bool tb_gate = false;
  {
    vsg_search_opts d;
    vsg_search_opts_default(&d);
    const char * const e = std::getenv("VSG_TB_GATE");
    tb_gate = (e == nullptr || e[0] != '0') && !lazy && !c->sp.fallback &&
              opts->maxsubs == d.maxsubs && opts->maxgaps == d.maxgaps && opts->mincols == d.mincols && opts->maxdiffs == d.maxdiffs &&
              opts->leftjust == 0 && opts->rightjust == 0 && opts->query_cov == d.query_cov && opts->target_cov == d.target_cov &&
              opts->maxid == d.maxid && opts->mid == d.mid && opts->iddef >= 0 && opts->iddef <= 4 && opt_weak_id <= opt_id &&
              opts->unoise == 0;
  }
  for (int64_t q = 0; q < nq; q++) { counts[q] = 0; }
  if (seqcount == 0 || nq == 0) { if (work) { work[0] = work[1] = work[2] = work[3] = 0; } return VSG_OK; }
  int const tophits = static_cast<int>(tophits64);
  // Lists longer than the shared-memory ranker holds are ranked in two passes (rank.cu, rank_all_*) and kept as CSR; a
  // sub-batch is then searched in pieces of at most `cand_budget` candidates (VSG_CAND_BUDGET: smaller pieces, for tests)
  bool const long_lists = tophits > 1024;
  int64_t cand_budget = CAND_VOLUME_BUDGET;
  if (const char * e = std::getenv("VSG_CAND_BUDGET")) { cand_budget = std::max<int64_t>(1, std::atoll(e)); }
  bool const trace_pieces = std::getenv("VSG_TRACE") != nullptr;
  // Both limits at least every list's length (e.g. --maxaccepts 0 --maxrejects 0): the candidate loop cannot stop before
  // a list ends (searchcore.cpp:915-918), so every candidate is aligned and the tail below may take them all in the
  // first round instead of in groups of eight
  bool const whole_lists = long_lists && maxaccepts >= tophits && maxrejects >= tophits;
  int const nstrands = opts->strand_both ? 2 : 1;
  if (opts->self != 0 && (opts->query_labels == nullptr || opts->target_labels == nullptr)) {
    Error::set("vsg_search_batch: --self needs query_labels and target_labels"); return VSG_EINVAL;
  }
  if (opts->idprefix < 0 || opts->idsuffix < 0) { Error::set("vsg_search_batch: idprefix/idsuffix must not be negative"); return VSG_EINVAL; }
  bool const content_filters = opts->idprefix > 0 || opts->idsuffix > 0 || opts->selfid != 0;

  // Sub-batches run on a few host threads, each with its own child context (stream + scratch):
  // while one thread replays accept/reject decisions or builds task lists, the kernels of the
  // others keep the GPU busy.  Results land in disjoint slots, so no ordering is needed.
  int64_t BATCH = 4096;
  if (const char * e = std::getenv("VSG_SUBBATCH")) { BATCH = std::max<int64_t>(256, std::atoll(e)); }
  int64_t const nbatches = (nq + BATCH - 1) / BATCH;
  int nthreads = 8;
  if (const char * e = std::getenv("VSG_HOST_THREADS")) { nthreads = std::max(1, std::atoi(e)); }
  nthreads = static_cast<int>(std::min<int64_t>(nthreads, nbatches));
  bool stagger = true;
  if (const char * e = std::getenv("VSG_STAGGER")) { stagger = std::atoi(e) != 0; }
  int64_t tail_pairs = 4096;  // the tail starts when the round's pairs + all remaining candidates fit in this (0: never)
  if (const char * e = std::getenv("VSG_TAIL_PAIRS")) { tail_pairs = std::max<int64_t>(0, std::atoll(e)); }
  while (static_cast<int>(c->children.size()) < nthreads) {
    vsg_ctx * ch = nullptr;
    int const r = vsg_ctx_create(c->device, &c->scoring, &ch);
    if (r != VSG_OK) { return r; }
    c->children.push_back(ch);
  }
  for (int t = 0; t < nthreads; t++) {
    c->children[static_cast<size_t>(t)]->dir_budget = std::max<size_t>(c->dir_budget / static_cast<size_t>(nthreads), static_cast<size_t>(1) << 30);
    c->children[static_cast<size_t>(t)]->fast_disabled = c->fast_disabled;
    c->children[static_cast<size_t>(t)]->ckpt_enabled = c->ckpt_enabled;
  }

  vsg_ctx * const parent = c;
  auto const t_call0 = std::chrono::steady_clock::now();
  auto run_batch = [&](vsg_ctx * c, int64_t sb0, int64_t bn_req, int64_t & total_pairs, int64_t & total_cells, int64_t & al_pairs, int64_t & al_cells) -> int {
  // host buffers live in the worker's context: a batch touches ~20 MB of them, and fresh pages per
  // batch (malloc -> mmap -> page faults) cost more than the bookkeeping itself
  if (!c->search_scratch) { c->search_scratch = std::make_shared<SearchScratch>(); }
  SearchScratch & sc = *static_cast<SearchScratch *>(c->search_scratch.get());
  auto & h_seqno = sc.h_seqno; auto & h_count = sc.h_count; auto & h_n = sc.h_n; auto & st = sc.st;
  Hit *& hits = sc.hits;  // bn*nstrands*tophits slots, deliberately uninitialised (each is zeroed when popped)
  auto & pq = sc.pq; auto & pt = sc.pt;
  auto & pstate = sc.pstate;  // which state each pair belongs to
  auto & px = sc.px;          // which of the state's hits
  auto & plead = sc.plead; auto & lead_tmp = sc.lead_tmp;
  int64_t tb_redone = 0;
  // tail mode (see below): one device call resolves every remaining candidate of the few queries still active
  auto & lq = sc.lq; auto & lt = sc.lt; auto & lstate = sc.lstate; auto & ldest = sc.ldest;
  auto & l_score = sc.l_score; auto & t_score = sc.t_score;
  auto & l_al = sc.l_al; auto & l_ma = sc.l_ma; auto & l_mi = sc.l_mi; auto & l_ga = sc.l_ga;
  auto & t_al = sc.t_al; auto & t_ma = sc.t_ma; auto & t_mi = sc.t_mi; auto & t_ga = sc.t_ga;
  auto & l_tr = sc.l_tr; auto & t_tr = sc.t_tr;
  auto & a_score = sc.a_score; auto & a_al = sc.a_al; auto & a_ma = sc.a_ma; auto & a_mi = sc.a_mi; auto & a_ga = sc.a_ga;
  auto & a_tr = sc.a_tr;
  auto & joined = sc.joined;
  VSG_CUDA_OK(cudaSetDevice(c->device));
  static const bool trace = std::getenv("VSG_TRACE") != nullptr;
  auto now = []() { return std::chrono::steady_clock::now(); };
  auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double, std::milli>(b - a).count();
  };
  double t_rank = 0, t_init = 0, t_gather = 0, t_align = 0, t_replay = 0, t_join = 0;
  auto tp0 = now();
  int64_t const sbn = std::min(bn_req, nq - sb0);
  vsg_seqset * rc_set = nullptr;
  struct RcGuard { vsg_seqset *& s; ~RcGuard() { if (s != nullptr) { vsg_seqset_destroy(s); s = nullptr; } } } rc_guard{rc_set};   // every exit
  if (nstrands == 2) {
    int r = seqset_revcomp(c, queries, q0 + sb0, sbn, &rc_set);
    if (r != VSG_OK) { return r; }
    // each strand is masked on its own (search.cpp:437-449); dust() upper-cases first, so the case the
    // reverse complement inherited from the masked plus strand does not matter
    if (opts->qmask_dust != 0 && (r = vsg_seqset_dust(c, rc_set)) != VSG_OK) { return r; }
  }
  // long lists: pass A for the whole sub-batch gives every list's length before anything large is allocated
  auto & all_T = sc.all_T; auto & all_K = sc.all_K;
  if (long_lists) {
    all_T.resize(static_cast<size_t>(sbn) * nstrands); all_K.resize(static_cast<size_t>(sbn) * nstrands);
    for (int s = 0; s < nstrands; s++) {
      int const r = rank_all_count(c, ix, s == 0 ? queries : rc_set, s == 0 ? q0 + sb0 : 0, sbn, minwordmatches, tophits,
                                   opts->mask_lower, all_T.data() + sbn * s, all_K.data() + sbn * s);
      if (r != VSG_OK) { return r; }
    }
  }
  // one piece of the sub-batch: queries [b0, b0 + bn) of the call, [rc0, rc0 + bn) of rc_set
  auto run_piece = [&](int64_t b0, int64_t bn, int64_t rc0) -> int {
    size_t const cells = static_cast<size_t>(bn) * tophits;
    auto & cand_at = sc.cand_at;
    cand_at.resize(static_cast<size_t>(bn) * nstrands);
    h_n.resize(static_cast<size_t>(bn) * nstrands);
    if (!long_lists) {
      h_seqno.resize(cells * nstrands); h_count.resize(cells * nstrands);
      if (content_filters) { sc.h_flags.resize(cells * nstrands); }
      for (size_t si = 0; si < cand_at.size(); si++) { cand_at[si] = si * static_cast<size_t>(tophits); }
    } else {
      size_t pos = 0;
      for (int s = 0; s < nstrands; s++) {
        for (int64_t q = 0; q < bn; q++) {
          size_t const si = static_cast<size_t>(s) * bn + q;
          cand_at[si] = pos;
          h_n[si] = std::min(all_K[static_cast<size_t>(s) * sbn + rc0 + q], tophits);
          pos += static_cast<size_t>(h_n[si]);
        }
      }
      h_seqno.resize(pos); h_count.resize(pos);
      if (content_filters) { sc.h_flags.resize(pos); }
    }
    // search_acceptable_unaligned for candidate `target` of the batch's query `ql` (searchcore.cpp:541-609)
    auto unaligned_ok = [&](int target, int64_t ql, int sqlen, unsigned content) -> bool {
      int64_t const qsize = opts->query_sizes != nullptr ? opts->query_sizes[b0 + ql] : 1;
      int64_t const tsize = opts->target_sizes != nullptr ? opts->target_sizes[target] : 1;
      bool const same_label = opts->self != 0 && opts->query_labels[b0 + ql] == opts->target_labels[target];
      return acceptable_unaligned(*opts, sqlen, db->h_len[static_cast<size_t>(target)], qsize, tsize, same_label, content);
    };
    for (int s = 0; s < nstrands && long_lists; s++) {
      uint32_t *d_seqno, *d_count; const int32_t * d_coff;
      const vsg_seqset * qset = (s == 0) ? queries : rc_set;
      int64_t const qq0 = (s == 0) ? q0 + b0 : rc0;
      size_t const at = cand_at[static_cast<size_t>(s) * bn], n = (s + 1 < nstrands ? cand_at[static_cast<size_t>(s + 1) * bn] : h_seqno.size()) - at;
      int r = rank_all_emit(c, ix, qset, qq0, bn, minwordmatches, tophits, opts->mask_lower, all_T.data() + sbn * s + rc0,
                            all_K.data() + sbn * s + rc0, &d_seqno, &d_count, &d_coff);
      if (r != VSG_OK) { return r; }
      if (n == 0) { continue; }
      VSG_CUDA_OK(cudaMemcpyAsync(h_seqno.data() + at, d_seqno, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaMemcpyAsync(h_count.data() + at, d_count, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, c->stream));
      if (content_filters) {
        if ((r = c->pre_flags.reserve(n + 16)) != VSG_OK) { return r; }
        VSG_CUDA_OK(cudaMemsetAsync(c->pre_flags.p, 0, n, c->stream));
        prefilter_kernel<true><<<static_cast<unsigned>((static_cast<int64_t>(n) * 32 + 255) / 256), 256, 0, c->stream>>>(
            qset->d, qq0, static_cast<int>(bn), db->d, d_seqno, d_coff, tophits, opts->idprefix, opts->idsuffix, opts->selfid,
            static_cast<uint8_t *>(c->pre_flags.p));
        count_launch();
        VSG_CUDA_OK(cudaMemcpyAsync(sc.h_flags.data() + at, c->pre_flags.p, n, cudaMemcpyDeviceToHost, c->stream));
      }
      VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
    }
    for (int s = 0; s < nstrands && !long_lists; s++) {
      uint32_t *d_seqno, *d_count; int32_t *d_n, *d_status;
      const vsg_seqset * qset = (s == 0) ? queries : rc_set;
      int64_t const qq0 = (s == 0) ? q0 + b0 : 0;
      int r = rank_enqueue(c, ix, qset, qq0, bn, minwordmatches, tophits, opts->mask_lower, &d_seqno, &d_count, &d_n, &d_status);
      if (r != VSG_OK) { return r; }
      int32_t status = 0;
      VSG_CUDA_OK(cudaMemcpyAsync(h_seqno.data() + cells * s, d_seqno, sizeof(uint32_t) * cells, cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaMemcpyAsync(h_count.data() + cells * s, d_count, sizeof(uint32_t) * cells, cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaMemcpyAsync(h_n.data() + bn * s, d_n, sizeof(int32_t) * bn, cudaMemcpyDeviceToHost, c->stream));
      if (content_filters) {
        if ((r = c->pre_flags.reserve(cells + 16)) != VSG_OK) { return r; }
        VSG_CUDA_OK(cudaMemsetAsync(c->pre_flags.p, 0, cells, c->stream));
        int64_t const nwarps = bn * tophits;
        prefilter_kernel<false><<<static_cast<unsigned>((nwarps * 32 + 255) / 256), 256, 0, c->stream>>>(
            qset->d, qq0, static_cast<int>(bn), db->d, d_seqno, d_n, tophits, opts->idprefix, opts->idsuffix, opts->selfid,
            static_cast<uint8_t *>(c->pre_flags.p));
        count_launch();
        VSG_CUDA_OK(cudaMemcpyAsync(sc.h_flags.data() + cells * s, c->pre_flags.p, cells, cudaMemcpyDeviceToHost, c->stream));
      }
      VSG_CUDA_OK(cudaMemcpyAsync(&status, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
      rank_collect_time(c);
      if (status != 0) {
        Error::set("vsg_search_batch: a query is longer than the device ranker supports (65 534 + wordlength nt)");
        return VSG_EINVAL;
      }
    }

    t_rank += ms(tp0, now()); tp0 = now();
    // one state per (query, strand); hits preallocated at one per candidate (a state never holds more)
    st.assign(static_cast<size_t>(bn) * nstrands, QState());
    size_t nhits = 0;
    for (size_t si = 0; si < st.size(); si++) {
      QState & S = st[si];
      S.ncand = h_n[si];
      S.cs = h_seqno.data() + cand_at[si];
      S.cc = h_count.data() + cand_at[si];
      S.cf = content_filters ? sc.h_flags.data() + cand_at[si] : nullptr;
      S.hit_base = static_cast<int64_t>(nhits);
      nhits += static_cast<size_t>(S.ncand);
    }
    if (nhits > sc.hits_cap) {
      std::free(hits);
      hits = static_cast<Hit *>(std::malloc(sizeof(Hit) * nhits));
      sc.hits_cap = hits != nullptr ? nhits : 0;
      if (hits == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
    }

    t_init += ms(tp0, now());
    bool any = true;
    bool tail_mode = false;
    bool gated_round = false;
    while (any) {
      gated_round = false;
      tp0 = now();
      any = false;
      pq.clear(); pt.clear(); pstate.clear(); px.clear(); plead.clear();
      // gather: run each active query's candidate loop up to its next align_delayed (searchcore.cpp:915-954)
      if (lazy) {
        // same decisions, alignments on demand: open the group the reference would hand to search16,
        // but align only the hit the replay is about to examine
        for (size_t si = 0; si < st.size(); si++) {
          QState & S = st[si];
          if (S.done) { continue; }
          int const strand = static_cast<int>(si / static_cast<size_t>(bn));
          int64_t const ql = static_cast<int64_t>(si % static_cast<size_t>(bn));
          int const sqlen = (strand == 0 ? queries->h_len[static_cast<size_t>(q0 + b0 + ql)] : rc_set->h_len[static_cast<size_t>(rc0 + ql)]);
          for (;;) {
            if (S.gpos < 0) {
              bool trigger = false;
              while ((S.finalized + S.delayed < maxaccepts + maxrejects - 1) && (S.rejects < maxrejects) &&
                     (S.accepts < maxaccepts) && (S.next < S.ncand)) {
                Hit & h = hits[static_cast<size_t>(S.hit_base) + S.hit_count];
                std::memset(&h, 0, sizeof(Hit));
                h.target = static_cast<int>(S.cs[S.next]); h.count = S.cc[S.next]; h.strand = strand;
                unsigned const content = S.cf != nullptr ? S.cf[S.next] : 0u;
                S.next++;
                if (unaligned_ok(h.target, ql, sqlen, content)) { S.delayed++; }
                else { h.rejected = true; }
                S.hit_count++;
                if (S.delayed == MAXDELAYED) { trigger = true; break; }
              }
              if (!trigger && S.delayed == 0) { S.done = true; break; }
              S.gpos = S.finalized;
              for (int x = S.finalized; x < S.hit_count; x++) {   // what the reference's search16 call covers
                Hit const & h = hits[static_cast<size_t>(S.hit_base) + x];
                if (!h.rejected) { total_pairs++; total_cells += static_cast<int64_t>(sqlen) * db->h_len[static_cast<size_t>(h.target)]; }
              }
            }
            bool need = false;
            while (S.gpos < S.hit_count && S.rejects < maxrejects && S.accepts < maxaccepts) {
              Hit const & h = hits[static_cast<size_t>(S.hit_base) + S.gpos];
              if (h.rejected) { S.rejects++; S.gpos++; continue; }
              need = true;
              break;
            }
            if (need) {
              // the group's first candidate alone (it is accepted most of the time); if the replay gets
              // past it, the rest of the group in one go — at most two device round trips per group
              int const xend = (S.gpos == S.finalized) ? S.gpos + 1 : S.hit_count;
              S.greq = 0;
              for (int x = S.gpos; x < xend; x++) {
                Hit const & h = hits[static_cast<size_t>(S.hit_base) + x];
                if (h.rejected) { continue; }
                pq.push_back(static_cast<uint32_t>(strand == 0 ? q0 + b0 + ql : rc0 + ql));
                pt.push_back(static_cast<uint32_t>(h.target));
                pstate.push_back(static_cast<int>(si));
                px.push_back(x);
                S.greq++;
              }
              S.gend = xend;
              S.waiting = true;
              any = true;
              break;
            }
            // group exhausted or a limit reached: align_delayed ends, the candidate loop resumes
            S.finalized = S.hit_count; S.delayed = 0; S.gpos = -1;
          }
        }
      } else
      for (size_t si = 0; si < st.size(); si++) {
        QState & S = st[si];
        if (S.done) { continue; }
        bool trigger = false;
        while ((S.finalized + S.delayed < maxaccepts + maxrejects - 1) && (S.rejects < maxrejects) &&
               (S.accepts < maxaccepts) && (S.next < S.ncand)) {
          Hit & h = hits[static_cast<size_t>(S.hit_base) + S.hit_count];
          std::memset(&h, 0, sizeof(Hit));
          h.target = static_cast<int>(S.cs[S.next]); h.count = S.cc[S.next];
          h.strand = static_cast<int>(si / static_cast<size_t>(bn));
          unsigned const content = S.cf != nullptr ? S.cf[S.next] : 0u;
          S.next++;
          {
            int const sstrand = static_cast<int>(si / static_cast<size_t>(bn));
            int64_t const sql = static_cast<int64_t>(si % static_cast<size_t>(bn));
            int const sqlen = (sstrand == 0 ? queries->h_len[static_cast<size_t>(q0 + b0 + sql)] : rc_set->h_len[static_cast<size_t>(rc0 + sql)]);
            if (unaligned_ok(h.target, sql, sqlen, content)) { S.delayed++; }
            else { h.rejected = true; }
          }
          S.hit_count++;
          if (S.delayed == MAXDELAYED) { trigger = true; break; }
        }
        if (!trigger && S.delayed == 0) { S.done = true; continue; }
        // align_delayed's search16 call: every not-yet-finalized, not pre-rejected hit
        int const strand = static_cast<int>(si / static_cast<size_t>(bn));
        int64_t const ql = static_cast<int64_t>(si % static_cast<size_t>(bn));
        // traceback on demand (align_ckpt.cuh): if accepting the group's first candidate ends this query's search,
        // the others are walked back only when that candidate turns out not to be accepted
        bool const gate_group = tb_gate && (S.accepts + 1 >= maxaccepts);
        int32_t leader = -1;
        for (int x = S.finalized; x < S.hit_count; x++) {
          Hit const & h = hits[static_cast<size_t>(S.hit_base) + x];
          if (!h.rejected) {
            plead.push_back(gate_group ? leader : -1);
            if (leader < 0) { leader = static_cast<int32_t>(pq.size()); }
            pq.push_back(static_cast<uint32_t>(strand == 0 ? q0 + b0 + ql : rc0 + ql));
            pt.push_back(static_cast<uint32_t>(h.target));
            pstate.push_back(static_cast<int>(si));
            px.push_back(x);
          }
        }
        S.waiting = true;
        any = true;
      }
      if (!any) { break; }
      size_t const np = pq.size();
      t_gather += ms(tp0, now()); tp0 = now();
      a_score.resize(np); a_al.resize(np); a_ma.resize(np); a_mi.resize(np); a_ga.resize(np); a_tr.resize(np * 4);
      // pairs of the plus strand index `queries`, those of the minus strand index rc_set: two calls
      // (states are ordered plus first, minus second, so pairs are too)
      auto device_align = [&](size_t n, const uint32_t * Q, const uint32_t * T, const int * state_of,
                              int16_t * o_sc, uint16_t * o_al, uint16_t * o_ma, uint16_t * o_mi, uint16_t * o_ga, int32_t * o_tr,
                              const int32_t * lead) -> int {
        size_t split = n;
        if (nstrands == 2) {
          split = 0;
          while (split < n && static_cast<int64_t>(state_of[split]) < bn) { split++; }
        }
        for (int part = 0; part < 2; part++) {
          size_t const lo = part == 0 ? 0 : split, hi = part == 0 ? split : n;
          if (hi <= lo) { continue; }
          const vsg_seqset * qset = part == 0 ? queries : rc_set;
          const int32_t * lead_part = nullptr;
          if (lead != nullptr) {
            // leaders as indices into this part's own pair list (a group never straddles the strands)
            lead_tmp.assign(lead + lo, lead + hi);
            if (lo > 0) { for (auto & v : lead_tmp) { if (v >= 0) { v -= static_cast<int32_t>(lo); } } }
            lead_part = lead_tmp.data();
          }
          int const r = align_pairs_gated(c, qset, db, static_cast<int64_t>(hi - lo), Q + lo, T + lo,
                                          o_sc + lo, o_al + lo, o_ma + lo, o_mi + lo, o_ga + lo, o_tr + 4 * lo, nullptr, 0, nullptr,
                                          lead_part, tb_force ? -1.0 : 100.0 * opt_id + 1e-7, opts->iddef);
          if (r != VSG_OK) { return r; }
        }
        return VSG_OK;
      };
      bool const from_cache = tail_mode;
      // what the tail shortcut would add to this round: every candidate the active queries have left
      auto count_extras = [&]() -> size_t {
        size_t extras = 0;
        for (size_t k = 0; k < np; k++) {
          if (k + 1 == np || pstate[k + 1] != pstate[k]) {
            QState const & S = st[static_cast<size_t>(pstate[k])];
            extras += static_cast<size_t>(std::max(0, S.ncand - (lazy ? S.gend : S.hit_count)));
          }
        }
        return extras;
      };
      if (tail_mode) {
        // every query still active had all its remaining candidates aligned when the tail began
        for (size_t k = 0; k < np; k++) {
          QState const & S = st[static_cast<size_t>(pstate[k])];
          size_t const ci = static_cast<size_t>(S.cache_off + px[k] - S.cache_first);
          a_score[k] = t_score[ci]; a_al[k] = t_al[ci]; a_ma[k] = t_ma[ci]; a_mi[k] = t_mi[ci]; a_ga[k] = t_ga[ci];
          for (int z = 0; z < 4; z++) { a_tr[4 * k + z] = t_tr[4 * ci + z]; }
        }
      } else if (tail_pairs > 0 && (whole_lists || (np <= static_cast<size_t>(tail_pairs) && np + count_extras() <= static_cast<size_t>(tail_pairs)))) {
        // TAIL: few queries are left and each would need up to five more rounds of eight candidates
        // (searchcore.cpp:915-954), every round a device round trip with almost nothing in it.  Align
        // all their remaining candidates now; later rounds replay from these results.  The decisions
        // (and work[0..1], the reference's own pairs) are unchanged; work[2..3] include the extras.
        lq.clear(); lt.clear(); lstate.clear(); ldest.clear();
        int64_t ncache = 0;
        for (size_t k = 0; k < np; k++) {
          lq.push_back(pq[k]); lt.push_back(pt[k]); lstate.push_back(pstate[k]); ldest.push_back(static_cast<int64_t>(k));
          if (k + 1 == np || pstate[k + 1] != pstate[k]) {
            size_t const si = static_cast<size_t>(pstate[k]);
            QState & S = st[si];
            int const first_extra = lazy ? S.gend : S.hit_count;
            int const strand = static_cast<int>(si / static_cast<size_t>(bn));
            int64_t const ql = static_cast<int64_t>(si % static_cast<size_t>(bn));
            int const sqlen = (strand == 0 ? queries->h_len[static_cast<size_t>(q0 + b0 + ql)] : rc_set->h_len[static_cast<size_t>(rc0 + ql)]);
            S.cache_first = first_extra; S.cache_off = static_cast<int>(ncache);
            for (int idx = first_extra; idx < S.ncand; idx++) {
              lq.push_back(pq[k]); lt.push_back(S.cs[idx]); lstate.push_back(pstate[k]); ldest.push_back(-(ncache + 1));
              al_cells += static_cast<int64_t>(sqlen) * db->h_len[static_cast<size_t>(S.cs[idx])];
              ncache++;
            }
          }
        }
        size_t const nl = lq.size();
        l_score.resize(nl); l_al.resize(nl); l_ma.resize(nl); l_mi.resize(nl); l_ga.resize(nl); l_tr.resize(nl * 4);
        size_t const nc = static_cast<size_t>(ncache);
        t_score.resize(nc); t_al.resize(nc); t_ma.resize(nc); t_mi.resize(nc); t_ga.resize(nc); t_tr.resize(nc * 4);
        int const r = device_align(nl, lq.data(), lt.data(), lstate.data(), l_score.data(), l_al.data(), l_ma.data(),
                                   l_mi.data(), l_ga.data(), l_tr.data(), nullptr);
        if (r != VSG_OK) { return r; }
        for (size_t k = 0; k < nl; k++) {
          if (ldest[k] >= 0) {
            size_t const d = static_cast<size_t>(ldest[k]);
            a_score[d] = l_score[k]; a_al[d] = l_al[k]; a_ma[d] = l_ma[k]; a_mi[d] = l_mi[k]; a_ga[d] = l_ga[k];
            for (int z = 0; z < 4; z++) { a_tr[4 * d + z] = l_tr[4 * k + z]; }
          } else {
            size_t const d = static_cast<size_t>(-ldest[k] - 1);
            t_score[d] = l_score[k]; t_al[d] = l_al[k]; t_ma[d] = l_ma[k]; t_mi[d] = l_mi[k]; t_ga[d] = l_ga[k];
            for (int z = 0; z < 4; z++) { t_tr[4 * d + z] = l_tr[4 * k + z]; }
          }
        }
        al_pairs += static_cast<int64_t>(nl);
        tail_mode = true;
      } else {
        gated_round = tb_gate && !lazy && plead.size() == np;
        int const r = device_align(np, pq.data(), pt.data(), pstate.data(), a_score.data(), a_al.data(), a_ma.data(),
                                   a_mi.data(), a_ga.data(), a_tr.data(), gated_round ? plead.data() : nullptr);
        if (r != VSG_OK) { return r; }
        al_pairs += static_cast<int64_t>(np);
      }
      if (!lazy) { total_pairs += static_cast<int64_t>(np); }
      t_align += ms(tp0, now()); tp0 = now();
      // replay: the second half of align_delayed (searchcore.cpp:780-880)
      size_t pi = 0;
      for (size_t si = 0; si < st.size(); si++) {
        QState & S = st[si];
        if (!S.waiting) { continue; }
        S.waiting = false;
        int64_t const ql = static_cast<int64_t>(si % static_cast<size_t>(bn));
        int const strand = static_cast<int>(si / static_cast<size_t>(bn));
        int const qlen = (strand == 0 ? queries->h_len[static_cast<size_t>(q0 + b0 + ql)] : rc_set->h_len[static_cast<size_t>(rc0 + ql)]);
        size_t i = pi;
        int const xlo = lazy ? S.gpos : S.finalized, xhi = lazy ? S.gend : S.hit_count;
        for (int x = xlo; x < xhi; x++) {
          Hit & h = hits[static_cast<size_t>(S.hit_base) + x];
          if (!h.rejected) {
            int64_t const cl = static_cast<int64_t>(qlen) * db->h_len[static_cast<size_t>(h.target)];
            if (!from_cache) { al_cells += cl; }
            if (!lazy) { total_cells += cl; }
          }
        }
        for (int x = xlo; x < xhi; x++) {
          if (S.rejects < maxrejects && S.accepts < maxaccepts) {
            Hit & h = hits[static_cast<size_t>(S.hit_base) + x];
            if (h.rejected) { S.rejects++; continue; }
            int64_t fb[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
            if (gated_round && plead[i] >= 0 && a_al[i] == 0xffffu && a_ma[i] == 0xffffu && a_mi[i] == 0xffffu) {
              // its walk was skipped because the device took the group's leader for accepted, yet the replay is here:
              // the two verdicts differ (a borderline identity); align this pair now
              const vsg_seqset * qset = strand == 0 ? queries : rc_set;
              int const r = vsg_align_pairs(c, qset, db, 1, &pq[i], &pt[i], &a_score[i], &a_al[i], &a_ma[i], &a_mi[i], &a_ga[i],
                                            &a_tr[4 * i], nullptr, 0, nullptr);
              if (r != VSG_OK) { return r; }
              tb_redone++;
            }
            bool const diverted = (a_score[i] == VSG_SCORE_SENTINEL);
            if (diverted) {
              // the reference's LinearMemoryAligner path (searchcore.cpp:806-832), host side of the boundary
              if (parent->fallback == nullptr ||
                  parent->fallback(parent->fallback_user, q0 + b0 + ql, strand, h.target, fb) != 0) {
                        Error::set("vsg_search_batch: a pair was deferred to the linear-memory aligner (core/linmemalign.cpp) "
                           "and no vsg_ctx_set_fallback callback resolved it");
                return VSG_EINVAL;
              }
            }
            int const dlen = db->h_len[static_cast<size_t>(h.target)];
            h.aligned = true;
            h.shortest = std::min(qlen, dlen);
            h.longest = std::max(qlen, dlen);
            int32_t trims4[4] = {a_tr[4 * i], a_tr[4 * i + 1], a_tr[4 * i + 2], a_tr[4 * i + 3]};
            int64_t nal = a_al[i], nma = a_ma[i], nmi = a_mi[i], nga = a_ga[i];
            h.nwscore = a_score[i];
            if (diverted) {
              h.nwscore = static_cast<int>(fb[0]); nal = fb[1]; nma = fb[2]; nmi = fb[3]; nga = fb[4];
              for (int z = 0; z < 4; z++) { trims4[z] = static_cast<int32_t>(fb[5 + z]); }
              h.forbidden_gap = fb[9] != 0;
            }
            h.nwalignmentlength = static_cast<int>(nal);
            h.nwdiff = static_cast<int>(nal - nma);
            h.nwgaps = static_cast<int>(nga);
            h.nwindels = static_cast<int>(nal - nma - nmi);
            h.matches = static_cast<int>(nal) - h.nwdiff;
            h.mismatches = h.nwdiff - h.nwindels;
            finish_hit(h, trims4, opts->iddef);
            int64_t const qsz = opts->query_sizes != nullptr ? opts->query_sizes[b0 + ql] : 1;
            int64_t const tsz = opts->target_sizes != nullptr ? opts->target_sizes[h.target] : 1;
            if (acceptable_aligned(h, opt_id, opt_weak_id, *opts, qlen, dlen, qsz, tsz)) { S.accepts++; } else { S.rejects++; }
            ++i;
          }
        }
        // the pairs of this state, examined or not, are consumed
        size_t mine = 0;
        while (pi + mine < np && static_cast<size_t>(pstate[pi + mine]) == si) { mine++; }
        pi += mine;
        if (lazy) { S.gpos = S.gend; }
        else { S.finalized = S.hit_count; S.delayed = 0; }
      }
      t_replay += ms(tp0, now());
    }

    tp0 = now();
    // search_joinhits + result records (search.cpp:466-488)
    for (int64_t q = 0; q < bn; q++) {
      joined.clear();
      for (int s = 0; s < nstrands; s++) {
        QState const & S = st[static_cast<size_t>(s) * bn + q];
        for (int x = 0; x < S.hit_count; x++) {
          Hit const & h = hits[static_cast<size_t>(S.hit_base) + x];
          if (h.accepted || h.weak) { joined.push_back(h); }
        }
      }
      std::stable_sort(joined.begin(), joined.end(), hit_less);
      int const n = static_cast<int>(std::min<int64_t>(static_cast<int64_t>(joined.size()), max_results));
      if (rows != nullptr) { rows[b0 + q].resize(static_cast<size_t>(n)); }
      for (int j = 0; j < n; j++) {
        Hit const & h = joined[static_cast<size_t>(j)];
        vsg_search_result & r = rows != nullptr ? rows[b0 + q][static_cast<size_t>(j)] : results[static_cast<size_t>(b0 + q) * max_results + j];
        r.target = h.target; r.matches = h.matches; r.mismatches = h.mismatches; r.gaps = h.nwgaps;
        r.alignment_length = h.nwalignmentlength;
        r.query_length = queries->h_len[static_cast<size_t>(q0 + b0 + q)];
        r.target_length = db->h_len[static_cast<size_t>(h.target)];
        r.accepted = h.accepted ? 1 : 0; r.strand = h.strand; r.nwscore = h.nwscore; r.id = h.id;
        r.internal_alignment_length = h.internal_alignmentlength; r.internal_gaps = h.internal_gaps;
      }
      counts[b0 + q] = n;
    }
    t_join += ms(tp0, now());
    return VSG_OK;
  };
  int pieces = 0;
  for (int64_t p0 = 0; p0 < sbn; pieces++) {
    // long lists: as many queries as fit the candidate budget (both strands), at least one
    int64_t p1 = sbn;
    if (long_lists) {
      int64_t vol = 0;
      for (p1 = p0; p1 < sbn; p1++) {
        int64_t v = 0;
        for (int s = 0; s < nstrands; s++) { v += all_K[static_cast<size_t>(s) * sbn + p1]; }
        if (p1 > p0 && vol + v > cand_budget) { break; }
        vol += v;
      }
    }
    int const r = run_piece(sb0 + p0, p1 - p0, p0);
    if (r != VSG_OK) { return r; }
    p0 = p1;
  }
  if (trace_pieces && long_lists) {
    std::fprintf(stderr, "[vsg trace] batch@%lld: %lld queries searched in %d pieces of at most %lld candidates\n",
                 static_cast<long long>(sb0), static_cast<long long>(sbn), pieces, static_cast<long long>(cand_budget));
  }
  if (trace) {
    std::fprintf(stderr, "[vsg trace] batch@%lld: rank %.1f init %.1f gather %.1f align %.1f replay %.1f join %.1f ms; done at %.1f ms; %lld skipped walks redone\n",
                 static_cast<long long>(sb0), t_rank, t_init, t_gather, t_align, t_replay, t_join, ms(t_call0, now()), static_cast<long long>(tb_redone));
  }
  return VSG_OK;
  };

  std::atomic<int64_t> next{0};
  std::vector<int> rcs(static_cast<size_t>(nthreads), VSG_OK);
  std::vector<std::string> msgs(static_cast<size_t>(nthreads));
  std::vector<int64_t> tp(static_cast<size_t>(nthreads), 0), tc(static_cast<size_t>(nthreads), 0), ap(static_cast<size_t>(nthreads), 0), ac(static_cast<size_t>(nthreads), 0);
  auto worker = [&](int t) {
    vsg_ctx * wc = c->children[static_cast<size_t>(t)];
    // Sub-batches are cut from a shared cursor.  A thread's FIRST one is shortened to (t+1)/nthreads of
    // the regular size: identical sub-batches started together run in lockstep (all threads rank, then
    // all gather on the host, then all align ...) and the device idles through every host phase;
    // staggered, some thread always has a kernel in flight.
    bool first = true;
    for (;;) {
      int64_t want = BATCH;
      if (first && stagger && nthreads > 1) { want = std::max<int64_t>(256, BATCH * (t + 1) / nthreads); }
      first = false;
      int64_t const b0 = next.fetch_add(want);
      if (b0 >= nq) { break; }
      int const r = run_batch(wc, b0, want, tp[static_cast<size_t>(t)], tc[static_cast<size_t>(t)], ap[static_cast<size_t>(t)], ac[static_cast<size_t>(t)]);
      if (r != VSG_OK) { rcs[static_cast<size_t>(t)] = r; msgs[static_cast<size_t>(t)] = vsg_last_error(); next.store(nq); break; }
    }
  };
  if (nthreads == 1) {
    worker(0);
  } else {
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; t++) { pool.emplace_back(worker, t); }
    for (auto & th : pool) { th.join(); }
  }
  for (int t = 0; t < nthreads; t++) {
    vsg_ctx * wc = c->children[static_cast<size_t>(t)];
    c->prof_cells += wc->prof_cells; c->prof_fast += wc->prof_fast; c->prof_exact += wc->prof_exact;
    c->prof_tb_skipped += wc->prof_tb_skipped;
    c->prof_fwd_launches += wc->prof_fwd_launches;
    c->prof_fwd_ms += wc->prof_fwd_ms; c->prof_tb_ms += wc->prof_tb_ms; c->prof_rank_ms += wc->prof_rank_ms;
    vsg_profile_reset(wc);
    total_pairs += tp[static_cast<size_t>(t)]; total_cells += tc[static_cast<size_t>(t)];
    aligned_pairs += ap[static_cast<size_t>(t)]; aligned_cells += ac[static_cast<size_t>(t)];
  }
  for (int t = 0; t < nthreads; t++) {
    if (rcs[static_cast<size_t>(t)] != VSG_OK) { Error::set(msgs[static_cast<size_t>(t)]); return rcs[static_cast<size_t>(t)]; }
  }
  if (work != nullptr) { work[0] = total_pairs; work[1] = total_cells; work[2] = aligned_pairs; work[3] = aligned_cells; }
  return VSG_OK;
}

extern "C" int vsg_search_batch(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * db,
                                const vsg_seqset * queries, int64_t q0, int64_t nq,
                                const vsg_search_opts * opts, vsg_search_result * results, int max_results,
                                int32_t * counts, int64_t * work)
{
  if (results == nullptr || max_results < 1) { Error::set("vsg_search_batch: bad argument"); return VSG_EINVAL; }
  return search_batch(c, ix, db, queries, q0, nq, opts, results, max_results, nullptr, counts, work);
}

int vsg::search_batch_rows(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * db, const vsg_seqset * queries, int64_t q0,
                           int64_t nq, const vsg_search_opts * opts, int64_t max_rows, std::vector<vsg_search_result> * rows,
                           int32_t * counts, int64_t * work)
{
  if (rows == nullptr || max_rows < 1) { Error::set("vsg_search_batch: bad argument"); return VSG_EINVAL; }
  return search_batch(c, ix, db, queries, q0, nq, opts, nullptr, max_rows, rows, counts, work);
}


// ---- all-against-all -----------------------------------------------------------------------------
extern "C" int vsg_allpairs_partition(const int32_t * len, int64_t n, int nparts, int64_t * bounds)
{
  if (n < 0 || nparts < 1 || bounds == nullptr || (n > 0 && len == nullptr)) { Error::set("vsg_allpairs_partition: bad argument"); return VSG_EINVAL; }
  // cells(i) = len[i] * sum_{j>i} len[j]
  std::vector<double> row(static_cast<size_t>(n));
  double suffix = 0.0, total = 0.0;
  for (int64_t i = n - 1; i >= 0; i--) { row[static_cast<size_t>(i)] = static_cast<double>(len[i]) * suffix; suffix += len[i]; total += row[static_cast<size_t>(i)]; }
  bounds[0] = 0;
  double acc = 0.0;
  int p = 1;
  for (int64_t i = 0; i < n && p < nparts; i++) {
    acc += row[static_cast<size_t>(i)];
    while (p < nparts && acc >= total * p / nparts) { bounds[p++] = i + 1; }
  }
  while (p <= nparts) { bounds[p++] = n; }
  return VSG_OK;
}

extern "C" int vsg_allpairs(vsg_ctx * c, const vsg_seqset * set, int64_t row0, int64_t nrows,
                            const vsg_search_opts * opts, vsg_pair_hit * hits, int64_t cap, int64_t * nhits,
                            int64_t * work)
{
  if (c == nullptr || set == nullptr || opts == nullptr || nhits == nullptr || (cap > 0 && hits == nullptr)) {
    Error::set("vsg_allpairs: bad argument");
    return VSG_EINVAL;
  }
  int64_t const n = set->d.n;
  if (row0 < 0 || nrows < 0 || row0 + nrows > n) { Error::set("vsg_allpairs: row range out of bounds"); return VSG_EINVAL; }
  if (opts->iddef < 0 || opts->iddef > 4) { Error::set("vsg_allpairs: iddef must be 0..4"); return VSG_EINVAL; }
  double const opt_id = opts->id;
  double const opt_weak_id = (opts->id >= 0.0 && opts->weak_id > opts->id) ? opts->id : opts->weak_id;
  *nhits = 0;

  // blocks of consecutive rows with about PAIRS_PER_BLOCK pairs each, handed to host threads that own
  // a child context each; every block writes its hits to a private vector, concatenated in row order
  int64_t const PAIRS_PER_BLOCK = 1 << 20;
  std::vector<int64_t> block_first;
  {
    int64_t acc = 0;
    block_first.push_back(row0);
    for (int64_t i = row0; i < row0 + nrows; i++) {
      acc += n - i - 1;
      if (acc >= PAIRS_PER_BLOCK && i + 1 < row0 + nrows) { block_first.push_back(i + 1); acc = 0; }
    }
    block_first.push_back(row0 + nrows);
  }
  int64_t const nblocks = static_cast<int64_t>(block_first.size()) - 1;
  int nthreads = 8;
  if (const char * e = std::getenv("VSG_HOST_THREADS")) { nthreads = std::max(1, std::atoi(e)); }
  nthreads = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(nthreads, nblocks)));
  while (static_cast<int>(c->children.size()) < nthreads) {
    vsg_ctx * ch = nullptr;
    int const r = vsg_ctx_create(c->device, &c->scoring, &ch);
    if (r != VSG_OK) { return r; }
    c->children.push_back(ch);
  }
  for (int t = 0; t < nthreads; t++) {
    c->children[static_cast<size_t>(t)]->dir_budget = std::max<size_t>(c->dir_budget / static_cast<size_t>(nthreads), static_cast<size_t>(1) << 30);
    c->children[static_cast<size_t>(t)]->fast_disabled = c->fast_disabled;
    c->children[static_cast<size_t>(t)]->ckpt_enabled = c->ckpt_enabled;
  }
  std::vector<std::vector<vsg_pair_hit>> out(static_cast<size_t>(nblocks));
  std::vector<int64_t> bpairs(static_cast<size_t>(nblocks), 0), bcells(static_cast<size_t>(nblocks), 0);

  auto run_block = [&](vsg_ctx * wc, int64_t bi) -> int {
    int64_t const r0 = block_first[static_cast<size_t>(bi)], r1 = block_first[static_cast<size_t>(bi) + 1];
    std::vector<uint32_t> pq, pt;
    int64_t cells = 0;
    {
      int64_t cap_pairs = 0;
      for (int64_t i = r0; i < r1; i++) { cap_pairs += n - i - 1; }
      pq.reserve(static_cast<size_t>(cap_pairs)); pt.reserve(static_cast<size_t>(cap_pairs));
    }
    for (int64_t i = r0; i < r1; i++) {
      int const ql = set->h_len[static_cast<size_t>(i)];
      int64_t tl = 0;
      for (int64_t j = i + 1; j < n; j++) {
        int const dl = set->h_len[static_cast<size_t>(j)];
        if (!acceptable_unaligned(*opts, ql, dl, 1, 1, false, 0u)) { continue; }  // allpairs_global.cpp:407-414 (defaults for the rest)
        pq.push_back(static_cast<uint32_t>(i)); pt.push_back(static_cast<uint32_t>(j)); tl += dl;
      }
      cells += static_cast<int64_t>(ql) * tl;
    }
    int64_t const np = static_cast<int64_t>(pq.size());
    if (np == 0) { return VSG_OK; }
    int64_t k = 0;
    std::vector<int16_t> sc(static_cast<size_t>(np));
    std::vector<uint16_t> al(static_cast<size_t>(np)), ma(static_cast<size_t>(np)), mi(static_cast<size_t>(np)), ga(static_cast<size_t>(np));
    std::vector<int32_t> tr(static_cast<size_t>(np) * 4);
    int const r = vsg_align_pairs(wc, set, set, np, pq.data(), pt.data(), sc.data(), al.data(), ma.data(), mi.data(), ga.data(),
                                  tr.data(), nullptr, 0, nullptr);
    if (r != VSG_OK) { return r; }
    std::vector<vsg_pair_hit> & o = out[static_cast<size_t>(bi)];
    k = 0;
    while (k < np) {
      int64_t const i = pq[static_cast<size_t>(k)];
      size_t const first = o.size();
      int const qlen = set->h_len[static_cast<size_t>(i)];
      for (; k < np && pq[static_cast<size_t>(k)] == i; k++) {
        int64_t const j = pt[static_cast<size_t>(k)];
        int64_t fb[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        bool const diverted = (sc[static_cast<size_t>(k)] == VSG_SCORE_SENTINEL);
        if (diverted && (c->fallback == nullptr || c->fallback(c->fallback_user, i, 0, j, fb) != 0)) {
          Error::set("vsg_allpairs: a pair was deferred to the linear-memory aligner (core/linmemalign.cpp) "
                     "and no vsg_ctx_set_fallback callback resolved it");
          return VSG_EINVAL;
        }
        Hit h;
        std::memset(&h, 0, sizeof h);
        int const dlen = set->h_len[static_cast<size_t>(j)];
        h.target = static_cast<int>(j); h.aligned = true;
        h.shortest = std::min(qlen, dlen); h.longest = std::max(qlen, dlen);
        int32_t trims4[4] = {tr[4 * static_cast<size_t>(k)], tr[4 * static_cast<size_t>(k) + 1], tr[4 * static_cast<size_t>(k) + 2], tr[4 * static_cast<size_t>(k) + 3]};
        int64_t nal = al[static_cast<size_t>(k)], nma = ma[static_cast<size_t>(k)], nmi = mi[static_cast<size_t>(k)], nga = ga[static_cast<size_t>(k)];
        h.nwscore = sc[static_cast<size_t>(k)];
        if (diverted) {
          h.nwscore = static_cast<int>(fb[0]); nal = fb[1]; nma = fb[2]; nmi = fb[3]; nga = fb[4];
          for (int z = 0; z < 4; z++) { trims4[z] = static_cast<int32_t>(fb[5 + z]); }
          h.forbidden_gap = fb[9] != 0;
        }
        h.nwalignmentlength = static_cast<int>(nal);
        h.nwdiff = static_cast<int>(nal - nma);
        h.nwgaps = static_cast<int>(nga);
        h.nwindels = static_cast<int>(nal - nma - nmi);
        h.matches = static_cast<int>(nal) - h.nwdiff;
        h.mismatches = h.nwdiff - h.nwindels;
        finish_hit(h, trims4, opts->iddef);
        if (acceptable_aligned(h, opt_id, opt_weak_id, *opts, qlen, dlen)) {
          vsg_pair_hit ph;
          ph.query = static_cast<int32_t>(i); ph.target = h.target; ph.matches = h.matches; ph.mismatches = h.mismatches;
          ph.gaps = h.nwgaps; ph.alignment_length = h.nwalignmentlength; ph.nwscore = h.nwscore;
          ph.internal_alignment_length = h.internal_alignmentlength; ph.id = h.id;
          o.push_back(ph);
        }
      }
      std::sort(o.begin() + static_cast<std::ptrdiff_t>(first), o.end(), [](const vsg_pair_hit & a, const vsg_pair_hit & b) {
        if (a.id != b.id) { return a.id > b.id; }
        return a.target < b.target;
      });
    }
    bpairs[static_cast<size_t>(bi)] = np; bcells[static_cast<size_t>(bi)] = cells;
    return VSG_OK;
  };

  std::atomic<int64_t> next{0};
  std::vector<int> rcs(static_cast<size_t>(nthreads), VSG_OK);
  std::vector<std::string> msgs(static_cast<size_t>(nthreads));
  auto worker = [&](int t) {
    vsg_ctx * wc = c->children[static_cast<size_t>(t)];
    cudaSetDevice(wc->device);
    for (;;) {
      int64_t const bi = next.fetch_add(1);
      if (bi >= nblocks) { break; }
      int const r = run_block(wc, bi);
      if (r != VSG_OK) { rcs[static_cast<size_t>(t)] = r; msgs[static_cast<size_t>(t)] = vsg_last_error(); next.store(nblocks); break; }
    }
  };
  if (nthreads == 1) { worker(0); }
  else {
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; t++) { pool.emplace_back(worker, t); }
    for (auto & th : pool) { th.join(); }
  }
  for (int t = 0; t < nthreads; t++) {
    vsg_ctx * wc = c->children[static_cast<size_t>(t)];
    c->prof_cells += wc->prof_cells; c->prof_fast += wc->prof_fast; c->prof_exact += wc->prof_exact;
    c->prof_tb_skipped += wc->prof_tb_skipped;
    c->prof_fwd_launches += wc->prof_fwd_launches;
    c->prof_fwd_ms += wc->prof_fwd_ms; c->prof_tb_ms += wc->prof_tb_ms; c->prof_rank_ms += wc->prof_rank_ms;
    vsg_profile_reset(wc);
    if (rcs[static_cast<size_t>(t)] != VSG_OK) { Error::set(msgs[static_cast<size_t>(t)]); return rcs[static_cast<size_t>(t)]; }
  }
  int64_t total = 0, tp = 0, tc = 0;
  for (int64_t bi = 0; bi < nblocks; bi++) { total += static_cast<int64_t>(out[static_cast<size_t>(bi)].size()); tp += bpairs[static_cast<size_t>(bi)]; tc += bcells[static_cast<size_t>(bi)]; }
  *nhits = total;
  if (work != nullptr) { work[0] = tp; work[1] = tc; }
  if (total > cap) { Error::set("vsg_allpairs: hit buffer too small"); return VSG_ECAP; }
  int64_t pos = 0;
  for (int64_t bi = 0; bi < nblocks; bi++) {
    auto const & o = out[static_cast<size_t>(bi)];
    if (!o.empty()) { std::memcpy(hits + pos, o.data(), sizeof(vsg_pair_hit) * o.size()); pos += static_cast<int64_t>(o.size()); }
  }
  return VSG_OK;
}
