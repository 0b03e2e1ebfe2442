// cluster.cu — the greedy centroid clustering driver of --cluster_fast on the device aligner and ranker.
//
// Replaces cluster_core_parallel / cluster_core_serial (reference core/cluster.cpp:877-1115) together with
// cluster_query_core (:162-189), evaluate_extra_hits (:601-856) and Dbindex::add_sequence
// (core/dbindex.cpp:121-148): sequences are taken in the caller's order (the reference sorts by length first,
// core/db.cpp:433-449) in ROUNDS of `round_size` consecutive sequences — the reference's --threads, which its
// results depend on (cluster.cpp:881-882).  Every round
//   1. ranks its queries against the centroids indexed so far (incremental device index, rank.cu) and runs
//      search_onequery's candidate loop for all of them in lock step, aligning the groups of <= 8 candidates the
//      reference hands to search16 in batched device calls (core/searchcore.cpp:884-957, 740-881);
//   2. walks the queries in order as the reference's serial pass does: centroids created EARLIER IN THE SAME
//      ROUND are inserted into a query's hit list by shared k-mer count and the list is re-evaluated
//      (evaluate_extra_hits), the best accepted hit decides (search_findbest2_byid, searchcore.cpp:960-991):
//      member of that centroid's cluster, or a new centroid, which is appended to the device index.
// Assignments, identities and alignment statistics are those of `vsearch --cluster_fast --threads round_size`.
//
// --strand both: every sequence is searched twice, as itself and as the reverse complement of the (already masked)
// sequence as stored, which is not masked again (cluster.cpp:162-189).  The session builds a MIRROR of the set once,
// in which entry 2i is sequence i and entry 2i+1 its reverse complement, so the 2 x round_size searches of a round are
// one contiguous query range: one ranking launch, one aligner call per lock-step iteration and one speculative batch
// cover both strands.  Each (sequence, strand) keeps its own hit list and counters; the serial pass runs
// evaluate_extra_hits for the plus and then the minus strand against the PLUS k-mers of the round's new centroids, and
// the best hit is taken over the plus hits, then the minus hits, ties to plus (search_findbest2_*).
#include "vsg_internal.h"
#include "hit_logic.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

namespace vsg {
struct CIndex;
int cindex_create(vsg_ctx * c, const vsg_seqset * set, int wordlength, int mask_lower, CIndex ** out);
void cindex_destroy(CIndex * ix);
int cindex_append(vsg_ctx * c, CIndex * ix, const uint32_t * seqnos, int n);
int seqset_strand_pairs(vsg_ctx * c, const vsg_seqset * src, vsg_seqset ** out);
int cindex_rank_enqueue(vsg_ctx * c, CIndex * ix, const vsg_seqset * queries, int64_t q0, int64_t nq, int minwordmatches,
                        int tophits, uint32_t ** d_seqno, uint32_t ** d_count, int32_t ** d_n, int32_t ** d_status);
const std::vector<uint32_t> & cindex_seqnos(const CIndex * ix);
}  // namespace vsg

using namespace vsg;

namespace {

struct CQuery {   // one searchinfo_s of the round: one sequence on one strand
  int seqno = 0, qlen = 0;
  int strand = 0;
  uint32_t qidx = 0;               // the query's entry in the session's query set (the mirror with --strand both)
  int ncand = 0, next = 0;
  const uint32_t * cs = nullptr;   // dense target numbers, best first
  const uint32_t * cc = nullptr;
  std::vector<Hit> hits;
  int accepts = 0, rejects = 0, finalized = 0, delayed = 0;
  bool done = false, waiting = false;
  std::vector<uint32_t> kmers;     // distinct unmasked k-mers (filled when an extra hit needs them)
  bool have_kmers = false;
  std::vector<uint64_t> bitmap;    // the same set as a 4^k-bit map (built when the query becomes a candidate centroid)
  bool have_bitmap = false;
};

// unique_count (core/unique.cpp:155-240): the distinct k-mers of the windows that hold no masked symbol.
// `stamp` (4^k words) de-duplicates without being cleared: a k-mer is new iff its stamp differs from `tag`.
void distinct_kmers(const uint8_t * sym, int len, int k, int mask_lower, std::vector<uint32_t> & stamp, uint32_t tag,
                    std::vector<uint32_t> & out)
{
  out.clear();
  uint32_t const mask = k < 16 ? ((1u << (2 * k)) - 1u) : 0xffffffffu;
  uint32_t v = 0;
  int good = 0;
  for (int i = 0; i < len; i++) {
    int const s = sym[i], c = s & 15;
    bool const single = (c == 1) | (c == 2) | (c == 4) | (c == 8);
    bool const bad = !single || (mask_lower && (s & 16));
    v = ((v << 2) | (c == 2 ? 1u : c == 4 ? 2u : c == 8 ? 3u : 0u)) & mask;
    good = bad ? 0 : good + 1;
    if (good >= k && stamp[v] != tag) { stamp[v] = tag; out.push_back(v); }
  }
}

// unique_count_shared (core/unique.cpp): how many of a's distinct k-mers are in the set `bm`
unsigned shared_count(const std::vector<uint32_t> & a, const std::vector<uint64_t> & bm)
{
  unsigned n = 0;
  for (uint32_t v : a) { n += static_cast<unsigned>((bm[v >> 6] >> (v & 63)) & 1u); }
  return n;
}

}  // namespace

struct vsg_cluster_session {
  vsg_ctx * c = nullptr;
  const vsg_seqset * set = nullptr;
  vsg_seqset * mirror = nullptr;                   // --strand both: entry 2i = sequence i, 2i+1 = its reverse complement
  const vsg_seqset * qset = nullptr;               // what the queries are read from: `mirror`, or `set` itself
  int nstr = 1;                                    // strands searched per sequence (entries per sequence in qset)
  vsg_search_opts opts;
  int64_t seqcount = 0, maxaccepts = 0, maxrejects = 0;
  int tophits = 0, k = 0, minwordmatches = 0, hit_capacity = 0;
  double opt_id = 0, opt_weak_id = 0;
  vsg::CIndex * ix = nullptr;                      // the centroids indexed so far
  int64_t total_pairs = 0, total_cells = 0, clusters = 0;
  int64_t next = 0;                                // first sequence not assigned yet
  std::vector<int32_t> cluster_of;                 // sequence -> cluster number (-1: not assigned yet)
  std::vector<uint32_t> stamp;                     // distinct_kmers' scratch
  uint32_t stamp_tag = 0;
  ~vsg_cluster_session()
  {
    if (ix != nullptr) { cindex_destroy(ix); }
    vsg_seqset_destroy(mirror);
  }
};

namespace {

// option checks and the clamps of cluster() (core/cluster.cpp:1213-1232); creates the (empty) incremental index
int session_setup(vsg_ctx * c, const vsg_seqset * set, const vsg_search_opts * opts, vsg_cluster_session & s)
{
  if (opts->idprefix != 0 || opts->idsuffix != 0 || opts->selfid != 0) { Error::set("vsg_cluster_fast: idprefix/idsuffix/selfid are not offered on this path"); return VSG_EINVAL; }
  if (opts->iddef < 0 || opts->iddef > 4) { Error::set("vsg_cluster_fast: iddef must be 0..4"); return VSG_EINVAL; }
  if (opts->self != 0 && opts->target_labels == nullptr) { Error::set("vsg_cluster_fast: --self needs target_labels (one per sequence)"); return VSG_EINVAL; }
  VSG_CUDA_OK(cudaSetDevice(c->device));
  int64_t const seqcount = set->d.n;
  if (seqcount > 0x7fffffff) { Error::set("vsg_cluster_fast: too many sequences"); return VSG_EINVAL; }
  // the clamps of cluster() (core/cluster.cpp:1213-1232)
  int64_t maxaccepts = opts->maxaccepts, maxrejects = opts->maxrejects < 0 ? 32 : opts->maxrejects;
  if (maxaccepts < 0) { Error::set("vsg_cluster_fast: maxaccepts must not be negative"); return VSG_EINVAL; }
  if (maxrejects == 0 || maxrejects > seqcount) { maxrejects = seqcount; }
  if (maxaccepts == 0 || maxaccepts > seqcount) { maxaccepts = seqcount; }
  int64_t const tophits64 = std::min<int64_t>(maxrejects + maxaccepts + MAXDELAYED, seqcount);
  if (tophits64 > 1024) { Error::set("vsg_cluster_fast: maxaccepts+maxrejects+8 > 1024 is not supported on the device ranker"); return VSG_EINVAL; }
  int const tophits = static_cast<int>(tophits64);
  int const k = opts->wordlength;
  if (k < 3 || k > 10) { Error::set("vsg_cluster_fast: the device index supports --wordlength 3..10"); return VSG_EINVAL; }
  int const minwordmatches = opts->minwordmatches < 0 ? minwordmatches_defaults[k] : opts->minwordmatches;
  double const opt_id = opts->id;
  double const opt_weak_id = (opts->id >= 0.0 && opts->weak_id > opts->id) ? opts->id : opts->weak_id;
  int const hit_capacity = static_cast<int>(std::min<int64_t>(maxaccepts + maxrejects - 1, tophits));   // cluster.cpp:616-618

  s.c = c; s.set = set; s.opts = *opts;
  s.seqcount = seqcount; s.maxaccepts = maxaccepts; s.maxrejects = maxrejects;
  s.tophits = tophits; s.k = k; s.minwordmatches = minwordmatches; s.hit_capacity = hit_capacity;
  s.opt_id = opt_id; s.opt_weak_id = opt_weak_id;
  s.cluster_of.assign(static_cast<size_t>(seqcount), -1);
  s.stamp.assign(static_cast<size_t>(1) << (2 * k), 0u);
  s.qset = set; s.nstr = 1;
  if (seqcount == 0) { return VSG_OK; }
  if (opts->strand_both != 0) {
    if (2 * seqcount > 0xffffffffLL) { Error::set("vsg_cluster_fast: too many sequences for --strand both"); return VSG_EINVAL; }
    int const rc = seqset_strand_pairs(c, set, &s.mirror);
    if (rc != VSG_OK) { return rc; }
    s.qset = s.mirror; s.nstr = 2;
  }
  return cindex_create(c, set, k, opts->mask_lower, &s.ix);
}

// cluster_core_parallel's rounds (core/cluster.cpp:877-1115) over the sequences [start, start + count); results[i] belongs
// to sequence start + i.  State that outlives the call (index, cluster numbers) lives in the session.
int session_rounds(vsg_cluster_session & s, int64_t const start, int64_t const count, int const round_size, vsg_cluster_result * results)
{
  vsg_ctx * const c = s.c;
  const vsg_seqset * const set = s.set;
  const vsg_seqset * const qset = s.qset;
  int const ns = s.nstr;
  const vsg_search_opts * const opts = &s.opts;
  int64_t const maxaccepts = s.maxaccepts, maxrejects = s.maxrejects;
  int const tophits = s.tophits, k = s.k, minwordmatches = s.minwordmatches, hit_capacity = s.hit_capacity;
  double const opt_id = s.opt_id, opt_weak_id = s.opt_weak_id;
  CIndex * const ix = s.ix;
  int64_t & total_pairs = s.total_pairs; int64_t & total_cells = s.total_cells; int64_t & clusters = s.clusters;
  std::vector<int32_t> & cluster_of = s.cluster_of;
  std::vector<uint32_t> & stamp = s.stamp;
  uint32_t & stamp_tag = s.stamp_tag;
  int rc = VSG_OK;
  auto size_of = [&](int seqno) -> int64_t { return opts->target_sizes != nullptr ? opts->target_sizes[seqno] : 1; };
  auto unaligned_ok = [&](int q, int qlen, int target) -> bool {
    bool const same_label = opts->self != 0 && opts->target_labels[q] == opts->target_labels[target];
    return acceptable_unaligned(*opts, qlen, set->h_len[static_cast<size_t>(target)], size_of(q), size_of(target), same_label, 0u);
  };

  std::vector<CQuery> rq(static_cast<size_t>(round_size) * ns);   // state u = (round-local sequence) * ns + strand
  std::vector<uint32_t> h_seqno, h_count;
  std::vector<int32_t> h_n;
  std::vector<uint32_t> pq, pt;
  std::vector<int> powner, px;
  std::vector<int16_t> a_score; std::vector<uint16_t> a_al, a_ma, a_mi, a_ga; std::vector<int32_t> a_tr;
  std::vector<uint8_t> round_sym;
  std::vector<uint32_t> new_centroids;
  const std::vector<uint32_t> & dense_to_seqno = cindex_seqnos(ix);

  // the statistics search16 returned for one (query, target) -> struct hit (searchcore.cpp:842-857 / cluster.cpp:786-809)
  auto fill_hit = [&](Hit & h, int qlen, int16_t sc, uint16_t al, uint16_t ma, uint16_t mi, uint16_t ga, const int32_t * tr,
                      int query, int strand, int & rcode) {
    int64_t fb[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    int32_t trims4[4] = {tr[0], tr[1], tr[2], tr[3]};
    int64_t nal = al, nma = ma, nmi = mi, nga = ga;
    h.nwscore = sc;
    if (sc == VSG_SCORE_SENTINEL) {   // the reference's LinearMemoryAligner path, host side of the boundary
      if (c->fallback == nullptr || c->fallback(c->fallback_user, query, strand, h.target, fb) != 0) {
        Error::set("vsg_cluster_fast: a pair was deferred to the linear-memory aligner (core/linmemalign.cpp) and no "
                   "vsg_ctx_set_fallback callback resolved it");
        rcode = VSG_EINVAL;
        return;
      }
      h.nwscore = static_cast<int>(fb[0]); nal = fb[1]; nma = fb[2]; nmi = fb[3]; nga = fb[4];
      for (int z = 0; z < 4; z++) { trims4[z] = static_cast<int32_t>(fb[5 + z]); }
      h.forbidden_gap = fb[9] != 0;
    }
    int const dlen = set->h_len[static_cast<size_t>(h.target)];
    h.aligned = true;
    h.shortest = std::min(qlen, dlen);
    h.longest = std::max(qlen, dlen);
    h.nwalignmentlength = static_cast<int>(nal);
    h.nwdiff = static_cast<int>(nal - nma);
    h.nwgaps = static_cast<int>(nga);
    h.nwindels = static_cast<int>(nal - nma - nmi);
    h.matches = static_cast<int>(nal) - h.nwdiff;
    h.mismatches = h.nwdiff - h.nwindels;
    finish_hit(h, trims4, opts->iddef);
  };

  static const bool trace = std::getenv("VSG_TRACE") != nullptr;
  auto now = []() { return std::chrono::steady_clock::now(); };
  auto ms_since = [](std::chrono::steady_clock::time_point a) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count(); };
  double t_rank = 0, t_groups = 0, t_spec = 0, t_serial = 0, t_append = 0;
  for (int64_t round0 = start; round0 < start + count; round0 += round_size) {
    int const nqr = static_cast<int>(std::min<int64_t>(round_size, start + count - round0));
    int const nu = nqr * ns;   // searches of the round: the round's sequences on every strand, in qset order
    auto tp = now();
    // ---- 1a. candidate ranking of the whole round (both strands) against the centroids indexed so far ----
    size_t const cells = static_cast<size_t>(nu) * tophits;
    h_seqno.resize(cells); h_count.resize(cells); h_n.resize(static_cast<size_t>(nu));
    {
      uint32_t *d_seqno, *d_count; int32_t *d_n, *d_status;
      if ((rc = cindex_rank_enqueue(c, ix, qset, round0 * ns, nu, minwordmatches, tophits, &d_seqno, &d_count, &d_n, &d_status)) != VSG_OK) { return rc; }
      int32_t status = 0;
      VSG_CUDA_OK(cudaMemcpyAsync(h_seqno.data(), d_seqno, sizeof(uint32_t) * cells, cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaMemcpyAsync(h_count.data(), d_count, sizeof(uint32_t) * cells, cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaMemcpyAsync(h_n.data(), d_n, sizeof(int32_t) * nu, cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaMemcpyAsync(&status, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
      if (status != 0) { Error::set("vsg_cluster_fast: a sequence is longer than the device ranker supports (65 534 + wordlength nt)"); return VSG_EINVAL; }
    }
    t_rank += ms_since(tp); tp = now();
    for (int u = 0; u < nu; u++) {
      CQuery & S = rq[static_cast<size_t>(u)];
      S.seqno = static_cast<int>(round0 + u / ns);
      S.strand = u % ns;
      S.qidx = static_cast<uint32_t>(round0 * ns + u);
      S.qlen = set->h_len[static_cast<size_t>(S.seqno)];
      S.ncand = h_n[static_cast<size_t>(u)]; S.next = 0;
      S.cs = h_seqno.data() + static_cast<size_t>(u) * tophits;
      S.cc = h_count.data() + static_cast<size_t>(u) * tophits;
      S.hits.clear();
      S.accepts = S.rejects = S.finalized = S.delayed = 0;
      S.done = false; S.waiting = false; S.have_kmers = false; S.have_bitmap = false;
    }
    // ---- 1b. search_onequery for every query and strand of the round, in lock step (searchcore.cpp:915-954) ----
    bool any = true;
    while (any) {
      any = false;
      pq.clear(); pt.clear(); powner.clear(); px.clear();
      for (int i = 0; i < nu; i++) {
        CQuery & S = rq[static_cast<size_t>(i)];
        if (S.done) { continue; }
        bool trigger = false;
        while ((S.finalized + S.delayed < maxaccepts + maxrejects - 1) && (S.rejects < maxrejects) &&
               (S.accepts < maxaccepts) && (S.next < S.ncand)) {
          Hit h;
          std::memset(&h, 0, sizeof(Hit));
          h.target = static_cast<int>(dense_to_seqno[S.cs[S.next]]); h.count = S.cc[S.next]; h.strand = S.strand;
          S.next++;
          if (unaligned_ok(S.seqno, S.qlen, h.target)) { S.delayed++; } else { h.rejected = true; }
          S.hits.push_back(h);
          if (S.delayed == MAXDELAYED) { trigger = true; break; }
        }
        if (!trigger && S.delayed == 0) { S.done = true; continue; }
        for (int x = S.finalized; x < static_cast<int>(S.hits.size()); x++) {   // align_delayed's search16 call
          if (!S.hits[static_cast<size_t>(x)].rejected) {
            pq.push_back(S.qidx); pt.push_back(static_cast<uint32_t>(S.hits[static_cast<size_t>(x)].target));
            powner.push_back(i); px.push_back(x);
          }
        }
        S.waiting = true;
        any = true;
      }
      if (!any) { break; }
      size_t const np = pq.size();
      a_score.resize(np); a_al.resize(np); a_ma.resize(np); a_mi.resize(np); a_ga.resize(np); a_tr.resize(np * 4);
      if (np > 0) {
        rc = vsg_align_pairs(c, qset, set, static_cast<int64_t>(np), pq.data(), pt.data(), a_score.data(), a_al.data(), a_ma.data(),
                             a_mi.data(), a_ga.data(), a_tr.data(), nullptr, 0, nullptr);
        if (rc != VSG_OK) { return rc; }
      }
      total_pairs += static_cast<int64_t>(np);
      for (size_t p = 0; p < np; p++) { total_cells += static_cast<int64_t>(qset->h_len[pq[p]]) * set->h_len[pt[p]]; }
      size_t pi = 0;
      for (int i = 0; i < nu; i++) {   // the second half of align_delayed (searchcore.cpp:780-880)
        CQuery & S = rq[static_cast<size_t>(i)];
        if (!S.waiting) { continue; }
        S.waiting = false;
        size_t a = pi;
        for (int x = S.finalized; x < static_cast<int>(S.hits.size()); x++) {
          if (S.rejects < maxrejects && S.accepts < maxaccepts) {
            Hit & h = S.hits[static_cast<size_t>(x)];
            if (h.rejected) { S.rejects++; continue; }
            int rcode = VSG_OK;
            fill_hit(h, S.qlen, a_score[a], a_al[a], a_ma[a], a_mi[a], a_ga[a], a_tr.data() + 4 * a, S.seqno, S.strand, rcode);
            if (rcode != VSG_OK) { return rcode; }
            if (acceptable_aligned(h, opt_id, opt_weak_id, *opts, S.qlen, set->h_len[static_cast<size_t>(h.target)], size_of(S.seqno), size_of(h.target))) { S.accepts++; } else { S.rejects++; }
            ++a;
          }
        }
        while (pi < np && powner[pi] == i) { pi++; }
        S.finalized = static_cast<int>(S.hits.size()); S.delayed = 0;
      }
    }
    t_groups += ms_since(tp); tp = now();
    // ---- 2. the serial pass (cluster.cpp:946-1025) ----
    new_centroids.clear();
    bool have_sym = false;
    std::vector<int64_t> sym_off;
    // u: a state of the round (sequence * ns + strand); the symbols are those of its qset entry, so a minus strand's
    // k-mers are those of the reverse complement, with the plus strand's masked windows mirrored
    auto need_kmers = [&](int u) -> int {
      CQuery & S = rq[static_cast<size_t>(u)];
      if (S.have_kmers) { return VSG_OK; }
      if (!have_sym) {
        // one download of the round's symbols (one copy when the sequences lie back to back, as they do for a packed set)
        int64_t const e0 = round0 * ns;
        sym_off.assign(static_cast<size_t>(nu) + 1, 0);
        bool contiguous = true;
        for (int z = 0; z < nu; z++) {
          size_t const sq = static_cast<size_t>(e0 + z);
          sym_off[static_cast<size_t>(z) + 1] = sym_off[static_cast<size_t>(z)] + qset->h_len[sq];
          if (z + 1 < nu && qset->h_off[sq + 1] != qset->h_off[sq] + qset->h_len[sq]) { contiguous = false; }
        }
        round_sym.resize(static_cast<size_t>(sym_off[static_cast<size_t>(nu)]) + 1);
        if (contiguous) {
          if (sym_off[static_cast<size_t>(nu)] > 0) {
            VSG_CUDA_OK(cudaMemcpyAsync(round_sym.data(), qset->d.sym + qset->h_off[static_cast<size_t>(e0)], static_cast<size_t>(sym_off[static_cast<size_t>(nu)]), cudaMemcpyDeviceToHost, c->stream));
          }
        } else {
          for (int z = 0; z < nu; z++) {
            int const l = qset->h_len[static_cast<size_t>(e0 + z)];
            if (l > 0) { VSG_CUDA_OK(cudaMemcpyAsync(round_sym.data() + sym_off[static_cast<size_t>(z)], qset->d.sym + qset->h_off[static_cast<size_t>(e0 + z)], static_cast<size_t>(l), cudaMemcpyDeviceToHost, c->stream)); }
          }
        }
        VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
        have_sym = true;
      }
      if (++stamp_tag == 0) { std::fill(stamp.begin(), stamp.end(), 0u); stamp_tag = 1; }
      distinct_kmers(round_sym.data() + sym_off[static_cast<size_t>(u)], S.qlen, k, opts->mask_lower, stamp, stamp_tag, S.kmers);
      S.have_kmers = true;
      return VSG_OK;
    };
    auto need_bitmap = [&](int j) -> int {   // j: a sequence of the round; its plus strand
      CQuery & C = rq[static_cast<size_t>(j) * ns];
      if (C.have_bitmap) { return VSG_OK; }
      int const r = need_kmers(j * ns);
      if (r != VSG_OK) { return r; }
      C.bitmap.assign(((static_cast<size_t>(1) << (2 * k)) + 63) / 64, 0);
      for (uint32_t v : C.kmers) { C.bitmap[v >> 6] |= static_cast<uint64_t>(1) << (v & 63); }
      C.have_bitmap = true;
      return VSG_OK;
    };
    // Speculative batch for the serial pass: a query without an accepted hit MAY found a cluster; every later
    // query of the round that shares enough k-mers with it MAY then have to be aligned against it
    // (evaluate_extra_hits aligns such pairs one at a time, cluster.cpp:741-752).  All those pairs go to the
    // device in one call; the serial pass below takes its alignments from here and falls back to a single-pair
    // call for anything not foreseen.  Decisions are unaffected; only alignments nobody asks for are extra work.
    struct Spec { int16_t sc; uint16_t al, ma, mi, ga; int32_t tr[4]; };
    std::vector<std::pair<uint64_t, Spec>> spec;   // key = (u << 32) | j: state u (sequence and strand) against sequence j, sorted
    {
      std::vector<int> maybe;
      for (int i = 0; i < nqr; i++) {
        int acc = 0;
        for (int st = 0; st < ns; st++) { acc += rq[static_cast<size_t>(i * ns + st)].accepts; }
        if (acc == 0) { maybe.push_back(i); }
      }
      pq.clear(); pt.clear();
      std::vector<uint64_t> keys;
      if (!maybe.empty() && nqr > 1) {
        for (int i = 1; i < nqr; i++) {
          for (int st = 0; st < ns; st++) {
            int const u = i * ns + st;
            for (int j : maybe) {
              if (j >= i) { break; }
              if ((rc = need_kmers(u)) != VSG_OK || (rc = need_bitmap(j)) != VSG_OK) { return rc; }
              CQuery & S = rq[static_cast<size_t>(u)];
              CQuery & C = rq[static_cast<size_t>(j) * ns];
              unsigned const shared = shared_count(S.kmers, C.bitmap);
              if (!(shared >= static_cast<unsigned>(minwordmatches) || shared >= S.kmers.size())) { continue; }
              if (!unaligned_ok(S.seqno, S.qlen, C.seqno)) { continue; }
              pq.push_back(S.qidx); pt.push_back(static_cast<uint32_t>(C.seqno));
              keys.push_back((static_cast<uint64_t>(u) << 32) | static_cast<uint64_t>(j));
            }
          }
        }
      }
      size_t const np = pq.size();
      if (np > 0) {
        a_score.resize(np); a_al.resize(np); a_ma.resize(np); a_mi.resize(np); a_ga.resize(np); a_tr.resize(np * 4);
        rc = vsg_align_pairs(c, qset, set, static_cast<int64_t>(np), pq.data(), pt.data(), a_score.data(), a_al.data(), a_ma.data(),
                             a_mi.data(), a_ga.data(), a_tr.data(), nullptr, 0, nullptr);
        if (rc != VSG_OK) { return rc; }
        spec.reserve(np);
        for (size_t p = 0; p < np; p++) {
          Spec sp1{a_score[p], a_al[p], a_ma[p], a_mi[p], a_ga[p], {a_tr[4 * p], a_tr[4 * p + 1], a_tr[4 * p + 2], a_tr[4 * p + 3]}};
          spec.emplace_back(keys[p], sp1);
        }
        std::sort(spec.begin(), spec.end(), [](const std::pair<uint64_t, Spec> & a, const std::pair<uint64_t, Spec> & b) { return a.first < b.first; });
      }
    }
    t_spec += ms_since(tp); tp = now();
    std::vector<int> extra_list;
    for (int i = 0; i < nqr; i++) {
      for (int st = 0; st < ns; st++) {   // the plus strand, then the minus strand (cluster.cpp:952-957)
        int const u = i * ns + st;
        CQuery & S = rq[static_cast<size_t>(u)];
        // evaluate_extra_hits (cluster.cpp:601-856)
        int added = 0;
        if (!extra_list.empty()) {
          if ((rc = need_kmers(u)) != VSG_OK) { return rc; }
          for (int j : extra_list) {
            CQuery & C = rq[static_cast<size_t>(j) * ns];   // the new centroid's PLUS k-mers (si_plus + extra_list[j])
            if ((rc = need_bitmap(j)) != VSG_OK) { return rc; }
            unsigned const shared = shared_count(S.kmers, C.bitmap);
            // search_enough_kmers (searchcore.cpp:252-257)
            if (!(shared >= static_cast<unsigned>(minwordmatches) || shared >= S.kmers.size())) { continue; }
            unsigned const length = static_cast<unsigned>(C.qlen);
            int x = static_cast<int>(S.hits.size());
            while (x > 0 && (S.hits[static_cast<size_t>(x) - 1].count < shared ||
                             (S.hits[static_cast<size_t>(x) - 1].count == shared &&
                              static_cast<unsigned>(set->h_len[static_cast<size_t>(S.hits[static_cast<size_t>(x) - 1].target)]) > length))) { --x; }
            if (x < hit_capacity) {
              if (static_cast<int>(S.hits.size()) >= hit_capacity) { S.hits.pop_back(); }
              Hit h;
              std::memset(&h, 0, sizeof(Hit));
              h.target = C.seqno; h.strand = S.strand; h.count = shared;
              S.hits.insert(S.hits.begin() + x, h);
              ++added;
            }
          }
        }
        if (added != 0) {
          S.rejects = 0; S.accepts = 0;
          for (Hit & h : S.hits) { h.accepted = false; h.rejected = false; }
          for (size_t t = 0; S.accepts < maxaccepts && S.rejects < maxrejects && t < S.hits.size(); ++t) {
            Hit & h = S.hits[t];
            if (!h.aligned) {
              if (unaligned_ok(S.seqno, S.qlen, h.target)) {
                uint32_t const q1 = S.qidx, t1 = static_cast<uint32_t>(h.target);
                int16_t sc; uint16_t al, ma, mi, ga; int32_t tr[4];
                // "only using 1 sequence" (cluster.cpp:741-752): from the speculative batch if it is a centroid of this round
                bool found = false;
                if (h.target >= round0) {
                  uint64_t const key = (static_cast<uint64_t>(u) << 32) | static_cast<uint64_t>(h.target - round0);
                  auto const it = std::lower_bound(spec.begin(), spec.end(), key, [](const std::pair<uint64_t, Spec> & a, uint64_t kk) { return a.first < kk; });
                  if (it != spec.end() && it->first == key) {
                    sc = it->second.sc; al = it->second.al; ma = it->second.ma; mi = it->second.mi; ga = it->second.ga;
                    for (int z = 0; z < 4; z++) { tr[z] = it->second.tr[z]; }
                    found = true;
                  }
                }
                if (!found) {
                  rc = vsg_align_pairs(c, qset, set, 1, &q1, &t1, &sc, &al, &ma, &mi, &ga, tr, nullptr, 0, nullptr);
                  if (rc != VSG_OK) { return rc; }
                }
                total_pairs++; total_cells += static_cast<int64_t>(S.qlen) * set->h_len[static_cast<size_t>(h.target)];
                int rcode = VSG_OK;
                fill_hit(h, S.qlen, sc, al, ma, mi, ga, tr, S.seqno, S.strand, rcode);
                if (rcode != VSG_OK) { return rcode; }
              } else {
                h.rejected = true;
                ++S.rejects;
              }
            }
            if (!h.rejected) {
              if (acceptable_aligned(h, opt_id, opt_weak_id, *opts, S.qlen, set->h_len[static_cast<size_t>(h.target)], size_of(S.seqno), size_of(h.target))) { ++S.accepts; } else { ++S.rejects; }
            }
          }
          size_t keep = S.hits.size();   // delete all undetermined hits from the first one on
          for (size_t t = S.hits.size(); t-- > 0;) { if (!S.hits[t].accepted && !S.hits[t].rejected) { keep = t; } }
          S.hits.resize(keep);
        }
      }
      // search_findbest2_byid (searchcore.cpp:960-991): the first hit that no other one precedes in the by-id order,
      // scanning the plus hits and then the minus hits, so that ties go to plus
      const Hit * best = nullptr;
      for (int st = 0; st < ns; st++) {
        for (const Hit & h : rq[static_cast<size_t>(i * ns + st)].hits) {
          // --sizeorder: search_findbest2_bysize (searchcore.cpp:994-1025)
          bool const better = best == nullptr ||
                              (opts->sizeorder != 0 ? hit_less_bysize(h, *best, size_of(h.target), size_of(best->target)) : hit_less(h, *best));
          if (better) { best = &h; }
        }
      }
      if (best != nullptr && !best->accepted) { best = nullptr; }
      int const seqno = static_cast<int>(round0 + i);
      vsg_cluster_result & r = results[static_cast<size_t>(seqno - start)];
      std::memset(&r, 0, sizeof r);
      if (best != nullptr) {
        r.cluster = cluster_of[static_cast<size_t>(best->target)];
        r.centroid = best->target;
        r.matches = best->matches; r.mismatches = best->mismatches; r.gaps = best->nwgaps;
        r.alignment_length = best->nwalignmentlength; r.nwscore = best->nwscore; r.strand = best->strand; r.id = best->id;
        cluster_of[static_cast<size_t>(seqno)] = r.cluster;
      } else {
        r.cluster = static_cast<int32_t>(clusters);
        r.centroid = -1;
        cluster_of[static_cast<size_t>(seqno)] = r.cluster;
        ++clusters;
        extra_list.push_back(i);
        new_centroids.push_back(static_cast<uint32_t>(seqno));   // indexed in plus orientation (add_sequence(seqno))
      }
    }
    t_serial += ms_since(tp); tp = now();
    // Dbindex::add_sequence for the round's new centroids (they were visible to the rest of the round as extras)
    if (!new_centroids.empty()) {
      if ((rc = cindex_append(c, ix, new_centroids.data(), static_cast<int>(new_centroids.size()))) != VSG_OK) { return rc; }
    }
    t_append += ms_since(tp);
  }
  if (trace) {
    std::fprintf(stderr, "[vsg trace] cluster rounds %lld..%lld, round %d: rank %.0f ms, candidate groups %.0f ms, speculative extras %.0f ms, "
                 "serial pass %.0f ms, index append %.0f ms; %lld pairs so far\n", static_cast<long long>(start), static_cast<long long>(start + count),
                 round_size, t_rank, t_groups, t_spec, t_serial, t_append, static_cast<long long>(total_pairs));
  }
  s.next = start + count;
  return VSG_OK;
}

}  // namespace

extern "C" int vsg_cluster_fast(vsg_ctx * c, const vsg_seqset * set, const vsg_search_opts * opts, int round_size,
                                vsg_cluster_result * results, int64_t * nclusters, int64_t * work)
{
  if (c == nullptr || set == nullptr || opts == nullptr || results == nullptr || round_size < 1) { Error::set("vsg_cluster_fast: bad argument"); return VSG_EINVAL; }
  if (nclusters != nullptr) { *nclusters = 0; }
  if (work != nullptr) { work[0] = work[1] = 0; }
  vsg_cluster_session s;
  int rc = session_setup(c, set, opts, s);
  if (rc != VSG_OK || s.seqcount == 0) { return rc; }
  if ((rc = session_rounds(s, 0, s.seqcount, round_size, results)) != VSG_OK) { return rc; }
  if (nclusters != nullptr) { *nclusters = s.clusters; }
  if (work != nullptr) { work[0] = s.total_pairs; work[1] = s.total_cells; }
  return VSG_OK;
}

// ---- the incremental form: cluster_session_init / cluster_assign_single / cluster_assign_batch (core/cluster.hpp:78-118) ----
extern "C" int vsg_cluster_session_create(vsg_ctx * c, const vsg_seqset * set, const vsg_search_opts * opts, vsg_cluster_session ** out)
{
  if (c == nullptr || set == nullptr || opts == nullptr || out == nullptr) { Error::set("vsg_cluster_session_create: null argument"); return VSG_EINVAL; }
  *out = nullptr;
  vsg_cluster_session * s = new (std::nothrow) vsg_cluster_session();
  if (s == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  int const rc = session_setup(c, set, opts, *s);
  if (rc != VSG_OK) { delete s; return rc; }
  *out = s;
  return VSG_OK;
}

extern "C" int vsg_cluster_session_assign(vsg_cluster_session * s, int64_t start, int64_t count, int round_size, vsg_cluster_result * results)
{
  if (s == nullptr || results == nullptr || round_size < 1 || count < 0) { Error::set("vsg_cluster_session_assign: bad argument"); return VSG_EINVAL; }
  if (start != s->next || start + count > s->seqcount) {
    Error::set("vsg_cluster_session_assign: ranges must be ascending, contiguous and inside the set (cluster.hpp:104-111)");
    return VSG_EINVAL;
  }
  if (count == 0) { return VSG_OK; }
  VSG_CUDA_OK(cudaSetDevice(s->c->device));
  return session_rounds(*s, start, count, round_size, results);
}

extern "C" int64_t vsg_cluster_session_clusters(const vsg_cluster_session * s) { return s != nullptr ? s->clusters : 0; }

extern "C" void vsg_cluster_session_destroy(vsg_cluster_session * s)
{
  if (s == nullptr) { return; }
  cudaSetDevice(s->c->device);
  delete s;
}
