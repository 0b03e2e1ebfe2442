// shim/cluster_session_vsg.cpp — seam 2, clustering half (SURVEY.md §8b): replacements for the reference's
// incremental clustering entry points
//     cluster_session_alloc / cluster_session_free / cluster_session_init / cluster_assign_single /
//     cluster_assign_batch / cluster_session_cleanup                  (src/core/cluster.hpp:78-118,
//                                                                      src/core/cluster.cpp:1597-1930)
// with the same signatures, the same result record (cluster.hpp:65-73) and the same error convention (fatal()),
// forwarding to a vsg_cluster_session of libvsg.so (include/vsg.h): the database is mirrored into HBM once at
// cluster_session_init, every call ranks / aligns / resolves its range in rounds on the device and the host
// (vsearch_b200/csrc/cluster.cu), the CIGARs of the assigned sequences come from one vsg_align_pairs call per
// range and strand.  The caller's Dbindex is not touched: the centroids' k-mer index lives on the device.  Link so that these
// definitions win over core/cluster.cpp.o's (oracle/Makefile weakens those six symbols).  See INTEGRATION.md.
#include "vsearch_api.h"
#include "core/cluster.hpp"
#include "core/linmemalign.hpp"
#include "utils/fatal.hpp"
#include "utils/reverse_complement.hpp"
#include "utils/string_alloc.hpp"

#include "vsg.h"

#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

namespace {

[[noreturn]] void die(const char * what)
{
  std::string const m = std::string("GPU cluster session: ") + what + ": " + vsg_last_error();
  fatal(m.c_str());
  std::abort();
}

}  // namespace

struct cluster_session_s {
  Parameters const * parameters = nullptr;
  Dbindex * dbindex = nullptr;
  Database const * db = nullptr;
  int seqcount = 0;
  vsg_ctx * ctx = nullptr;
  vsg_seqset * set = nullptr;
  vsg_cluster_session * session = nullptr;
  vsg_search_opts opts;
  std::vector<int64_t> sizes, labels;
};

namespace {

// the reference's own answer for a pair its 16-bit aligner defers (core/cluster.cpp:786-809 via searchcore.cpp:806-832);
// strand 1 aligns the reverse complement of the query, as cluster_query_core searches it (cluster.cpp:178-181)
struct Lma {
  std::string cigar;
  int64_t out[10];
};
void lma_align(cluster_session_s const & cs, int64_t query, int32_t strand, int64_t target, Lma & r)
{
  Parameters const & p = *cs.parameters;
  char const * q = cs.db->getsequence(static_cast<uint64_t>(query));
  char const * const d = cs.db->getsequence(static_cast<uint64_t>(target));
  auto const ql = static_cast<int64_t>(cs.db->getsequencelen(static_cast<uint64_t>(query)));
  std::vector<char> rc;
  if (strand != 0) {
    rc.resize(static_cast<size_t>(ql) + 1);
    reverse_complement(rc.data(), q, ql);
    q = rc.data();
  }
  auto const dl = static_cast<int64_t>(cs.db->getsequencelen(static_cast<uint64_t>(target)));
  struct Scoring scoring = scoring_from_options(p);
  LinearMemoryAligner lma(scoring);
  char * const cigar = xstrdup(lma.align(q, d, ql, dl));
  int64_t sc = 0, al = 0, ma = 0, mi = 0, ga = 0;
  lma.alignstats(cigar, q, d, &sc, &al, &ma, &mi, &ga);
  r.cigar = cigar;
  r.out[0] = sc; r.out[1] = al; r.out[2] = ma; r.out[3] = mi; r.out[4] = ga;
  auto run_at = [&](char const * s, int64_t & len, char & op) {
    len = 0;
    while (*s >= '0' && *s <= '9') { len = len * 10 + (*s - '0'); ++s; }
    if (len == 0) { len = 1; }
    op = *s;
  };
  int64_t l0 = 0, l1 = 0; char o0 = 0, o1 = 0;
  size_t const n = std::strlen(cigar);
  r.out[5] = r.out[6] = r.out[7] = r.out[8] = 0;
  if (n > 0) {
    run_at(cigar, l0, o0);
    size_t st = n - 1;
    while (st > 0 && cigar[st - 1] >= '0' && cigar[st - 1] <= '9') { st--; }
    run_at(cigar + st, l1, o1);
    if (o0 == 'D') { r.out[5] = l0; } else if (o0 == 'I') { r.out[6] = l0; }
    if (o1 == 'D') { r.out[7] = l1; } else if (o1 == 'I') { r.out[8] = l1; }
  }
  r.out[9] = 0;
  xfree(cigar);
}

int lma_fallback(void * user, int64_t query, int32_t strand, int64_t target, int64_t * out)
{
  Lma r;
  lma_align(*static_cast<cluster_session_s *>(user), query, strand, target, r);
  std::memcpy(out, r.out, sizeof r.out);
  return 0;
}

void label_into(char (&dst)[1024], Database const & db, int seqno)
{
  std::snprintf(dst, sizeof dst, "%.*s", static_cast<int>(db.getheaderlen(static_cast<uint64_t>(seqno))),
                db.getheader(static_cast<uint64_t>(seqno)));
}

void assign_range(cluster_session_s * cs, int start, int count, int round_size, cluster_result_s * results)
{
  if (count <= 0) { return; }
  if (cs->seqcount != static_cast<int>(cs->db->getsequencecount())) {
    fatal("cluster_assign_batch: the database changed since cluster_session_init(); re-initialize the clustering session.");
  }
  std::vector<vsg_cluster_result> r(static_cast<size_t>(count));
  if (vsg_cluster_session_assign(cs->session, start, count, round_size, r.data()) != VSG_OK) { die("vsg_cluster_session_assign"); }
  // CIGARs of the assigned sequences: one batched call per strand; a strand-1 record's CIGAR is that of the reverse
  // complement (the range's reverse complements, made on the device, entry i = sequence start + i)
  struct Batch {
    std::vector<uint32_t> q, t;
    int64_t cap = 64;
    std::vector<int16_t> sc; std::vector<uint16_t> al, ma, mi, ga;
    std::vector<char> cig;
    std::vector<int64_t> coff;
    size_t next = 0;
  } b[2];
  for (int i = 0; i < count; i++) {
    vsg_cluster_result const & x = r[static_cast<size_t>(i)];
    if (x.centroid >= 0) {
      Batch & B = b[x.strand != 0 ? 1 : 0];
      B.q.push_back(static_cast<uint32_t>(x.strand != 0 ? i : start + i)); B.t.push_back(static_cast<uint32_t>(x.centroid));
      B.cap += static_cast<int64_t>(cs->db->getsequencelen(static_cast<uint64_t>(start + i))) +
               static_cast<int64_t>(cs->db->getsequencelen(static_cast<uint64_t>(x.centroid))) + 1;
    }
  }
  vsg_seqset * rc = nullptr;
  if (!b[1].q.empty() && vsg_seqset_revcomp(cs->ctx, cs->set, start, count, &rc) != VSG_OK) { die("vsg_seqset_revcomp"); }
  for (int st = 0; st < 2; st++) {
    Batch & B = b[st];
    size_t const np = B.q.size();
    B.sc.resize(np); B.al.resize(np); B.ma.resize(np); B.mi.resize(np); B.ga.resize(np);
    B.cig.resize(static_cast<size_t>(B.cap)); B.coff.resize(np + 1);
    if (np > 0 && vsg_align_pairs(cs->ctx, st != 0 ? rc : cs->set, cs->set, static_cast<int64_t>(np), B.q.data(), B.t.data(), B.sc.data(),
                                  B.al.data(), B.ma.data(), B.mi.data(), B.ga.data(), nullptr, B.cig.data(), B.cap, B.coff.data()) != VSG_OK) {
      die("vsg_align_pairs");
    }
  }
  vsg_seqset_destroy(rc);
  for (int i = 0; i < count; i++) {
    cluster_result_s & out = results[i];
    std::memset(&out, 0, sizeof out);
    vsg_cluster_result const & x = r[static_cast<size_t>(i)];
    out.cluster_id = x.cluster;
    if (x.centroid < 0) {
      out.is_centroid = true;
      out.centroid_seqno = start + i;
      out.identity = 100.0;
      label_into(out.centroid_label, *cs->db, start + i);
    } else {
      out.is_centroid = false;
      out.centroid_seqno = x.centroid;
      out.identity = x.id;
      label_into(out.centroid_label, *cs->db, x.centroid);
      int const st = x.strand != 0 ? 1 : 0;
      Batch & B = b[st];
      size_t const pi = B.next++;
      std::string text;
      if (B.sc[pi] == SHRT_MAX) { Lma l; lma_align(*cs, start + i, st, x.centroid, l); text = l.cigar; }   // the deferred pair's CIGAR
      else { text = B.cig.data() + B.coff[pi]; }
      int const n = std::snprintf(out.cigar, sizeof out.cigar, "%s", text.c_str());
      out.cigar_truncated = (n >= static_cast<int>(sizeof out.cigar));
    }
  }
}

}  // namespace

auto cluster_session_alloc() -> struct cluster_session_s * { return new cluster_session_s{}; }

auto cluster_session_cleanup(struct cluster_session_s * cs) -> void
{
  if (cs == nullptr) { return; }
  if (cs->session != nullptr) { vsg_cluster_session_destroy(cs->session); cs->session = nullptr; }
  if (cs->set != nullptr) { vsg_seqset_destroy(cs->set); cs->set = nullptr; }
  if (cs->ctx != nullptr) { vsg_ctx_destroy(cs->ctx); cs->ctx = nullptr; }
}

auto cluster_session_free(struct cluster_session_s * cs) -> void
{
  if (cs != nullptr) { cluster_session_cleanup(cs); delete cs; }
}

auto cluster_session_init(struct cluster_session_s * cs, struct Parameters const & parameters,
                          struct Dbindex & dbindex, struct Database const & db) -> void
{
  cluster_session_cleanup(cs);
  Parameters const & p = parameters;
  cs->parameters = &p; cs->dbindex = &dbindex; cs->db = &db;
  cs->seqcount = static_cast<int>(db.getsequencecount());

  vsg_scoring sco;
  int64_t const v[14] = {p.opt_match, p.opt_mismatch,
                         p.opt_gap_open_query_left, p.opt_gap_open_target_left,
                         p.opt_gap_open_query_interior, p.opt_gap_open_target_interior,
                         p.opt_gap_open_query_right, p.opt_gap_open_target_right,
                         p.opt_gap_extension_query_left, p.opt_gap_extension_target_left,
                         p.opt_gap_extension_query_interior, p.opt_gap_extension_target_interior,
                         p.opt_gap_extension_query_right, p.opt_gap_extension_target_right};
  std::memcpy(sco.v, v, sizeof v);
  sco.n_mismatch = p.opt_n_mismatch ? 1 : 0;
  const char * const dev = std::getenv("VSG_DEVICE");
  if (vsg_ctx_create(dev != nullptr ? std::atoi(dev) : 0, &sco, &cs->ctx) != VSG_OK) { die("vsg_ctx_create"); }

  uint64_t const n = db.getsequencecount();
  std::vector<int64_t> off(n);
  std::vector<int32_t> len(n);
  uint64_t total = 0;
  for (uint64_t i = 0; i < n; i++) { off[i] = static_cast<int64_t>(total); len[i] = static_cast<int32_t>(db.getsequencelen(i)); total += db.getsequencelen(i); }
  std::vector<char> cat(total + 1);
  cs->sizes.resize(n); cs->labels.resize(n);
  std::unordered_map<std::string, int64_t> label_of;
  for (uint64_t i = 0; i < n; i++) {
    std::memcpy(cat.data() + off[i], db.getsequence(i), static_cast<size_t>(len[i]));   // case = the database's soft mask
    cs->sizes[i] = static_cast<int64_t>(db.getabundance(i));
    auto const it = label_of.emplace(std::string(db.getheader(i)), static_cast<int64_t>(label_of.size()));
    cs->labels[i] = it.first->second;
  }
  if (vsg_seqset_create(cs->ctx, cat.data(), off.data(), len.data(), static_cast<int64_t>(n), 1, &cs->set) != VSG_OK) { die("vsg_seqset_create"); }

  vsg_search_opts & o = cs->opts;
  vsg_search_opts_default(&o);
  o.id = p.opt_id; o.weak_id = p.opt_weak_id;
  o.maxaccepts = static_cast<int32_t>(p.opt_maxaccepts); o.maxrejects = static_cast<int32_t>(p.opt_maxrejects);
  o.wordlength = static_cast<int32_t>(dbindex.wordlength);
  o.minwordmatches = static_cast<int32_t>(p.opt_minwordmatches);
  o.iddef = static_cast<int32_t>(p.opt_iddef);
  o.mask_lower = (p.opt_qmask != Masking::none) ? 1 : 0;
  o.minqt = p.opt_minqt; o.maxqt = p.opt_maxqt; o.minsl = p.opt_minsl; o.maxsl = p.opt_maxsl;
  o.maxid = p.opt_maxid; o.mid = p.opt_mid; o.query_cov = p.opt_query_cov; o.target_cov = p.opt_target_cov;
  o.maxsubs = p.opt_maxsubs; o.maxgaps = p.opt_maxgaps; o.mincols = p.opt_mincols; o.maxdiffs = p.opt_maxdiffs;
  o.leftjust = p.opt_leftjust != 0 ? 1 : 0; o.rightjust = p.opt_rightjust != 0 ? 1 : 0;
  o.unoise = (p.opt_cluster_unoise != nullptr) ? 1 : 0; o.unoise_alpha = p.opt_unoise_alpha;
  o.sizeorder = p.opt_sizeorder ? 1 : 0;
  o.strand_both = p.opt_strand ? 1 : 0;
  o.maxqsize = p.opt_maxqsize; o.mintsize = p.opt_mintsize;
  o.minsizeratio = p.opt_minsizeratio; o.maxsizeratio = p.opt_maxsizeratio;
  o.self = p.opt_self != 0 ? 1 : 0;
  o.query_sizes = cs->sizes.data(); o.target_sizes = cs->sizes.data();
  o.query_labels = cs->labels.data(); o.target_labels = cs->labels.data();
  vsg_ctx_set_fallback(cs->ctx, lma_fallback, cs);
  if (vsg_cluster_session_create(cs->ctx, cs->set, &o, &cs->session) != VSG_OK) { die("vsg_cluster_session_create"); }
}

auto cluster_assign_single(struct cluster_session_s * cs, int seqno, struct cluster_result_s * result) -> void
{
  assign_range(cs, seqno, 1, 1, result);
}

auto cluster_assign_batch(struct cluster_session_s * cs, int start_seqno, int count, struct cluster_result_s * results) -> void
{
  int const round = static_cast<int>(cs->parameters->opt_threads) > 0 ? static_cast<int>(cs->parameters->opt_threads) : 1;
  assign_range(cs, start_seqno, count, round, results);
}
