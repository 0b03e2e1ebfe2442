// group.cu — several GPUs behind ONE process: the database is uploaded once, copied peer to peer
// (NVLink / NVSwitch) to every other device, indexed on each, and queries / all-pairs rows are sharded
// across the devices with no data-path collective (SURVEY.md §8e).  The reference is a single process
// (LIBRARY_API.md:138-156): this is what lets a drop-in of search_batch() use all the GPUs of a box
// (shim/search_batch_vsg.cpp with VSG_DEVICES=0,1,...).  bench.py's multi-GPU runs keep one process per
// GPU with an NCCL broadcast, as its contract asks; both end in the same per-device calls.
#include "vsg_internal.h"

#include <algorithm>
#include <chrono>
#include <cstring>
#include <thread>

using namespace vsg;

struct vsg_group {
  std::vector<int> devices;
  std::vector<vsg_ctx *> ctx;
  std::vector<vsg_seqset *> db;
  std::vector<vsg_index *> index;
  int wordlength = 8, mask_lower = 0;
  double upload_ms = 0.0, broadcast_ms = 0.0, index_ms = 0.0;
  int64_t broadcast_bytes = 0;
  vsg_fallback_fn fallback = nullptr;   // the application's routine; query indices are those of the whole call
  void * fallback_user = nullptr;
};

namespace {

double now_ms()
{
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// a copy of `src` (resident on another device) in ctx's HBM: packed symbols, offsets and lengths travel
// device to device; the small host-side metadata is shared as is
int clone_seqset(vsg_ctx * c, const vsg_seqset * src, vsg_seqset ** out)
{
  *out = nullptr;
  VSG_CUDA_OK(cudaSetDevice(c->device));
  vsg_seqset * s = new (std::nothrow) vsg_seqset();
  if (s == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  s->device = c->device;
  s->h_len = src->h_len;
  s->h_nonacgt = src->h_nonacgt;
  s->h_off = src->h_off;
  s->total = src->total;
  int64_t const n = src->d.n;
  int rc;
  if ((rc = s->b_sym.reserve(static_cast<size_t>(src->total) + 64)) != VSG_OK ||
      (rc = s->b_off.reserve(sizeof(int64_t) * static_cast<size_t>(n) + 8)) != VSG_OK ||
      (rc = s->b_len.reserve(sizeof(int32_t) * static_cast<size_t>(n) + 8)) != VSG_OK) {
    vsg_seqset_destroy(s);
    return rc;
  }
  if (src->total > 0) {
    VSG_CUDA_OK(cudaMemcpyPeerAsync(s->b_sym.p, c->device, src->d.sym, src->device, static_cast<size_t>(src->total), c->stream));
  }
  if (n > 0) {
    VSG_CUDA_OK(cudaMemcpyPeerAsync(s->b_off.p, c->device, src->d.off, src->device, sizeof(int64_t) * static_cast<size_t>(n), c->stream));
    VSG_CUDA_OK(cudaMemcpyPeerAsync(s->b_len.p, c->device, src->d.len, src->device, sizeof(int32_t) * static_cast<size_t>(n), c->stream));
  }
  s->d.sym = static_cast<uint8_t *>(s->b_sym.p);
  s->d.off = static_cast<int64_t *>(s->b_off.p);
  s->d.len = static_cast<int32_t *>(s->b_len.p);
  s->d.n = n;
  *out = s;
  return VSG_OK;
}

}  // namespace

extern "C" int vsg_group_create(const int * devices, int ndev, const vsg_scoring * scoring, const char * cat,
                                const int64_t * off, const int32_t * len, int64_t n, int wordlength, int mask_lower,
                                int dust_db, vsg_group ** out)
{
  if (devices == nullptr || ndev < 1 || scoring == nullptr || out == nullptr) { Error::set("vsg_group_create: bad argument"); return VSG_EINVAL; }
  *out = nullptr;
  vsg_group * g = new (std::nothrow) vsg_group();
  if (g == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  g->wordlength = wordlength;
  g->mask_lower = (mask_lower != 0 || dust_db != 0) ? 1 : 0;
  int rc = VSG_OK;
  for (int i = 0; i < ndev && rc == VSG_OK; i++) {
    vsg_ctx * c = nullptr;
    rc = vsg_ctx_create(devices[i], scoring, &c);
    if (rc == VSG_OK) { g->devices.push_back(devices[i]); g->ctx.push_back(c); }
  }
  if (rc != VSG_OK) { vsg_group_destroy(g); return rc; }
  g->db.assign(static_cast<size_t>(ndev), nullptr);
  g->index.assign(static_cast<size_t>(ndev), nullptr);
  // 1. one upload (+ optional DUST) on the first device
  double t0 = now_ms();
  rc = vsg_seqset_create(g->ctx[0], cat, off, len, n, 1, &g->db[0]);
  if (rc == VSG_OK && dust_db != 0) { rc = vsg_seqset_dust(g->ctx[0], g->db[0]); }
  if (rc != VSG_OK) { vsg_group_destroy(g); return rc; }
  g->upload_ms = now_ms() - t0;
  // 2. device-to-device copies to the others, all in flight together
  t0 = now_ms();
  for (int i = 1; i < ndev; i++) {
    // direct peer access where the topology offers it (cudaMemcpyPeer stages through the host otherwise)
    int can = 0;
    cudaDeviceCanAccessPeer(&can, devices[i], devices[0]);
    if (can != 0) {
      cudaSetDevice(devices[i]);
      cudaError_t const e = cudaDeviceEnablePeerAccess(devices[0], 0);
      if (e != cudaSuccess) { cudaGetLastError(); }   // already enabled
    }
    rc = clone_seqset(g->ctx[static_cast<size_t>(i)], g->db[0], &g->db[static_cast<size_t>(i)]);
    if (rc != VSG_OK) { vsg_group_destroy(g); return rc; }
    g->broadcast_bytes += g->db[0]->total + static_cast<int64_t>(12) * n;
  }
  for (int i = 1; i < ndev; i++) {
    if ((rc = vsg_ctx_sync(g->ctx[static_cast<size_t>(i)])) != VSG_OK) { vsg_group_destroy(g); return rc; }
  }
  g->broadcast_ms = now_ms() - t0;
  // 3. every device builds its own index (a few ms; cheaper than shipping 2 B per posting)
  t0 = now_ms();
  std::vector<int> rcs(static_cast<size_t>(ndev), VSG_OK);
  std::vector<std::string> msgs(static_cast<size_t>(ndev));
  std::vector<std::thread> pool;
  for (int i = 0; i < ndev; i++) {
    pool.emplace_back([&, i]() {
      rcs[static_cast<size_t>(i)] = vsg_index_create(g->ctx[static_cast<size_t>(i)], g->db[static_cast<size_t>(i)], wordlength, g->mask_lower,
                                                     &g->index[static_cast<size_t>(i)]);
      if (rcs[static_cast<size_t>(i)] != VSG_OK) { msgs[static_cast<size_t>(i)] = vsg_last_error(); }
    });
  }
  for (auto & th : pool) { th.join(); }
  g->index_ms = now_ms() - t0;
  for (int i = 0; i < ndev; i++) {
    if (rcs[static_cast<size_t>(i)] != VSG_OK) { Error::set(msgs[static_cast<size_t>(i)]); rc = rcs[static_cast<size_t>(i)]; vsg_group_destroy(g); return rc; }
  }
  *out = g;
  return VSG_OK;
}

extern "C" void vsg_group_destroy(vsg_group * g)
{
  if (g == nullptr) { return; }
  for (auto * ix : g->index) { if (ix != nullptr) { vsg_index_destroy(ix); } }
  for (auto * s : g->db) { if (s != nullptr) { vsg_seqset_destroy(s); } }
  for (auto * c : g->ctx) { if (c != nullptr) { vsg_ctx_destroy(c); } }
  delete g;
}

extern "C" int vsg_group_size(const vsg_group * g) { return g != nullptr ? static_cast<int>(g->ctx.size()) : 0; }
extern "C" vsg_ctx * vsg_group_ctx(vsg_group * g, int i) { return (g != nullptr && i >= 0 && i < static_cast<int>(g->ctx.size())) ? g->ctx[static_cast<size_t>(i)] : nullptr; }
extern "C" vsg_seqset * vsg_group_db(vsg_group * g, int i) { return (g != nullptr && i >= 0 && i < static_cast<int>(g->db.size())) ? g->db[static_cast<size_t>(i)] : nullptr; }
extern "C" vsg_index * vsg_group_index(vsg_group * g, int i) { return (g != nullptr && i >= 0 && i < static_cast<int>(g->index.size())) ? g->index[static_cast<size_t>(i)] : nullptr; }

extern "C" int vsg_group_stats(const vsg_group * g, double * ms3, int64_t * broadcast_bytes)
{
  if (g == nullptr || ms3 == nullptr) { return VSG_EINVAL; }
  ms3[0] = g->upload_ms; ms3[1] = g->broadcast_ms; ms3[2] = g->index_ms;
  if (broadcast_bytes != nullptr) { *broadcast_bytes = g->broadcast_bytes; }
  return VSG_OK;
}

extern "C" int vsg_group_set_fallback(vsg_group * g, vsg_fallback_fn fn, void * user)
{
  if (g == nullptr) { return VSG_EINVAL; }
  g->fallback = fn; g->fallback_user = user;
  for (auto * c : g->ctx) { vsg_ctx_set_fallback(c, fn, user); }   // vsg_group_allpairs: indices are global already
  return VSG_OK;
}

namespace {
// a device sees its slice of the queries: hand the application the index within the whole call
struct SliceFallback { vsg_fallback_fn fn; void * user; int64_t base; };
int slice_fallback(void * u, int64_t query, int32_t strand, int64_t target, int64_t * out)
{
  SliceFallback const * w = static_cast<SliceFallback *>(u);
  return w->fn(w->user, query + w->base, strand, target, out);
}
}  // namespace

// vsg_group_search; the rows of query q go to results[q * max_results ...] or, with rows != nullptr, to rows[q]
static int group_search(vsg_group * g, const char * qcat, const int64_t * qoff, const int32_t * qlen, int64_t nq,
                        int dust_queries, const vsg_search_opts * opts, vsg_search_result * results, int64_t max_results,
                        std::vector<vsg_search_result> * rows, int32_t * counts, int64_t * work)
{
  if (g == nullptr || opts == nullptr || counts == nullptr || nq < 0 ||
      (nq > 0 && (qcat == nullptr || qoff == nullptr || qlen == nullptr))) { Error::set("vsg_group_search: bad argument"); return VSG_EINVAL; }
  int const nd = static_cast<int>(g->ctx.size());
  if (work != nullptr) { work[0] = work[1] = work[2] = work[3] = 0; }
  if (nq == 0) { return VSG_OK; }
  // contiguous query ranges of equal nucleotide count (the DP work per query is proportional to its length)
  std::vector<int64_t> bounds(static_cast<size_t>(nd) + 1, nq);
  {
    double total = 0.0;
    for (int64_t i = 0; i < nq; i++) { total += qlen[i]; }
    bounds[0] = 0;
    double acc = 0.0;
    int p = 1;
    for (int64_t i = 0; i < nq && p < nd; i++) {
      acc += qlen[i];
      while (p < nd && acc >= total * p / nd) { bounds[static_cast<size_t>(p++)] = i + 1; }
    }
  }
  std::vector<int> rcs(static_cast<size_t>(nd), VSG_OK);
  std::vector<std::string> msgs(static_cast<size_t>(nd));
  std::vector<int64_t> w(static_cast<size_t>(nd) * 4, 0);
  auto run = [&](int d) {
    int64_t const b0 = bounds[static_cast<size_t>(d)], b1 = bounds[static_cast<size_t>(d) + 1];
    if (b1 <= b0) { return; }
    vsg_ctx * c = g->ctx[static_cast<size_t>(d)];
    // this device's slice, rebased: offsets relative to its first sequence
    int64_t const base = qoff[b0];
    std::vector<int64_t> off(static_cast<size_t>(b1 - b0));
    for (int64_t i = b0; i < b1; i++) { off[static_cast<size_t>(i - b0)] = qoff[i] - base; }
    vsg_seqset * q = nullptr;
    int rc = vsg_seqset_create(c, qcat + base, off.data(), qlen + b0, b1 - b0, 1, &q);
    if (rc == VSG_OK && dust_queries != 0) { rc = vsg_seqset_dust(c, q); }
    SliceFallback sf{g->fallback, g->fallback_user, b0};
    if (g->fallback != nullptr) { vsg_ctx_set_fallback(c, slice_fallback, &sf); }
    vsg_search_opts o = *opts;
    if (o.query_sizes != nullptr) { o.query_sizes += b0; }
    if (o.query_labels != nullptr) { o.query_labels += b0; }
    if (rc == VSG_OK && rows != nullptr) {
      rc = search_batch_rows(c, g->index[static_cast<size_t>(d)], g->db[static_cast<size_t>(d)], q, 0, b1 - b0, &o,
                             max_results, rows + b0, counts + b0, w.data() + 4 * d);
    } else if (rc == VSG_OK) {
      rc = vsg_search_batch(c, g->index[static_cast<size_t>(d)], g->db[static_cast<size_t>(d)], q, 0, b1 - b0, &o,
                            results + static_cast<size_t>(b0) * max_results, static_cast<int>(max_results), counts + b0, w.data() + 4 * d);
    }
    if (rc != VSG_OK) { rcs[static_cast<size_t>(d)] = rc; msgs[static_cast<size_t>(d)] = vsg_last_error(); }
    if (g->fallback != nullptr) { vsg_ctx_set_fallback(c, g->fallback, g->fallback_user); }
    if (q != nullptr) { vsg_seqset_destroy(q); }
  };
  if (nd == 1) { run(0); }
  else {
    std::vector<std::thread> pool;
    for (int d = 0; d < nd; d++) { pool.emplace_back(run, d); }
    for (auto & th : pool) { th.join(); }
  }
  for (int d = 0; d < nd; d++) {
    if (rcs[static_cast<size_t>(d)] != VSG_OK) { Error::set(msgs[static_cast<size_t>(d)]); return rcs[static_cast<size_t>(d)]; }
    if (work != nullptr) { for (int z = 0; z < 4; z++) { work[z] += w[static_cast<size_t>(4 * d + z)]; } }
  }
  return VSG_OK;
}

extern "C" int vsg_group_search(vsg_group * g, const char * qcat, const int64_t * qoff, const int32_t * qlen, int64_t nq,
                                int dust_queries, const vsg_search_opts * opts, vsg_search_result * results, int max_results,
                                int32_t * counts, int64_t * work)
{
  if (results == nullptr) { Error::set("vsg_group_search: bad argument"); return VSG_EINVAL; }
  return group_search(g, qcat, qoff, qlen, nq, dust_queries, opts, results, max_results, nullptr, counts, work);
}

int vsg::group_search_rows(vsg_group * g, const char * qcat, const int64_t * qoff, const int32_t * qlen, int64_t nq,
                           int dust_queries, const vsg_search_opts * opts, int64_t max_rows, std::vector<vsg_search_result> * rows,
                           int32_t * counts, int64_t * work)
{
  if (rows == nullptr) { Error::set("vsg_group_search: bad argument"); return VSG_EINVAL; }
  return group_search(g, qcat, qoff, qlen, nq, dust_queries, opts, nullptr, max_rows, rows, counts, work);
}

extern "C" int vsg_group_allpairs(vsg_group * g, const vsg_search_opts * opts, vsg_pair_hit * hits, int64_t cap,
                                  int64_t * nhits, int64_t * work)
{
  if (g == nullptr || opts == nullptr || nhits == nullptr || (cap > 0 && hits == nullptr)) { Error::set("vsg_group_allpairs: bad argument"); return VSG_EINVAL; }
  int const nd = static_cast<int>(g->ctx.size());
  const vsg_seqset * set = g->db[0];
  int64_t const n = set->d.n;
  *nhits = 0;
  if (work != nullptr) { work[0] = work[1] = 0; }
  // row ranges of equal DP work (triangle balancing), one per device
  std::vector<int64_t> bounds(static_cast<size_t>(nd) + 1, 0);
  int rc = vsg_allpairs_partition(set->h_len.data(), n, nd, bounds.data());
  if (rc != VSG_OK) { return rc; }
  // every device writes into its own stretch of the caller's buffer, sized by its share of the pairs
  std::vector<int64_t> cap_off(static_cast<size_t>(nd) + 1, 0);
  {
    double total_pairs = 0.0;
    std::vector<double> pr(static_cast<size_t>(nd));
    for (int d = 0; d < nd; d++) {
      double p = 0.0;
      for (int64_t i = bounds[static_cast<size_t>(d)]; i < bounds[static_cast<size_t>(d) + 1]; i++) { p += static_cast<double>(n - i - 1); }
      pr[static_cast<size_t>(d)] = p; total_pairs += p;
    }
    for (int d = 0; d < nd; d++) {
      int64_t const share = total_pairs > 0 ? static_cast<int64_t>(static_cast<double>(cap) * pr[static_cast<size_t>(d)] / total_pairs) : 0;
      cap_off[static_cast<size_t>(d) + 1] = std::min<int64_t>(cap, cap_off[static_cast<size_t>(d)] + share);
    }
    cap_off[static_cast<size_t>(nd)] = cap;
  }
  std::vector<int> rcs(static_cast<size_t>(nd), VSG_OK);
  std::vector<std::string> msgs(static_cast<size_t>(nd));
  std::vector<int64_t> got(static_cast<size_t>(nd), 0), w(static_cast<size_t>(nd) * 2, 0);
  auto run = [&](int d) {
    int64_t const r0 = bounds[static_cast<size_t>(d)], r1 = bounds[static_cast<size_t>(d) + 1];
    if (r1 <= r0) { return; }
    int const r = vsg_allpairs(g->ctx[static_cast<size_t>(d)], g->db[static_cast<size_t>(d)], r0, r1 - r0, opts,
                               hits + cap_off[static_cast<size_t>(d)], cap_off[static_cast<size_t>(d) + 1] - cap_off[static_cast<size_t>(d)],
                               &got[static_cast<size_t>(d)], w.data() + 2 * d);
    if (r != VSG_OK) { rcs[static_cast<size_t>(d)] = r; msgs[static_cast<size_t>(d)] = vsg_last_error(); }
  };
  if (nd == 1) { run(0); }
  else {
    std::vector<std::thread> pool;
    for (int d = 0; d < nd; d++) { pool.emplace_back(run, d); }
    for (auto & th : pool) { th.join(); }
  }
  int64_t pos = 0;
  for (int d = 0; d < nd; d++) {
    if (rcs[static_cast<size_t>(d)] != VSG_OK) { Error::set(msgs[static_cast<size_t>(d)]); return rcs[static_cast<size_t>(d)]; }
    // compact the per-device stretches into one list in row order
    if (cap_off[static_cast<size_t>(d)] != pos && got[static_cast<size_t>(d)] > 0) {
      std::memmove(hits + pos, hits + cap_off[static_cast<size_t>(d)], sizeof(vsg_pair_hit) * static_cast<size_t>(got[static_cast<size_t>(d)]));
    }
    pos += got[static_cast<size_t>(d)];
    if (work != nullptr) { work[0] += w[static_cast<size_t>(2 * d)]; work[1] += w[static_cast<size_t>(2 * d + 1)]; }
  }
  *nhits = pos;
  return VSG_OK;
}
