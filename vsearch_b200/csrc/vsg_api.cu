// vsg_api.cu — host side of libvsg.so: contexts, sequence sets in HBM, and the batched aligner
// entry point vsg_align_pairs (replaces search16_init/qprep/search16/exit,
// reference core/align_simd.cpp:1282-2060; see include/vsg.h for the per-function mapping).
#include "align_kernels.cuh"
#include "align_ckpt.cuh"

#include <cub/cub.cuh>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <chrono>

namespace vsg {

static thread_local std::string g_last_error;
void Error::set(const std::string & m) { g_last_error = m; }

static std::atomic<int64_t> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// Device buffers come from a small per-device cache of freed blocks: query batches, reverse
// complements and scratch come and go every call, and cudaMalloc/cudaFree are expensive —
// dramatically so once NCCL has enabled peer access between the GPUs of a box.
namespace {
struct PoolKey { int device; size_t cls; bool operator<(const PoolKey & o) const { return device != o.device ? device < o.device : cls < o.cls; } };
std::mutex g_pool_mutex;
std::multimap<PoolKey, void *> g_pool;
size_t size_class(size_t bytes)
{
  size_t const GB = static_cast<size_t>(1) << 30;
  if (bytes > GB) { return (bytes + GB - 1) / GB * GB; }
  size_t c = 1 << 16;
  while (c < bytes) { c <<= 1; }
  return c;
}
}  // namespace

int DevBuf::reserve(size_t bytes)
{
  if (bytes <= cap) { return VSG_OK; }
  release();
  int dev = 0;
  cudaGetDevice(&dev);
  size_t const want = size_class(bytes + 256);
  {
    std::lock_guard<std::mutex> const lock(g_pool_mutex);
    auto it = g_pool.find(PoolKey{dev, want});
    if (it != g_pool.end()) { p = it->second; cap = want; g_pool.erase(it); return VSG_OK; }
  }
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    // give the cache back to the driver and retry once
    cudaGetLastError();
    {
      std::lock_guard<std::mutex> const lock(g_pool_mutex);
      for (auto it = g_pool.begin(); it != g_pool.end();) {
        if (it->first.device == dev) { cudaFree(it->second); it = g_pool.erase(it); } else { ++it; }
      }
    }
    e = cudaMalloc(&p, want);
  }
  if (e != cudaSuccess) {
    p = nullptr;
    Error::set(std::string("cudaMalloc(") + std::to_string(want) + "): " + cudaGetErrorString(e));
    return VSG_ENOMEM;
  }
  cap = want;
  return VSG_OK;
}
void DevBuf::release()
{
  if (p == nullptr) { return; }
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> const lock(g_pool_mutex);
  g_pool.emplace(PoolKey{dev, cap}, p);
  p = nullptr; cap = 0;
}

int PinBuf::reserve(size_t bytes)
{
  if (bytes <= cap) { return VSG_OK; }
  if (p != nullptr) { cudaFreeHost(p); p = nullptr; cap = 0; }
  size_t const want = bytes + bytes / 8 + 256;
  cudaError_t const e = cudaMallocHost(&p, want);
  if (e != cudaSuccess) {
    p = nullptr;
    Error::set(std::string("cudaMallocHost(") + std::to_string(want) + "): " + cudaGetErrorString(e));
    return VSG_ENOMEM;
  }
  cap = want;
  return VSG_OK;
}
void PinBuf::release() { if (p != nullptr) { cudaFreeHost(p); p = nullptr; cap = 0; } }

// scope guards for the error paths (VSG_CUDA_OK returns from the middle of a function)
namespace {
struct ScopedBuf { DevBuf b; ~ScopedBuf() { b.release(); } };
struct SeqsetGuard { vsg_seqset * s; ~SeqsetGuard() { if (s != nullptr) { vsg_seqset_destroy(s); } } vsg_seqset * release() { vsg_seqset * r = s; s = nullptr; return r; } };
struct CtxGuard { vsg_ctx * c; ~CtxGuard() { if (c != nullptr) { vsg_ctx_destroy(c); } } vsg_ctx * release() { vsg_ctx * r = c; c = nullptr; return r; } };
}  // namespace

// ---- scoring ---------------------------------------------------------------------------------
static int16_t clamp_cell(int64_t v, int64_t limit, bool & fb)
{
  if (v > limit) { fb = true; return static_cast<int16_t>(limit); }
  if (v < -limit) { fb = true; return static_cast<int16_t>(-limit); }
  return static_cast<int16_t>(v);
}

static bool ambiguous4(unsigned c) { return !(c == 1 || c == 2 || c == 4 || c == 8); }

static void build_score_params(const vsg_scoring & s, ScoreParams & p)
{
  bool fb = false;
  int64_t const slim = 32767, plim = 32767 / 5;  // align_simd.cpp:1256-1257
  p.match = clamp_cell(s.v[0], slim, fb);
  p.mismatch = clamp_cell(s.v[1], slim, fb);
  for (int k = 0; k < 6; k++) {
    p.go[k] = clamp_cell(s.v[2 + k], plim, fb);
    p.ge[k] = clamp_cell(s.v[8 + k], plim, fb);
  }
  p.n_mismatch = s.n_mismatch != 0 ? 1 : 0;
  p.fallback = fb ? 1 : 0;
  for (unsigned i = 0; i < 16; i++) {
    for (unsigned j = 0; j < 16; j++) {
      int16_t v;
      if (p.n_mismatch && (i == 15 || j == 15)) { v = p.mismatch; }
      else if (ambiguous4(i) || ambiguous4(j)) { v = 0; }
      else if (i == j) { v = p.match; }
      else { v = p.mismatch; }
      p.S[i][j] = v;
    }
  }
  int gpmax = 0;
  for (int k = 0; k < 6; k++) { gpmax = std::max(gpmax, p.go[k] + p.ge[k]); }
  p.score_min = static_cast<int16_t>(-32768 + gpmax);  // align_simd.cpp:1432-1444
}

// The shifted scoring of the checkpoint kernels (align_ckpt.cuh): c = ceil(smax / 2), S2 = S - 2c <= 0, ge2 = ge + c.
// Same alignment problem, every cell of anti-diagonal i+j lowered by c*(i+j+2); false if a value leaves int16.
static bool shifted_params(const ScoreParams & p, ScoreParams & q)
{
  q = p;
  int smax = 0;
  for (int i = 0; i < 16; i++) { for (int j = 0; j < 16; j++) { smax = std::max<int>(smax, p.S[i][j]); } }
  int const c = (smax + 1) / 2;
  q.shift = c;
  bool ok = true;
  auto fit = [&](int v) -> int16_t { if (v < -32767 || v > 32767) { ok = false; } return static_cast<int16_t>(v); };
  for (int i = 0; i < 16; i++) { for (int j = 0; j < 16; j++) { q.S[i][j] = fit(p.S[i][j] - 2 * c); } }
  for (int k = 0; k < 6; k++) { q.ge[k] = fit(p.ge[k] + c); }
  q.match = fit(p.match - 2 * c);
  q.mismatch = fit(p.mismatch - 2 * c);
  if (q.match < q.mismatch) { ok = false; }   // tb_ckpt.h scores ACGT pairs as mismatch + e * (match - mismatch)
  return ok;
}

// search16_fits, align_simd.cpp:130-134
static inline bool fits16(int64_t q, int64_t d) { return (q + d <= 65535) && (q * d <= 25000000LL); }

// Rows per lane and strip count for a query of length Q.
static inline void fast_shape(int Q, bool general, int & R, int & nstrips)
{
  nstrips = (Q + 32 * FAST_RMAX - 1) / (32 * FAST_RMAX);
  R = (Q + 32 * nstrips - 1) / (32 * nstrips);
  if (R < 1) { R = 1; }
  if (general) { R = R <= 4 ? 4 : (R <= 8 ? 8 : 16); }
  nstrips = (Q + 32 * R - 1) / (32 * R);
}

// Can the biased 16-bit wavefront kernel represent every intermediate of a (Qpad x D) problem
// exactly, and is the reference's overflow flag provably silent?  Bounds (penalties >= 0):
//   every H, incl. both boundaries and the reference's <= 3 padding columns, is
//     >= -(G + Qpad*Rm) - G - (D+4)*Rm            (left column, then one gap along the row)
//     <= Smax * min(Qpad, D+4)
//   E, F and the temporaries (h-QR, e-R, diag+S) stay within 2G+|Smin| below / Smax above that.
struct FastBound { bool valid; int64_t G, Rm, smax, smin; };
static FastBound fast_bound_of(const ScoreParams & sp)
{
  FastBound fb{true, 0, 0, 0, 0};
  for (int k = 0; k < 6; k++) {
    if (sp.go[k] < 0 || sp.ge[k] < 0) { fb.valid = false; }
    fb.G = std::max<int64_t>(fb.G, sp.go[k] + sp.ge[k]);
    fb.Rm = std::max<int64_t>(fb.Rm, sp.ge[k]);
  }
  for (int i = 0; i < 16; i++) {
    for (int j = 0; j < 16; j++) {
      fb.smax = std::max<int64_t>(fb.smax, sp.S[i][j]);
      fb.smin = std::min<int64_t>(fb.smin, sp.S[i][j]);
    }
  }
  return fb;
}
static inline bool fast_path_ok(const FastBound & fb, int Qpad, int D)
{
  if (!fb.valid) { return false; }
  int64_t const lb = -(fb.G + static_cast<int64_t>(Qpad) * fb.Rm) - fb.G - static_cast<int64_t>(D + 4) * fb.Rm - 2 * fb.G + fb.smin;
  int64_t const ub = fb.smax * std::min<int64_t>(Qpad, D + 4) + fb.smax;
  return lb > -32700 && ub < 32700;  // inside the reference's own no-overflow range (score_min = SHRT_MIN + G, SHRT_MAX)
}

}  // namespace vsg

using namespace vsg;

// ---- misc C ABI ------------------------------------------------------------------------------
extern "C" const char * vsg_last_error(void) { return g_last_error.c_str(); }
extern "C" const char * vsg_version(void) { return "vsearch_b200 0.1 (sm_100a)"; }
extern "C" int64_t vsg_launch_count(void) { return g_launches.load(); }

// ---- context ---------------------------------------------------------------------------------
extern "C" int vsg_ctx_create(int device, const vsg_scoring * scoring, vsg_ctx ** out)
{
  if (out == nullptr || scoring == nullptr) { Error::set("vsg_ctx_create: null argument"); return VSG_EINVAL; }
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    Error::set(std::string("no CUDA device available: ") + cudaGetErrorString(e) +
               " (libvsg has no CPU fallback)");
    return VSG_ENODEVICE;
  }
  if (device < 0 || device >= ndev) { Error::set("vsg_ctx_create: bad device ordinal"); return VSG_EINVAL; }
  VSG_CUDA_OK(cudaSetDevice(device));
  vsg_ctx * c = new (std::nothrow) vsg_ctx();
  if (c == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  CtxGuard guard{c};
  c->device = device;
  c->scoring = *scoring;
  build_score_params(*scoring, c->sp);
  c->sp.shift = 0;
  c->ckpt_enabled = shifted_params(c->sp, c->sp2);
  if (const char * ck = std::getenv("VSG_CKPT")) { if (ck[0] == '0') { c->ckpt_enabled = false; } }
  const char * df = std::getenv("VSG_DISABLE_FAST");
  c->fast_disabled = (df != nullptr && df[0] == '1');
  const char * db = std::getenv("VSG_DIR_BUDGET_MB");
  if (db != nullptr && std::atoll(db) > 0) { c->dir_budget = static_cast<size_t>(std::atoll(db)) << 20; }
  else {
    // scratch for direction bits / checkpoints: at most 64 GiB, and no more than 40 % of what the device has free
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && free_b > 0) {
      c->dir_budget = std::max<size_t>(std::min<size_t>(c->dir_budget, free_b / 5 * 2), static_cast<size_t>(256) << 20);
    }
  }
  VSG_CUDA_OK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  for (auto & ev : c->ev) { VSG_CUDA_OK(cudaEventCreate(&ev)); }
  // the fast kernel leans on VIMNMX.S16x2 predicate semantics: check them on this device once
  int * d_bad = nullptr;
  VSG_CUDA_OK(cudaMalloc(&d_bad, sizeof(int)));
  dpx_selftest_kernel<<<1, 1, 0, c->stream>>>(d_bad, 5, 9, 7, 9, -3, -10, -4, 2);
  count_launch();
  int bad = -1;
  VSG_CUDA_OK(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  cudaFree(d_bad);
  if (bad != 0) {
    Error::set("DPX self-test failed (code " + std::to_string(bad) + "): __vibmax_u16x2/__vadd2/__viaddmax_u16x2/__vimax3_u16x2 semantics differ");
    return VSG_ECUDA;
  }
  *out = guard.release();
  return VSG_OK;
}

extern "C" void vsg_ctx_destroy(vsg_ctx * c)
{
  if (c == nullptr) { return; }
  for (vsg_ctx * ch : c->children) { vsg_ctx_destroy(ch); }
  c->children.clear();
  cudaSetDevice(c->device);
  if (c->stream != nullptr) { cudaStreamSynchronize(c->stream); }
  for (DevBuf * b : {&c->dir, &c->bnd, &c->he, &c->cigar_scratch, &c->cigar_dense, &c->stats,
                     &c->tasks_fast, &c->tasks_exact, &c->pairs, &c->cigar_len, &c->cigar_offs,
                     &c->cub_tmp, &c->rank_tmp, &c->rank_scratch, &c->pre_flags, &c->ticket,
                     &c->rall_q, &c->rall_hist, &c->rall_keys, &c->rall_out, &c->rall_tmp}) { b->release(); }
  for (PinBuf * b : {&c->h_tasks, &c->h_stats}) { b->release(); }
  for (auto & ev : c->ev) { if (ev != nullptr) { cudaEventDestroy(ev); } }
  for (auto & ev : c->ev_pool) { cudaEventDestroy(ev); }
  if (c->stream != nullptr) { cudaStreamDestroy(c->stream); }
  delete c;
}

extern "C" int vsg_ctx_set_fallback(vsg_ctx * c, vsg_fallback_fn fn, void * user)
{
  if (c == nullptr) { return VSG_EINVAL; }
  c->fallback = fn;
  c->fallback_user = user;
  return VSG_OK;
}

extern "C" void * vsg_ctx_stream(vsg_ctx * c) { return c != nullptr ? static_cast<void *>(c->stream) : nullptr; }

extern "C" int vsg_ctx_sync(vsg_ctx * c)
{
  if (c == nullptr) { return VSG_EINVAL; }
  VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  return VSG_OK;
}

// ---- sequence sets ---------------------------------------------------------------------------
extern "C" int vsg_seqset_create(vsg_ctx * c, const char * cat, const int64_t * off, const int32_t * len,
                                 int64_t n, int host, vsg_seqset ** out)
{
  if (c == nullptr || out == nullptr || n < 0 || (n > 0 && (cat == nullptr || off == nullptr || len == nullptr))) {
    Error::set("vsg_seqset_create: bad argument");
    return VSG_EINVAL;
  }
  *out = nullptr;
  VSG_CUDA_OK(cudaSetDevice(c->device));
  vsg_seqset * s = new (std::nothrow) vsg_seqset();
  if (s == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  SeqsetGuard guard{s};   // destroys s on every early return
  s->device = c->device;
  s->h_len.resize(static_cast<size_t>(n));
  std::vector<int64_t> h_off(static_cast<size_t>(n));
  if (host != 0) {
    if (n > 0) {
      std::memcpy(s->h_len.data(), len, sizeof(int32_t) * static_cast<size_t>(n));
      std::memcpy(h_off.data(), off, sizeof(int64_t) * static_cast<size_t>(n));
    }
  } else if (n > 0) {
    VSG_CUDA_OK(cudaMemcpyAsync(s->h_len.data(), len, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, c->stream));
    VSG_CUDA_OK(cudaMemcpyAsync(h_off.data(), off, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, c->stream));
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  }
  int64_t total = 0;
  for (int64_t i = 0; i < n; i++) {
    if (s->h_len[i] < 0 || h_off[i] < 0) { Error::set("vsg_seqset_create: negative length/offset"); return VSG_EINVAL; }
    total = std::max<int64_t>(total, h_off[i] + s->h_len[i]);
  }
  s->total = total;
  s->h_off = h_off;
  int rc;
  if ((rc = s->b_sym.reserve(static_cast<size_t>(total) + 64)) != VSG_OK ||
      (rc = s->b_off.reserve(sizeof(int64_t) * static_cast<size_t>(n) + 8)) != VSG_OK ||
      (rc = s->b_len.reserve(sizeof(int32_t) * static_cast<size_t>(n) + 8)) != VSG_OK) {
    return rc;
  }
  const char * d_ascii = cat;
  ScopedBuf tmp_ascii_g;
  DevBuf & tmp_ascii = tmp_ascii_g.b;
  if (host != 0 && total > 0) {
    if ((rc = tmp_ascii.reserve(static_cast<size_t>(total))) != VSG_OK) { return rc; }
    VSG_CUDA_OK(cudaMemcpyAsync(tmp_ascii.p, cat, static_cast<size_t>(total), cudaMemcpyHostToDevice, c->stream));
    d_ascii = static_cast<const char *>(tmp_ascii.p);
  }
  if (n > 0) {
    VSG_CUDA_OK(cudaMemcpyAsync(s->b_off.p, h_off.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice, c->stream));
    VSG_CUDA_OK(cudaMemcpyAsync(s->b_len.p, s->h_len.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, c->stream));
  }
  s->d.sym = static_cast<uint8_t *>(s->b_sym.p);
  s->d.off = static_cast<int64_t *>(s->b_off.p);
  s->d.len = static_cast<int32_t *>(s->b_len.p);
  s->d.n = n;
  s->h_nonacgt.assign(static_cast<size_t>(n), 0);
  if (total > 0) {
    int64_t const blocks = (total + 255) / 256;
    encode_kernel<<<static_cast<unsigned>(blocks), 256, 0, c->stream>>>(d_ascii, static_cast<uint8_t *>(s->b_sym.p), total);
    count_launch();
  }
  if (n > 0) {
    ScopedBuf flag_g;
    DevBuf & flag = flag_g.b;
    if ((rc = flag.reserve(static_cast<size_t>(n))) != VSG_OK) { return rc; }
    int64_t const blocks = (n * 32 + 255) / 256;
    nonacgt_kernel<<<static_cast<unsigned>(blocks), 256, 0, c->stream>>>(s->d, static_cast<uint8_t *>(flag.p));
    count_launch();
    VSG_CUDA_OK(cudaMemcpyAsync(s->h_nonacgt.data(), flag.p, static_cast<size_t>(n), cudaMemcpyDeviceToHost, c->stream));
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
    flag.release();
  } else {
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  }
  tmp_ascii.release();
  VSG_CUDA_OK(cudaGetLastError());
  *out = guard.release();
  return VSG_OK;
}

extern "C" void vsg_seqset_destroy(vsg_seqset * s)
{
  if (s == nullptr) { return; }
  cudaSetDevice(s->device);
  s->b_sym.release(); s->b_off.release(); s->b_len.release();
  delete s;
}

namespace vsg {
int seqset_revcomp(vsg_ctx * c, const vsg_seqset * src, int64_t q0, int64_t n, vsg_seqset ** out)
{
  *out = nullptr;
  vsg_seqset * s = new (std::nothrow) vsg_seqset();
  if (s == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  SeqsetGuard guard{s};
  s->device = c->device;
  s->h_len.assign(src->h_len.begin() + q0, src->h_len.begin() + q0 + n);
  s->h_nonacgt.assign(src->h_nonacgt.begin() + q0, src->h_nonacgt.begin() + q0 + n);
  std::vector<int64_t> h_off(static_cast<size_t>(n));
  int64_t total = 0;
  for (int64_t i = 0; i < n; i++) { h_off[static_cast<size_t>(i)] = total; total += s->h_len[static_cast<size_t>(i)]; }
  s->total = total;
  s->h_off = h_off;
  int rc;
  if ((rc = s->b_sym.reserve(static_cast<size_t>(total) + 64)) != VSG_OK ||
      (rc = s->b_off.reserve(sizeof(int64_t) * static_cast<size_t>(n) + 8)) != VSG_OK ||
      (rc = s->b_len.reserve(sizeof(int32_t) * static_cast<size_t>(n) + 8)) != VSG_OK) {
    return rc;
  }
  s->d.sym = static_cast<uint8_t *>(s->b_sym.p);
  s->d.off = static_cast<int64_t *>(s->b_off.p);
  s->d.len = static_cast<int32_t *>(s->b_len.p);
  s->d.n = n;
  if (n > 0) {
    VSG_CUDA_OK(cudaMemcpyAsync(s->b_off.p, h_off.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice, c->stream));
    VSG_CUDA_OK(cudaMemcpyAsync(s->b_len.p, s->h_len.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, c->stream));
    int64_t const blocks = (n * 32 + 255) / 256;
    revcomp_kernel<<<static_cast<unsigned>(blocks), 256, 0, c->stream>>>(src->d, q0, n, s->d.off, static_cast<uint8_t *>(s->b_sym.p));
    count_launch();
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));  // h_off goes out of scope
  }
  *out = guard.release();
  return VSG_OK;
}

// the query set of a --strand both clustering: 2n entries, 2i = sequence i as stored (case = its mask), 2i + 1 = its
// reverse complement, back to back, so that the two strands of consecutive sequences form one contiguous range
int seqset_strand_pairs(vsg_ctx * c, const vsg_seqset * src, vsg_seqset ** out)
{
  *out = nullptr;
  vsg_seqset * s = new (std::nothrow) vsg_seqset();
  if (s == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  SeqsetGuard guard{s};
  int64_t const n = src->d.n, m = 2 * n;
  s->device = c->device;
  s->h_len.resize(static_cast<size_t>(m));
  s->h_off.resize(static_cast<size_t>(m));
  s->h_nonacgt.resize(static_cast<size_t>(m));
  int64_t total = 0;
  for (int64_t i = 0; i < n; i++) {
    int32_t const l = src->h_len[static_cast<size_t>(i)];
    for (int64_t e = 2 * i; e < 2 * i + 2; e++) {
      s->h_len[static_cast<size_t>(e)] = l;
      s->h_off[static_cast<size_t>(e)] = total;
      s->h_nonacgt[static_cast<size_t>(e)] = src->h_nonacgt[static_cast<size_t>(i)];
      total += l;
    }
  }
  s->total = total;
  int rc;
  if ((rc = s->b_sym.reserve(static_cast<size_t>(total) + 64)) != VSG_OK ||
      (rc = s->b_off.reserve(sizeof(int64_t) * static_cast<size_t>(m) + 8)) != VSG_OK ||
      (rc = s->b_len.reserve(sizeof(int32_t) * static_cast<size_t>(m) + 8)) != VSG_OK) {
    return rc;
  }
  s->d.sym = static_cast<uint8_t *>(s->b_sym.p);
  s->d.off = static_cast<int64_t *>(s->b_off.p);
  s->d.len = static_cast<int32_t *>(s->b_len.p);
  s->d.n = m;
  if (n > 0) {
    VSG_CUDA_OK(cudaMemcpyAsync(s->b_off.p, s->h_off.data(), sizeof(int64_t) * m, cudaMemcpyHostToDevice, c->stream));
    VSG_CUDA_OK(cudaMemcpyAsync(s->b_len.p, s->h_len.data(), sizeof(int32_t) * m, cudaMemcpyHostToDevice, c->stream));
    int64_t const blocks = (n * 32 + 255) / 256;
    strand_pairs_kernel<<<static_cast<unsigned>(blocks), 256, 0, c->stream>>>(src->d, s->d.off, static_cast<uint8_t *>(s->b_sym.p));
    count_launch();
    VSG_CUDA_OK(cudaGetLastError());
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  }
  *out = guard.release();
  return VSG_OK;
}
}  // namespace vsg

extern "C" int vsg_seqset_revcomp(vsg_ctx * c, const vsg_seqset * src, int64_t q0, int64_t n, vsg_seqset ** out)
{
  if (c == nullptr || src == nullptr || out == nullptr || q0 < 0 || n < 0 || q0 + n > src->d.n) {
    Error::set("vsg_seqset_revcomp: bad argument");
    return VSG_EINVAL;
  }
  *out = nullptr;
  if (src->device != c->device) { Error::set("vsg_seqset_revcomp: the set belongs to another device"); return VSG_EINVAL; }
  VSG_CUDA_OK(cudaSetDevice(c->device));
  return seqset_revcomp(c, src, q0, n, out);
}

extern "C" int64_t vsg_seqset_count(const vsg_seqset * s) { return s != nullptr ? s->d.n : 0; }

// ---- the aligner -----------------------------------------------------------------------------
namespace {

template <int R, bool G, bool M>
void launch_fast_one(vsg_ctx * c, const DevSeqs & qs, const DevSeqs & ts, const FastTask * d_tasks, int n)
{
  int const blocks = (n + FAST_WARPS - 1) / FAST_WARPS;
  constexpr size_t dyn = fast_dyn_smem(R, G);
  if (dyn > 48 * 1024) {  // opt in to > 48 KB of dynamic shared memory (per device, cheap: set every time)
    cudaFuncSetAttribute(nw_fast_kernel<R, G, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(dyn));
  }
  nw_fast_kernel<R, G, M><<<blocks, FAST_WARPS * 32, dyn, c->stream>>>(
      c->sp, qs, ts, d_tasks, n, static_cast<uint8_t *>(c->dir.p), static_cast<uint2 *>(c->bnd.p),
      static_cast<int32_t *>(c->stats.p));
  count_launch();
}

// multi: the tasks' queries need more than one strip of 32*R rows (only possible for R > 8)
void launch_fast(vsg_ctx * c, int R, bool general, bool multi, const DevSeqs & qs, const DevSeqs & ts,
                 const FastTask * d_tasks, int n)
{
  if (general) {
    switch (R) {
      case 4: launch_fast_one<4, true, false>(c, qs, ts, d_tasks, n); break;
      case 8: launch_fast_one<8, true, false>(c, qs, ts, d_tasks, n); break;
      default: launch_fast_one<16, true, true>(c, qs, ts, d_tasks, n); break;
    }
    return;
  }
  switch (R) {
#define VSG_CASE(r) case r: launch_fast_one<r, false, false>(c, qs, ts, d_tasks, n); break;
    VSG_CASE(1) VSG_CASE(2) VSG_CASE(3) VSG_CASE(4) VSG_CASE(5) VSG_CASE(6) VSG_CASE(7) VSG_CASE(8)
#undef VSG_CASE
#define VSG_CASE(r) case r: if (multi) { launch_fast_one<r, false, true>(c, qs, ts, d_tasks, n); } \
                            else { launch_fast_one<r, false, false>(c, qs, ts, d_tasks, n); } break;
    VSG_CASE(9) VSG_CASE(10) VSG_CASE(11) VSG_CASE(12) VSG_CASE(13) VSG_CASE(14) VSG_CASE(15)
    default: if (multi) { launch_fast_one<16, false, true>(c, qs, ts, d_tasks, n); }
             else { launch_fast_one<16, false, false>(c, qs, ts, d_tasks, n); } break;
#undef VSG_CASE
  }
}

// checkpoint forward kernel (align_ckpt.cuh): plain-ACGT tasks use the per-lane profile up to 8 rows per lane and
// the lane-replicated table above; tasks with IUPAC symbols the 16x16x16 table at 4, 8 or 16 rows per lane
template <int R, int MODE>
void launch_ckpt_one(vsg_ctx * c, const DevSeqs & qs, const DevSeqs & ts, const FastTask * d_tasks, int n)
{
  int const blocks = (n + FAST_WARPS - 1) / FAST_WARPS;
  constexpr size_t dyn = ck_dyn_smem(R, MODE);
  if (dyn > 48 * 1024) {
    cudaFuncSetAttribute(nw_ckpt_kernel<R, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(dyn));
  }
  nw_ckpt_kernel<R, MODE><<<blocks, FAST_WARPS * 32, dyn, c->stream>>>(
      c->sp2, qs, ts, d_tasks, n, static_cast<uint2 *>(c->dir.p), static_cast<uint2 *>(c->bnd.p),
      static_cast<int32_t *>(c->stats.p));
  count_launch();
}

void launch_ckpt(vsg_ctx * c, int R, bool general, const DevSeqs & qs, const DevSeqs & ts, const FastTask * d_tasks, int n)
{
  if (general) {
    switch (R) {
      case 4: launch_ckpt_one<4, CK_GEN>(c, qs, ts, d_tasks, n); break;
      case 8: launch_ckpt_one<8, CK_GEN>(c, qs, ts, d_tasks, n); break;
      default: launch_ckpt_one<16, CK_GEN>(c, qs, ts, d_tasks, n); break;
    }
    return;
  }
  static const bool force_lut = std::getenv("VSG_CK_LUT") != nullptr;   // experiment: table variant (more resident warps) for R <= 8 too
  if (force_lut && R == 8) { launch_ckpt_one<8, CK_LUT>(c, qs, ts, d_tasks, n); return; }
  switch (R) {
#define VSG_CASE(r) case r: launch_ckpt_one<r, CK_PROF>(c, qs, ts, d_tasks, n); break;
    VSG_CASE(1) VSG_CASE(2) VSG_CASE(3) VSG_CASE(4) VSG_CASE(5) VSG_CASE(6) VSG_CASE(7) VSG_CASE(8)
#undef VSG_CASE
#define VSG_CASE(r) case r: launch_ckpt_one<r, CK_LUT>(c, qs, ts, d_tasks, n); break;
    VSG_CASE(9) VSG_CASE(10) VSG_CASE(11) VSG_CASE(12) VSG_CASE(13) VSG_CASE(14) VSG_CASE(15)
    default: launch_ckpt_one<16, CK_LUT>(c, qs, ts, d_tasks, n); break;
#undef VSG_CASE
  }
}

int launch_tb_ckpt_tasks(vsg_ctx * c, int R, bool general, const DevSeqs & qs, const DevSeqs & ts, const FastTask * d_tasks, int n,
                         const TbGate & gate)
{
  // a grid that fills the device once (the kernel hands further pairs out itself), fewer blocks for small calls
  int rc;
  if ((rc = c->ticket.reserve(64)) != VSG_OK) { return rc; }
  VSG_CUDA_OK(cudaMemsetAsync(c->ticket.p, 0, sizeof(int), c->stream));
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
  int const nthr = gate.ids != nullptr ? gate.nids : 2 * n;
  if (nthr == 0) { return VSG_OK; }
  int const want = (nthr + TB_CK_THREADS - 1) / TB_CK_THREADS;
  static int const refill = [] { const char * e = std::getenv("VSG_TB_REFILL"); return e != nullptr ? std::atoi(e) : 0; }();
  int const tbase = refill > 0 ? 0 : nthr;   // >= the number of pairs: every thread does its own pair only
  if (R <= 8) {
    cudaFuncSetAttribute(traceback_ckpt_tasks_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tb_ck_smem(8)));
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, traceback_ckpt_tasks_kernel<8>, TB_CK_THREADS, tb_ck_smem(8));
    int const blocks = refill > 0 ? std::min(want, std::max(1, per_sm) * sms * refill) : want;
    traceback_ckpt_tasks_kernel<8><<<blocks, TB_CK_THREADS, tb_ck_smem(8), c->stream>>>(
        c->sp2, qs, ts, d_tasks, n, R, general ? 1 : 0, static_cast<const uint2 *>(c->dir.p), static_cast<const uint2 *>(c->bnd.p),
        static_cast<int32_t *>(c->stats.p), static_cast<int *>(c->ticket.p), tbase, gate);
  } else {
    cudaFuncSetAttribute(traceback_ckpt_tasks_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tb_ck_smem(16)));
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, traceback_ckpt_tasks_kernel<16>, TB_CK_THREADS, tb_ck_smem(16));
    int const blocks = refill > 0 ? std::min(want, std::max(1, per_sm) * sms * refill) : want;
    traceback_ckpt_tasks_kernel<16><<<blocks, TB_CK_THREADS, tb_ck_smem(16), c->stream>>>(
        c->sp2, qs, ts, d_tasks, n, R, general ? 1 : 0, static_cast<const uint2 *>(c->dir.p), static_cast<const uint2 *>(c->bnd.p),
        static_cast<int32_t *>(c->stats.p), static_cast<int *>(c->ticket.p), tbase, gate);
  }
  count_launch();
  return VSG_OK;
}

// A chunk = the tasks whose direction blocks share the scratch buffer at the same time.
struct ClassRun { int R; bool general, multi, ckpt; size_t first; int count; };  // a run of one kernel class in all_fast
struct ChunkPlan {
  std::vector<ClassRun> runs;
  size_t exact_first = 0; int exact_count = 0;
  size_t pair_first = 0; int pair_count = 0;  // descriptors (CIGAR mode only)
  uint64_t dir_bytes = 0, bnd_elems = 0, he_elems = 0, cigar_bytes = 0;
  int64_t cells = 0, nfast = 0, nexact = 0;
};

struct ChunkBuilder {  // the chunk being filled
  std::vector<FastTask> fast[2][3][FAST_RMAX + 1];  // [general][0 = one strip, direction bits; 1 = several strips; 2 = checkpoints][rows per lane]
  std::vector<ExactTask> exact;
  uint64_t dir_bytes = 0, bnd_elems = 0, he_elems = 0, cigar_bytes = 0;
  int64_t cells = 0, nfast = 0, nexact = 0;
  int npairdesc = 0;
  bool empty() const { return nfast == 0 && nexact == 0; }
};

inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

}  // namespace

extern "C" int vsg_align_pairs(vsg_ctx * c, const vsg_seqset * queries, const vsg_seqset * targets,
                               int64_t npairs, const uint32_t * qidx, const uint32_t * tidx,
                               int16_t * score, uint16_t * aligned, uint16_t * matches,
                               uint16_t * mismatches, uint16_t * gaps, int32_t * trims,
                               char * cigar_buf, int64_t cigar_cap, int64_t * cigar_off)
{
  return vsg::align_pairs_gated(c, queries, targets, npairs, qidx, tidx, score, aligned, matches, mismatches, gaps, trims,
                                cigar_buf, cigar_cap, cigar_off, nullptr, 0.0, 2);
}

// leader_of (optional, npairs entries, statistics-only calls): traceback on demand, see align_ckpt.cuh (TbGate).  A pair
// whose walk was skipped comes back with aligned = matches = mismatches = 0xffff.
int vsg::align_pairs_gated(vsg_ctx * c, const vsg_seqset * queries, const vsg_seqset * targets,
                           int64_t npairs, const uint32_t * qidx, const uint32_t * tidx,
                           int16_t * score, uint16_t * aligned, uint16_t * matches,
                           uint16_t * mismatches, uint16_t * gaps, int32_t * trims,
                           char * cigar_buf, int64_t cigar_cap, int64_t * cigar_off,
                           const int32_t * leader_of, double gate_threshold, int gate_iddef)
{
  if (c == nullptr || queries == nullptr || targets == nullptr || npairs < 0 ||
      (npairs > 0 && (qidx == nullptr || tidx == nullptr || score == nullptr))) {
    Error::set("vsg_align_pairs: bad argument");
    return VSG_EINVAL;
  }
  if (npairs > (1LL << 30)) { Error::set("vsg_align_pairs: too many pairs in one call"); return VSG_EINVAL; }
  if (queries->device != c->device || targets->device != c->device) { Error::set("vsg_align_pairs: sequence set lives on another device than the context"); return VSG_EINVAL; }
  VSG_CUDA_OK(cudaSetDevice(c->device));
  static const bool trace = std::getenv("VSG_TRACE") != nullptr;
  auto const t_begin = std::chrono::steady_clock::now();
  bool const want_cigar = (cigar_buf != nullptr);
  if (want_cigar && cigar_off == nullptr) { Error::set("vsg_align_pairs: cigar_off required with cigar_buf"); return VSG_EINVAL; }
  if (npairs == 0) { if (want_cigar) { cigar_off[0] = 0; } return VSG_OK; }

  int rc;
  // final home of the per-pair statistics: pinned, written by one D2H at the end (GPU pairs) and by
  // the host directly (pairs resolved without DP)
  if ((rc = c->h_stats.reserve(sizeof(int32_t) * VSG_STAT_WORDS * static_cast<size_t>(npairs))) != VSG_OK) { return rc; }
  if ((rc = c->stats.reserve(sizeof(int32_t) * VSG_STAT_WORDS * static_cast<size_t>(npairs) + 64)) != VSG_OK) { return rc; }
  int32_t * const hs = static_cast<int32_t *>(c->h_stats.p);
  struct HostPair { int64_t slot; int32_t st[VSG_STAT_WORDS]; };
  std::vector<HostPair> host_pairs;
  std::vector<std::string> cigars;
  if (want_cigar) { cigars.resize(static_cast<size_t>(npairs)); }

  ScoreParams const & sp = c->sp;
  FastBound const fbound = fast_bound_of(sp);
  FastBound const fbound2 = fast_bound_of(c->sp2);
  // Small calls are latency-bound (the cluster driver's rounds, the tail rounds of a search).  For sequences of
  // similar length one thread regenerating ~40 tiles takes a few hundred microseconds whatever the batch size while
  // walking stored direction bits takes tens: below VSG_CKPT_MIN_PAIRS pairs (default 2048) such pairs use the
  // direction-bit kernels.  A target several times longer than the query turns that around — the walk over stored
  // bits pays one dependent HBM load per column of the end gap, the regenerated tiles cross it 32 columns at a time
  // — so those pairs stay on the checkpoint kernels at any call size.  Both paths are bit-identical
  // (tests/test_stress_gpu.py runs either).
  const char * const ckpt_min_env = std::getenv("VSG_CKPT_MIN_PAIRS");   // read per call: tests switch it
  int64_t const ckpt_min_pairs = ckpt_min_env != nullptr ? std::atoll(ckpt_min_env) : 2048LL;
  bool const ckpt_any_size = c->ckpt_enabled && npairs >= ckpt_min_pairs;
  std::vector<FastTask> all_fast;
  std::vector<ExactTask> all_exact;
  std::vector<PairDesc> all_pairs;  // CIGAR mode only
  std::vector<ChunkPlan> plans;
  ChunkBuilder cb;
  all_fast.reserve(static_cast<size_t>(npairs) / 2 + 16);
  struct Cand { int64_t slot; uint32_t t; int32_t d; bool general; };
  std::vector<Cand> group_fast;

  auto host_pair = [&](int64_t slot) -> int32_t * {
    host_pairs.emplace_back();
    host_pairs.back().slot = slot;
    std::memset(host_pairs.back().st, 0, sizeof(int32_t) * VSG_STAT_WORDS);
    return host_pairs.back().st;
  };

  auto close_chunk = [&]() {
    if (cb.empty()) { return; }
    ChunkPlan pl;
    for (int gm = 0; gm < 6; gm++) {
      int const g = gm / 3, m = gm % 3;
      for (int R = 1; R <= FAST_RMAX; R++) {
        auto & v = cb.fast[g][m][R];
        if (v.empty()) { continue; }
        // longest first: the tail of the grid is made of the short ones
        auto const longer = [](const FastTask & a, const FastTask & b) { return a.dmax > b.dmax; };
        if (!std::is_sorted(v.begin(), v.end(), longer)) { std::sort(v.begin(), v.end(), longer); }
        pl.runs.push_back(ClassRun{R, g != 0, m == 1, m == 2, all_fast.size(), static_cast<int>(v.size())});
        all_fast.insert(all_fast.end(), v.begin(), v.end());
        v.clear();
      }
    }
    pl.exact_first = all_exact.size(); pl.exact_count = static_cast<int>(cb.exact.size());
    all_exact.insert(all_exact.end(), cb.exact.begin(), cb.exact.end());
    cb.exact.clear();
    pl.pair_first = all_pairs.size() - static_cast<size_t>(cb.npairdesc); pl.pair_count = cb.npairdesc;
    pl.dir_bytes = cb.dir_bytes; pl.bnd_elems = cb.bnd_elems; pl.he_elems = cb.he_elems; pl.cigar_bytes = cb.cigar_bytes;
    pl.cells = cb.cells; pl.nfast = cb.nfast; pl.nexact = cb.nexact;
    plans.push_back(std::move(pl));
    cb.dir_bytes = cb.bnd_elems = cb.he_elems = cb.cigar_bytes = 0;
    cb.cells = cb.nfast = cb.nexact = 0; cb.npairdesc = 0;
  };

  auto add_pairdesc = [&](uint32_t q, uint32_t t, int kind, int64_t slot, int R, int half, int dmax, uint64_t dir_off, uint64_t aux_off = 0) {
    if (!want_cigar) { return; }
    PairDesc pd{};
    pd.q = q; pd.t = t; pd.dir_off = dir_off; pd.kind = kind; pd.out = static_cast<int32_t>(slot);
    pd.R = R; pd.half = half; pd.dmax = dmax; pd.aux_off = aux_off;
    pd.cigar_off = cb.cigar_bytes;
    cb.cigar_bytes += static_cast<uint64_t>(queries->h_len[q]) + static_cast<uint64_t>(targets->h_len[t]) + 2;
    all_pairs.push_back(pd);
    cb.npairdesc++;
  };

  // ---- plan: resolve trivial pairs on the host, group by query, pair targets two by two ----------
  int64_t i = 0;
  while (i < npairs) {
    uint32_t const q = qidx[i];
    if (q >= static_cast<uint64_t>(queries->d.n)) { Error::set("vsg_align_pairs: query index out of range"); return VSG_EINVAL; }
    int64_t j = i;
    while (j < npairs && qidx[j] == q) { j++; }
    int const Q = queries->h_len[q];
    bool const q_general = queries->h_nonacgt[q] != 0;
    group_fast.clear();
    for (int64_t k = i; k < j; k++) {
      uint32_t const t = tidx[k];
      if (t >= static_cast<uint64_t>(targets->d.n)) { Error::set("vsg_align_pairs: target index out of range"); return VSG_EINVAL; }
      int const D = targets->h_len[t];
      if (sp.fallback) { host_pair(k)[VSG_STAT_SCORE] = VSG_SCORE_SENTINEL; continue; }  // align_simd.cpp:1463-1479
      if (Q == 0) {                                                                      // align_simd.cpp:1481-1539
        int32_t * s = host_pair(k);
        if (!fits16(0, D)) { s[VSG_STAT_SCORE] = VSG_SCORE_SENTINEL; continue; }
        s[VSG_STAT_ALIGNED] = D; s[VSG_STAT_GAPS] = D;
        if (D > 0) {
          int64_t const a = -static_cast<int64_t>(sp.go[T_L]) - static_cast<int64_t>(D) * sp.ge[T_L];
          int64_t const b = -static_cast<int64_t>(sp.go[T_R]) - static_cast<int64_t>(D) * sp.ge[T_R];
          s[VSG_STAT_SCORE] = static_cast<int16_t>(std::max(a, b));
          s[VSG_STAT_TRIM_LEFT] = -D; s[VSG_STAT_TRIM_RIGHT] = -D;
          if (want_cigar) { cigars[static_cast<size_t>(k)] = std::to_string(D) + "I"; }
          s[VSG_STAT_CIGARLEN] = static_cast<int32_t>(std::to_string(D).size() + 1);
        }
        continue;
      }
      if (D == 0 || !fits16(Q, D)) { host_pair(k)[VSG_STAT_SCORE] = VSG_SCORE_SENTINEL; continue; }  // :1867-1882
      bool const general = q_general || targets->h_nonacgt[t] != 0;
      int R, ns;
      fast_shape(Q, general, R, ns);
      if (!c->fast_disabled && fast_path_ok(fbound, ns * 32 * R, D)) {
        group_fast.push_back(Cand{k, t, D, general});
      } else {
        uint64_t const dirb = align_up(static_cast<uint64_t>(Q) * D, 16);
        if (!cb.empty() && cb.dir_bytes + dirb > c->dir_budget) { close_chunk(); }
        ExactTask et{};
        et.q = q; et.t = t; et.out = static_cast<int32_t>(k);
        et.dir_off = cb.dir_bytes; et.he_off = cb.he_elems;
        add_pairdesc(q, t, 1, k, 0, 0, 0, cb.dir_bytes);
        cb.dir_bytes += dirb;
        cb.he_elems += 2ULL * Q;
        cb.exact.push_back(et);
        cb.cells += static_cast<int64_t>(Q) * D; cb.nexact++;
      }
    }
    if (!group_fast.empty()) {
      // similar lengths together (a warp runs for the longer of its two targets)
      auto const by_len = [](const Cand & a, const Cand & b) {
        if (a.general != b.general) { return a.general < b.general; }
        if (a.d != b.d) { return a.d > b.d; }
        return a.slot < b.slot;
      };
      if (!std::is_sorted(group_fast.begin(), group_fast.end(), by_len)) { std::sort(group_fast.begin(), group_fast.end(), by_len); }
      size_t k = 0;
      while (k < group_fast.size()) {
        Cand const & a = group_fast[k];
        bool const pair2 = (k + 1 < group_fast.size()) && (group_fast[k + 1].general == a.general);
        Cand const & b = pair2 ? group_fast[k + 1] : a;
        int R, ns;
        fast_shape(Q, a.general, R, ns);
        int const dmax = std::max(a.d, b.d);
        // single-strip tasks go through the checkpoint kernel (no direction bits; align_ckpt.cuh) when its
        // shifted scoring stays inside the exact range too
        bool const ck = (ns == 1) && c->ckpt_enabled && (ckpt_any_size || dmax >= 3 * Q) && fast_path_ok(fbound2, 32 * R, dmax);
        uint64_t const dirb = ck ? ck_row_elems(dmax) * sizeof(uint2) : static_cast<uint64_t>(ns) * fast_strip_bytes(dmax, R);
        uint64_t const auxe = ck ? ck_col_elems(dmax, R) : (ns > 1 ? static_cast<uint64_t>(dmax) : 0);
        if (!cb.empty() && cb.dir_bytes + dirb + (cb.bnd_elems + auxe) * sizeof(uint2) > c->dir_budget) { close_chunk(); }
        FastTask ft{};
        ft.q = q; ft.tlo = a.t; ft.thi = b.t;
        ft.out_lo = static_cast<int32_t>(a.slot);
        ft.out_hi = pair2 ? static_cast<int32_t>(b.slot) : -1;
        ft.dmax = dmax;
        ft.dir_off = ck ? cb.dir_bytes / sizeof(uint2) : cb.dir_bytes;   // checkpoints: uint2 element offsets
        ft.bnd_off = cb.bnd_elems;
        int const gbit = a.general ? 2 : 0;
        add_pairdesc(q, a.t, ck ? 2 : 0, a.slot, R, ck ? gbit : 0, dmax, ft.dir_off, ft.bnd_off);
        if (pair2) { add_pairdesc(q, b.t, ck ? 2 : 0, b.slot, R, ck ? (gbit | 1) : 1, dmax, ft.dir_off, ft.bnd_off); }
        cb.dir_bytes += align_up(dirb, 32);
        cb.bnd_elems += auxe;
        cb.fast[a.general ? 1 : 0][ck ? 2 : (ns > 1 ? 1 : 0)][R].push_back(ft);
        cb.cells += static_cast<int64_t>(Q) * a.d + (pair2 ? static_cast<int64_t>(Q) * b.d : 0);
        cb.nfast += pair2 ? 2 : 1;
        k += pair2 ? 2 : 1;
      }
    }
    i = j;
  }
  close_chunk();
  auto const t_planned = std::chrono::steady_clock::now();

  // ---- upload every task of the call once; size the scratch for the largest chunk ----------------
  uint64_t max_dir = 0, max_bnd = 0, max_he = 0, max_cig = 0;
  for (auto const & pl : plans) {
    max_dir = std::max(max_dir, pl.dir_bytes); max_bnd = std::max(max_bnd, pl.bnd_elems);
    max_he = std::max(max_he, pl.he_elems); max_cig = std::max(max_cig, pl.cigar_bytes);
  }
  if (!plans.empty()) {
    if ((rc = c->dir.reserve(max_dir + 256)) != VSG_OK) { return rc; }
    if ((rc = c->bnd.reserve(sizeof(uint2) * (max_bnd + 1))) != VSG_OK) { return rc; }
    if ((rc = c->he.reserve(sizeof(int16_t) * (max_he + 1))) != VSG_OK) { return rc; }
    if ((rc = c->tasks_fast.reserve(sizeof(FastTask) * (all_fast.size() + 1))) != VSG_OK) { return rc; }
    if ((rc = c->tasks_exact.reserve(sizeof(ExactTask) * (all_exact.size() + 1))) != VSG_OK) { return rc; }
    size_t const fb = sizeof(FastTask) * all_fast.size(), eb = sizeof(ExactTask) * all_exact.size();
    if ((rc = c->h_tasks.reserve(fb + eb + 64)) != VSG_OK) { return rc; }
    char * hp = static_cast<char *>(c->h_tasks.p);
    if (fb > 0) {
      std::memcpy(hp, all_fast.data(), fb);
      VSG_CUDA_OK(cudaMemcpyAsync(c->tasks_fast.p, hp, fb, cudaMemcpyHostToDevice, c->stream));
    }
    if (eb > 0) {
      std::memcpy(hp + fb, all_exact.data(), eb);
      VSG_CUDA_OK(cudaMemcpyAsync(c->tasks_exact.p, hp + fb, eb, cudaMemcpyHostToDevice, c->stream));
    }
  }
  // traceback on demand: per checkpoint run, the pair ids of the leaders (and ungated pairs) and of the followers
  bool const gated = leader_of != nullptr && !want_cigar && !plans.empty();
  struct GateRun { size_t lead_first, lead_count, foll_first, foll_count; };
  std::vector<std::vector<GateRun>> gate_runs;
  int const * d_gate_ids = nullptr;
  int32_t const * d_leader = nullptr;
  if (gated) {
    std::vector<int> ids;
    ids.reserve(static_cast<size_t>(npairs));
    gate_runs.resize(plans.size());
    for (size_t ci = 0; ci < plans.size(); ci++) {
      for (auto const & run : plans[ci].runs) {
        GateRun g{ids.size(), 0, 0, 0};
        if (run.ckpt) {
          for (int pass = 0; pass < 2; pass++) {
            if (pass == 1) { g.lead_count = ids.size() - g.lead_first; g.foll_first = ids.size(); }
            for (int k = 0; k < run.count; k++) {
              FastTask const & ft = all_fast[run.first + static_cast<size_t>(k)];
              for (int half = 0; half < 2; half++) {
                int32_t const slot = half ? ft.out_hi : ft.out_lo;
                if (slot < 0) { continue; }
                bool const follower = leader_of[slot] >= 0;
                if (follower == (pass == 1)) { ids.push_back(2 * k + half); }
              }
            }
          }
          g.foll_count = ids.size() - g.foll_first;
        }
        gate_runs[ci].push_back(g);
      }
    }
    if ((rc = c->gate.reserve(sizeof(int) * (ids.size() + static_cast<size_t>(npairs)) + 64)) != VSG_OK) { return rc; }
    int * const dg = static_cast<int *>(c->gate.p);
    // pageable sources: both copies are staged before cudaMemcpyAsync returns
    if (!ids.empty()) { VSG_CUDA_OK(cudaMemcpyAsync(dg, ids.data(), sizeof(int) * ids.size(), cudaMemcpyHostToDevice, c->stream)); }
    VSG_CUDA_OK(cudaMemcpyAsync(dg + ids.size(), leader_of, sizeof(int32_t) * static_cast<size_t>(npairs), cudaMemcpyHostToDevice, c->stream));
    d_gate_ids = dg;
    d_leader = dg + ids.size();
    // "not computed" everywhere until a kernel says otherwise
    VSG_CUDA_OK(cudaMemsetAsync(c->stats.p, 0xff, sizeof(int32_t) * VSG_STAT_WORDS * static_cast<size_t>(npairs), c->stream));
  }
  // events: 3 per chunk
  while (c->ev_pool.size() < 3 * plans.size()) {
    cudaEvent_t e;
    VSG_CUDA_OK(cudaEventCreate(&e));
    c->ev_pool.push_back(e);
  }

  FastTask * const d_fast = static_cast<FastTask *>(c->tasks_fast.p);
  ExactTask * const d_exact = static_cast<ExactTask *>(c->tasks_exact.p);
  int32_t * const d_stats = static_cast<int32_t *>(c->stats.p);
  uint8_t * const d_dir = static_cast<uint8_t *>(c->dir.p);

  for (size_t ci = 0; ci < plans.size(); ci++) {
    ChunkPlan const & pl = plans[ci];
    VSG_CUDA_OK(cudaEventRecord(c->ev_pool[3 * ci], c->stream));
    for (auto const & run : pl.runs) {
      if (run.ckpt) { launch_ckpt(c, run.R, run.general, queries->d, targets->d, d_fast + run.first, run.count); }
      else { launch_fast(c, run.R, run.general, run.multi, queries->d, targets->d, d_fast + run.first, run.count); }
    }
    if (pl.exact_count > 0) {
      nw_exact_kernel<<<(pl.exact_count + 63) / 64, 64, 0, c->stream>>>(sp, queries->d, targets->d, d_exact + pl.exact_first,
                                                                        pl.exact_count, d_dir, static_cast<int16_t *>(c->he.p), d_stats);
      count_launch();
    }
    VSG_CUDA_OK(cudaEventRecord(c->ev_pool[3 * ci + 1], c->stream));
    if (!want_cigar) {
      TbGate const no_gate{nullptr, 0, nullptr, 0, 2, 0.0};
      if (gated) {
        // phase 1: leaders and ungated pairs of every checkpoint run (their verdicts must be in before any follower looks)
        for (size_t ri = 0; ri < pl.runs.size(); ri++) {
          auto const & run = pl.runs[ri];
          if (!run.ckpt) { continue; }
          GateRun const & g = gate_runs[ci][ri];
          TbGate const g1{d_gate_ids + g.lead_first, static_cast<int>(g.lead_count), d_leader, 1, gate_iddef, gate_threshold};
          if ((rc = launch_tb_ckpt_tasks(c, run.R, run.general, queries->d, targets->d, d_fast + run.first, run.count, g1)) != VSG_OK) { return rc; }
        }
      }
      for (size_t ri = 0; ri < pl.runs.size(); ri++) {
        auto const & run = pl.runs[ri];
        if (run.ckpt) {
          if (gated) {
            GateRun const & g = gate_runs[ci][ri];
            TbGate const g2{d_gate_ids + g.foll_first, static_cast<int>(g.foll_count), d_leader, 2, gate_iddef, gate_threshold};
            if ((rc = launch_tb_ckpt_tasks(c, run.R, run.general, queries->d, targets->d, d_fast + run.first, run.count, g2)) != VSG_OK) { return rc; }
            continue;
          }
          if ((rc = launch_tb_ckpt_tasks(c, run.R, run.general, queries->d, targets->d, d_fast + run.first, run.count, no_gate)) != VSG_OK) { return rc; }
          continue;
        }
        int const nthr = 2 * run.count;
        traceback_fast_tasks_kernel<<<(nthr + 127) / 128, 128, 0, c->stream>>>(sp, queries->d, targets->d, d_fast + run.first,
                                                                               run.count, run.R, d_dir, d_stats);
        count_launch();
      }
      if (pl.exact_count > 0) {
        traceback_exact_tasks_kernel<<<(pl.exact_count + 127) / 128, 128, 0, c->stream>>>(sp, queries->d, targets->d,
                                                                                         d_exact + pl.exact_first, pl.exact_count, d_dir, d_stats);
        count_launch();
      }
      VSG_CUDA_OK(cudaEventRecord(c->ev_pool[3 * ci + 2], c->stream));
    } else {
      // CIGAR texts: descriptors up, traceback with text, dense packing, texts home — per chunk
      int const np = pl.pair_count;
      if ((rc = c->pairs.reserve(sizeof(PairDesc) * (static_cast<size_t>(np) + 1))) != VSG_OK) { return rc; }
      if ((rc = c->cigar_scratch.reserve(pl.cigar_bytes + 64)) != VSG_OK) { return rc; }
      if ((rc = c->cigar_dense.reserve(pl.cigar_bytes + 64)) != VSG_OK) { return rc; }
      if ((rc = c->cigar_len.reserve(sizeof(int64_t) * (static_cast<size_t>(np) + 1))) != VSG_OK) { return rc; }
      if ((rc = c->cigar_offs.reserve(sizeof(int64_t) * (static_cast<size_t>(np) + 1))) != VSG_OK) { return rc; }
      PairDesc const * hpairs = all_pairs.data() + pl.pair_first;
      PairDesc * d_pairs = static_cast<PairDesc *>(c->pairs.p);
      VSG_CUDA_OK(cudaMemcpyAsync(d_pairs, hpairs, sizeof(PairDesc) * np, cudaMemcpyHostToDevice, c->stream));
      traceback_kernel<true><<<(np + 127) / 128, 128, 0, c->stream>>>(sp, queries->d, targets->d, d_pairs, np, d_dir,
                                                                      static_cast<char *>(c->cigar_scratch.p), d_stats);
      count_launch();
      bool ck8 = false, ck16 = false;
      for (auto const & run : pl.runs) { if (run.ckpt) { (run.R <= 8 ? ck8 : ck16) = true; } }
      int const tbb = (np + TB_CK_THREADS - 1) / TB_CK_THREADS;
      if (ck8) {
        cudaFuncSetAttribute(traceback_ckpt_pairs_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tb_ck_smem(8)));
        traceback_ckpt_pairs_kernel<8><<<tbb, TB_CK_THREADS, tb_ck_smem(8), c->stream>>>(c->sp2, queries->d, targets->d, d_pairs, np,
            static_cast<const uint2 *>(c->dir.p), static_cast<const uint2 *>(c->bnd.p), static_cast<char *>(c->cigar_scratch.p), d_stats);
        count_launch();
      }
      if (ck16) {
        cudaFuncSetAttribute(traceback_ckpt_pairs_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tb_ck_smem(16)));
        traceback_ckpt_pairs_kernel<16><<<tbb, TB_CK_THREADS, tb_ck_smem(16), c->stream>>>(c->sp2, queries->d, targets->d, d_pairs, np,
            static_cast<const uint2 *>(c->dir.p), static_cast<const uint2 *>(c->bnd.p), static_cast<char *>(c->cigar_scratch.p), d_stats);
        count_launch();
      }
      VSG_CUDA_OK(cudaEventRecord(c->ev_pool[3 * ci + 2], c->stream));
      cigar_len_kernel<<<(np + 255) / 256, 256, 0, c->stream>>>(d_pairs, d_stats, np, static_cast<int64_t *>(c->cigar_len.p));
      count_launch();
      size_t tmp_bytes = 0;
      cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, static_cast<int64_t *>(c->cigar_len.p),
                                    static_cast<int64_t *>(c->cigar_offs.p), np, c->stream);
      if ((rc = c->cub_tmp.reserve(tmp_bytes + 16)) != VSG_OK) { return rc; }
      cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp_bytes, static_cast<int64_t *>(c->cigar_len.p),
                                    static_cast<int64_t *>(c->cigar_offs.p), np, c->stream);
      count_launch();
      cigar_gather_kernel<<<np, 64, 0, c->stream>>>(d_pairs, np, queries->d, targets->d, d_stats,
                                                    static_cast<int64_t *>(c->cigar_offs.p),
                                                    static_cast<char *>(c->cigar_scratch.p), static_cast<char *>(c->cigar_dense.p));
      count_launch();
      std::vector<int64_t> h_offs(static_cast<size_t>(np)), h_lens(static_cast<size_t>(np));
      VSG_CUDA_OK(cudaMemcpyAsync(h_offs.data(), c->cigar_offs.p, sizeof(int64_t) * np, cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaMemcpyAsync(h_lens.data(), c->cigar_len.p, sizeof(int64_t) * np, cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
      int64_t const total = np > 0 ? h_offs[static_cast<size_t>(np) - 1] + h_lens[static_cast<size_t>(np) - 1] : 0;
      std::vector<char> dense(static_cast<size_t>(total) + 1);
      if (total > 0) {
        VSG_CUDA_OK(cudaMemcpyAsync(dense.data(), c->cigar_dense.p, static_cast<size_t>(total), cudaMemcpyDeviceToHost, c->stream));
        VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
      }
      for (int p = 0; p < np; p++) { cigars[static_cast<size_t>(hpairs[p].out)] = std::string(dense.data() + h_offs[static_cast<size_t>(p)]); }
    }
  }
  if (!plans.empty()) {
    VSG_CUDA_OK(cudaMemcpyAsync(hs, d_stats, sizeof(int32_t) * VSG_STAT_WORDS * static_cast<size_t>(npairs), cudaMemcpyDeviceToHost, c->stream));
  }
  VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  VSG_CUDA_OK(cudaGetLastError());
  for (size_t ci = 0; ci < plans.size(); ci++) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_pool[3 * ci], c->ev_pool[3 * ci + 1]) == cudaSuccess) { c->prof_fwd_ms += ms; }
    if (cudaEventElapsedTime(&ms, c->ev_pool[3 * ci + 1], c->ev_pool[3 * ci + 2]) == cudaSuccess) { c->prof_tb_ms += ms; }
    c->prof_cells += plans[ci].cells; c->prof_fast += plans[ci].nfast; c->prof_exact += plans[ci].nexact;
    c->prof_fwd_launches += static_cast<int64_t>(plans[ci].runs.size()) + (plans[ci].exact_count > 0 ? 1 : 0);
  }
  for (auto const & hp : host_pairs) { std::memcpy(hs + static_cast<size_t>(hp.slot) * VSG_STAT_WORDS, hp.st, sizeof(int32_t) * VSG_STAT_WORDS); }

  int64_t cpos = 0;
  for (int64_t k = 0; k < npairs; k++) {
    int32_t const * s = hs + static_cast<size_t>(k) * VSG_STAT_WORDS;
    if (gated && leader_of[k] >= 0 && s[VSG_STAT_ALIGNED] == -1 && s[VSG_STAT_MATCHES] == -1) { c->prof_tb_skipped++; }
    score[k] = static_cast<int16_t>(s[VSG_STAT_SCORE]);
    if (aligned != nullptr) { aligned[k] = static_cast<uint16_t>(s[VSG_STAT_ALIGNED]); }
    if (matches != nullptr) { matches[k] = static_cast<uint16_t>(s[VSG_STAT_MATCHES]); }
    if (mismatches != nullptr) { mismatches[k] = static_cast<uint16_t>(s[VSG_STAT_MISMATCHES]); }
    if (gaps != nullptr) { gaps[k] = static_cast<uint16_t>(s[VSG_STAT_GAPS]); }
    if (trims != nullptr) {
      int const tl = s[VSG_STAT_TRIM_LEFT], tr = s[VSG_STAT_TRIM_RIGHT];
      trims[4 * k + 0] = tl > 0 ? tl : 0;   // leading D  -> trim_q_left
      trims[4 * k + 1] = tl < 0 ? -tl : 0;  // leading I  -> trim_t_left
      trims[4 * k + 2] = tr > 0 ? tr : 0;
      trims[4 * k + 3] = tr < 0 ? -tr : 0;
    }
    if (want_cigar) {
      std::string const & cg = cigars[static_cast<size_t>(k)];
      if (cpos + static_cast<int64_t>(cg.size()) + 1 > cigar_cap) { Error::set("vsg_align_pairs: cigar buffer too small"); return VSG_ECAP; }
      cigar_off[k] = cpos;
      std::memcpy(cigar_buf + cpos, cg.c_str(), cg.size() + 1);
      cpos += static_cast<int64_t>(cg.size()) + 1;
    }
  }
  if (want_cigar) { cigar_off[npairs] = cpos; }
  if (trace) {
    auto const t_end = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[vsg trace] align_pairs %lld pairs, %zu chunk(s): plan %.1f ms, total %.1f ms\n",
                 static_cast<long long>(npairs), plans.size(),
                 std::chrono::duration<double, std::milli>(t_planned - t_begin).count(),
                 std::chrono::duration<double, std::milli>(t_end - t_begin).count());
  }
  return VSG_OK;
}

namespace vsg {
// Integer issue peak of an SM: independent chains, half of them a packed DPX instruction (VIADDMNMX.U16x2, ALU
// pipe), half a 32-bit multiply-add (IMAD, FMA pipe) — the mix the checkpoint forward kernel is made of.  Each pipe
// alone issues 0.5 warp-instructions per clock per SM sub-partition, together they reach the issue limit of 1
// (tools/pipe_probe.cu, profiles/pipe_probe_r02.txt).  Operands come from the other chains so that nothing folds.
__global__ void int_peak_kernel(uint32_t * out, uint32_t seed, uint32_t one, int iters)
{
  uint32_t a[8];
#pragma unroll
  for (int k = 0; k < 8; k++) { a[k] = seed * (threadIdx.x + 1) + k * 0x00030005u; }
  for (int it = 0; it < iters; it++) {
    uint32_t n[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      if (k & 1) { asm volatile("mad.lo.u32 %0, %1, %2, %3;" : "=r"(n[k]) : "r"(a[k]), "r"(one), "r"(a[(k + 2) & 7])); }
      else { n[k] = __viaddmax_u16x2(a[k], a[(k + 2) & 7], a[(k + 4) & 7]); }
    }
#pragma unroll
    for (int k = 0; k < 8; k++) { a[k] = n[k]; }
  }
  uint32_t r = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) { r ^= a[k]; }
  if (r == 0x12345678u) { out[0] = r; }
}
}  // namespace vsg

extern "C" int vsg_measure_int_peak(vsg_ctx * c, double * packed_lane_ops_per_s)
{
  if (c == nullptr || packed_lane_ops_per_s == nullptr) { return VSG_EINVAL; }
  VSG_CUDA_OK(cudaSetDevice(c->device));
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
  int rc;
  if ((rc = c->cub_tmp.reserve(64)) != VSG_OK) { return rc; }
  int const iters = 8192, threads = 256, blocks = sms * 8;
  double best = 0.0;
  for (int rep = 0; rep < 4; rep++) {
    VSG_CUDA_OK(cudaEventRecord(c->ev[4], c->stream));
    int_peak_kernel<<<blocks, threads, 0, c->stream>>>(static_cast<uint32_t *>(c->cub_tmp.p), 3u + rep, 1u, iters);
    count_launch();
    VSG_CUDA_OK(cudaEventRecord(c->ev[5], c->stream));
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
    double const ops = 8.0 * iters * static_cast<double>(threads) * blocks;  // one instruction per chain and iteration
    if (rep > 0) { best = std::max(best, ops / (ms * 1e-3)); }
  }
  *packed_lane_ops_per_s = best;
  return VSG_OK;
}

extern "C" int vsg_profile_reset(vsg_ctx * c)
{
  if (c == nullptr) { return VSG_EINVAL; }
  c->prof_cells = c->prof_fast = c->prof_exact = c->prof_fwd_launches = c->prof_tb_skipped = 0;
  c->prof_fwd_ms = c->prof_tb_ms = c->prof_rank_ms = 0.f;
  return VSG_OK;
}

extern "C" int vsg_profile_get(vsg_ctx * c, vsg_profile * out)
{
  if (c == nullptr || out == nullptr) { return VSG_EINVAL; }
  out->cells = c->prof_cells; out->fast_pairs = c->prof_fast; out->exact_pairs = c->prof_exact;
  out->fwd_launches = c->prof_fwd_launches;
  out->fwd_ms = c->prof_fwd_ms; out->traceback_ms = c->prof_tb_ms; out->rank_ms = c->prof_rank_ms;
  out->reserved = 0.f;
  out->tb_skipped = c->prof_tb_skipped;
  return VSG_OK;
}
