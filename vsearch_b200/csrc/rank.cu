// rank.cu — k-mer index in HBM and the candidate ranker (sm_100a).
//
// Replaces, for whole batches of queries at once,
//   unique_count            (reference core/unique.cpp:155-353)   distinct unmasked k-mers of a sequence
//   Dbindex::prepare/add_*  (core/dbindex.cpp:121-255)            k-mer -> targets postings
//   search_topscores        (core/searchcore.cpp:260-340)         per-target shared-k-mer counts,
//                                                                 threshold, best `tophits` targets
//   minheap_*               (core/minheap.cpp:82-263)             order: count desc, length asc, seqno asc
//
// Layout.  The database is cut into SHARDS of at most 32766 consecutive targets (static index; 32768 for the cluster
// driver's incremental one).  A shard stores CSR postings; in the static index every k-mer has two sub-lists, its even
// and its odd targets, and a posting is the BYTE OFFSET of the target's counter word as a u16 (half the bytes of the
// reference's u32 lists; the reference's per-k-mer bitmaps for very frequent k-mers, dbindex.cpp:212-229, are a storage
// variant with the same meaning and are not needed).  --wordlength 3..10: list heads for all 2 * 4^k sub-lists;
// 11..15: only the sub-lists that exist, found by binary search (build_sparse_shard).
// One CTA ranks one query: for every shard it zeroes 32768 16-bit counters in SHARED memory, turns the postings of
// the query's distinct k-mers into shared-memory atomic adds — the runs of all k-mers laid end to end as one stream
// of 16-byte vectors that the 16 warps split evenly (every lane busy every round) —, scans the counters against a
// running threshold and appends the survivors as 64-bit sort keys to a candidate list that is sorted and cut to
// `tophits` at the end (and whenever a crowd of ties fills it up).  HBM traffic per query is the postings themselves
// (2 B each) — the counters never leave the SM.
#include "vsg_internal.h"

#include <cub/cub.cuh>
#include <thrust/iterator/transform_iterator.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace vsg {

constexpr int SHARD_BITS = 15;
constexpr int SHARD = 1 << SHARD_BITS;  // targets per shard
constexpr int RANK_THREADS = 512;
#ifndef VSG_RANK_U
#define VSG_RANK_U 4      // posting vectors (of 8) a lane holds at a time
#endif
#ifndef VSG_RANK_ROLL
#define VSG_RANK_ROLL 0   // 1: refill a slot as soon as it has been applied (measured: no gain, see DESIGN experiment log)
#endif
#ifndef VSG_RANK_ZFUSE
#define VSG_RANK_ZFUSE 1  // clear the counters behind the last scan of a shard instead of in a pass of its own
#endif
constexpr int KMER_CAP = 2048;          // distinct-k-mer capacity per query (query length <= 2047 + k)
constexpr int CAND_CAP = 2048;          // candidate keys held in shared memory
constexpr int TOPHITS_MAX = 1024;
constexpr int RANK_PREFETCH = 3;         // k-mers (per warp) between the L2 prefetch of a list and its use
constexpr int SCAN_SEG_WORDS = 512;     // counters are scanned 1024 at a time (<= 1024 new candidates)
constexpr int COUNTER_WORDS = SHARD / 2 + 1;
// Static index: a shard holds 32766 targets and its postings are stored as the BYTE OFFSET of the target's counter
// word (two 16-bit counters per word: offset = (local target & ~1) * 2 <= 65528); every k-mer has two sub-lists,
// the even and the odd targets, each padded to a multiple of 8 entries with offset 65532 = word 16383, which no
// target owns.  Turning a posting into its counter update then takes no arithmetic at all: the address is the
// posting, the increment (1 or 0x10000) is a constant of the sub-list.
constexpr int SHARD_STATIC = SHARD - 2;
constexpr uint16_t POST_PAD = 65532;

struct ShardDev {
  const uint32_t * start;  // 4^k + 1 list offsets (incremental index: where this shard's part of every list begins)
  const uint16_t * post;   // shard-local target numbers (static index)
  int32_t t0;              // first target of the shard
  int32_t nt;              // targets in the shard
  // incremental index (cluster driver): lists of 32-bit target numbers in creation order, this shard's part of
  // list km is post32[start[km] .. end[km])
  const uint32_t * end;
  const uint32_t * post32;
  // sparse static index (--wordlength 11..15): the sorted (k-mer << 1 | target parity) keys of the sub-lists that
  // exist in this shard; sub-list i is post[start[i] .. start[i + 1]).  nr == 0: dense (start indexed by 2 * k-mer)
  const uint32_t * rkeys;
  uint32_t nr;
  uint32_t reserved;
};

__device__ __forceinline__ bool sym_bad(int s, int mask_lower)
{
  int const c = s & 15;
  bool const single = (c == 1) | (c == 2) | (c == 4) | (c == 8);
  return !single || (mask_lower && (s & 16));
}
__device__ __forceinline__ uint32_t sym_2bit(int s)
{
  int const c = s & 15;
  return (c == 2) ? 1u : (c == 4) ? 2u : (c == 8) ? 3u : 0u;
}

// k-mer ending at position p (p >= k-1); returns false when the window holds a masked symbol
__device__ __forceinline__ bool kmer_at(const uint8_t * __restrict__ s, int p, int k, int mask_lower,
                                        uint32_t & out)
{
  uint32_t v = 0;
  bool bad = false;
  for (int j = p - k + 1; j <= p; j++) {
    int const c = s[j];
    bad |= sym_bad(c, mask_lower);
    v = (v << 2) | sym_2bit(c);
  }
  out = v;
  return !bad;
}

// ---- index build: pass 1 counts, pass 2 fills; one CTA per target, shared-memory bitmap dedupe ----
template <bool FILL>
__global__ void index_build_kernel(DevSeqs db, int t0, int nt, int k, int mask_lower, int split,
                                   uint32_t * __restrict__ count /* pass1: counts; pass2: fill cursors */,
                                   const uint32_t * __restrict__ start, uint16_t * __restrict__ post)
{
  extern __shared__ uint32_t bitmap[];
  int const lt = blockIdx.x;
  if (lt >= nt) { return; }
  int const words = (1 << (2 * k)) >> 5;
  for (int i = threadIdx.x; i < (words > 0 ? words : 1); i += blockDim.x) { bitmap[i] = 0; }
  __syncthreads();
  int64_t const t = static_cast<int64_t>(t0) + lt;
  const uint8_t * __restrict__ s = db.sym + db.off[t];
  int const len = db.len[t];
  for (int p = k - 1 + threadIdx.x; p < len; p += blockDim.x) {
    uint32_t km;
    if (kmer_at(s, p, k, mask_lower, km)) {
      uint32_t const bit = 1u << (km & 31);
      uint32_t const old = atomicOr(&bitmap[km >> 5], bit);
      if ((old & bit) == 0) {  // first occurrence in this target
        uint32_t const list = split ? 2u * km + static_cast<uint32_t>(lt & 1) : km;   // static index: even / odd targets apart
        if (FILL) {
          uint32_t const pos = atomicAdd(&count[list], 1u);
          post[static_cast<size_t>(start[list]) + pos] = static_cast<uint16_t>((lt & ~1) << 1);
        } else {
          atomicAdd(&count[list], 1u);
        }
      }
    }
  }
}

// lists are padded to a multiple of 8 entries so that every list starts on a 16-byte boundary
__global__ void pad_counts_kernel(uint32_t * __restrict__ count, int n)
{
  int const i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { count[i] = (count[i] + 7u) & ~7u; }
}
__global__ void fill_u16_kernel(uint16_t * __restrict__ p, size_t n, uint16_t v)
{
  size_t const i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) { p[i] = v; }
}

// per-k-mer totals over the shards built so far (vsg_udb_load checks them against the file's word counts)
__global__ void add_totals_kernel(const uint32_t * __restrict__ count /* 2 per k-mer */, uint32_t * __restrict__ totals, size_t hashsize)
{
  size_t const i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < hashsize) { totals[i] += count[2 * i] + count[2 * i + 1]; }
}

// ---- sparse build (--wordlength 11..15: 4^k list heads per shard would dwarf the postings) --------------------------
// One 46-bit key per window: k-mer (30 bits) | target parity | local target >> 1 (14 bits); windows that hold a masked
// symbol, and the first k-1 positions of a target, get SPARSE_INVALID, which sorts behind every real key.  Sorting the
// keys and dropping duplicates IS the per-target de-duplication (unique_count_hash, core/unique.cpp:243-334: its
// CityHash table is only the device that finds the distinct k-mers) and the grouping by list in one go.
constexpr uint64_t SPARSE_INVALID = 1ull << 45;
__global__ void sparse_keys_kernel(DevSeqs db, int t0, int nt, int k, int mask_lower, const int64_t * __restrict__ cum,
                                   uint64_t * __restrict__ keys)
{
  int const lt = blockIdx.x;
  if (lt >= nt) { return; }
  int64_t const t = static_cast<int64_t>(t0) + lt;
  const uint8_t * __restrict__ s = db.sym + db.off[t];
  int const len = db.len[t];
  uint64_t * __restrict__ out = keys + cum[lt];
  uint64_t const low = (static_cast<uint64_t>(lt & 1) << 14) | static_cast<uint64_t>(lt >> 1);
  for (int p = threadIdx.x; p < len; p += blockDim.x) {
    uint64_t key = SPARSE_INVALID;
    uint32_t km;
    if (p >= k - 1 && kmer_at(s, p, k, mask_lower, km)) { key = (static_cast<uint64_t>(km) << 15) | low; }
    out[p] = key;
  }
}
struct SparseRunOf {   // key -> sub-list id (k-mer << 1 | parity); the invalid key maps to 0x80000000
  __host__ __device__ uint32_t operator()(uint64_t key) const { return static_cast<uint32_t>(key >> 14); }
};
struct PadTo8 {
  __host__ __device__ uint32_t operator()(uint32_t n) const { return (n + 7u) & ~7u; }
};
// sub-list r: its distinct keys ukeys[src[r] .. src[r] + cnt[r]) become counter offsets at post[dst[r] ...]
__global__ void sparse_scatter_kernel(const uint64_t * __restrict__ ukeys, const uint32_t * __restrict__ rkeys,
                                      const uint32_t * __restrict__ cnt, const uint32_t * __restrict__ src,
                                      const uint32_t * __restrict__ dst, uint32_t nr, uint16_t * __restrict__ post,
                                      uint32_t * __restrict__ totals)
{
  uint32_t const r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nr) { return; }
  uint32_t const n = cnt[r], a = src[r], b = dst[r];
  for (uint32_t i = 0; i < n; i++) { post[b + i] = static_cast<uint16_t>((ukeys[a + i] & 0x3fffu) << 2); }
  if (totals != nullptr) { atomicAdd(&totals[rkeys[r] >> 1], n); }
}

// Order inside a list does not matter to the counts, only to the speed of the shared-memory atomics that apply it:
// the ranker's warp turns a list into counter updates 32 postings at a time — lane L holds vector blk*32 + L of the
// list and instruction j of a vector round updates posting 8*(blk*32 + L) + j of every lane.  Those 32 postings are a
// "row"; a row whose postings fall into 32 different shared-memory banks (bank = bits 2..6 of the stored counter offset) is applied in one pass, one with collisions is replayed.  This kernel sorts every list
// by bank and deals the sorted postings out down the rows' lanes, so that the members of one row lie a whole
// list / 32 apart in bank order: a row only collides where a bank holds more than 1/32 of the list.
constexpr int BANK_ORDER_CAP = 8192;   // longer lists (a k-mer in a quarter of the shard) are left as they are
__global__ void __launch_bounds__(128)
list_bank_order_kernel(const uint32_t * __restrict__ start, uint16_t * __restrict__ post, int nlists)
{
  __shared__ uint16_t src[BANK_ORDER_CAP];
  __shared__ uint32_t hist[32], cursor[32];
  for (int li = blockIdx.x; li < nlists; li += gridDim.x) {
    uint32_t const b = start[li];
    int const n = static_cast<int>(start[li + 1] - b);   // a multiple of 8
    if (n <= 32 || n > BANK_ORDER_CAP) { continue; }      // uniform per block
    uint16_t * const lp = post + b;
    if (threadIdx.x < 32) { hist[threadIdx.x] = 0; }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      uint16_t const x = lp[i];
      src[i] = x;
      atomicAdd(&hist[(x >> 2) & 31], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      uint32_t const v = hist[threadIdx.x];
      uint32_t incl = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { uint32_t const o = __shfl_up_sync(0xffffffffu, incl, d); if (threadIdx.x >= d) { incl += o; } }
      cursor[threadIdx.x] = incl - v;
    }
    __syncthreads();
    int const nv = n >> 3, full = nv >> 5, rem = nv & 31;   // vectors; whole 32-vector blocks; lanes used in the last block
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      uint16_t const x = src[i];
      int const si = static_cast<int>(atomicAdd(&cursor[(x >> 2) & 31], 1u));   // rank in bank order
      // positions in the order (lane, block, posting of the vector)
      int const vr = si >> 3, j = si & 7;
      int lane, blk;
      if (vr < rem * (full + 1)) { lane = vr / (full + 1); blk = vr % (full + 1); }
      else { int const v2 = vr - rem * (full + 1); lane = rem + v2 / full; blk = v2 % full; }
      lp[8 * (blk * 32 + lane) + j] = x;
    }
    __syncthreads();
  }
}

// ---- bitonic sort helpers on shared memory (descending for keys, ascending for k-mers) ----------
template <typename T, bool DESC>
__device__ void bitonic_sort_shared(T * a, int n /* power of two */)
{
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < (n >> 1); i += blockDim.x) {
        int const lo = 2 * i - (i & (stride - 1));
        int const hi = lo + stride;
        bool const up = ((lo & size) == 0);
        T const x = a[lo], y = a[hi];
        bool const sw = DESC ? (up ? (x < y) : (x > y)) : (up ? (x > y) : (x < y));
        if (sw) { a[lo] = y; a[hi] = x; }
      }
    }
  }
  __syncthreads();
}

__device__ __forceinline__ int next_pow2(int v)
{
  int p = 1;
  while (p < v) { p <<= 1; }
  return p;
}

// key: larger = better.  count (15 bits) | ~length (25 bits) | ~seqno (24 bits)
__device__ __forceinline__ uint64_t make_key(uint32_t count, uint32_t len, uint32_t seqno)
{
  uint32_t const l = len > 0x1ffffffu ? 0x1ffffffu : len;
  if (count > 32767u) { count = 32767u; }  // the reference saturates its counters (searchcore.cpp:306-315)
  return (static_cast<uint64_t>(count) << 49) | (static_cast<uint64_t>(0x1ffffffu - l) << 24) |
         static_cast<uint64_t>(0xffffffu - seqno);
}

// What a rank_kernel launch computes per query.
//   RANK_TOP:   the best `tophits` candidates, sorted, into out_seqno / out_count (row qi * tophits), their number to out_n.
//   RANK_COUNT: (ranking without the TOPHITS_MAX ceiling, pass A) a histogram of the saturated counts >= minmatches over
//               all shards, in this CTA's `hist` row; from it the threshold T (the largest count with at least tophits
//               targets at or above it, else minmatches) to qT[qi] and the exact number K of targets >= T to out_n[qi].
//   RANK_EMIT:  (pass B) the unsorted keys of the K targets with count >= qT[qi] to keys[key_off[qi] ...]; a count that
//               differs from key_off[qi + 1] - key_off[qi] sets *status to 2.
enum { RANK_TOP = 0, RANK_COUNT = 1, RANK_EMIT = 2 };

template <bool INCR, int MODE = RANK_TOP>
__global__ void __launch_bounds__(RANK_THREADS, 2)
rank_kernel(DevSeqs qs, int64_t q0, int nq, DevSeqs db, const ShardDev * __restrict__ shards, int nshards,
            int k, int mask_lower, int minwordmatches, int tophits,
            uint32_t * __restrict__ out_seqno, uint32_t * __restrict__ out_count, int32_t * __restrict__ out_n,
            int32_t * __restrict__ status, uint32_t * __restrict__ scratch, size_t scratch_stride, int bitmap_words, int flat,
            uint32_t * __restrict__ qT = nullptr, const int32_t * __restrict__ key_off = nullptr,
            uint64_t * __restrict__ keys = nullptr, uint32_t * __restrict__ hist_rows = nullptr, int hist_stride = 0)
{
  extern __shared__ __align__(16) unsigned char smem[];
  uint64_t * const cand = reinterpret_cast<uint64_t *>(smem);                     // CAND_CAP
  uint32_t * const counters = reinterpret_cast<uint32_t *>(smem + CAND_CAP * 8);  // COUNTER_WORDS (+pad)
  uint32_t * const kmers = counters + COUNTER_WORDS + 3;                          // KMER_CAP
  uint32_t * const lbeg = kmers + KMER_CAP;                                       // KMER_CAP
  uint32_t * const llen = lbeg + KMER_CAP;                                        // KMER_CAP
  uint32_t * const cum = llen + KMER_CAP;                                         // KMER_CAP + 1 (static index, flat stream)
  __shared__ int s_ncand, s_nk, s_T, s_K;
  __shared__ int s_wsum[RANK_THREADS / 32];

  int const lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NWARPS = RANK_THREADS / 32;

  bool clean = false;   // the counters are all zero (left so by the previous shard's last scan)
  for (int qi = blockIdx.x; qi < nq; qi += gridDim.x) {
    int64_t const q = q0 + qi;
    const uint8_t * __restrict__ s = qs.sym + qs.off[q];
    int const len = qs.len[q];
    int const nwin = len - k + 1;
    if (threadIdx.x == 0) { s_ncand = 0; s_nk = 0; }
    bool const longq = nwin > KMER_CAP;
    if (longq && (scratch == nullptr || nwin > 65535)) {
      if (threadIdx.x == 0) { out_n[qi] = 0; atomicExch(status, 1); }
      continue;
    }
    int np2, nk, nchunks = 1;
    uint32_t * gk = nullptr;
    if (!longq) {
      // 1. the query's k-mers, sorted, duplicates and masked windows invalidated (0xffffffff)
      np2 = next_pow2(nwin > 1 ? nwin : 1);
      for (int i = threadIdx.x; i < np2; i += blockDim.x) {
        uint32_t km = 0xffffffffu;
        if (i < nwin) {
          uint32_t v;
          if (kmer_at(s, i + k - 1, k, mask_lower, v)) { km = v; }
        }
        kmers[i] = km;
      }
      bitonic_sort_shared<uint32_t, false>(kmers, np2);
      int mine = 0;
      for (int i = threadIdx.x; i < np2; i += blockDim.x) {
        uint32_t const v = kmers[i];
        bool const keep = (v != 0xffffffffu) && (i == 0 || kmers[i - 1] != v);
        lbeg[i] = keep ? 1u : 0u;  // temporary keep flag
        mine += keep;
      }
      __syncthreads();
      for (int i = threadIdx.x; i < np2; i += blockDim.x) { if (lbeg[i] == 0u) { kmers[i] = 0xffffffffu; } }
      atomicAdd(&s_nk, mine);
      __syncthreads();
      nk = s_nk;
    } else {
      // 1'. long query: de-duplicate through a 4^k-bit map in this CTA's HBM scratch, collect the
      //     distinct k-mers in a list there, and feed them through shared memory KMER_CAP at a time
      uint32_t * const bm = scratch + static_cast<size_t>(blockIdx.x) * scratch_stride;
      gk = bm + bitmap_words;
      if (k <= 10) {
        for (int i = threadIdx.x; i < bitmap_words; i += blockDim.x) { bm[i] = 0; }
        __syncthreads();
        for (int p = threadIdx.x; p < nwin; p += blockDim.x) {
          uint32_t v;
          if (kmer_at(s, p + k - 1, k, mask_lower, v)) {
            uint32_t const bit = 1u << (v & 31);
            uint32_t const old = atomicOr(&bm[v >> 5], bit);
            if ((old & bit) == 0) { gk[atomicAdd(&s_nk, 1)] = v; }
          }
        }
      } else {
        // wordlength 11..15: a 4^k-bit map per CTA is out of reach; an open-addressing table of bitmap_words (a power
        // of two >= twice the windows) slots does what unique_count_hash's table does (core/unique.cpp:243-334)
        uint32_t const hmask = static_cast<uint32_t>(bitmap_words) - 1u;
        for (int i = threadIdx.x; i < bitmap_words; i += blockDim.x) { bm[i] = 0xffffffffu; }
        __syncthreads();
        for (int p = threadIdx.x; p < nwin; p += blockDim.x) {
          uint32_t v;
          if (kmer_at(s, p + k - 1, k, mask_lower, v)) {
            uint32_t slot = (v * 2654435761u) >> 7 & hmask;
            for (;;) {
              uint32_t const old = atomicCAS(&bm[slot], 0xffffffffu, v);
              if (old == 0xffffffffu) { gk[atomicAdd(&s_nk, 1)] = v; break; }
              if (old == v) { break; }
              slot = (slot + 1u) & hmask;
            }
          }
        }
      }
      __threadfence_block();
      __syncthreads();
      nk = s_nk;
      nchunks = nk > 0 ? (nk + KMER_CAP - 1) / KMER_CAP : 1;
      np2 = 1;
    }
    // search_topscores: count >= min(minwordmatches, kmersamplecount)  (searchcore.cpp:320)
    uint32_t const minmatches = static_cast<uint32_t>(minwordmatches < nk ? minwordmatches : nk);
    // RUNNING THRESHOLD (queries with np2 + nk + 1 <= KMER_CAP, i.e. up to ~1000 nt): hist[c] counts,
    // over the shards seen so far, the targets whose k-mer count is c; T = the largest count with at
    // least `tophits` targets at or above it.  A target below T can never reach the final list, so
    // only counts >= T are turned into candidate keys: a few dozen per shard instead of the ~3 % of
    // all targets that pass the reference's fixed threshold (searchcore.cpp:320), no overflow sorts.
    bool const running = MODE == RANK_TOP && !longq && (np2 + nk + 1 <= KMER_CAP);
    // RANK_COUNT: counts saturate at 32767 as the reference's do, so min(nk, 32767) + 1 bins (HBM: a long query's
    // bins do not fit in shared memory)
    int const hbins = (nk < 32767 ? nk : 32767) + 1;
    uint32_t * const qhist = MODE == RANK_COUNT ? hist_rows + static_cast<size_t>(blockIdx.x) * hist_stride : nullptr;
    if constexpr (MODE == RANK_COUNT) { for (int i = threadIdx.x; i < hbins; i += blockDim.x) { qhist[i] = 0; } }
    // RANK_EMIT: T of this query and the room pass A counted for it
    uint32_t const emit_T = MODE == RANK_EMIT ? qT[qi] : 0u;
    int const emit_n = MODE == RANK_EMIT ? key_off[qi + 1] - key_off[qi] : 0;
    uint32_t * const hist = kmers + np2;  // nk + 1 bins in the unused tail of the k-mer array
    if (running) {
      for (int i = threadIdx.x; i <= nk; i += blockDim.x) { hist[i] = 0; }
      if (threadIdx.x == 0) { s_T = static_cast<int>(minmatches); }
    }
    // visits every counter >= thr of the current shard: f(count, local target)
    // zero != 0: the counters are cleared behind the scan (the next shard then skips its clearing pass)
    auto scan_counters = [&](int nt, uint32_t thr, int zero, auto && f) {
      int const nvec = (((nt + 1) >> 1) + 3) >> 2;
      uint32_t const below = thr > 0 ? ((thr - 1) | ((thr - 1) << 16)) : 0u;
      uint4 * __restrict__ cv = reinterpret_cast<uint4 *>(counters);
      if (zero != 0 && threadIdx.x == 0) { counters[(POST_PAD >> 2)] = 0; }   // where the padding entries of the lists land
      for (int vi = threadIdx.x; vi < nvec; vi += blockDim.x) {
        uint4 const x = cv[vi];
        if (zero != 0) { cv[vi] = make_uint4(0u, 0u, 0u, 0u); }
        uint32_t const w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int u = 0; u < 4; u++) {
          // some half above thr-1?  (thr == 0: everything passes)
          if (thr > 0 && __vmaxu2(w[u], below) == below) { continue; }
          uint32_t const c0 = w[u] & 0xffffu, c1 = w[u] >> 16;
          int const lt0 = 2 * (4 * vi + u), lt1 = lt0 + 1;
          if (c0 >= thr && lt0 < nt) { f(c0, lt0); }
          if (c1 >= thr && lt1 < nt) { f(c1, lt1); }
        }
      }
    };

    for (int sh = 0; sh < nshards; sh++) {
      ShardDev const S = shards[sh];
      // 2. zero the counters; fetch the bounds of every k-mer's posting list in this shard
      if (!clean) { for (int i = threadIdx.x; i < COUNTER_WORDS; i += blockDim.x) { counters[i] = 0; } }
      clean = false;
      for (int chunk = 0; chunk < nchunks; chunk++) {
      if (longq) {
        int const cn = nk > 0 ? min(KMER_CAP, nk - chunk * KMER_CAP) : 1;
        for (int i = threadIdx.x; i < cn; i += blockDim.x) { kmers[i] = nk > 0 ? gk[chunk * KMER_CAP + i] : 0xffffffffu; }
        np2 = cn;
        __syncthreads();
      }
      for (int i = threadIdx.x; i < np2; i += blockDim.x) {
        uint32_t const km = kmers[i];
        uint32_t b = 0, n = 0;
        if (km != 0xffffffffu) {
          if (INCR) { b = S.start[km]; n = S.end[km] - b; }
          else if (S.nr == 0u) {
            // even sub-list [b, mid), odd sub-list [mid, end): lengths in vectors of 8, both in one word
            b = S.start[2 * km];
            uint32_t const mid = S.start[2 * km + 1], e = S.start[2 * km + 2];
            n = ((mid - b) >> 3) | (((e - mid) >> 3) << 16);
          } else {
            // sparse shard: lower bound of the even sub-list's key among the sub-lists that exist; the odd one, if
            // present, is its neighbour, so the pair is one contiguous run of postings either way
            uint32_t const want = km << 1;
            uint32_t lo = 0, hi = S.nr;
            while (lo < hi) {
              uint32_t const mid = (lo + hi) >> 1;
              if (__ldg(S.rkeys + mid) < want) { lo = mid + 1; } else { hi = mid; }
            }
            b = S.start[lo];
            uint32_t na = 0, nb = 0, i = lo;
            if (i < S.nr && __ldg(S.rkeys + i) == want) { na = (S.start[i + 1] - S.start[i]) >> 3; i++; }
            if (i < S.nr && __ldg(S.rkeys + i) == (want | 1u)) { nb = (S.start[i + 1] - S.start[i]) >> 3; }
            n = na | (nb << 16);
          }
        }
        lbeg[i] = b; llen[i] = n;
      }
      __syncthreads();
      // 3. postings -> counters (targets within a list are distinct, lists collide -> shared-memory
      //    atomics).  Lists are 16-byte aligned and padded, so a lane pulls 8 targets per 128-bit
      //    load.  A warp walks the two sub-lists of a k-mer at a time and issues up to three loads per lane and
      //    sub-list before it touches a counter: six independent HBM requests per lane hide the latency that a
      //    one-list-at-a-time loop exposes once per list.  Padding entries land in counter word 16383, which
      //    no target of a static shard owns.
      if constexpr (INCR) {
        // unpadded lists of 32-bit target numbers: one warp per list, coalesced loads
        for (int li = warp; li < np2; li += NWARPS) {
          uint32_t const n = llen[li];
          const uint32_t * __restrict__ pl = S.post32 + lbeg[li];
          for (uint32_t e = lane; e < n; e += 32) {
            uint32_t const a = __ldg(pl + e) - static_cast<uint32_t>(S.t0);
            atomicAdd(&counters[a >> 1], (a & 1) ? 0x10000u : 1u);
          }
        }
      }
#ifdef VSG_RANK_LEGACY
      else if (flat != 0) {
#else
      else {
#endif
        // FLAT VECTOR STREAM.  The even and the odd sub-list of a k-mer are one contiguous run of 16-byte vectors, and
        // the runs of all the query's k-mers, laid end to end, form one virtual stream of Vtot vectors.  Each warp
        // takes a contiguous 1/16 of the stream and walks it 32 vectors per round — every lane always has a vector
        // (a per-k-mer loop leaves most lanes idle on the second trip of a 36-vector sub-list and pays its set-up
        // 243 times per shard).  Per run i, with c_i its position in the stream:
        //   cum[i]  = c_i + n_i          where the run ends
        //   lbeg[i] = first vector - c_i  so that stream position + lbeg = the vector's index in the shard's postings
        //   llen[i] = c_i + na_i         positions below it hold even targets (increment 1), the rest odd ones (0x10000)
        // A lane finds its first run by one binary search and then walks forward (runs average two rounds).
        uint32_t Vtot;
        {
          // 3a. exclusive prefix sum of the run lengths (in vectors)
          int const per = (np2 + RANK_THREADS - 1) / RANK_THREADS;   // <= 4
          int const i0 = threadIdx.x * per;
          uint32_t nn[KMER_CAP / RANK_THREADS], bb[KMER_CAP / RANK_THREADS];
          uint32_t sum = 0;
#pragma unroll
          for (int u = 0; u < KMER_CAP / RANK_THREADS; u++) {
            bool const in = u < per && i0 + u < np2;
            nn[u] = in ? llen[i0 + u] : 0u;
            bb[u] = in ? lbeg[i0 + u] : 0u;
            sum += (nn[u] & 0xffffu) + (nn[u] >> 16);
          }
          uint32_t incl = sum;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { uint32_t const o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) { incl += o; } }
          if (lane == 31) { s_wsum[warp] = static_cast<int>(incl); }
          __syncthreads();
          uint32_t wbase = 0, total = 0;
#pragma unroll
          for (int w2 = 0; w2 < NWARPS; w2++) { uint32_t const v = static_cast<uint32_t>(s_wsum[w2]); if (w2 < warp) { wbase += v; } total += v; }
          uint32_t c0 = wbase + incl - sum;
#pragma unroll
          for (int u = 0; u < KMER_CAP / RANK_THREADS; u++) {
            if (u < per && i0 + u < np2) {
              uint32_t const na = nn[u] & 0xffffu, n = na + (nn[u] >> 16);
              lbeg[i0 + u] = (bb[u] >> 3) - c0;
              llen[i0 + u] = c0 + na;
              cum[i0 + u] = c0 + n;
              c0 += n;
            }
          }
          Vtot = total;
          __syncthreads();
        }
        uint32_t const per_w = ((Vtot + NWARPS * 32 - 1) / (NWARPS * 32)) * 32;
        uint32_t const wbeg = static_cast<uint32_t>(warp) * per_w;
        uint32_t const wend = min(Vtot, wbeg + per_w);
        if (wbeg < wend) {
          constexpr int U = VSG_RANK_U;   // vectors (of 8 postings) held per lane
          const uint4 * __restrict__ pbase = reinterpret_cast<const uint4 *>(S.post);
          uint32_t const cnt_sa = static_cast<uint32_t>(__cvta_generic_to_shared(counters));
          // the run holding this lane's first vector: the first whose end lies beyond it
          uint32_t const v_first = min(wbeg + static_cast<uint32_t>(lane), wend - 1);
          int lo = 0, hi = np2 - 1;
          while (lo < hi) {
            int const mid = (lo + hi) >> 1;
            if (cum[mid] <= v_first) { lo = mid + 1; } else { hi = mid; }
          }
          // sa walks the run arrays as a shared-memory byte address of lbeg[s]; llen and cum lie KMER_CAP words further each
          uint32_t sa = static_cast<uint32_t>(__cvta_generic_to_shared(lbeg + lo));
          uint32_t ce = cum[lo];
          // U loads per lane are issued back to back, then turned into counter updates; the other 31 warps of the SM
          // cover the wait (VSG_RANK_ROLL refills each slot right after its use instead: measured equal).
          uint4 cur[U];
          uint32_t inc[U];
          auto fetch = [&](int u, uint32_t vv) {
            inc[u] = 0u;
            if (vv < wend) {
              while (vv >= ce) {
                sa += 4u;
                asm("ld.shared.u32 %0, [%1+%2];" : "=r"(ce) : "r"(sa), "n"(2 * KMER_CAP * 4));
              }
              uint32_t vb, sp;
              asm("ld.shared.u32 %0, [%1];" : "=r"(vb) : "r"(sa));
              asm("ld.shared.u32 %0, [%1+%2];" : "=r"(sp) : "r"(sa), "n"(KMER_CAP * 4));
              cur[u] = __ldg(pbase + static_cast<uint32_t>(vb + vv));
              inc[u] = vv < sp ? 1u : 0x10000u;
            }
          };
          auto apply = [&](int u) {
            if (inc[u] != 0u) {
              uint32_t const w[4] = {cur[u].x, cur[u].y, cur[u].z, cur[u].w};
#pragma unroll
              for (int k2 = 0; k2 < 4; k2++) {
                // the postings ARE the byte offsets of their counter words
                asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(cnt_sa + (w[k2] & 0xffffu)), "r"(inc[u]));
                asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(cnt_sa + (w[k2] >> 16)), "r"(inc[u]));
              }
            }
          };
#if VSG_RANK_ROLL
#pragma unroll
          for (int u = 0; u < U; u++) { fetch(u, wbeg + 32u * u + static_cast<uint32_t>(lane)); }
          for (uint32_t v0 = wbeg; v0 < wend; v0 += 32u * U) {
#pragma unroll
            for (int u = 0; u < U; u++) {
              apply(u);
              fetch(u, v0 + 32u * (U + u) + static_cast<uint32_t>(lane));
            }
          }
#else
          for (uint32_t v0 = wbeg; v0 < wend; v0 += 32u * U) {
#pragma unroll
            for (int u = 0; u < U; u++) { fetch(u, v0 + 32u * u + static_cast<uint32_t>(lane)); }
#pragma unroll
            for (int u = 0; u < U; u++) { apply(u); }
          }
#endif
        }
#ifdef VSG_RANK_LEGACY
      } else {
        // (A/B reference, VSG_RANK_FLAT=0) a warp takes one k-mer at a time: list a = its even targets (increment 1),
        // list b = its odd targets (increment 0x10000)
        auto pair_len = [&](int li) -> uint32_t {
          uint32_t const na = llen[li] & 0xffffu, nb = llen[li] >> 16;
          return na > nb ? na : nb;
        };
        // One register buffer of six vectors (three per list): as soon as a vector has been turned into
        // counter updates its slot is refilled from the NEXT (k-mer, offset), so six loads per lane
        // stay in flight without a second buffer (48 data registers would not leave room in the 64
        // this kernel may use at two 512-thread CTAs per SM).
        struct ListPair { uint32_t na, nb; const uint4 * pa; const uint4 * pb; };
        auto bounds_of = [&](int li) -> ListPair {
          ListPair lp;
          lp.na = llen[li] & 0xffffu;
          lp.nb = llen[li] >> 16;
          lp.pa = reinterpret_cast<const uint4 *>(S.post + lbeg[li]);
          lp.pb = lp.pa + lp.na;
          return lp;
        };
        int li = warp;
        uint32_t base = 0;
        bool have = li < np2;
        uint4 cur[6];
        uint32_t valid = 0;
        if (have) {
          ListPair const lp = bounds_of(li);
#pragma unroll
          for (int u = 0; u < 6; u++) {
            uint32_t const e = lane + 32u * (u % 3);
            if (e < (u < 3 ? lp.na : lp.nb)) { cur[u] = __ldg((u < 3 ? lp.pa : lp.pb) + e); valid |= 1u << u; }
          }
        }
        while (have) {
          int nli = li;
          uint32_t nbase = base + 96;
          if (nbase >= pair_len(li)) { nli = li + NWARPS; nbase = 0; }
          bool const nhave = nli < np2;
          if (nbase == 0) {
            // the register buffer only reaches one k-mer ahead, less than a trip to HBM takes: pull the k-mer three
            // turns ahead into L2 now (its two sub-lists are one contiguous run of 128-byte lines, one line per lane)
            int const pli = nli + RANK_PREFETCH * NWARPS;
            if (pli < np2) {
              uint32_t const pn = (llen[pli] & 0xffffu) + (llen[pli] >> 16);   // vectors of 16 bytes
              if (8u * lane < pn) {
                asm volatile("prefetch.global.L2 [%0];" :: "l"(S.post + lbeg[pli] + 64u * lane));
              }
            }
          }
          ListPair lp{0u, 0u, nullptr, nullptr};
          if (nhave) { lp = bounds_of(nli); }
          uint32_t nvalid = 0;
#pragma unroll
          for (int u = 0; u < 6; u++) {
            if ((valid & (1u << u)) != 0u) {
              uint32_t const w[4] = {cur[u].x, cur[u].y, cur[u].z, cur[u].w};
              uint32_t const inc = u < 3 ? 1u : 0x10000u;
#pragma unroll
              for (int k = 0; k < 4; k++) {
                uint32_t const a = w[k] & 0xffffu, b = w[k] >> 16;   // byte offsets of the counter words
                atomicAdd(reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(counters) + a), inc);
                atomicAdd(reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(counters) + b), inc);
              }
            }
            uint32_t const e = nbase + lane + 32u * (u % 3);
            if (e < (u < 3 ? lp.na : lp.nb)) { cur[u] = __ldg((u < 3 ? lp.pa : lp.pb) + e); nvalid |= 1u << u; }
          }
          valid = nvalid;
          li = nli; base = nbase; have = nhave;
        }
      }
#else
      }
#endif
      __syncthreads();
      }  // chunk
      if constexpr (MODE != RANK_TOP) {
        if (MODE == RANK_COUNT || emit_n > 0) {
          scan_counters(S.nt, MODE == RANK_COUNT ? minmatches : emit_T, VSG_RANK_ZFUSE, [&](uint32_t c, int lt) {
            if constexpr (MODE == RANK_COUNT) {
              atomicAdd(&qhist[c < 32767u ? c : 32767u], 1u);
            } else {
              int const t = S.t0 + lt;
              int const pos = atomicAdd(&s_ncand, 1);
              if (pos < emit_n) { keys[key_off[qi] + pos] = make_key(c, static_cast<uint32_t>(db.len[t]), static_cast<uint32_t>(t)); }
            }
          });
          clean = VSG_RANK_ZFUSE != 0;
        }
        __syncthreads();
        continue;  // next shard
      }
      int const nwords = (S.nt + 1) >> 1;
      uint32_t thr = minmatches;
      if (running) {
        // 4r. histogram of this shard's counts >= T, new T, then keys for counts >= new T only
        uint32_t const T0 = static_cast<uint32_t>(s_T);
        scan_counters(S.nt, T0, 0, [&](uint32_t c, int) { atomicAdd(&hist[c], 1u); });
        __syncthreads();
        if (warp == 0) {
          int acc = 0, T = static_cast<int>(T0), K = -1;
          for (int top = nk; top >= static_cast<int>(T0); top -= 32) {
            int const b = top - lane;
            int v = b >= static_cast<int>(T0) ? static_cast<int>(hist[b]) : 0;
            // inclusive prefix over lanes = suffix over bins (lane 0 is the highest bin)
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { int const o = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) { v += o; } }
            unsigned const hit = __ballot_sync(0xffffffffu, acc + v >= tophits);
            if (hit != 0u) {
              int const first = __ffs(hit) - 1;
              T = top - first;
              K = acc + __shfl_sync(0xffffffffu, v, first);
              break;
            }
            acc += __shfl_sync(0xffffffffu, v, 31);
          }
          if (K < 0) { K = acc; }  // fewer than tophits targets so far: keep them all
          if (lane == 0) { s_T = T; s_K = K; }
        }
        int const level = s_ncand;
        __syncthreads();
        uint32_t const T1 = static_cast<uint32_t>(s_T);
        int const K = s_K;
        if (level + K <= CAND_CAP) {
          // at most K targets (all shards so far) are >= T1, so at most K keys are appended here
          scan_counters(S.nt, T1, VSG_RANK_ZFUSE, [&](uint32_t c, int lt) {
            int const t = S.t0 + lt;
            cand[atomicAdd(&s_ncand, 1)] = make_key(c, static_cast<uint32_t>(db.len[t]), static_cast<uint32_t>(t));
          });
          clean = VSG_RANK_ZFUSE != 0;
          __syncthreads();
          continue;  // next shard
        }
        thr = T1;  // a crowd of ties at T1: the sort-and-cut path below, from T1 up
      } else {
      // 4. threshold scan.  Common case: count the survivors, one block-wide prefix sum, write them
      //    straight to their slots (no barrier per segment).  Only if they would not fit does the
      //    segmented sort-and-cut path below run.
      {
        int mycount = 0;
        for (int wi = threadIdx.x; wi < nwords; wi += blockDim.x) {
          uint32_t const w = counters[wi];
          mycount += ((w & 0xffffu) >= minmatches && 2 * wi < S.nt) + ((w >> 16) >= minmatches && 2 * wi + 1 < S.nt);
        }
        int incl = mycount;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int const o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) { incl += o; } }
        if (lane == 31) { s_wsum[warp] = incl; }
        __syncthreads();
        int wbase = 0, total = 0;
        for (int w2 = 0; w2 < NWARPS; w2++) { int const v = s_wsum[w2]; if (w2 < warp) { wbase += v; } total += v; }
        int const level = s_ncand;
        __syncthreads();
        if (level + total <= CAND_CAP) {
          int pos = level + wbase + incl - mycount;
          for (int wi = threadIdx.x; wi < nwords; wi += blockDim.x) {
            uint32_t const w = counters[wi];
            uint32_t const c0 = w & 0xffffu, c1 = w >> 16;
            int const lt0 = 2 * wi, lt1 = 2 * wi + 1;
            if (c0 >= minmatches && lt0 < S.nt) {
              int const t = S.t0 + lt0;
              cand[pos++] = make_key(c0, static_cast<uint32_t>(db.len[t]), static_cast<uint32_t>(t));
            }
            if (c1 >= minmatches && lt1 < S.nt) {
              int const t = S.t0 + lt1;
              cand[pos++] = make_key(c1, static_cast<uint32_t>(db.len[t]), static_cast<uint32_t>(t));
            }
          }
          if (threadIdx.x == 0) { s_ncand = level + total; }
          __syncthreads();
          continue;  // next shard
        }
      }
      }
      // 4b. segmented scan with sort-and-cut when the candidate list could overflow
      for (int seg = 0; seg < nwords; seg += SCAN_SEG_WORDS) {
        // every thread must take the same decision: read the fill level, then fence the read off
        // from the appends of threads that are already past this point
        int const level = s_ncand;
        __syncthreads();
        if (level + 2 * SCAN_SEG_WORDS > CAND_CAP) {
          int const m = level;
          int const p2 = next_pow2(m);
          for (int i = m + threadIdx.x; i < p2; i += blockDim.x) { cand[i] = 0; }
          bitonic_sort_shared<uint64_t, true>(cand, p2);
          if (threadIdx.x == 0) { s_ncand = m < tophits ? m : tophits; }
          __syncthreads();
        }
        int const wend = min(seg + SCAN_SEG_WORDS, nwords);
        for (int wi = seg + threadIdx.x; wi < wend; wi += blockDim.x) {
          uint32_t const w = counters[wi];
          uint32_t const c0 = w & 0xffffu, c1 = w >> 16;
          int const lt0 = 2 * wi, lt1 = 2 * wi + 1;
          if (c0 >= thr && lt0 < S.nt) {
            int const t = S.t0 + lt0;
            cand[atomicAdd(&s_ncand, 1)] = make_key(c0, static_cast<uint32_t>(db.len[t]), static_cast<uint32_t>(t));
          }
          if (c1 >= thr && lt1 < S.nt) {
            int const t = S.t0 + lt1;
            cand[atomicAdd(&s_ncand, 1)] = make_key(c1, static_cast<uint32_t>(db.len[t]), static_cast<uint32_t>(t));
          }
        }
        __syncthreads();
      }
    }
    if constexpr (MODE == RANK_COUNT) {
      // suffix sums over the bins from the top: T = the first bin where they reach tophits
      __syncthreads();
      if (warp == 0) {
        int const lo = static_cast<int>(minmatches);
        int acc = 0, T = lo, K = -1;
        for (int top = hbins - 1; top >= lo; top -= 32) {
          int const b = top - lane;
          int v = b >= lo ? static_cast<int>(qhist[b]) : 0;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { int const o = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) { v += o; } }
          unsigned const hit = __ballot_sync(0xffffffffu, acc + v >= tophits);
          if (hit != 0u) {
            int const first = __ffs(hit) - 1;
            T = top - first;
            K = acc + __shfl_sync(0xffffffffu, v, first);
            break;
          }
          acc += __shfl_sync(0xffffffffu, v, 31);
        }
        if (K < 0) { K = acc; }   // fewer than tophits targets: all of them
        if (lane == 0) { qT[qi] = static_cast<uint32_t>(T); out_n[qi] = K; }
      }
      __syncthreads();
      continue;  // next query
    }
    if constexpr (MODE == RANK_EMIT) {
      if (threadIdx.x == 0 && s_ncand != emit_n) { atomicExch(status, 2); }
      __syncthreads();
      continue;  // next query
    }
    // 5. final order.  Usually far more targets pass the k-mer threshold than are wanted: find the
    //    count T of the tophits-th best with a histogram, keep count >= T, sort only those.
    int m = s_ncand;
    __syncthreads();
    if (running) {
      if (m > 2 * tophits) {
        // keys below the final T were appended while T was still lower: drop them before sorting
        uint64_t const tkey = static_cast<uint64_t>(static_cast<uint32_t>(s_T)) << 49;
        uint64_t mine[CAND_CAP / RANK_THREADS];
        int cnt = 0;
        for (int i = threadIdx.x; i < m; i += blockDim.x) { uint64_t const kx = cand[i]; if (kx >= tkey) { mine[cnt++] = kx; } }
        if (threadIdx.x == 0) { s_ncand = 0; }
        __syncthreads();
        int base = cnt > 0 ? atomicAdd(&s_ncand, cnt) : 0;
        for (int i = 0; i < cnt; i++) { cand[base + i] = mine[i]; }
        __syncthreads();
        m = s_ncand;
      }
    } else if (m > 2 * tophits && nk + 1 <= 2 * KMER_CAP) {
      uint32_t * const hist = lbeg;  // 2 * KMER_CAP words available, counts are <= nk <= KMER_CAP
      int const nb = nk + 1;
      for (int i = threadIdx.x; i < nb; i += blockDim.x) { hist[i] = 0; }
      __syncthreads();
      for (int i = threadIdx.x; i < m; i += blockDim.x) { atomicAdd(&hist[static_cast<uint32_t>(cand[i] >> 49)], 1u); }
      __syncthreads();
      if (warp == 0) {
        int acc = 0, T = 0;
        for (int top = nb - 1; top >= 0; top -= 32) {
          int const b = top - lane;
          int v = b >= 0 ? static_cast<int>(hist[b]) : 0;
          // inclusive prefix over lanes = suffix over bins (lane 0 is the highest bin)
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { int const o = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) { v += o; } }
          unsigned const hit = __ballot_sync(0xffffffffu, acc + v >= tophits);
          if (hit != 0u) { T = top - (__ffs(hit) - 1); break; }
          acc += __shfl_sync(0xffffffffu, v, 31);
        }
        if (lane == 0) { s_nk = T; s_ncand = 0; }
      }
      __syncthreads();
      uint64_t const tkey = static_cast<uint64_t>(static_cast<uint32_t>(s_nk)) << 49;
      // compact in place: read everything first, then write the survivors
      uint64_t mine[CAND_CAP / RANK_THREADS];
      int cnt = 0;
      for (int i = threadIdx.x; i < m; i += blockDim.x) { uint64_t const kx = cand[i]; if (kx >= tkey) { mine[cnt++] = kx; } }
      __syncthreads();
      int base = cnt > 0 ? atomicAdd(&s_ncand, cnt) : 0;
      for (int i = 0; i < cnt; i++) { cand[base + i] = mine[i]; }
      __syncthreads();
      m = s_ncand;
    }
    int const p2 = next_pow2(m > 1 ? m : 1);
    for (int i = m + threadIdx.x; i < p2; i += blockDim.x) { cand[i] = 0; }
    bitonic_sort_shared<uint64_t, true>(cand, p2);
    int const nout = m < tophits ? m : tophits;
    for (int i = threadIdx.x; i < nout; i += blockDim.x) {
      uint64_t const key = cand[i];
      out_seqno[static_cast<size_t>(qi) * tophits + i] = 0xffffffu - static_cast<uint32_t>(key & 0xffffffu);
      out_count[static_cast<size_t>(qi) * tophits + i] = static_cast<uint32_t>(key >> 49);
    }
    if (threadIdx.x == 0) { out_n[qi] = nout; }
    __syncthreads();
  }
}

constexpr size_t RANK_SMEM = CAND_CAP * 8 + (COUNTER_WORDS + 3) * 4 + KMER_CAP * 4 * 4 + 4;   // 114 708 B: two CTAs fit an SM's 227 KB

}  // namespace vsg

using namespace vsg;

struct vsg_index {
  int device = 0;
  int k = 8;
  int mask_lower = 0;
  int64_t ntargets = 0;
  const vsg_seqset * db = nullptr;
  std::vector<DevBuf> b_start, b_post, b_rkeys;
  std::vector<ShardDev> h_shards;
  DevBuf b_shards;
  int64_t total_postings = 0;
};

extern "C" void vsg_index_destroy(vsg_index * ix);
namespace vsg {

static void shard_bank_order(vsg_ctx * c, const uint32_t * start, uint16_t * post, size_t nlists)
{
  static bool const bank_order = [] { const char * e = std::getenv("VSG_BANK_ORDER"); return e == nullptr || e[0] != '0'; }();
  if (!bank_order || nlists == 0) { return; }
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
  list_bank_order_kernel<<<static_cast<int>(std::min<size_t>(nlists, static_cast<size_t>(sms) * 32)), 128, 0, c->stream>>>(start, post, static_cast<int>(nlists));
  count_launch();
}

// dense shard (k <= 10): start[2 * 4^k + 1], two sub-lists per k-mer
static int build_dense_shard(vsg_ctx * c, vsg_index * ix, int sh, int t0, int nt, DevBuf & cnt, DevBuf & tmp, uint32_t * d_totals)
{
  const vsg_seqset * db = ix->db;
  int const k = ix->k;
  size_t const hashsize = static_cast<size_t>(1) << (2 * k);
  size_t const bitmap_bytes = std::max<size_t>(hashsize / 8, 4);
  size_t const nlists = 2 * hashsize;   // even and odd targets of every k-mer
  int rc;
  // list offsets are 32-bit: a shard's postings (at most one per nucleotide) plus the padding of its lists must fit
  int64_t nuc = 0;
  for (int i = 0; i < nt; i++) { nuc += db->h_len[static_cast<size_t>(t0) + static_cast<size_t>(i)]; }
  if (nuc + 7 * static_cast<int64_t>(nlists) >= (static_cast<int64_t>(1) << 32) - 64) {
    Error::set("vsg_index_create: a shard of 32766 targets holds 2^32 nucleotides or more");
    return VSG_EINVAL;
  }
  DevBuf & bs = ix->b_start[static_cast<size_t>(sh)];
  if ((rc = bs.reserve(sizeof(uint32_t) * (nlists + 1))) != VSG_OK) { return rc; }
  VSG_CUDA_OK(cudaMemsetAsync(cnt.p, 0, sizeof(uint32_t) * (nlists + 1), c->stream));
  index_build_kernel<false><<<nt, 128, bitmap_bytes, c->stream>>>(db->d, t0, nt, k, ix->mask_lower, 1,
                                                                  static_cast<uint32_t *>(cnt.p), nullptr, nullptr);
  count_launch();
  if (d_totals != nullptr) {
    add_totals_kernel<<<static_cast<unsigned>((hashsize + 255) / 256), 256, 0, c->stream>>>(static_cast<const uint32_t *>(cnt.p), d_totals, hashsize);
    count_launch();
  }
  pad_counts_kernel<<<static_cast<unsigned>((nlists + 255) / 256), 256, 0, c->stream>>>(static_cast<uint32_t *>(cnt.p), static_cast<int>(nlists));
  count_launch();
  size_t tb = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tb, static_cast<uint32_t *>(cnt.p), static_cast<uint32_t *>(bs.p),
                                static_cast<int>(nlists + 1), c->stream);
  if ((rc = tmp.reserve(tb + 16)) != VSG_OK) { return rc; }
  cub::DeviceScan::ExclusiveSum(tmp.p, tb, static_cast<uint32_t *>(cnt.p), static_cast<uint32_t *>(bs.p),
                                static_cast<int>(nlists + 1), c->stream);
  count_launch();
  uint32_t total = 0;
  VSG_CUDA_OK(cudaMemcpyAsync(&total, static_cast<uint32_t *>(bs.p) + nlists, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  DevBuf & bp = ix->b_post[static_cast<size_t>(sh)];
  if ((rc = bp.reserve(sizeof(uint16_t) * (static_cast<size_t>(total) + 64))) != VSG_OK) { return rc; }
  VSG_CUDA_OK(cudaMemsetAsync(cnt.p, 0, sizeof(uint32_t) * (nlists + 1), c->stream));
  if (total > 0) {
    fill_u16_kernel<<<static_cast<unsigned>((static_cast<size_t>(total) + 255) / 256), 256, 0, c->stream>>>(
        static_cast<uint16_t *>(bp.p), static_cast<size_t>(total), POST_PAD);
    count_launch();
  }
  index_build_kernel<true><<<nt, 128, bitmap_bytes, c->stream>>>(db->d, t0, nt, k, ix->mask_lower, 1,
                                                                 static_cast<uint32_t *>(cnt.p),
                                                                 static_cast<uint32_t *>(bs.p),
                                                                 static_cast<uint16_t *>(bp.p));
  count_launch();
  if (total > 0) { shard_bank_order(c, static_cast<const uint32_t *>(bs.p), static_cast<uint16_t *>(bp.p), nlists); }
  ShardDev sd{};
  sd.start = static_cast<uint32_t *>(bs.p); sd.post = static_cast<uint16_t *>(bp.p); sd.t0 = t0; sd.nt = nt;
  ix->h_shards.push_back(sd);
  ix->total_postings += total;
  return VSG_OK;
}

// sparse shard (k 11..15): sort the windows' keys, drop duplicates, run-length encode the sub-lists
struct SparseScratch { DevBuf keys0, keys1, runs, cum, num, tmp; void release() { keys0.release(); keys1.release(); runs.release(); cum.release(); num.release(); tmp.release(); } };
static int build_sparse_shard(vsg_ctx * c, vsg_index * ix, int sh, int t0, int nt, SparseScratch & w, uint32_t * d_totals)
{
  const vsg_seqset * db = ix->db;
  int rc;
  // window slots of the shard's targets back to back, whatever the layout of the sequence set
  std::vector<int64_t> cum(static_cast<size_t>(nt) + 1, 0);
  for (int i = 0; i < nt; i++) { cum[static_cast<size_t>(i) + 1] = cum[static_cast<size_t>(i)] + db->h_len[static_cast<size_t>(t0) + static_cast<size_t>(i)]; }
  int64_t const W = cum[static_cast<size_t>(nt)];
  if (W >= (static_cast<int64_t>(1) << 31) - 64) { Error::set("vsg_index_create: a shard of 32766 targets holds 2^31 nucleotides or more (wordlength > 10)"); return VSG_EINVAL; }
  DevBuf & bs = ix->b_start[static_cast<size_t>(sh)];
  DevBuf & bp = ix->b_post[static_cast<size_t>(sh)];
  DevBuf & bk = ix->b_rkeys[static_cast<size_t>(sh)];
  int const n = static_cast<int>(W);
  uint32_t nr = 0, total = 0;
  if (n > 0) {
    if ((rc = w.keys0.reserve(sizeof(uint64_t) * (static_cast<size_t>(n) + 8))) != VSG_OK ||
        (rc = w.keys1.reserve(sizeof(uint64_t) * (static_cast<size_t>(n) + 8))) != VSG_OK ||
        (rc = w.cum.reserve(sizeof(int64_t) * (static_cast<size_t>(nt) + 1))) != VSG_OK ||
        (rc = w.num.reserve(64)) != VSG_OK) { return rc; }
    uint64_t * const k0 = static_cast<uint64_t *>(w.keys0.p);
    uint64_t * const k1 = static_cast<uint64_t *>(w.keys1.p);
    uint32_t * const d_num = static_cast<uint32_t *>(w.num.p);
    VSG_CUDA_OK(cudaMemcpyAsync(w.cum.p, cum.data(), sizeof(int64_t) * (static_cast<size_t>(nt) + 1), cudaMemcpyHostToDevice, c->stream));
    sparse_keys_kernel<<<nt, 128, 0, c->stream>>>(db->d, t0, nt, ix->k, ix->mask_lower, static_cast<const int64_t *>(w.cum.p), k0);
    count_launch();
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));   // `cum` (pageable) has been consumed
    size_t tb = 0, tb2 = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, tb, k0, k1, n, 0, 46, c->stream);
    cub::DeviceSelect::Unique(nullptr, tb2, k1, k0, d_num, n, c->stream);
    if ((rc = w.tmp.reserve(std::max(tb, tb2) + 64)) != VSG_OK) { return rc; }
    cub::DeviceRadixSort::SortKeys(w.tmp.p, tb, k0, k1, n, 0, 46, c->stream);
    count_launch();
    cub::DeviceSelect::Unique(w.tmp.p, tb2, k1, k0, d_num, n, c->stream);
    count_launch();
    uint32_t nu = 0;
    VSG_CUDA_OK(cudaMemcpyAsync(&nu, d_num, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
    // k0[0 .. nu): the distinct keys in order, closed by the invalid key if any window was unusable.
    // Sub-lists = runs of key >> 14; the invalid key's run has id 0x80000000 and comes last.
    if ((rc = w.runs.reserve(sizeof(uint32_t) * 2 * (static_cast<size_t>(nu) + 2))) != VSG_OK ||
        (rc = bk.reserve(sizeof(uint32_t) * (static_cast<size_t>(nu) + 2))) != VSG_OK) { return rc; }
    uint32_t * const rcnt = static_cast<uint32_t *>(w.runs.p);
    uint32_t * const rsrc = rcnt + nu + 2;
    uint32_t * const rkeys = static_cast<uint32_t *>(bk.p);
    VSG_CUDA_OK(cudaMemsetAsync(rcnt, 0, sizeof(uint32_t) * 2 * (static_cast<size_t>(nu) + 2), c->stream));
    uint32_t nruns = 0;
    if (nu > 0) {
      auto runs_in = thrust::make_transform_iterator(static_cast<const uint64_t *>(k0), SparseRunOf());
      size_t tb3 = 0;
      cub::DeviceRunLengthEncode::Encode(nullptr, tb3, runs_in, rkeys, rcnt, d_num, static_cast<int>(nu), c->stream);
      if ((rc = w.tmp.reserve(tb3 + 64)) != VSG_OK) { return rc; }
      cub::DeviceRunLengthEncode::Encode(w.tmp.p, tb3, runs_in, rkeys, rcnt, d_num, static_cast<int>(nu), c->stream);
      count_launch();
      VSG_CUDA_OK(cudaMemcpyAsync(&nruns, d_num, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
      if (nruns > 0) {
        uint32_t lastkey = 0;
        VSG_CUDA_OK(cudaMemcpyAsync(&lastkey, rkeys + (nruns - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
        if (lastkey >= 0x80000000u) { nruns--; }
      }
    }
    nr = nruns;
    if (nr > 0) {
      if ((rc = bs.reserve(sizeof(uint32_t) * (static_cast<size_t>(nr) + 2))) != VSG_OK) { return rc; }
      // source offsets (plain counts) and destination offsets (counts padded to vectors of 8) of every sub-list
      size_t tb4 = 0, tb5 = 0;
      auto padded = thrust::make_transform_iterator(static_cast<const uint32_t *>(rcnt), PadTo8());
      cub::DeviceScan::ExclusiveSum(nullptr, tb4, rcnt, rsrc, static_cast<int>(nr + 1), c->stream);
      cub::DeviceScan::ExclusiveSum(nullptr, tb5, padded, static_cast<uint32_t *>(bs.p), static_cast<int>(nr + 1), c->stream);
      if ((rc = w.tmp.reserve(std::max(tb4, tb5) + 64)) != VSG_OK) { return rc; }
      cub::DeviceScan::ExclusiveSum(w.tmp.p, tb4, rcnt, rsrc, static_cast<int>(nr + 1), c->stream);
      count_launch();
      cub::DeviceScan::ExclusiveSum(w.tmp.p, tb5, padded, static_cast<uint32_t *>(bs.p), static_cast<int>(nr + 1), c->stream);
      count_launch();
      VSG_CUDA_OK(cudaMemcpyAsync(&total, static_cast<uint32_t *>(bs.p) + nr, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
      VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
      if ((rc = bp.reserve(sizeof(uint16_t) * (static_cast<size_t>(total) + 64))) != VSG_OK) { return rc; }
      fill_u16_kernel<<<static_cast<unsigned>((static_cast<size_t>(total) + 255) / 256), 256, 0, c->stream>>>(
          static_cast<uint16_t *>(bp.p), static_cast<size_t>(total), POST_PAD);
      count_launch();
      sparse_scatter_kernel<<<(nr + 127) / 128, 128, 0, c->stream>>>(k0, rkeys, rcnt, rsrc, static_cast<const uint32_t *>(bs.p), nr,
                                                                    static_cast<uint16_t *>(bp.p), d_totals);
      count_launch();
      shard_bank_order(c, static_cast<const uint32_t *>(bs.p), static_cast<uint16_t *>(bp.p), nr);
      VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
    }
  }
  if (nr == 0) {
    // no usable window in the whole shard: one empty sub-list under a key no k-mer has
    if ((rc = bs.reserve(16)) != VSG_OK || (rc = bp.reserve(128)) != VSG_OK || (rc = bk.reserve(16)) != VSG_OK) { return rc; }
    VSG_CUDA_OK(cudaMemsetAsync(bs.p, 0, 16, c->stream));
    VSG_CUDA_OK(cudaMemsetAsync(bk.p, 0xff, 16, c->stream));
    nr = 1;
  }
  ShardDev sd{};
  sd.t0 = t0; sd.nt = nt;
  sd.start = static_cast<uint32_t *>(bs.p); sd.post = static_cast<uint16_t *>(bp.p);
  sd.rkeys = static_cast<uint32_t *>(bk.p); sd.nr = nr;
  ix->h_shards.push_back(sd);
  ix->total_postings += total;
  return VSG_OK;
}

// d_totals (optional): 4^k words on the device, zeroed by the caller; receives the number of targets holding each k-mer
int index_create_counts(vsg_ctx * c, const vsg_seqset * db, int wordlength, int mask_lower, uint32_t * d_totals, vsg_index ** out)
{
  if (c == nullptr || db == nullptr || out == nullptr) { Error::set("vsg_index_create: null argument"); return VSG_EINVAL; }
  *out = nullptr;
  if (wordlength < 3 || wordlength > 15) {
    Error::set("vsg_index_create: --wordlength must be in 3..15");
    return VSG_EINVAL;
  }
  if (db->device != c->device) { Error::set("vsg_index_create: the sequence set lives on another device than the context"); return VSG_EINVAL; }
  if (db->d.n > (1 << 24)) { Error::set("vsg_index_create: more than 2^24 targets"); return VSG_EINVAL; }
  VSG_CUDA_OK(cudaSetDevice(c->device));
  int const k = wordlength;
  bool const sparse = k > 10;
  size_t const hashsize = static_cast<size_t>(1) << (2 * k);
  if (!sparse) {
    size_t const bitmap_bytes = std::max<size_t>(hashsize / 8, 4);
    if (bitmap_bytes > 48 * 1024) {
      VSG_CUDA_OK(cudaFuncSetAttribute(index_build_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bitmap_bytes)));
      VSG_CUDA_OK(cudaFuncSetAttribute(index_build_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bitmap_bytes)));
    }
  }
  vsg_index * ix = new (std::nothrow) vsg_index();
  if (ix == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  ix->device = c->device; ix->k = wordlength; ix->mask_lower = mask_lower; ix->ntargets = db->d.n; ix->db = db;
  int const nshards = static_cast<int>((db->d.n + SHARD_STATIC - 1) / SHARD_STATIC);
  ix->b_start.resize(static_cast<size_t>(nshards));
  ix->b_post.resize(static_cast<size_t>(nshards));
  ix->b_rkeys.resize(static_cast<size_t>(nshards));
  DevBuf cnt, tmp;
  SparseScratch w;
  int rc = VSG_OK;
  if (!sparse) { rc = cnt.reserve(sizeof(uint32_t) * (2 * hashsize + 1)); }
  for (int sh = 0; sh < nshards && rc == VSG_OK; sh++) {
    int const t0 = sh * SHARD_STATIC;
    int const nt = static_cast<int>(std::min<int64_t>(SHARD_STATIC, db->d.n - t0));
    rc = sparse ? build_sparse_shard(c, ix, sh, t0, nt, w, d_totals) : build_dense_shard(c, ix, sh, t0, nt, cnt, tmp, d_totals);
  }
  if (rc == VSG_OK) { rc = ix->b_shards.reserve(sizeof(ShardDev) * (ix->h_shards.size() + 1)); }
  cudaError_t e = cudaSuccess;
  if (rc == VSG_OK && !ix->h_shards.empty()) {
    e = cudaMemcpyAsync(ix->b_shards.p, ix->h_shards.data(), sizeof(ShardDev) * ix->h_shards.size(), cudaMemcpyHostToDevice, c->stream);
  }
  if (rc == VSG_OK && e == cudaSuccess) { e = cudaStreamSynchronize(c->stream); }
  if (rc == VSG_OK && e == cudaSuccess) { e = cudaGetLastError(); }
  cnt.release(); tmp.release(); w.release();
  if (rc == VSG_OK && e != cudaSuccess) { Error::set(std::string("vsg_index_create: ") + cudaGetErrorString(e)); rc = VSG_ECUDA; }
  if (rc != VSG_OK) { vsg_index_destroy(ix); return rc; }
  *out = ix;
  return VSG_OK;
}
}  // namespace vsg

extern "C" int vsg_index_create(vsg_ctx * c, const vsg_seqset * db, int wordlength, int mask_lower,
                                vsg_index ** out)
{
  return vsg::index_create_counts(c, db, wordlength, mask_lower, nullptr, out);
}

extern "C" void vsg_index_destroy(vsg_index * ix)
{
  if (ix == nullptr) { return; }
  cudaSetDevice(ix->device);
  for (auto & b : ix->b_start) { b.release(); }
  for (auto & b : ix->b_post) { b.release(); }
  for (auto & b : ix->b_rkeys) { b.release(); }
  ix->b_shards.release();
  delete ix;
}

namespace vsg {
const vsg_seqset * index_db(const vsg_index * ix) { return ix->db; }
int index_wordlength(const vsg_index * ix) { return ix->k; }

void rank_collect_time(vsg_ctx * c);

// launch geometry of a static-index ranking and the HBM scratch of queries with more than KMER_CAP windows
struct RankLaunch {
  int grid = 0, maxlen = 0, bitmap_words = 1;
  uint32_t * scratch = nullptr;
  size_t stride = 0;
};
static int rank_launch_setup(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq, RankLaunch & L)
{
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
  L.grid = static_cast<int>(std::min<int64_t>(nq, static_cast<int64_t>(sms) * 2));
  // queries with more than KMER_CAP windows de-duplicate their k-mers in HBM scratch
  L.maxlen = 0;
  for (int64_t q = q0; q < q0 + nq; q++) { L.maxlen = std::max(L.maxlen, queries->h_len[static_cast<size_t>(q)]); }
  L.scratch = nullptr;
  L.stride = 0;
  L.bitmap_words = std::max(1, (1 << (2 * std::min(ix->k, 10))) >> 5);
  if (ix->k > 10) { L.bitmap_words = 4096; while (L.bitmap_words < 2 * L.maxlen) { L.bitmap_words <<= 1; } }   // hash slots (power of two)
  if (L.maxlen - ix->k + 1 > KMER_CAP) {
    L.stride = static_cast<size_t>(L.bitmap_words) + static_cast<size_t>(L.maxlen) + 8;
    int const rc = c->rank_scratch.reserve(sizeof(uint32_t) * L.stride * static_cast<size_t>(L.grid));
    if (rc != VSG_OK) { return rc; }
    L.scratch = static_cast<uint32_t *>(c->rank_scratch.p);
  }
  return VSG_OK;
}
static int rank_flat_mode()
{
  static int const rank_flat = [] { const char * e = std::getenv("VSG_RANK_FLAT"); return (e == nullptr || e[0] != '0') ? 1 : 0; }();
  return rank_flat;
}
static int rank_check_args(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq)
{
  if (q0 < 0 || nq < 0 || q0 + nq > queries->d.n) { Error::set("vsg_rank: query range out of bounds"); return VSG_EINVAL; }
  if (queries->device != c->device || ix->device != c->device) { Error::set("vsg_rank: sequence set / index lives on another device than the context"); return VSG_EINVAL; }
  return VSG_OK;
}

// device-side results left in ctx->rank_tmp: [seqno nq*tophits][count nq*tophits][n nq][status 1]
int rank_enqueue(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq,
                 int minwordmatches, int tophits, int mask_lower, uint32_t ** d_seqno, uint32_t ** d_count,
                 int32_t ** d_n, int32_t ** d_status)
{
  if (tophits < 1 || tophits > TOPHITS_MAX) { Error::set("vsg_rank: tophits must be in 1..1024"); return VSG_EINVAL; }
  int rc;
  if ((rc = rank_check_args(c, ix, queries, q0, nq)) != VSG_OK) { return rc; }
  if (nq > (1 << 30) / tophits) { Error::set("vsg_rank: batch too large"); return VSG_EINVAL; }
  size_t const cells = static_cast<size_t>(nq) * tophits;
  if ((rc = c->rank_tmp.reserve(sizeof(uint32_t) * (2 * cells + nq + 4))) != VSG_OK) { return rc; }
  *d_seqno = static_cast<uint32_t *>(c->rank_tmp.p);
  *d_count = *d_seqno + cells;
  *d_n = reinterpret_cast<int32_t *>(*d_count + cells);
  *d_status = *d_n + nq;
  VSG_CUDA_OK(cudaMemsetAsync(*d_status, 0, sizeof(int32_t), c->stream));
  if (nq == 0) { return VSG_OK; }
  cudaStream_t const rs = c->stream;
  VSG_CUDA_OK(cudaFuncSetAttribute(rank_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(RANK_SMEM)));
  RankLaunch L;
  if ((rc = rank_launch_setup(c, ix, queries, q0, nq, L)) != VSG_OK) { return rc; }
  VSG_CUDA_OK(cudaEventRecord(c->ev[4], rs));
  rank_kernel<false><<<L.grid, RANK_THREADS, RANK_SMEM, rs>>>(
      queries->d, q0, static_cast<int>(nq), ix->db->d, static_cast<const ShardDev *>(ix->b_shards.p),
      static_cast<int>(ix->h_shards.size()), ix->k, mask_lower, minwordmatches, tophits, *d_seqno, *d_count, *d_n,
      *d_status, L.scratch, L.stride, L.bitmap_words, rank_flat_mode());
  count_launch();
  VSG_CUDA_OK(cudaEventRecord(c->ev[5], rs));
  c->rank_pending = true;
  return VSG_OK;
}

// ---- ranking without the TOPHITS_MAX ceiling ------------------------------------------------------------------------
// RANK_TOP keeps its candidate keys in shared memory (CAND_CAP) and cuts them with an in-block sort, which is what makes
// the default limits fast; longer lists (--maxaccepts 0, --maxrejects 0, large limits) are ranked in two passes over the
// same counting code instead:
//   rank_all_count  pass A: per query the threshold T and the exact number K of targets with count >= T (host arrays);
//                   the caller sizes its work from K before anything large is allocated
//   rank_all_emit   pass B: the K keys of every query of a range into one buffer, one segmented sort (descending), the
//                   first min(K, tophits) keys of each query as CSR (seqno, count) on the device
// Equal to search_topscores + minheap: the keys carry the heap's order, and every target with count >= T is sorted, so
// ties at the cut are broken as the heap breaks them.
__global__ void rank_all_gather_kernel(const uint64_t * __restrict__ keys, const int32_t * __restrict__ koff,
                                       const int32_t * __restrict__ coff, int nq, uint32_t * __restrict__ seqno,
                                       uint32_t * __restrict__ count)
{
  for (int qi = blockIdx.x; qi < nq; qi += gridDim.x) {
    int const n = coff[qi + 1] - coff[qi];
    const uint64_t * __restrict__ kq = keys + koff[qi];
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      uint64_t const key = kq[j];
      seqno[coff[qi] + j] = 0xffffffu - static_cast<uint32_t>(key & 0xffffffu);
      count[coff[qi] + j] = static_cast<uint32_t>(key >> 49);
    }
  }
}

int rank_all_count(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq,
                   int minwordmatches, int tophits, int mask_lower, uint32_t * h_T, int32_t * h_K)
{
  if (tophits < 1) { Error::set("vsg_rank: tophits must be at least 1"); return VSG_EINVAL; }
  int rc;
  if ((rc = rank_check_args(c, ix, queries, q0, nq)) != VSG_OK) { return rc; }
  if (nq == 0) { return VSG_OK; }
  if (nq > (1 << 28)) { Error::set("vsg_rank: batch too large"); return VSG_EINVAL; }
  if ((rc = c->rall_q.reserve(sizeof(uint32_t) * (2 * static_cast<size_t>(nq) + 4))) != VSG_OK) { return rc; }
  uint32_t * const d_T = static_cast<uint32_t *>(c->rall_q.p);
  int32_t * const d_K = reinterpret_cast<int32_t *>(d_T + nq);
  int32_t * const d_status = d_K + nq;
  cudaStream_t const rs = c->stream;
  VSG_CUDA_OK(cudaMemsetAsync(d_status, 0, sizeof(int32_t), rs));
  VSG_CUDA_OK(cudaFuncSetAttribute(rank_kernel<false, RANK_COUNT>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(RANK_SMEM)));
  RankLaunch L;
  if ((rc = rank_launch_setup(c, ix, queries, q0, nq, L)) != VSG_OK) { return rc; }
  int const hstride = (std::min(std::max(L.maxlen - ix->k + 1, 0), 32767) + 1 + 31) & ~31;
  if ((rc = c->rall_hist.reserve(sizeof(uint32_t) * static_cast<size_t>(hstride) * static_cast<size_t>(L.grid))) != VSG_OK) { return rc; }
  VSG_CUDA_OK(cudaEventRecord(c->ev[4], rs));
  rank_kernel<false, RANK_COUNT><<<L.grid, RANK_THREADS, RANK_SMEM, rs>>>(
      queries->d, q0, static_cast<int>(nq), ix->db->d, static_cast<const ShardDev *>(ix->b_shards.p),
      static_cast<int>(ix->h_shards.size()), ix->k, mask_lower, minwordmatches, tophits, nullptr, nullptr, d_K,
      d_status, L.scratch, L.stride, L.bitmap_words, rank_flat_mode(), d_T, nullptr, nullptr,
      static_cast<uint32_t *>(c->rall_hist.p), hstride);
  count_launch();
  VSG_CUDA_OK(cudaEventRecord(c->ev[5], rs));
  c->rank_pending = true;
  int32_t status = 0;
  VSG_CUDA_OK(cudaMemcpyAsync(h_T, d_T, sizeof(uint32_t) * static_cast<size_t>(nq), cudaMemcpyDeviceToHost, rs));
  VSG_CUDA_OK(cudaMemcpyAsync(h_K, d_K, sizeof(int32_t) * static_cast<size_t>(nq), cudaMemcpyDeviceToHost, rs));
  VSG_CUDA_OK(cudaMemcpyAsync(&status, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, rs));
  VSG_CUDA_OK(cudaStreamSynchronize(rs));
  VSG_CUDA_OK(cudaGetLastError());
  rank_collect_time(c);
  if (status != 0) { Error::set("vsg_rank: a query is longer than the device ranker supports (65 534 + wordlength nt)"); return VSG_EINVAL; }
  return VSG_OK;
}

int rank_all_emit(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq,
                  int minwordmatches, int tophits, int mask_lower, const uint32_t * h_T, const int32_t * h_K,
                  uint32_t ** d_seqno, uint32_t ** d_count, const int32_t ** d_coff)
{
  *d_seqno = nullptr; *d_count = nullptr; *d_coff = nullptr;
  int rc;
  if ((rc = rank_check_args(c, ix, queries, q0, nq)) != VSG_OK) { return rc; }
  if (nq == 0) { return VSG_OK; }
  // key offsets, candidate offsets, T, n, status
  size_t const n1 = static_cast<size_t>(nq) + 1;
  std::vector<int32_t> h(2 * n1 + 2 * static_cast<size_t>(nq) + 1, 0);
  int64_t kt = 0, ct = 0;
  for (int64_t i = 0; i < nq; i++) {
    h[static_cast<size_t>(i)] = static_cast<int32_t>(kt);
    h[n1 + static_cast<size_t>(i)] = static_cast<int32_t>(ct);
    h[2 * n1 + static_cast<size_t>(i)] = static_cast<int32_t>(h_T[i]);
    kt += h_K[i];
    ct += std::min<int64_t>(h_K[i], tophits);
    if (kt > INT32_MAX - 64) { Error::set("vsg_rank: more than 2^31 candidate keys in one call"); return VSG_EINVAL; }
  }
  h[static_cast<size_t>(nq)] = static_cast<int32_t>(kt);
  h[n1 + static_cast<size_t>(nq)] = static_cast<int32_t>(ct);
  if ((rc = c->rall_q.reserve(sizeof(int32_t) * h.size())) != VSG_OK ||
      (rc = c->rall_keys.reserve(sizeof(uint64_t) * (2 * static_cast<size_t>(kt) + 2))) != VSG_OK ||
      (rc = c->rall_out.reserve(sizeof(uint32_t) * (2 * static_cast<size_t>(ct) + 2))) != VSG_OK) { return rc; }
  int32_t * const d_koff = static_cast<int32_t *>(c->rall_q.p);
  int32_t * const d_cand_off = d_koff + n1;
  uint32_t * const d_T = reinterpret_cast<uint32_t *>(d_cand_off + n1);
  int32_t * const d_n = reinterpret_cast<int32_t *>(d_T + nq);
  int32_t * const d_status = d_n + nq;
  uint64_t * const keys0 = static_cast<uint64_t *>(c->rall_keys.p);
  uint64_t * const keys1 = keys0 + kt + 1;
  uint32_t * const out = static_cast<uint32_t *>(c->rall_out.p);
  cudaStream_t const rs = c->stream;
  // pageable source: staged before the call returns
  VSG_CUDA_OK(cudaMemcpyAsync(d_koff, h.data(), sizeof(int32_t) * h.size(), cudaMemcpyHostToDevice, rs));
  VSG_CUDA_OK(cudaFuncSetAttribute(rank_kernel<false, RANK_EMIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(RANK_SMEM)));
  RankLaunch L;
  if ((rc = rank_launch_setup(c, ix, queries, q0, nq, L)) != VSG_OK) { return rc; }
  VSG_CUDA_OK(cudaEventRecord(c->ev[4], rs));
  rank_kernel<false, RANK_EMIT><<<L.grid, RANK_THREADS, RANK_SMEM, rs>>>(
      queries->d, q0, static_cast<int>(nq), ix->db->d, static_cast<const ShardDev *>(ix->b_shards.p),
      static_cast<int>(ix->h_shards.size()), ix->k, mask_lower, minwordmatches, tophits, nullptr, nullptr, d_n,
      d_status, L.scratch, L.stride, L.bitmap_words, rank_flat_mode(), d_T, d_koff, keys0, nullptr, 0);
  count_launch();
  if (kt > 0) {
    size_t tb = 0;
    VSG_CUDA_OK(cub::DeviceSegmentedSort::SortKeysDescending(nullptr, tb, keys0, keys1, static_cast<int>(kt), static_cast<int>(nq),
                                                             d_koff, d_koff + 1, rs));
    if ((rc = c->rall_tmp.reserve(tb + 16)) != VSG_OK) { return rc; }
    VSG_CUDA_OK(cub::DeviceSegmentedSort::SortKeysDescending(c->rall_tmp.p, tb, keys0, keys1, static_cast<int>(kt), static_cast<int>(nq),
                                                             d_koff, d_koff + 1, rs));
    count_launch();
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
    rank_all_gather_kernel<<<static_cast<int>(std::min<int64_t>(nq, static_cast<int64_t>(sms) * 8)), 256, 0, rs>>>(
        keys1, d_koff, d_cand_off, static_cast<int>(nq), out, out + ct);
    count_launch();
  }
  VSG_CUDA_OK(cudaEventRecord(c->ev[5], rs));
  c->rank_pending = true;
  int32_t status = 0;
  VSG_CUDA_OK(cudaMemcpyAsync(&status, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, rs));
  VSG_CUDA_OK(cudaStreamSynchronize(rs));
  VSG_CUDA_OK(cudaGetLastError());
  rank_collect_time(c);
  if (status == 1) { Error::set("vsg_rank: a query is longer than the device ranker supports (65 534 + wordlength nt)"); return VSG_EINVAL; }
  if (status != 0) { Error::set("vsg_rank: the second ranking pass found another number of candidates than the first"); return VSG_ECUDA; }
  *d_seqno = out;
  *d_count = out + ct;
  *d_coff = d_cand_off;
  return VSG_OK;
}

// call after the stream has been synchronised
void rank_collect_time(vsg_ctx * c)
{
  if (c->rank_pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]) == cudaSuccess) { c->prof_rank_ms += ms; }
    c->rank_pending = false;
  }
}
}  // namespace vsg

extern "C" int vsg_rank(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * queries, int64_t q0, int64_t nq,
                        int minwordmatches, int tophits, int mask_lower, uint32_t * cand_seqno,
                        uint32_t * cand_count, int32_t * ncand)
{
  if (c == nullptr || ix == nullptr || queries == nullptr || cand_seqno == nullptr || cand_count == nullptr || ncand == nullptr) {
    Error::set("vsg_rank: null argument");
    return VSG_EINVAL;
  }
  VSG_CUDA_OK(cudaSetDevice(c->device));
  if (tophits > TOPHITS_MAX) {
    // the caller's dense rows, filled from the CSR of rank_all_emit a key budget at a time
    std::vector<uint32_t> T(static_cast<size_t>(std::max<int64_t>(nq, 0)));
    std::vector<int32_t> K(T.size());
    int rc = rank_all_count(c, ix, queries, q0, nq, minwordmatches, tophits, mask_lower, T.data(), K.data());
    if (rc != VSG_OK) { return rc; }
    std::vector<uint32_t> hs, hc;
    for (int64_t i0 = 0; i0 < nq;) {
      int64_t i1 = i0, vol = 0;
      while (i1 < nq && (i1 == i0 || vol + K[static_cast<size_t>(i1)] <= CAND_VOLUME_BUDGET)) { vol += K[static_cast<size_t>(i1++)]; }
      uint32_t *d_seqno, *d_count;
      const int32_t * d_coff;
      if ((rc = rank_all_emit(c, ix, queries, q0 + i0, i1 - i0, minwordmatches, tophits, mask_lower, T.data() + i0, K.data() + i0,
                              &d_seqno, &d_count, &d_coff)) != VSG_OK) { return rc; }
      int64_t ct = 0;
      for (int64_t i = i0; i < i1; i++) { ct += std::min<int64_t>(K[static_cast<size_t>(i)], tophits); }
      hs.resize(static_cast<size_t>(ct)); hc.resize(static_cast<size_t>(ct));
      if (ct > 0) {
        VSG_CUDA_OK(cudaMemcpyAsync(hs.data(), d_seqno, sizeof(uint32_t) * static_cast<size_t>(ct), cudaMemcpyDeviceToHost, c->stream));
        VSG_CUDA_OK(cudaMemcpyAsync(hc.data(), d_count, sizeof(uint32_t) * static_cast<size_t>(ct), cudaMemcpyDeviceToHost, c->stream));
        VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
      }
      size_t pos = 0;
      for (int64_t i = i0; i < i1; i++) {
        int const n = static_cast<int>(std::min<int64_t>(K[static_cast<size_t>(i)], tophits));
        std::memcpy(cand_seqno + static_cast<size_t>(i) * tophits, hs.data() + pos, sizeof(uint32_t) * static_cast<size_t>(n));
        std::memcpy(cand_count + static_cast<size_t>(i) * tophits, hc.data() + pos, sizeof(uint32_t) * static_cast<size_t>(n));
        ncand[i] = n;
        pos += static_cast<size_t>(n);
      }
      i0 = i1;
    }
    return VSG_OK;
  }
  uint32_t *d_seqno, *d_count; int32_t *d_n, *d_status;
  int rc = rank_enqueue(c, ix, queries, q0, nq, minwordmatches, tophits, mask_lower, &d_seqno, &d_count, &d_n, &d_status);
  if (rc != VSG_OK) { return rc; }
  size_t const cells = static_cast<size_t>(nq) * tophits;
  int32_t status = 0;
  if (nq > 0) {
    VSG_CUDA_OK(cudaMemcpyAsync(cand_seqno, d_seqno, sizeof(uint32_t) * cells, cudaMemcpyDeviceToHost, c->stream));
    VSG_CUDA_OK(cudaMemcpyAsync(cand_count, d_count, sizeof(uint32_t) * cells, cudaMemcpyDeviceToHost, c->stream));
    VSG_CUDA_OK(cudaMemcpyAsync(ncand, d_n, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, c->stream));
  }
  VSG_CUDA_OK(cudaMemcpyAsync(&status, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  VSG_CUDA_OK(cudaGetLastError());
  rank_collect_time(c);
  if (status != 0) {
    Error::set("vsg_rank: a query is longer than the device ranker supports (65 534 + wordlength nt)");
    return VSG_EINVAL;
  }
  return VSG_OK;
}


// ---------------------------------------------------------------------------------------------
// Incremental index of the cluster driver: replaces Dbindex::prepare + Dbindex::add_sequence
// (core/dbindex.cpp:121-148, 163-255) for a set of targets that GROWS (the centroids).  Targets get
// dense numbers in creation order; list km holds the numbers of the targets containing k-mer km, in
// creation order, inside a CSR whose per-list CAPACITY is the number of sequences of the whole set that
// contain km (every sequence could become a centroid) — counted once, as the reference's counting pass
// does for its bitmap/list sizing.  Shards of 32768 targets are contiguous ranges of every list; the
// list positions at a shard boundary are snapshotted when the boundary is crossed.
// ---------------------------------------------------------------------------------------------
namespace vsg {

__global__ void cindex_append_kernel(DevSeqs db, const uint32_t * __restrict__ seqnos, int n, uint32_t first_id, int k,
                                     int mask_lower, uint32_t * __restrict__ cursor, uint32_t * __restrict__ post32,
                                     int32_t * __restrict__ clen)
{
  extern __shared__ uint32_t bitmap[];
  int const ci = blockIdx.x;
  if (ci >= n) { return; }
  int const words = (1 << (2 * k)) >> 5;
  for (int i = threadIdx.x; i < (words > 0 ? words : 1); i += blockDim.x) { bitmap[i] = 0; }
  __syncthreads();
  int64_t const t = seqnos[ci];
  const uint8_t * __restrict__ s = db.sym + db.off[t];
  int const len = db.len[t];
  if (threadIdx.x == 0) { clen[first_id + ci] = len; }
  for (int p = k - 1 + threadIdx.x; p < len; p += blockDim.x) {
    uint32_t km;
    if (kmer_at(s, p, k, mask_lower, km)) {
      uint32_t const bit = 1u << (km & 31);
      uint32_t const old = atomicOr(&bitmap[km >> 5], bit);
      if ((old & bit) == 0) { post32[atomicAdd(&cursor[km], 1u)] = first_id + static_cast<uint32_t>(ci); }
    }
  }
}

struct CIndex {
  int device = 0, k = 8, mask_lower = 0;
  const vsg_seqset * set = nullptr;
  int64_t ncent = 0;                 // targets added so far
  DevBuf b_start, b_cursor, b_post, b_clen, b_shards, b_seqnos;
  std::vector<DevBuf> b_begin;       // list positions at the start of shard s >= 1
  std::vector<uint32_t> h_seqno;     // dense target number -> sequence number
};

int cindex_create(vsg_ctx * c, const vsg_seqset * set, int wordlength, int mask_lower, CIndex ** out)
{
  *out = nullptr;
  if (wordlength < 3 || wordlength > 10) { Error::set("cluster index: the device index supports --wordlength 3..10"); return VSG_EINVAL; }
  VSG_CUDA_OK(cudaSetDevice(c->device));
  CIndex * ix = new (std::nothrow) CIndex();
  if (ix == nullptr) { Error::set("out of host memory"); return VSG_ENOMEM; }
  ix->device = c->device; ix->k = wordlength; ix->mask_lower = mask_lower; ix->set = set;
  size_t const hashsize = static_cast<size_t>(1) << (2 * wordlength);
  size_t const bitmap_bytes = std::max<size_t>(hashsize / 8, 4);
  if (bitmap_bytes > 48 * 1024) {
    VSG_CUDA_OK(cudaFuncSetAttribute(index_build_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bitmap_bytes)));
    VSG_CUDA_OK(cudaFuncSetAttribute(cindex_append_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bitmap_bytes)));
  }
  int rc;
  DevBuf cnt, tmp;
  if ((rc = cnt.reserve(sizeof(uint32_t) * (hashsize + 1))) != VSG_OK ||
      (rc = ix->b_start.reserve(sizeof(uint32_t) * (hashsize + 1))) != VSG_OK ||
      (rc = ix->b_cursor.reserve(sizeof(uint32_t) * (hashsize + 1))) != VSG_OK ||
      (rc = ix->b_clen.reserve(sizeof(int32_t) * (static_cast<size_t>(set->d.n) + 1))) != VSG_OK) { delete ix; return rc; }
  // capacity of every list = the number of sequences of the whole set that contain the k-mer
  VSG_CUDA_OK(cudaMemsetAsync(cnt.p, 0, sizeof(uint32_t) * (hashsize + 1), c->stream));
  int64_t const n = set->d.n;
  for (int64_t t0 = 0; t0 < n; t0 += 1 << 20) {
    int const nt = static_cast<int>(std::min<int64_t>(1 << 20, n - t0));
    index_build_kernel<false><<<nt, 128, bitmap_bytes, c->stream>>>(set->d, static_cast<int>(t0), nt, wordlength, mask_lower, 0,
                                                                    static_cast<uint32_t *>(cnt.p), nullptr, nullptr);
    count_launch();
  }
  size_t tb = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tb, static_cast<uint32_t *>(cnt.p), static_cast<uint32_t *>(ix->b_start.p), static_cast<int>(hashsize + 1), c->stream);
  if ((rc = tmp.reserve(tb + 16)) != VSG_OK) { delete ix; return rc; }
  cub::DeviceScan::ExclusiveSum(tmp.p, tb, static_cast<uint32_t *>(cnt.p), static_cast<uint32_t *>(ix->b_start.p), static_cast<int>(hashsize + 1), c->stream);
  count_launch();
  // 64-bit check of the total: offsets are 32-bit
  {
    std::vector<uint32_t> h(hashsize);
    VSG_CUDA_OK(cudaMemcpyAsync(h.data(), cnt.p, sizeof(uint32_t) * hashsize, cudaMemcpyDeviceToHost, c->stream));
    VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
    uint64_t total = 0;
    for (uint32_t v : h) { total += v; }
    if (total > 0xfffffff0ull) { cnt.release(); tmp.release(); delete ix; Error::set("cluster index: more than 2^32 k-mer occurrences in the sequence set"); return VSG_EINVAL; }
    if ((rc = ix->b_post.reserve(sizeof(uint32_t) * (total + 64))) != VSG_OK) { cnt.release(); tmp.release(); delete ix; return rc; }
  }
  VSG_CUDA_OK(cudaMemcpyAsync(ix->b_cursor.p, ix->b_start.p, sizeof(uint32_t) * (hashsize + 1), cudaMemcpyDeviceToDevice, c->stream));
  VSG_CUDA_OK(cudaStreamSynchronize(c->stream));
  cnt.release(); tmp.release();
  *out = ix;
  return VSG_OK;
}

void cindex_destroy(CIndex * ix)
{
  if (ix == nullptr) { return; }
  cudaSetDevice(ix->device);
  for (DevBuf * b : {&ix->b_start, &ix->b_cursor, &ix->b_post, &ix->b_clen, &ix->b_shards, &ix->b_seqnos}) { b->release(); }
  for (auto & b : ix->b_begin) { b.release(); }
  delete ix;
}

// Dbindex::add_sequence for a batch of new targets (ascending sequence numbers); enqueued on c->stream
int cindex_append(vsg_ctx * c, CIndex * ix, const uint32_t * seqnos, int n)
{
  if (n <= 0) { return VSG_OK; }
  size_t const hashsize = static_cast<size_t>(1) << (2 * ix->k);
  size_t const bitmap_bytes = std::max<size_t>(hashsize / 8, 4);
  int rc;
  int done = 0;
  while (done < n) {
    // never across a shard boundary in one launch: a shard's part of every list must be contiguous
    int64_t const room = SHARD - (ix->ncent % SHARD);
    int const m = static_cast<int>(std::min<int64_t>(n - done, room));
    if (sizeof(uint32_t) * static_cast<size_t>(m) + 16 > ix->b_seqnos.cap) {
      VSG_CUDA_OK(cudaStreamSynchronize(c->stream));   // the buffer is about to be replaced: let earlier launches finish with it
      if ((rc = ix->b_seqnos.reserve(sizeof(uint32_t) * static_cast<size_t>(std::max(m, 4096)) + 16)) != VSG_OK) { return rc; }
    }
    // the upload below reuses one small buffer: order it after the previous launch on the same stream
    VSG_CUDA_OK(cudaMemcpyAsync(ix->b_seqnos.p, seqnos + done, sizeof(uint32_t) * static_cast<size_t>(m), cudaMemcpyHostToDevice, c->stream));
    cindex_append_kernel<<<m, 128, bitmap_bytes, c->stream>>>(ix->set->d, static_cast<const uint32_t *>(ix->b_seqnos.p), m,
                                                              static_cast<uint32_t>(ix->ncent), ix->k, ix->mask_lower,
                                                              static_cast<uint32_t *>(ix->b_cursor.p), static_cast<uint32_t *>(ix->b_post.p),
                                                              static_cast<int32_t *>(ix->b_clen.p));
    count_launch();   // (the copy above is from pageable memory: staged before cudaMemcpyAsync returns)
    for (int i = 0; i < m; i++) { ix->h_seqno.push_back(seqnos[done + i]); }
    ix->ncent += m;
    done += m;
    if (ix->ncent % SHARD == 0) {
      ix->b_begin.emplace_back();
      if ((rc = ix->b_begin.back().reserve(sizeof(uint32_t) * (hashsize + 1))) != VSG_OK) { return rc; }
      VSG_CUDA_OK(cudaMemcpyAsync(ix->b_begin.back().p, ix->b_cursor.p, sizeof(uint32_t) * (hashsize + 1), cudaMemcpyDeviceToDevice, c->stream));
    }
  }
  return VSG_OK;
}

const std::vector<uint32_t> & cindex_seqnos(const CIndex * ix) { return ix->h_seqno; }

// search_topscores of queries [q0, q0+nq) of `queries` against the targets added so far; results as rank_enqueue,
// candidate numbers are DENSE target numbers (CIndex::h_seqno maps them back)
int cindex_rank_enqueue(vsg_ctx * c, CIndex * ix, const vsg_seqset * queries, int64_t q0, int64_t nq, int minwordmatches,
                        int tophits, uint32_t ** d_seqno, uint32_t ** d_count, int32_t ** d_n, int32_t ** d_status)
{
  if (tophits < 1 || tophits > TOPHITS_MAX) { Error::set("cluster ranker: tophits must be in 1..1024"); return VSG_EINVAL; }
  size_t const cells = static_cast<size_t>(nq) * tophits;
  int rc;
  if ((rc = c->rank_tmp.reserve(sizeof(uint32_t) * (2 * cells + nq + 4))) != VSG_OK) { return rc; }
  *d_seqno = static_cast<uint32_t *>(c->rank_tmp.p);
  *d_count = *d_seqno + cells;
  *d_n = reinterpret_cast<int32_t *>(*d_count + cells);
  *d_status = *d_n + nq;
  VSG_CUDA_OK(cudaMemsetAsync(*d_status, 0, sizeof(int32_t), c->stream));
  if (nq == 0) { return VSG_OK; }
  int const nshards = static_cast<int>((ix->ncent + SHARD - 1) / SHARD);
  if (nshards == 0) {   // nothing indexed yet: no candidates
    VSG_CUDA_OK(cudaMemsetAsync(*d_n, 0, sizeof(int32_t) * nq, c->stream));
    return VSG_OK;
  }
  std::vector<ShardDev> sh(static_cast<size_t>(nshards));
  for (int s = 0; s < nshards; s++) {
    ShardDev & sd = sh[static_cast<size_t>(s)];
    sd.start = static_cast<const uint32_t *>(s == 0 ? ix->b_start.p : ix->b_begin[static_cast<size_t>(s) - 1].p);
    sd.end = static_cast<const uint32_t *>(s + 1 < nshards || ix->ncent % SHARD == 0 ? ix->b_begin[static_cast<size_t>(s)].p : ix->b_cursor.p);
    sd.post = nullptr; sd.post32 = static_cast<const uint32_t *>(ix->b_post.p);
    sd.rkeys = nullptr; sd.nr = 0; sd.reserved = 0;
    sd.t0 = s * SHARD;
    sd.nt = static_cast<int32_t>(std::min<int64_t>(SHARD, ix->ncent - static_cast<int64_t>(s) * SHARD));
  }
  if ((rc = ix->b_shards.reserve(sizeof(ShardDev) * sh.size())) != VSG_OK) { return rc; }
  // pageable source: staged before the call returns, so `sh` may go out of scope
  VSG_CUDA_OK(cudaMemcpyAsync(ix->b_shards.p, sh.data(), sizeof(ShardDev) * sh.size(), cudaMemcpyHostToDevice, c->stream));
  VSG_CUDA_OK(cudaFuncSetAttribute(rank_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(RANK_SMEM)));
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
  int const grid = static_cast<int>(std::min<int64_t>(nq, static_cast<int64_t>(sms) * 2));
  DevSeqs lens{nullptr, nullptr, static_cast<const int32_t *>(ix->b_clen.p), ix->ncent};   // target lengths by dense number
  int maxlen = 0;
  for (int64_t q = q0; q < q0 + nq; q++) { maxlen = std::max(maxlen, queries->h_len[static_cast<size_t>(q)]); }
  uint32_t * d_scratch = nullptr;
  size_t stride = 0;
  int const bitmap_words = std::max(1, (1 << (2 * ix->k)) >> 5);
  if (maxlen - ix->k + 1 > KMER_CAP) {
    stride = static_cast<size_t>(bitmap_words) + static_cast<size_t>(maxlen) + 8;
    if ((rc = c->rank_scratch.reserve(sizeof(uint32_t) * stride * static_cast<size_t>(grid))) != VSG_OK) { return rc; }
    d_scratch = static_cast<uint32_t *>(c->rank_scratch.p);
  }
  rank_kernel<true><<<grid, RANK_THREADS, RANK_SMEM, c->stream>>>(
      queries->d, q0, static_cast<int>(nq), lens, static_cast<const ShardDev *>(ix->b_shards.p), nshards, ix->k, ix->mask_lower,
      minwordmatches, tophits, *d_seqno, *d_count, *d_n, *d_status, d_scratch, stride, bitmap_words, 0);
  count_launch();
  return VSG_OK;
}

}  // namespace vsg
