// vsg_internal.h — shared between the CUDA translation units of libvsg.so (not installed).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <memory>
#include <string>
#include <vector>

#include "../../include/vsg.h"

namespace vsg {

// ---------------------------------------------------------------------------------------------
// Scoring as the kernels see it (built once per context from vsg_scoring; the 16-bit clamping and
// the "defer everything" flag follow core/align_simd.cpp:1264-1277, 1316-1373).
// ---------------------------------------------------------------------------------------------
enum { Q_L = 0, T_L = 1, Q_I = 2, T_I = 3, Q_R = 4, T_R = 5 };

struct ScoreParams {
  int16_t S[16][16];  // substitution matrix over 4-bit codes (align_simd.cpp:1319-1342)
  int16_t go[6];      // gap open   {q_l,t_l,q_i,t_i,q_r,t_r}
  int16_t ge[6];      // gap extend {q_l,t_l,q_i,t_i,q_r,t_r}
  int16_t match, mismatch;
  int16_t score_min;  // SHRT_MIN + max(0, all six open+extend) (align_simd.cpp:1432-1444)
  int16_t n_mismatch;
  int32_t fallback;   // a value did not fit a 16-bit cell: every pair is deferred
  int32_t shift;      // anti-diagonal shift c of a SHIFTED scoring (align_ckpt.cuh): S - 2c, ge + c; 0 = the caller's own
};

// One symbol per byte in HBM: bits 0-3 = 4-bit IUPAC code (utils/maps.cpp:75-118),
// bit 4 = lower case (soft-masked).  That is everything the aligner (code) and the k-mer
// sampler (code is a single base? lower case?) need from the ASCII byte.
struct DevSeqs {
  const uint8_t * sym;
  const int64_t * off;
  const int32_t * len;
  int64_t n;
};

// A unit of forward-DP work for one warp: one query against two targets, one per 16-bit half of
// every packed register (thi == tlo when the query has an odd number of targets; the duplicate
// half's output slot is -1).
struct FastTask {
  uint32_t q;
  uint32_t tlo, thi;
  int32_t out_lo, out_hi;  // pair slots (index into the per-batch stats array), -1 = discard
  int32_t dmax;            // max(dlen_lo, dlen_hi)
  uint64_t dir_off;        // byte offset of this task's direction block
  uint64_t bnd_off;        // element offset (uint2) of the strip-boundary row, if strips > 1
};

struct ExactTask {
  uint32_t q, t;
  int32_t out;
  int32_t pad;
  uint64_t dir_off;  // qlen*dlen bytes, row-major, one byte per cell
  uint64_t he_off;   // 2*qlen int16
};

// What the traceback kernel needs to find a pair's direction bits.
struct PairDesc {
  uint32_t q, t;
  uint64_t dir_off;
  int32_t kind;   // 0 = fast layout, 1 = exact layout, 2 = checkpoints (align_ckpt.cuh): dir_off / aux_off are uint2 element offsets
  int32_t out;    // pair slot in the stats array
  int32_t R;      // fast: rows per lane
  int32_t half;   // fast: 0 = low nibble, 1 = high nibble; checkpoints: bit 0 = half, bit 1 = general alphabet
  int32_t dmax;   // fast: steps per strip = dmax + 31
  uint64_t cigar_off;  // scratch region for the reversed CIGAR (qlen+dlen+2 bytes)
  uint64_t aux_off;    // checkpoints: element offset of the task's column checkpoints
};

struct Error {
  static void set(const std::string & m);
};

#define VSG_CUDA_OK(call)                                                                 \
  do {                                                                                    \
    cudaError_t e__ = (call);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      vsg::Error::set(std::string(#call) + ": " + cudaGetErrorString(e__));               \
      return VSG_ECUDA;                                                                   \
    }                                                                                     \
  } while (0)

// growable device / pinned buffers
struct DevBuf {
  void * p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes);
  void release();
};
struct PinBuf {
  void * p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes);
  void release();
};

void count_launch(int n = 1);

// Candidate lists longer than the shared-memory ranker's 1 024 entries are ranked and searched in pieces of at most this
// many candidate keys (summed over the queries and strands of a piece): 8 MB of keys on the device and, in
// vsg_search_batch, about 150 MB of host hit records per worker thread.
constexpr int64_t CAND_VOLUME_BUDGET = int64_t(1) << 20;

// vsg_align_pairs with traceback on demand (align_ckpt.cuh, TbGate): leader_of[k] = index of pair k's group leader in
// this call, or -1; threshold = 100 * --id (+ margin); skipped pairs return aligned = matches = mismatches = 0xffff
int align_pairs_gated(vsg_ctx * c, const vsg_seqset * queries, const vsg_seqset * targets,
                      int64_t npairs, const uint32_t * qidx, const uint32_t * tidx,
                      int16_t * score, uint16_t * aligned, uint16_t * matches,
                      uint16_t * mismatches, uint16_t * gaps, int32_t * trims,
                      char * cigar_buf, int64_t cigar_cap, int64_t * cigar_off,
                      const int32_t * leader_of, double gate_threshold, int gate_iddef);

// vsg_search_batch / vsg_group_search with the rows of query q (at most max_rows) in rows[q] instead of a dense
// nq x max_results array: memory in proportion to the rows produced, whatever the limits (vsg_usearch_stream)
int search_batch_rows(vsg_ctx * c, const vsg_index * ix, const vsg_seqset * db, const vsg_seqset * queries, int64_t q0,
                      int64_t nq, const vsg_search_opts * opts, int64_t max_rows, std::vector<vsg_search_result> * rows,
                      int32_t * counts, int64_t * work);
int group_search_rows(vsg_group * g, const char * qcat, const int64_t * qoff, const int32_t * qlen, int64_t nq,
                      int dust_queries, const vsg_search_opts * opts, int64_t max_rows, std::vector<vsg_search_result> * rows,
                      int32_t * counts, int64_t * work);

}  // namespace vsg

struct vsg_seqset {
  vsg::DevSeqs d{};
  std::vector<int32_t> h_len;       // host copy of lengths
  std::vector<int64_t> h_off;       // host copy of offsets
  std::vector<uint8_t> h_nonacgt;   // 1 if the sequence holds a symbol outside ACGTU
  vsg::DevBuf b_sym, b_off, b_len;
  int device = 0;
  int64_t total = 0;
};

struct vsg_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  vsg_scoring scoring{};
  vsg::ScoreParams sp{};
  vsg::ScoreParams sp2{};      // the shifted scoring the checkpoint kernels run with (align_ckpt.cuh)
  bool ckpt_enabled = true;    // VSG_CKPT=0 routes single-strip pairs through the direction-bit kernel instead (A/B, tests)
  bool fast_disabled = false;  // VSG_DISABLE_FAST=1 (tests force the exact kernel)
  // scratch
  vsg::DevBuf dir, bnd, he, cigar_scratch, cigar_dense, stats, tasks_fast, tasks_exact, pairs,
      cigar_len, cigar_offs, cub_tmp, rank_tmp, rank_scratch, pre_flags, ticket, gate,
      rall_q, rall_hist, rall_keys, rall_out, rall_tmp;   // ranking without the tophits ceiling (rank.cu)
  vsg::PinBuf h_tasks, h_stats;
  size_t dir_budget = (size_t)64 << 30;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  // cumulative profile since the last vsg_profile_reset (kernel times from cudaEvents on `stream`)
  int64_t prof_cells = 0, prof_fast = 0, prof_exact = 0, prof_fwd_launches = 0, prof_tb_skipped = 0;
  float prof_fwd_ms = 0.f, prof_tb_ms = 0.f, prof_rank_ms = 0.f;
  bool rank_pending = false;
  std::vector<cudaEvent_t> ev_pool;  // 3 per chunk of an align call
  vsg_fallback_fn fallback = nullptr;  // host-side aligner for SHRT_MAX pairs
  void * fallback_user = nullptr;
  std::vector<vsg_ctx *> children;  // per-host-thread contexts of vsg_search_batch
  std::shared_ptr<void> search_scratch;  // host buffers of vsg_search_batch's driver, kept between calls
};
