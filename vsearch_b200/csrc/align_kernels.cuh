// align_kernels.cuh — device code of the batched global aligner (sm_100a).
//
// Three kernels replace the reference's search16 (core/align_simd.cpp:1447-2060):
//
//  nw_fast_kernel<R,GENERAL>   one WARP aligns one query against TWO targets at once.  Every
//      32-bit register holds the same DP quantity for both targets as two 16-bit halves
//      (VIMNMX.S16x2 / VIADD.16x2 are native on sm_100a).  Lane l owns query rows
//      [l*R, l*R+R) and walks the target columns as an anti-diagonal wavefront: at step s it is at
//      column s-l, takes H/F of the row above from lane l-1 by warp shuffle and keeps its own H/E
//      column in registers, so DP state never touches memory.  Substitution scores come from a
//      shared-memory table (replicated per lane -> conflict free), per-column data (table offset,
//      target-gap penalties, top-boundary values) from a 64-entry shared-memory ring the warp
//      refills with coalesced loads every 32 steps.  The four direction bits per cell
//      (align_simd.cpp:710-717) fall out of the max instructions' predicates and are stored as
//      R bytes per lane per step, 128*RW contiguous bytes per warp per step.  Queries longer than
//      32*R rows run as several strips that hand the boundary row over through HBM.
//      Arithmetic is exact integer arithmetic in a biased (+0x8000) unsigned 16-bit representation; the host only
//      sends a pair here when a bound on every intermediate proves that neither saturation nor the
//      reference's overflow flag can occur (vsg_api.cu: fast_path_ok), in which case the
//      reference's saturating arithmetic is plain integer arithmetic too.
//
//  nw_exact_kernel             one THREAD per pair, 32-bit arithmetic with explicit clamps that
//      reproduces the reference's saturating 16-bit lanes bit for bit, including the blocks of four
//      columns, the zero-padded last block and the sticky h_min/h_max overflow flag
//      (align_simd.cpp:825-826, 1735-1752, 2029-2051).  Used for every pair the bound cannot clear.
//
//  traceback_kernel            one thread per pair walks the stored direction bits exactly as
//      backtrack16 does (align_simd.cpp:1132-1245) and emits statistics, terminal-gap trims and
//      (optionally) the run-length CIGAR.
#pragma once

#include "vsg_internal.h"

#include <type_traits>

namespace vsg {

// every DP value v is held as the unsigned halfword v + 0x8000: the whole non-saturating range of
// the reference's signed cells, ordered correctly under UNSIGNED compares, and never negative, so
// 32-bit adds/subtracts of packed pairs cannot carry between the halves
constexpr uint32_t BIAS = 0x8000u;
constexpr uint32_t BIAS2 = 0x80008000u;
constexpr int FAST_WARPS = 4;        // warps per CTA
constexpr int FAST_RMAX = 16;        // rows per lane
constexpr int RING = 64;             // column records per warp

__host__ __device__ inline int fast_rw(int R) { return R <= 4 ? 1 : (R <= 8 ? 2 : 4); }
// Direction bytes of one strip.  Layout: a lane's direction words of 4/RW consecutive wavefront
// steps form one 16-byte TILE (RW = 1: four steps, RW = 2: two, RW = 4: one); the tiles of the 32
// lanes of a step group lie back to back, so the warp writes a group with one fully coalesced
// 512-byte store.  A diagonal move of the traceback (one row up = same lane one byte down, one
// column left = one step back) stays inside the tile, which the traceback keeps in registers:
// one 16-byte load serves up to 4/RW steps of the walk.
__host__ __device__ inline size_t fast_strip_bytes(int dmax, int R)
{
  return static_cast<size_t>((dmax + 31 + 3) & ~3) * 32 * fast_rw(R) * 4;
}

__device__ __forceinline__ uint32_t pk2(int lo, int hi)
{
  return (static_cast<uint32_t>(lo) & 0xffffu) | (static_cast<uint32_t>(hi) << 16);
}
__device__ __forceinline__ uint32_t pk1(int v) { return pk2(v, v); }

// per-halfword unsigned max; ORs bit_lo / bit_hi into w where b > a strictly (i.e. NOT a >= b)
__device__ __forceinline__ uint32_t max_flag(uint32_t a, uint32_t b, uint32_t & w,
                                             uint32_t bit_lo, uint32_t bit_hi)
{
  bool ph, pl;
  uint32_t const m = __vibmax_u16x2(a, b, &ph, &pl);  // VIMNMX.U16x2 with predicate outputs
  if (!pl) { w |= bit_lo; }
  if (!ph) { w |= bit_hi; }
  return m;
}

// shared-memory loads by 32-bit shared-window address: keeps ptxas from re-deriving the generic
// base address (S2R/S2UR/LEA chains) inside the hot loop
__device__ __forceinline__ uint32_t lds32(uint32_t a)
{
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t a)
{
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}

__device__ __forceinline__ int code_to_2bit(int c4) { return (c4 == 2) ? 1 : (c4 == 4) ? 2 : (c4 == 8) ? 3 : 0; }

// Semantics self-test of the DPX intrinsic the fast kernel leans on (run once per context).
// Inputs arrive as kernel arguments so that nothing is folded at compile time.
__global__ void dpx_selftest_kernel(int * bad, int a0, int a1, int b0, int b1, int c0, int c1, int d0, int d1)
{
  bool ph, pl;
  // halves: lo = (5 vs 7) -> max 7, pred(a>=b)=false ; hi = (9 vs 9) -> pred true
  uint32_t m = __vibmax_u16x2(pk2(a0, a1), pk2(b0, b1), &ph, &pl);
  int b = 0;
  if (m != pk2(7, 9) || pl || !ph) { b |= 1; }
  // large halves (unsigned order): lo = (0xfffd vs 0xfffc) -> pred true; hi = (0x0002 vs 0xfff6) -> 0xfff6, pred false
  m = __vibmax_u16x2(pk2(c0, d1), pk2(d0, c1), &ph, &pl);
  if (m != pk2(-3, -10) || !pl || ph) { b |= 2; }
  if (__vadd2(pk2(c0, 100), pk2(d1, -7)) != pk2(-1, 93)) { b |= 4; }
  // the fused forms of the checkpoint kernel: per-half wrapping add, unsigned max (VIADDMNMX.U16x2, VIMNMX3.U16x2)
  // lo: max(0xfffd + 0xfff6 (= -3 - 10 -> 0xfff3), 0x0002) = 0xfff3 ; hi: max(100 - 4, 96 + 1) = 97
  if (__viaddmax_u16x2(pk2(c0, 100), pk2(c1, d0), pk2(d1, 97)) != pk2(-13, 97)) { b |= 8; }
  if (__vimax3_u16x2(pk2(a0, a1), pk2(b0, b1), pk2(d1, c1)) != pk2(7, -10)) { b |= 16; }
  *bad = b;
}

// shared memory the fast kernel needs beyond its static arrays (the per-lane score profile)
__host__ __device__ constexpr bool fast_has_profile(int R, bool general) { return !general && R <= 8; }
__host__ __device__ constexpr size_t fast_dyn_smem(int R, bool general)
{
  return fast_has_profile(R, general) ? static_cast<size_t>(FAST_WARPS) * 16 * ((R + 3) / 4) * 32 * 16 : 0;
}

template <int R, bool GENERAL, bool MULTI>
__global__ void __launch_bounds__(FAST_WARPS * 32)
nw_fast_kernel(const __grid_constant__ ScoreParams sp, DevSeqs qs, DevSeqs ts,
               const FastTask * __restrict__ tasks, int ntasks,
               uint8_t * __restrict__ dir, uint2 * __restrict__ bnd, int32_t * __restrict__ stats)
{
  constexpr int RW = (R <= 4 ? 1 : (R <= 8 ? 2 : 4));
  // PROF: plain-ACGT classes with <= 8 rows per lane read their substitution scores from a per-lane
  // PROFILE (target-pair code x the lane's own rows) so that one 128-bit load serves four rows
  constexpr bool PROF = fast_has_profile(R, GENERAL);
  constexpr int RQ = (R + 3) / 4;
  constexpr int LUT_WORDS = GENERAL ? 4096 : (PROF ? 32 : 64 * 32);
  // MULTI: the query needs several strips (only queries longer than 32*FAST_RMAX rows do)
  extern __shared__ uint4 prof_mem[];
  __shared__ uint32_t lut[LUT_WORDS];
  // every column record is stored twice, RING entries apart, so that the 32 consecutive records a
  // lane reads during a chunk are contiguous (no wrap-around arithmetic per step)
  __shared__ uint4 ringA[FAST_WARPS][2 * RING];
  __shared__ uint32_t ringB[FAST_WARPS][2 * RING];

  int const lane = threadIdx.x & 31;
  int const wib = threadIdx.x >> 5;

  if (!PROF) {
    // substitution table: both halves looked up at once
    for (int e = threadIdx.x; e < LUT_WORDS; e += blockDim.x) {
      if (GENERAL) {
        int const q = e >> 8, dlo = e & 15, dhi = (e >> 4) & 15;
        lut[e] = pk2(sp.S[dlo][q], sp.S[dhi][q]);
      } else {
        int const ent = e >> 5;  // replicated for the 32 lanes: word = ent*32 + lane
        int const q = 1 << (ent >> 4), dlo = 1 << (ent & 3), dhi = 1 << ((ent >> 2) & 3);
        lut[e] = pk2(sp.S[dlo][q], sp.S[dhi][q]);
      }
    }
    __syncthreads();
  }

  int const w = blockIdx.x * FAST_WARPS + wib;
  if (w >= ntasks) { return; }
  FastTask const tk = tasks[w];

  int const Q = qs.len[tk.q];
  uint8_t const * __restrict__ qsym = qs.sym + qs.off[tk.q];
  int const Dlo = ts.len[tk.tlo], Dhi = ts.len[tk.thi];
  uint8_t const * __restrict__ dlo_p = ts.sym + ts.off[tk.tlo];
  uint8_t const * __restrict__ dhi_p = ts.sym + ts.off[tk.thi];
  int const dmax = tk.dmax;
  int const nsteps = dmax + 31;
  int const strip_rows = 32 * R;
  int const nstrips = MULTI ? (Q + strip_rows - 1) / strip_rows : 1;
  size_t const strip_bytes = fast_strip_bytes(dmax, R);

  int const QRqi = sp.go[Q_I] + sp.ge[Q_I], Rqi = sp.ge[Q_I];
  int const QRqr = sp.go[Q_R] + sp.ge[Q_R], Rqr = sp.ge[Q_R];
  int const QRti = sp.go[T_I] + sp.ge[T_I], Rti = sp.ge[T_I];
  int const QRtr = sp.go[T_R] + sp.ge[T_R], Rtr = sp.ge[T_R];
  int const gotl = sp.go[T_L], getl = sp.ge[T_L];
  int const goql = sp.go[Q_L], geql = sp.ge[Q_L];

  // where the final score H(Q-1, D-1) lives
  int const klast = (Q - 1) / strip_rows;
  int const llast = ((Q - 1) % strip_rows) / R;
  int const rlast = (Q - 1) % R;
  int score_lo = 0, score_hi = 0;

  uint4 * const rA = ringA[wib];
  uint32_t * const rB = ringB[wib];
  uint2 * const mybnd = bnd + tk.bnd_off;
  uint32_t const lut_s = static_cast<uint32_t>(__cvta_generic_to_shared(lut));
  uint32_t const rA_s = static_cast<uint32_t>(__cvta_generic_to_shared(rA));
  uint32_t const rB_s = static_cast<uint32_t>(__cvta_generic_to_shared(rB));
  // this lane's column of the profile: entry (tp, r4) sits at prof_s + (tp*RQ + r4)*512
  uint4 * const myprof = prof_mem + static_cast<size_t>(wib) * 16 * RQ * 32 + lane;
  uint32_t const prof_s = static_cast<uint32_t>(__cvta_generic_to_shared(myprof));

  for (int strip = 0; strip < nstrips; strip++) {
    int const row0 = strip * strip_rows + lane * R;

    uint32_t Hl[R], E[R], rowoff[PROF ? 1 : R], QRq[R], Rq[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
      int const i = row0 + r;
      bool const last = (i == Q - 1);
      QRq[r] = pk1(last ? QRqr : QRqi);
      Rq[r] = pk1(last ? Rqr : Rqi);
      Hl[r] = BIAS2 - pk1(gotl + (i + 1) * getl);  // H(i,-1)     (align_simd.cpp:852-853)
      E[r] = Hl[r] - QRq[r];                       // E(i,0)      (align_simd.cpp:855-857)
      // per-row constants must live in registers: without this ptxas re-derives the "is this the
      // query's last row" select (compare + select + repack) for every row of every step
      asm volatile("" : "+r"(QRq[r]), "+r"(Rq[r]));
    }
    if (PROF) {
      // rows beyond the query's end score like 'A' (their cells are never read)
      int code[RQ * 4];
#pragma unroll
      for (int r = 0; r < RQ * 4; r++) {
        int const i = row0 + r;
        code[r] = (r < R && i < Q) ? (1 << code_to_2bit(qsym[i] & 15)) : 1;
      }
      for (int tp = 0; tp < 16; tp++) {
        int const dlo = 1 << (tp & 3), dhi = 1 << (tp >> 2);
#pragma unroll
        for (int r4 = 0; r4 < RQ; r4++) {
          uint4 v;
          v.x = pk2(sp.S[dlo][code[4 * r4 + 0]], sp.S[dhi][code[4 * r4 + 0]]);
          v.y = pk2(sp.S[dlo][code[4 * r4 + 1]], sp.S[dhi][code[4 * r4 + 1]]);
          v.z = pk2(sp.S[dlo][code[4 * r4 + 2]], sp.S[dhi][code[4 * r4 + 2]]);
          v.w = pk2(sp.S[dlo][code[4 * r4 + 3]], sp.S[dhi][code[4 * r4 + 3]]);
          myprof[(tp * RQ + r4) * 32] = v;   // read back by this lane only: no barrier needed
        }
      }
    } else {
#pragma unroll
      for (int r = 0; r < R; r++) {
        int const i = row0 + r;
        int const code = (i < Q) ? (qsym[i] & 15) : 0;
        rowoff[r] = lut_s + (GENERAL ? static_cast<uint32_t>(code) * 1024u
                                     : (static_cast<uint32_t>(code_to_2bit(code)) * 16u * 32u + lane) * 4u);
        asm volatile("" : "+r"(rowoff[r]));
      }
    }
    // H(row0-1,-1): the diagonal input of this lane's first row at column 0
    uint32_t diag_in = (row0 == 0) ? BIAS2 : BIAS2 - pk1(gotl + row0 * getl);
    uint32_t Hout = BIAS2, Fout = BIAS2;
    uint8_t * const dstrip = dir + tk.dir_off + static_cast<size_t>(strip) * strip_bytes;
    bool const write_bnd = MULTI && (strip + 1 < nstrips) && (lane == 31);
    bool const capture = (strip == klast) && (lane == llast);
    // the steps at which the lane that owns the last row passes the targets' last columns
    int const cap_lo = (strip == klast) ? Dlo - 1 + llast : -1;
    int const cap_hi = (strip == klast) ? Dhi - 1 + llast : -1;

    // one step of the wavefront: this lane's R rows of column c.  EDGE steps may find the lane
    // outside the matrix (ramp-up / ramp-down) and may have to pick up the final score; steady
    // steps (all 32 lanes inside, no score to capture) skip those tests.
    struct Words { uint32_t v[RW]; };  // the direction words one lane produces in one step
    auto step = [&](auto edge_tag, int c, uint32_t aA, uint32_t aB, Words & out) -> bool {
      constexpr bool EDGE = decltype(edge_tag)::value;
      uint32_t hin = __shfl_up_sync(0xffffffffu, Hout, 1);
      uint32_t fin = __shfl_up_sync(0xffffffffu, Fout, 1);
      if (!EDGE || (c >= 0 && c < dmax)) {
        uint4 const rec = lds128(aA);
        if (lane == 0) { hin = rec.w; fin = lds32(aB); }

        // H(i-1,j-1) + S for every row first: the old column is dead before the new one is
        // produced (no register rotation at the loop edge) and these adds are off the F chain
        uint32_t t[R];
        if (PROF) {
          uint32_t const pa = prof_s + rec.x;
#pragma unroll
          for (int r4 = 0; r4 < RQ; r4++) {
            uint4 const S4 = lds128(pa + r4 * 512u);
            uint32_t const Sv[4] = {S4.x, S4.y, S4.z, S4.w};
#pragma unroll
            for (int u = 0; u < 4; u++) {
              int const r = 4 * r4 + u;
              if (r < R) { t[r] = __vadd2(r == 0 ? diag_in : Hl[r - 1], Sv[u]); }
            }
          }
        } else {
#pragma unroll
          for (int r = 0; r < R; r++) {
            uint32_t const S = lds32(rowoff[r] + rec.x);
            t[r] = __vadd2(r == 0 ? diag_in : Hl[r - 1], S);
          }
        }
        uint32_t F = fin;
        uint32_t wd[RW];
#pragma unroll
        for (int kk = 0; kk < RW; kk++) { wd[kk] = 0; }

#pragma unroll
        for (int r = 0; r < R; r++) {
          // the 8 flags of this row-step go to a register of their own (a short dependency chain
          // per row instead of one 32-deep chain per word, which made ptxas park predicates in
          // P2R/ISETP pairs); one multiply-add per row merges it into the output word
          uint32_t fb = 0;
          uint32_t const m1 = max_flag(t[r], F, fb, 1u, 16u);     // up:   F > h
          uint32_t const h = max_flag(m1, E[r], fb, 2u, 32u);     // left: E > h
          Hl[r] = h;
          uint32_t const hf = h - rec.y;                          // H - QR_t
          uint32_t const f = F - rec.z;                           // F - R_t
          F = max_flag(hf, f, fb, 4u, 64u);                       // extup:   f > hf
          uint32_t const he = h - QRq[r];
          uint32_t const e = E[r] - Rq[r];
          E[r] = max_flag(he, e, fb, 8u, 128u);                   // extleft: e > he
          wd[r >> 2] = fb * (1u << (8u * (r & 3))) + wd[r >> 2];
        }
        Hout = Hl[R - 1];
        Fout = F;
        diag_in = hin;

#pragma unroll
        for (int kk = 0; kk < RW; kk++) { out.v[kk] = wd[kk]; }

        if (MULTI && write_bnd) { __stcg(mybnd + c, make_uint2(Hout, Fout)); }

        if (EDGE && capture && (c == Dlo - 1 || c == Dhi - 1)) {
          uint32_t v = 0;
#pragma unroll
          for (int r = 0; r < R; r++) { if (r == rlast) { v = Hl[r]; } }
          if (c == Dlo - 1) { score_lo = static_cast<int>(v & 0xffffu) - static_cast<int>(BIAS); }
          if (c == Dhi - 1) { score_hi = static_cast<int>(v >> 16) - static_cast<int>(BIAS); }
        }
        return true;
      }
      return false;
    };

    // the tile this lane writes for steps [g*SPT, g*SPT + SPT) starts at dwords + g * 128
    constexpr int SPT = 4 / RW;
    uint32_t * const dwords = reinterpret_cast<uint32_t *>(dstrip) + static_cast<size_t>(lane) * 4;
    for (int s0 = 0; s0 < nsteps; s0 += 32) {
      {
        // refill the ring with columns [s0, s0+32): one column per lane, coalesced
        __syncwarp();
        int const cc = s0 + lane;
        if (cc < dmax) {
          int const a = (cc < Dlo) ? (dlo_p[cc] & 15) : 0;
          int const b = (cc < Dhi) ? (dhi_p[cc] & 15) : 0;
          uint4 rec;
          rec.x = GENERAL ? static_cast<uint32_t>(a + 16 * b) * 4u
                          : static_cast<uint32_t>(code_to_2bit(a) + 4 * code_to_2bit(b)) * (PROF ? RQ * 512u : 128u);
          // target-gap penalties: right-end values from the target's last column on
          // (align_simd.cpp:1741-1751)
          rec.y = pk2(cc >= Dlo - 1 ? QRtr : QRti, cc >= Dhi - 1 ? QRtr : QRti);
          rec.z = pk2(cc >= Dlo - 1 ? Rtr : Rti, cc >= Dhi - 1 ? Rtr : Rti);
          uint32_t fin0;
          if (!MULTI || strip == 0) {
            rec.w = BIAS2 - pk1(goql + (cc + 1) * geql);  // H(-1,c)  (align_simd.cpp:1895-1901)
            fin0 = rec.w - rec.y;                         // F(0,c)   (align_simd.cpp:830-833)
          } else {
            uint2 const v = __ldcg(mybnd + cc);
            rec.w = v.x;
            fin0 = v.y;
          }
          int const slot = cc & (RING - 1);
          rA[slot] = rec; rA[slot + RING] = rec;
          rB[slot] = fin0; rB[slot + RING] = fin0;
        }
        __syncwarp();
      }
      // this lane's records for the chunk start at column s0 - lane
      uint32_t const slot0 = static_cast<uint32_t>(s0 - lane) & (RING - 1);
      uint32_t aA = rA_s + slot0 * 16u, aB = rB_s + slot0 * 4u;
      bool const steady = (s0 >= 32) && (s0 + 31 < dmax) &&
                          (static_cast<unsigned>(cap_lo - s0) >= 32u) && (static_cast<unsigned>(cap_hi - s0) >= 32u);
      if (steady) {
        constexpr int UNR = (RW == 1) ? 4 : 2;  // steps per trip: a whole tile (RW <= 2) or two (RW == 4)
#pragma unroll 1
        for (int k0 = 0; k0 < 32; k0 += UNR) {
          Words b[UNR];
#pragma unroll
          for (int u = 0; u < UNR; u++) {
            step(std::false_type{}, s0 - lane + k0 + u, aA + (k0 + u) * 16u, aB + (k0 + u) * 4u, b[u]);
          }
          uint4 * const tp = reinterpret_cast<uint4 *>(dwords + static_cast<size_t>((s0 + k0) / SPT) * 128);
          if (RW == 1) { tp[0] = make_uint4(b[0].v[0], b[1].v[0], b[UNR > 2 ? 2 : 0].v[0], b[UNR > 3 ? 3 : 0].v[0]); }
          else if (RW == 2) { tp[0] = make_uint4(b[0].v[0], b[0].v[1], b[1].v[0], b[1].v[1]); }
          else {
#pragma unroll
            for (int u = 0; u < UNR; u++) { tp[32 * u] = make_uint4(b[u].v[0], b[u].v[1], b[u].v[RW > 2 ? 2 : 0], b[u].v[RW > 3 ? 3 : 0]); }
          }
        }
      } else {
        int const kend = min(32, nsteps - s0);
        int c = s0 - lane;
        for (int k = 0; k < kend; k++, c++, aA += 16u, aB += 4u) {
          Words w1;
          if (step(std::true_type{}, c, aA, aB, w1)) {
            uint32_t const * const wd = w1.v;
            int const sg = s0 + k;
            uint32_t * const dp = dwords + static_cast<size_t>(sg / SPT) * 128 + (sg % SPT) * RW;
            if (RW == 1) { dp[0] = wd[0]; }
            else if (RW == 2) { *reinterpret_cast<uint2 *>(dp) = make_uint2(wd[0], wd[1]); }
            else { *reinterpret_cast<uint4 *>(dp) = make_uint4(wd[0], wd[1], wd[RW > 2 ? 2 : 0], wd[RW > 3 ? 3 : 0]); }
          }
        }
      }
    }
    __syncwarp();
  }

  if (lane == llast) {
    if (tk.out_lo >= 0) { stats[static_cast<size_t>(tk.out_lo) * VSG_STAT_WORDS + VSG_STAT_SCORE] = score_lo; }
    if (tk.out_hi >= 0) { stats[static_cast<size_t>(tk.out_hi) * VSG_STAT_WORDS + VSG_STAT_SCORE] = score_hi; }
  }
}

// ---------------------------------------------------------------------------------------------
// exact kernel: bit-for-bit model of one saturating 16-bit lane, one thread per pair
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int sat16(int x) { return x > 32767 ? 32767 : (x < -32768 ? -32768 : x); }

__global__ void nw_exact_kernel(const __grid_constant__ ScoreParams sp, DevSeqs qs, DevSeqs ts,
                                const ExactTask * __restrict__ tasks, int ntasks,
                                uint8_t * __restrict__ dir, int16_t * __restrict__ he,
                                int32_t * __restrict__ stats)
{
  int const w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= ntasks) { return; }
  ExactTask const tk = tasks[w];
  int const Q = qs.len[tk.q];
  int const D = ts.len[tk.t];
  uint8_t const * __restrict__ qsym = qs.sym + qs.off[tk.q];
  uint8_t const * __restrict__ dsym = ts.sym + ts.off[tk.t];
  uint8_t * __restrict__ dp = dir + tk.dir_off;
  int16_t * __restrict__ Hcol = he + tk.he_off;
  int16_t * __restrict__ Ecol = Hcol + Q;

  int const QRqi = sp.go[Q_I] + sp.ge[Q_I], Rqi = sp.ge[Q_I];
  int const QRqr = sp.go[Q_R] + sp.ge[Q_R], Rqr = sp.ge[Q_R];
  int const QRti = sp.go[T_I] + sp.ge[T_I], Rti = sp.ge[T_I];
  int const QRtr = sp.go[T_R] + sp.ge[T_R], Rtr = sp.ge[T_R];
  int const QRtl = sp.go[T_L] + sp.ge[T_L], Rtl = sp.ge[T_L];
  int const Rql = sp.ge[Q_L];

  int H[4], F[4], Sm[4] = {0, 0, 0, 0};
  H[0] = 0;
  for (int k = 1; k < 4; k++) { H[k] = static_cast<int16_t>(-sp.go[Q_L] - k * sp.ge[Q_L]); }
  for (int k = 0; k < 4; k++) { F[k] = static_cast<int16_t>(-sp.go[Q_L] - (k + 1) * sp.ge[Q_L]); }

  bool overflow = false;
  int const nblocks = (D + 3) / 4;
  for (int b = 0; b < nblocks; b++) {
    int sym[4], QRt[4], Rt[4], h[4], f[4], n[4] = {0, 0, 0, 0};
    bool const ends = (4 * b + 4 >= D);
    for (int k = 0; k < 4; k++) {
      int const j = 4 * b + k;
      sym[k] = j < D ? (dsym[j] & 15) : 0;
      bool const right = ends && (k >= ((D + 3) & 3));
      QRt[k] = right ? sat16(QRti + sat16(QRtr - QRti)) : QRti;
      Rt[k] = right ? sat16(Rti + sat16(Rtr - Rti)) : Rti;
      h[k] = H[k];
      f[k] = sat16(F[k] - QRt[k]);
    }
    int h_min = 0, h_max = 0;
    int M = QRtl;
    for (int i = 0; i < Q; i++) {
      bool const last = (i == Q - 1);
      int h4 = 0, E;
      if (b == 0) {
        if (!last) {
          h4 = sat16(0 - M);
          E = sat16(sat16(0 - M) - QRqi);
          M = sat16(M + Rtl);
        } else {
          E = sat16(sat16(0 - M) - QRqr);
        }
      } else {
        if (!last) { h4 = Hcol[i]; }
        E = Ecol[i];
      }
      int const QRq = last ? QRqr : QRqi;
      int const Rq = last ? Rqr : Rqi;
      int const qc = qsym[i] & 15;
      for (int k = 0; k < 4; k++) {
        int Hc = sat16(h[k] + sp.S[sym[k]][qc]);
        int bits = 0;
        if (f[k] > Hc) { bits |= 1; }
        Hc = max(Hc, f[k]);
        if (E > Hc) { bits |= 2; }
        Hc = max(Hc, E);
        h_min = min(h_min, Hc);
        h_max = max(h_max, Hc);
        n[k] = Hc;
        int const HF = sat16(Hc - QRt[k]);
        f[k] = sat16(f[k] - Rt[k]);
        if (f[k] > HF) { bits |= 4; }
        f[k] = max(f[k], HF);
        int const HE = sat16(Hc - QRq);
        E = sat16(E - Rq);
        if (E > HE) { bits |= 8; }
        E = max(E, HE);
        int const j = 4 * b + k;
        if (j < D) { dp[static_cast<size_t>(i) * D + j] = static_cast<uint8_t>(bits); }
      }
      Hcol[i] = static_cast<int16_t>(n[3]);
      Ecol[i] = static_cast<int16_t>(E);
      h[0] = h4; h[1] = n[0]; h[2] = n[1]; h[3] = n[2];
    }
    for (int k = 0; k < 4; k++) { Sm[k] = n[k]; }
    if (h_min <= sp.score_min || h_max >= 32767) { overflow = true; }
    H[0] = sat16(H[3] - Rql); H[1] = sat16(H[0] - Rql); H[2] = sat16(H[1] - Rql); H[3] = sat16(H[2] - Rql);
    F[0] = sat16(F[3] - Rql); F[1] = sat16(F[0] - Rql); F[2] = sat16(F[1] - Rql); F[3] = sat16(F[2] - Rql);
  }
  stats[static_cast<size_t>(tk.out) * VSG_STAT_WORDS + VSG_STAT_SCORE] =
      overflow ? VSG_SCORE_SENTINEL : Sm[(D + 3) & 3];
}

// ---------------------------------------------------------------------------------------------
// traceback (backtrack16, align_simd.cpp:1132-1245) + trims + optional CIGAR text
// ---------------------------------------------------------------------------------------------
struct DirReader {
  uint8_t const * base;
  int kind, R, RW, half, D;
  size_t strip_bytes;
  int strip_rows;
  // position of the current row i, kept incrementally (the walk only ever moves one row up)
  int l = 0, r = 0, sh = 0;        // fast layout: lane, row within the lane, log2(steps per tile)
  size_t row_base = 0;             // fast: strip offset; exact: i * D
  // the 16-byte tile read last (fast layout): consecutive traceback steps mostly stay inside it
  size_t tile_at = ~static_cast<size_t>(0);
  uint4 tile = {0u, 0u, 0u, 0u};
  __device__ __forceinline__ void start(int i)
  {
    if (kind == 1) { row_base = static_cast<size_t>(i) * D; return; }
    int const strip = i / strip_rows;
    int const il = i - strip * strip_rows;
    l = il / R;
    r = il - l * R;
    row_base = static_cast<size_t>(strip) * strip_bytes;
    sh = RW == 1 ? 2 : (RW == 2 ? 1 : 0);
  }
  __device__ __forceinline__ void up()  // i -> i - 1
  {
    if (kind == 1) { row_base -= static_cast<size_t>(D); return; }
    if (--r < 0) {
      r = R - 1;
      if (--l < 0) { l = 31; row_base -= strip_bytes; }
    }
  }
  __device__ __forceinline__ int get(int j)
  {
    if (kind == 1) { return base[row_base + j]; }
    int const sg = j + l;  // wavefront step at which lane l visits column j
    int const g = sg >> sh;
    size_t const a = row_base + (static_cast<size_t>(g) * 32 + l) * 16;
    if (a != tile_at) {
      tile = __ldg(reinterpret_cast<const uint4 *>(base + a));
      tile_at = a;
    }
    int const idx = (sg - (g << sh)) * (RW * 4) + r;  // byte within the tile
    int const wsel = idx >> 2;
    uint32_t const w = wsel == 0 ? tile.x : (wsel == 1 ? tile.y : (wsel == 2 ? tile.z : tile.w));
    int const v = static_cast<int>((w >> (8 * (idx & 3))) & 0xffu);
    return half ? (v >> 4) : (v & 15);
  }
};

// four sequence symbols at a time for the traceback's backward walk (a thread's loads are not
// coalesced with its neighbours': every load instruction costs the warp 32 memory transactions)
struct SymCache {
  uintptr_t at = 0;  // address of the aligned 4-byte word held
  uint32_t w = 0;
  __device__ __forceinline__ int get(uint8_t const * __restrict__ p, int i)
  {
    // the aligned word around p[i] lies inside the symbol buffer's allocation (device allocations
    // start and end on coarser boundaries than 4 bytes)
    uintptr_t const a = reinterpret_cast<uintptr_t>(p + i);
    uintptr_t const wa = a & ~static_cast<uintptr_t>(3);
    if (wa != at) { at = wa; w = __ldg(reinterpret_cast<const uint32_t *>(wa)); }
    return static_cast<int>((w >> (8 * (a & 3))) & 15u);
  }
};

struct CigarWriter {
  char * end;   // next byte is written at --end
  char op;
  int run;
  int len;
  bool text;
  __device__ __forceinline__ void flush()
  {
    if (op != 0 && run != 0) {
      int n = 1;
      if (text) { *--end = op; }
      if (run > 1) {
        int v = run;
        while (v > 0) {
          if (text) { *--end = static_cast<char>('0' + (v % 10)); }
          v /= 10;
          n++;
        }
      }
      len += n;
    }
  }
  __device__ __forceinline__ void push(char o)
  {
    if (o == op) { run++; return; }
    if (text) { flush(); }  // statistics-only walks need the open run (op, run), not the text length
    op = o;
    run = 1;
  }
  __device__ __forceinline__ void push_n(char o, int n)
  {
    if (o == op) { run += n; return; }
    if (text) { flush(); }
    op = o;
    run = n;
  }
};

template <bool TEXT>
__device__ __forceinline__ void traceback_one(const ScoreParams & sp, const DevSeqs & qs, const DevSeqs & ts,
                                              const PairDesc & pd, uint8_t const * __restrict__ dir,
                                              char * __restrict__ cigar_scratch, int32_t * __restrict__ stats)
{
  int32_t * const st = stats + static_cast<size_t>(pd.out) * VSG_STAT_WORDS;
  if (st[VSG_STAT_SCORE] == VSG_SCORE_SENTINEL) {
    st[VSG_STAT_ALIGNED] = 0; st[VSG_STAT_MATCHES] = 0; st[VSG_STAT_MISMATCHES] = 0;
    st[VSG_STAT_GAPS] = 0; st[VSG_STAT_TRIM_LEFT] = 0; st[VSG_STAT_TRIM_RIGHT] = 0;
    st[VSG_STAT_CIGARLEN] = 0;
    if (TEXT) { cigar_scratch[pd.cigar_off] = 0; }
    return;
  }
  int const Q = qs.len[pd.q];
  int const D = ts.len[pd.t];
  uint8_t const * __restrict__ qsym = qs.sym + qs.off[pd.q];
  uint8_t const * __restrict__ dsym = ts.sym + ts.off[pd.t];

  SymCache qc, tc;
  DirReader rd;
  rd.base = dir + pd.dir_off;
  rd.kind = pd.kind; rd.R = pd.R; rd.RW = fast_rw(pd.R); rd.half = pd.half; rd.D = D;
  rd.strip_rows = 32 * pd.R;
  rd.strip_bytes = fast_strip_bytes(pd.dmax, pd.R);

  CigarWriter cw;
  cw.text = TEXT;
  cw.end = TEXT ? (cigar_scratch + pd.cigar_off + Q + D + 1) : nullptr;
  if (TEXT) { *--cw.end = 0; }
  cw.op = 0; cw.run = 0; cw.len = 0;

  int aligned = 0, matches = 0, mismatches = 0, gaps = 0;
  int i = Q - 1, j = D - 1;
  rd.start(i);
  char op = 0;
  int last_run_op = 0;  // op of the run that ends the alignment (first one pushed)
  int last_run = 0;
  bool first_run_open = true;

  while (i >= 0 && j >= 0) {
    aligned++;
    int const b = rd.get(j);
    // backtrack16's priorities (align_simd.cpp:1150-1190) as selects: the lanes of a warp walk
    // unrelated alignments, so every branch here is a divergent one
    bool const ext_i = (op == 'I') && (b & 8);
    bool const ext_d = !ext_i && (op == 'D') && (b & 4);
    bool const open_i = !ext_i && !ext_d && (b & 2);
    bool const open_d = !ext_i && !ext_d && !open_i && (b & 1);
    bool const is_i = ext_i || open_i, is_d = ext_d || open_d;
    gaps += ((open_i && op != 'I') || (open_d && op != 'D')) ? 1 : 0;
    if (!is_i && !is_d) {
      int const a = qc.get(qsym, i), c = tc.get(dsym, j);
      bool const hit = (a & c) != 0 && !(sp.n_mismatch && (a == 15 || c == 15));
      matches += hit ? 1 : 0;
      mismatches += hit ? 0 : 1;
    }
    char const nop = is_i ? 'I' : (is_d ? 'D' : 'M');
    if (!is_i) { i--; rd.up(); }
    if (!is_d) { j--; }
    if (first_run_open) {
      if (last_run == 0 || nop == last_run_op) { last_run_op = nop; last_run++; }
      else { first_run_open = false; }
    }
    cw.push(nop);
    op = nop;
  }
  while (i >= 0) {
    aligned++;
    if (op != 'D') { gaps++; }
    i--;
    if (first_run_open) {
      if (last_run == 0 || last_run_op == 'D') { last_run_op = 'D'; last_run++; }
      else { first_run_open = false; }
    }
    cw.push('D');
    op = 'D';
  }
  while (j >= 0) {
    aligned++;
    if (op != 'I') { gaps++; }
    j--;
    if (first_run_open) {
      if (last_run == 0 || last_run_op == 'I') { last_run_op = 'I'; last_run++; }
      else { first_run_open = false; }
    }
    cw.push('I');
    op = 'I';
  }
  // the run still open in the writer is the alignment's FIRST (leftmost) run
  int const first_op = cw.op, first_run = cw.run;
  cw.flush();

  st[VSG_STAT_ALIGNED] = aligned;
  st[VSG_STAT_MATCHES] = matches;
  st[VSG_STAT_MISMATCHES] = mismatches;
  st[VSG_STAT_GAPS] = gaps;
  st[VSG_STAT_TRIM_LEFT] = first_op == 'D' ? first_run : (first_op == 'I' ? -first_run : 0);
  st[VSG_STAT_TRIM_RIGHT] = last_run_op == 'D' ? last_run : (last_run_op == 'I' ? -last_run : 0);
  st[VSG_STAT_CIGARLEN] = cw.len;
  // the text (if any) sits right-aligned: it ends with its NUL at region + Q + D
}

template <bool TEXT>
__global__ void traceback_kernel(const __grid_constant__ ScoreParams sp, DevSeqs qs, DevSeqs ts,
                                 const PairDesc * __restrict__ pairs, int npairs,
                                 uint8_t const * __restrict__ dir, char * __restrict__ cigar_scratch,
                                 int32_t * __restrict__ stats)
{
  int const p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npairs) { return; }
  PairDesc const pd = pairs[p];
  if (pd.kind == 2) { return; }  // checkpoint layout: traceback_ckpt_pairs_kernel's (align_ckpt.cuh)
  traceback_one<TEXT>(sp, qs, ts, pd, dir, cigar_scratch, stats);
}

// statistics-only traceback straight from the forward tasks (no per-pair descriptors to build,
// upload or read): thread 2k / 2k+1 = first / second target of task k
__global__ void traceback_fast_tasks_kernel(const __grid_constant__ ScoreParams sp, DevSeqs qs, DevSeqs ts,
                                            const FastTask * __restrict__ tasks, int ntasks, int R,
                                            uint8_t const * __restrict__ dir, int32_t * __restrict__ stats)
{
  int const id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= 2 * ntasks) { return; }
  FastTask const tk = tasks[id >> 1];
  int const half = id & 1;
  int const out = half ? tk.out_hi : tk.out_lo;
  if (out < 0) { return; }
  PairDesc pd;
  pd.q = tk.q; pd.t = half ? tk.thi : tk.tlo; pd.dir_off = tk.dir_off; pd.kind = 0; pd.out = out;
  pd.R = R; pd.half = half; pd.dmax = tk.dmax; pd.cigar_off = 0;
  traceback_one<false>(sp, qs, ts, pd, dir, nullptr, stats);
}

__global__ void traceback_exact_tasks_kernel(const __grid_constant__ ScoreParams sp, DevSeqs qs, DevSeqs ts,
                                             const ExactTask * __restrict__ tasks, int ntasks,
                                             uint8_t const * __restrict__ dir, int32_t * __restrict__ stats)
{
  int const id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= ntasks) { return; }
  ExactTask const tk = tasks[id];
  PairDesc pd;
  pd.q = tk.q; pd.t = tk.t; pd.dir_off = tk.dir_off; pd.kind = 1; pd.out = tk.out;
  pd.R = 1; pd.half = 0; pd.dmax = 0; pd.cigar_off = 0;
  traceback_one<false>(sp, qs, ts, pd, dir, nullptr, stats);
}

// CIGAR texts sit right-aligned in their scratch regions; pack them densely (NUL-terminated)
__global__ void cigar_gather_kernel(const PairDesc * __restrict__ pairs, int npairs, DevSeqs qs,
                                    DevSeqs ts, const int32_t * __restrict__ stats,
                                    const int64_t * __restrict__ dense_off,
                                    const char * __restrict__ scratch, char * __restrict__ dense)
{
  int const p = blockIdx.x;
  if (p >= npairs) { return; }
  PairDesc const pd = pairs[p];
  int const len = stats[static_cast<size_t>(pd.out) * VSG_STAT_WORDS + VSG_STAT_CIGARLEN];
  char * const dst = dense + dense_off[p];
  if (len == 0) {
    if (threadIdx.x == 0) { dst[0] = 0; }
    return;
  }
  int const Q = qs.len[pd.q], D = ts.len[pd.t];
  char const * const src = scratch + pd.cigar_off + (Q + D) - len;
  for (int k = threadIdx.x; k <= len; k += blockDim.x) { dst[k] = src[k]; }
}

__global__ void cigar_len_kernel(const PairDesc * __restrict__ pairs, const int32_t * __restrict__ stats,
                                 int npairs, int64_t * __restrict__ lens)
{
  int const p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < npairs) {
    lens[p] = stats[static_cast<size_t>(pairs[p].out) * VSG_STAT_WORDS + VSG_STAT_CIGARLEN] + 1;
  }
}

// ASCII -> symbol byte (4-bit code | lower-case flag), per-sequence non-ACGTU flag
__device__ __forceinline__ int ascii_to_code(int c)
{
  int const u = (c >= 'a' && c <= 'z') ? c - 32 : c;
  switch (u) {
    case 'A': return 1; case 'C': return 2; case 'G': return 4; case 'T': case 'U': return 8;
    case 'M': return 3; case 'R': return 5; case 'S': return 6; case 'V': return 7;
    case 'W': return 9; case 'Y': return 10; case 'H': return 11; case 'K': return 12;
    case 'D': return 13; case 'B': return 14; case 'N': return 15;
    default: return 0;
  }
}

__global__ void encode_kernel(const char * __restrict__ ascii, uint8_t * __restrict__ sym, int64_t total)
{
  int64_t const i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < total) {
    int const c = static_cast<unsigned char>(ascii[i]);
    int const lower = (c >= 'a' && c <= 'z') ? 16 : 0;
    sym[i] = static_cast<uint8_t>(ascii_to_code(c) | lower);
  }
}

// the complement of one symbol (reference chrmap_complement, utils/maps.cpp:121-151): the complement of a 4-bit
// IUPAC code is its bit reversal; non-IUPAC bytes become 'N' (upper case); case is kept.
__device__ __forceinline__ uint8_t complement_sym(int s)
{
  int const c = s & 15;
  if (c == 0) { return 15; }
  return static_cast<uint8_t>(((c & 1) << 3) | ((c & 2) << 1) | ((c & 4) >> 1) | ((c & 8) >> 3) | (s & 16));
}

// reverse complement of sequences [q0, q0+n) of `src` into a compact set (reference
// utils/reverse_complement.cpp:71-84 + chrmap_complement)
__global__ void revcomp_kernel(DevSeqs src, int64_t q0, int64_t n, const int64_t * __restrict__ dst_off,
                               uint8_t * __restrict__ dst)
{
  int64_t const w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  int const lane = threadIdx.x & 31;
  if (w >= n) { return; }
  uint8_t const * p = src.sym + src.off[q0 + w];
  int const len = src.len[q0 + w];
  uint8_t * o = dst + dst_off[w];
  for (int i = lane; i < len; i += 32) { o[i] = complement_sym(p[len - 1 - i]); }
}

// the strand mirror of a whole set: sequence w of `src` goes to entry 2w of the output (as stored) and its reverse
// complement to entry 2w + 1, both at dst_off; one warp per sequence
__global__ void strand_pairs_kernel(DevSeqs src, const int64_t * __restrict__ dst_off, uint8_t * __restrict__ dst)
{
  int64_t const w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  int const lane = threadIdx.x & 31;
  if (w >= src.n) { return; }
  uint8_t const * p = src.sym + src.off[w];
  int const len = src.len[w];
  uint8_t * fwd = dst + dst_off[2 * w];
  uint8_t * rev = dst + dst_off[2 * w + 1];
  for (int i = lane; i < len; i += 32) {
    fwd[i] = p[i];
    rev[i] = complement_sym(p[len - 1 - i]);
  }
}

__global__ void nonacgt_kernel(DevSeqs s, uint8_t * __restrict__ flag)
{
  int64_t const w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  int const lane = threadIdx.x & 31;
  if (w >= s.n) { return; }
  uint8_t const * p = s.sym + s.off[w];
  int const n = s.len[w];
  int bad = 0;
  for (int i = lane; i < n; i += 32) {
    int const c = p[i] & 15;
    bad |= !(c == 1 || c == 2 || c == 4 || c == 8);
  }
  bad = __any_sync(0xffffffffu, bad);
  if (lane == 0) { flag[w] = static_cast<uint8_t>(bad); }
}

}  // namespace vsg
