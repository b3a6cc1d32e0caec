// Dense FP64 linear algebra of the gamma draw (update_gamma!, src/gibbs.jl:420-438), batched over chains:
//   G_c = X diag(S_c) X' + I          -> k_gram_syrk : FP64 tensor-core (DMMA m8n8k4) SYRK, ring of TMA tensor-map boxes + mbarriers
//   G_c = L_c L_c', w = L_c^-1 rhs    -> blocked left-looking Cholesky: k_augment / k_chol_update (DMMA) / k_potf2_inv /
//                                        k_trsm_dmma (DMMA) / k_small_tile; the forward solve rides along as a bordering row
//   a4  = L_c^-T w                    -> k_bwd_stream (the factor streamed once through a ring of TMA boxes); above
//                                        N = 8192 k_bwd_cluster (the same stream split over a cluster of 8 CTAs)
//   X v, X' a4 (all chains at once)   -> k_xmma (tall-skinny DMMA GEMM, deterministic split-K)
// tcgen05 has no FP64 kind, so the Blackwell tensor path for this contraction is the warp-level DMMA.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cuda.h>
#include "bnr_engine.cuh"
#include "bnr_kernels.h"

namespace bnr {

// ------------------------------------------------------------------------------------------------------------
// small PTX helpers
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
// -x by flipping the sign bit (an integer op: the FP64 pipe is what the DMMA loop is bound by)
__device__ __forceinline__ double neg_bits(double x) {
  return __longlong_as_double(__double_as_longlong(x) ^ (long long)0x8000000000000000ull);
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem));
}

// ------------------------------------------------------------------------------------------------------------
// mbarrier / bulk-copy (TMA engine) helpers
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 2-D tiled TMA load (SASS: UTMALDG): one request moves a whole (box_inner rows) x (16 k) operand tile; the box is
// 4 rows wider than the tile, which IS the shared-memory padding (row pitch == 4 mod 16 doubles: conflict-free fragments)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, int x, int y, unsigned long long* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(
                   smem_u32(smem_dst)), "l"((unsigned long long)tm), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}
// contiguous global -> shared copy by the TMA engine, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------------------------
// SYRK on FP64 tensor cores.
//   MODE 0:  C_c[i][j] = sum_k A[i][k] s_c[k] A[j][k] + (i==j)      A = X (shared by all chains), K = qp
//   MODE 1:  C_c[i][j] -= sum_{k < nk*16} L_c[i][k] L_c[j][k]        left-looking Cholesky update of block column J
//   MODE 2:  C_c[i][j]  = sum_{k < 128} C_c[i][k] Linv_c[j][k]       panel solve with the inverted diagonal block
// The operand is "k-major": element (row, k) at A[row + ld*k] (rows contiguous) - exactly how X (column-major
// n x q) and a column panel of the column-major G are stored, so a 128-row x 16-k tile is sixteen contiguous
// 1 KB rows = one box of a 2-D tensor map {rows, k}.  A dedicated producer warp loads one box per operand and stage
// into a 4-stage shared-memory ring (cp.async.bulk.tensor.2d, completion on "full" mbarriers); the 8 consumer warps
// never execute a block-wide barrier in the main loop - they wait on "full", issue DMMA m8n8k4, and release the
// stage on "empty".
// CTA tile 128 x 128, k-step 16.  The MMA "M" dimension runs along j (columns of C) and "N" along i (rows of C), so
// every accumulator pair is two consecutive rows of one column of the column-major C -> 16-byte stores.  Strictly
// lower tiles use a column-strip warp layout (syrk_strip_tile: 2 column fragments x all row fragments per warp),
// diagonal tiles compute only their lower triangle, balanced over the warps (syrk_diag_tile).  Shared rows are
// padded to 132 doubles (== 4 mod 16) which makes the (row, k) fragment loads bank-conflict free.
// The per-chain scale s_c[k] is applied to the operand with the fewest fragments per warp (2): DMUL shares the
// FP64 pipe with DMMA.  Work that cannot contribute is skipped: the symmetric half of diagonal tiles and row
// fragments that lie entirely in the zero padding beyond n.  The boxes are 132 rows wide (4 more than the tile):
// the box pitch is the padded row stride, at the price of 3 % more L2 traffic.
// NOTE the ring is written by the TMA engine behind the compiler's back: the consumer-side pointers into it must NOT
// be __restrict__ (with a compile-time trip count the compiler then reuses the fragments of a stage's previous
// occupant); the "memory" clobber of mbar_wait is what orders the fragment loads after the hand-shake.
// grid = (C, k-splits, tiles), block = 384 (2 consumer warpgroups + 1 producer warpgroup, registers re-balanced with
// setmaxnreg: 232 per consumer thread, 40 per producer thread); dynamic smem = SYRK_SMEM.
// ------------------------------------------------------------------------------------------------------------
constexpr int SY_BT = 128;        // tile edge
#ifndef BNR_SY_BK
#define BNR_SY_BK 16
#endif
#ifndef BNR_SY_STAGES
#define BNR_SY_STAGES 4
#endif
constexpr int SY_BK = BNR_SY_BK;  // k-step
constexpr int SY_LDS = 132;       // smem row stride in doubles (== 4 mod 16 -> conflict-free fragment loads)
constexpr int SY_STAGES = BNR_SY_STAGES;
constexpr int SYRK_MAX_SPLITS = 8;
constexpr int SY_STAGE_DBL = 2 * SY_BK * SY_LDS + SY_BK;   // two operand tiles + 16 scales
constexpr int SY_THREADS = 384;   // 2 consumer warpgroups + 1 producer warpgroup (one active lane)
constexpr int SY_PRODUCER_REGS = 40, SY_CONSUMER_REGS = 232;   // 128*40 + 256*232 = 64512 = 384*168
constexpr size_t SYRK_SMEM = (size_t)SY_STAGES * SY_STAGE_DBL * sizeof(double) + 2 * SY_STAGES * sizeof(unsigned long long);

// Diagonal tiles: only the lower triangle of the 128 x 128 tile is needed.  Seen as 16 x 16 fragments of 8 x 8,
// fragment column j holds 16 - j useful fragments; warp W takes columns W and 15 - W (17 fragments, the same for
// every warp), so the symmetric half is skipped AND the four SM sub-partitions stay evenly loaded.  W is a template
// parameter: every loop bound and register index is static, no predicated DMMA.
// acc[t], t < 16-W : fragment (row-fragment W+t, column-fragment W);  t >= 16-W : (row-fragment t-1, column 15-W).
template <int MODE, int W>
__device__ __forceinline__ void syrk_diag_frags(const double* sj, const double* ss, int k4,
                                                int lk, int lr, double (&a2)[2], double (&bfr)[16 - W]) {
  const int kr = k4 * 4 + lk;
  const double* row = sj + kr * SY_LDS + lr;
  // the scale rides on the two column-operand fragments (2 DMULs) rather than on the 16 - W row-operand fragments:
  // DMUL shares the FP64 pipe with DMMA, so every multiply saved is tensor throughput gained
  if (MODE == 0) {
    const double sk = ss[kr];
    a2[0] = row[W * 8] * sk;
    a2[1] = row[(15 - W) * 8] * sk;
  } else if (MODE == 1) {
    // C -= A A': the accumulators start from C (syrk_diag_tile) and the column operand enters negated
    a2[0] = neg_bits(row[W * 8]);
    a2[1] = neg_bits(row[(15 - W) * 8]);
  } else {
    a2[0] = row[W * 8];
    a2[1] = row[(15 - W) * 8];
  }
#pragma unroll
  for (int i = 0; i < 16 - W; ++i) bfr[i] = row[(W + i) * 8];
}

template <int MODE, int W>
__device__ __forceinline__ void syrk_diag_tile(const double* smem, unsigned long long* full,
                                               unsigned long long* empty, int nk, int lk, int lr, int lane,
                                               double* __restrict__ Cc, int np, int i0, double diag_add) {
  constexpr int NA = 16 - W;        // fragments of column W
  double acc[17][2];
  if (MODE == 1) {
    // MODE 1 updates C in place.  Its 17 fragments are loaded NOW, as independent 16-byte loads that overlap the
    // pipeline fill: the old load-subtract-store epilogue serialised them (a later load may alias an earlier store),
    // which cost ~25 us per CTA once G (512 MB) lives in HBM -- half of all stall samples of k_chol_update.
#pragma unroll
    for (int t = 0; t < 17; ++t) {
      const int jf = (t < NA) ? W : 15 - W;
      const int ifr = (t < NA) ? W + t : t - 1;
      const double2 v = *reinterpret_cast<const double2*>(Cc + (size_t)(i0 + jf * 8 + lr) * np + i0 + ifr * 8 + 2 * lk);
      acc[t][0] = v.x; acc[t][1] = v.y;
    }
  } else {
#pragma unroll
    for (int t = 0; t < 17; ++t) acc[t][0] = acc[t][1] = 0.0;
  }
  double a2[2][2], bfr[2][NA];
  mbar_wait(&full[0], 0);
  const double* sj = smem;
  syrk_diag_frags<MODE, W>(sj, sj + 2 * SY_BK * SY_LDS, 0, lk, lr, a2[0], bfr[0]);
  for (int kt = 0; kt < nk; ++kt) {
#pragma unroll
    for (int k4 = 0; k4 < SY_BK / 4; ++k4) {
      const int cur = k4 & 1, nxt = cur ^ 1;
      if (k4 + 1 < SY_BK / 4) {
        syrk_diag_frags<MODE, W>(sj, sj + 2 * SY_BK * SY_LDS, k4 + 1, lk, lr, a2[nxt], bfr[nxt]);
      } else if (kt + 1 < nk) {
        mbar_wait(&full[(kt + 1) % SY_STAGES], ((kt + 1) / SY_STAGES) & 1);
        const double* nj = smem + (size_t)((kt + 1) % SY_STAGES) * SY_STAGE_DBL;
        syrk_diag_frags<MODE, W>(nj, nj + 2 * SY_BK * SY_LDS, 0, lk, lr, a2[nxt], bfr[nxt]);
      }
#pragma unroll
      for (int t = 0; t < NA; ++t) dmma884(acc[t][0], acc[t][1], a2[cur][0], bfr[cur][t]);
#pragma unroll
      for (int t = NA; t < 17; ++t) dmma884(acc[t][0], acc[t][1], a2[cur][1], bfr[cur][t - 1 - W]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[kt % SY_STAGES]);
    sj = smem + (size_t)((kt + 1) % SY_STAGES) * SY_STAGE_DBL;
  }
#pragma unroll
  for (int t = 0; t < 17; ++t) {
    const int jf = (t < NA) ? W : 15 - W;
    const int ifr = (t < NA) ? W + t : t - 1;
    const int j = i0 + jf * 8 + lr;                   // diagonal tile: j0 == i0
    const int i = i0 + ifr * 8 + 2 * lk;
    double2* p = reinterpret_cast<double2*>(Cc + (size_t)j * np + i);
    double2 v;
    if (MODE == 0) {
      v.x = acc[t][0] + (i == j ? diag_add : 0.0);
      v.y = acc[t][1] + (i + 1 == j ? diag_add : 0.0);
    } else {
      v.x = acc[t][0];               // MODE 1: C - A A' accumulated in place
      v.y = acc[t][1];
    }
    *p = v;
  }
}

// Off-diagonal tiles, "column-strip" warp layout: warp w owns the two 8-column fragments 2w, 2w+1 of the tile
// (columns j0 + 16w .. j0 + 16w + 15 of C) and ALL NF 8-row fragments of the i operand, i.e. 2 x NF DMMAs per k4-step.
// Compared with a 64 x 32 warp tile this (a) halves the DMULs: the per-chain scale rides on the 2 column-operand
// fragments, (b) lets a tile of the last block row stop at the last fragment that holds a valid row (NF < 16):
// the zero padding of n up to a multiple of 128 costs no tensor work.
template <int MODE, int NF>
__device__ __forceinline__ void syrk_strip_frags(const double* sj, const double* si, const double* ss, int k4,
                                                 int f0, int f1, int lk, int lr, int ldi,
                                                 double (&af)[2], double (&bf)[NF]) {
  const int kr = k4 * 4 + lk;
  const double* rj = sj + kr * SY_LDS + lr;
  const double* ri = si + kr * ldi + lr;
  if (MODE == 0) {
    const double sk = ss[kr];
    af[0] = rj[f0 * 8] * sk;
    af[1] = rj[f1 * 8] * sk;
  } else if (MODE == 1) {
    af[0] = neg_bits(rj[f0 * 8]);    // C -= A_i A_j': accumulators start from C, the 2-fragment operand enters negated
    af[1] = neg_bits(rj[f1 * 8]);
  } else {
    af[0] = rj[f0 * 8];
    af[1] = rj[f1 * 8];
  }
#pragma unroll
  for (int nf = 0; nf < NF; ++nf) bf[nf] = ri[nf * 8];
}

// MODE 2 (panel solve, the j operand is the lower-triangular inverse of the diagonal block): output column j' only
// needs k <= j', so warp w takes the column fragments w and 15 - w (instead of 2w, 2w + 1) and stops feeding each of
// them once k passes its last column: 2w + 2 and 32 - 2w k4-steps -- 34 of 64 for every warp, balanced.
template <int MODE, int NF>
__device__ __forceinline__ void syrk_strip_tile(const double* smem, unsigned long long* full,
                                                unsigned long long* empty, int nk, int warp, int lk, int lr, int lane,
                                                double* __restrict__ Cc, int np, int i0, int j0, int ldi) {
  double acc[2][NF][2];
  const int f0 = (MODE == 2) ? warp : 2 * warp, f1 = (MODE == 2) ? 15 - warp : 2 * warp + 1;
  if (MODE == 1) {
    // in-place update: the tile's current values are the initial accumulators (see syrk_diag_tile)
#pragma unroll
    for (int mf = 0; mf < 2; ++mf) {
      const int j = j0 + (mf == 0 ? f0 : f1) * 8 + lr;
#pragma unroll
      for (int nf = 0; nf < NF; ++nf) {
        const double2 v = *reinterpret_cast<const double2*>(Cc + (size_t)j * np + i0 + nf * 8 + 2 * lk);
        acc[mf][nf][0] = v.x; acc[mf][nf][1] = v.y;
      }
    }
  } else {
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < NF; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
  }
  const int lim0 = 2 * f0 + 2, lim1 = 2 * f1 + 2;       // MODE 2: k4-steps that can still reach the fragment
  double af[2][2], bf[2][NF];
  mbar_wait(&full[0], 0);
  const double* sj = smem;
  syrk_strip_frags<MODE, NF>(sj, sj + SY_BK * SY_LDS, sj + 2 * SY_BK * SY_LDS, 0, f0, f1, lk, lr, ldi, af[0], bf[0]);
  for (int kt = 0; kt < nk; ++kt) {
#pragma unroll
    for (int k4 = 0; k4 < SY_BK / 4; ++k4) {
      const int cur = k4 & 1, nxt = cur ^ 1;
      if (k4 + 1 < SY_BK / 4) {
        syrk_strip_frags<MODE, NF>(sj, sj + SY_BK * SY_LDS, sj + 2 * SY_BK * SY_LDS, k4 + 1, f0, f1, lk, lr, ldi, af[nxt], bf[nxt]);
      } else if (kt + 1 < nk) {
        mbar_wait(&full[(kt + 1) % SY_STAGES], ((kt + 1) / SY_STAGES) & 1);
        const double* nj = smem + (size_t)((kt + 1) % SY_STAGES) * SY_STAGE_DBL;
        syrk_strip_frags<MODE, NF>(nj, nj + SY_BK * SY_LDS, nj + 2 * SY_BK * SY_LDS, 0, f0, f1, lk, lr, ldi, af[nxt], bf[nxt]);
      }
      if (MODE == 2) {
        const int k4g = kt * (SY_BK / 4) + k4;
        if (k4g < lim0) {
#pragma unroll
          for (int nf = 0; nf < NF; ++nf) dmma884(acc[0][nf][0], acc[0][nf][1], af[cur][0], bf[cur][nf]);
        }
        if (k4g < lim1) {
#pragma unroll
          for (int nf = 0; nf < NF; ++nf) dmma884(acc[1][nf][0], acc[1][nf][1], af[cur][1], bf[cur][nf]);
        }
      } else {
#pragma unroll
        for (int nf = 0; nf < NF; ++nf) {
          dmma884(acc[0][nf][0], acc[0][nf][1], af[cur][0], bf[cur][nf]);
          dmma884(acc[1][nf][0], acc[1][nf][1], af[cur][1], bf[cur][nf]);
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[kt % SY_STAGES]);
    sj = smem + (size_t)((kt + 1) % SY_STAGES) * SY_STAGE_DBL;
  }
#pragma unroll
  for (int mf = 0; mf < 2; ++mf) {
    const int j = j0 + (mf == 0 ? f0 : f1) * 8 + lr;
#pragma unroll
    for (int nf = 0; nf < NF; ++nf) {
      const int i = i0 + nf * 8 + 2 * lk;
      double2* p = reinterpret_cast<double2*>(Cc + (size_t)j * np + i);
      double2 v;
      v.x = acc[mf][nf][0];          // MODE 1: C - A_i A_j' accumulated in place
      v.y = acc[mf][nf][1];
      *p = v;
    }
  }
}

// Operands arrive as tensor-map boxes: the j operand through tmj at (row jx, k-row jy0 + 16 kt), the i operand through
// tmi at (row i0, k-row iy0 + 16 kt); jy0 / iy0 carry the chain, the first contributing column and the k-split offset.
template <int MODE>
__device__ __forceinline__ void
syrk_body(const CUtensorMap* tmj, const CUtensorMap* tmi, int jy0, int iy0, const double* __restrict__ scale,
          size_t scale_stride, double* __restrict__ Cm, size_t c_chain_stride, int np, int nvalid, int nk, int origin,
          double diag_add, int part = 0, int nstrip = 1, int tile_index = 0) {
  extern __shared__ __align__(128) double smem[];
  unsigned long long* full = reinterpret_cast<unsigned long long*>(smem + (size_t)SY_STAGES * SY_STAGE_DBL);
  unsigned long long* empty = full + SY_STAGES;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.x;          // chains vary fastest: the 64 CTAs that share one X tile run back to back (L2 reuse)
  int ib, jb;
  if (MODE == 0) {
    // tile_index enumerates the lower-triangular tiles by decreasing cost, so that the tail of the grid is made of
    // cheap CTAs: the strictly-lower (full-cost) tiles, the diagonal (half-cost) ones, and last the strictly-lower
    // tiles of a SHORT last row block (<= 32 valid rows: a quarter of the DMMAs)
    const int T = np / SY_BT;
    const bool short_last = T > 1 && nvalid - (T - 1) * SY_BT <= 32;
    const int noff = short_last ? (T - 1) * (T - 2) / 2 : T * (T - 1) / 2;
#ifdef SYRK_LAB_ONLY_DIAG
    const int t = tile_index + noff;
#else
    const int t = tile_index;
#endif
    if (t < noff) {
      ib = (int)((1.0 + sqrt(1.0 + 8.0 * t)) * 0.5);
      while (ib * (ib - 1) / 2 > t) --ib;
      while ((ib + 1) * ib / 2 <= t) ++ib;
      jb = t - ib * (ib - 1) / 2;
    } else if (t < noff + T) {
      ib = jb = t - noff;
    } else {
      ib = T - 1;
      jb = t - noff - T;
    }
  } else {
    // MODE 1 (Cholesky update of block column jb = origin) and MODE 2 (panel solve of block column jb): the CTAs of a
    // launch cover the row blocks part, part + 1, ... of that column (part >= jb; part == jb includes the diagonal tile)
    // When the launch has too few tiles to occupy the GPU (few chains: the latency-bound regime) every tile is cut
    // into nstrip (2 or 4) row strips of 128 / nstrip rows, one CTA each: the same fragments in the same k order
    // (bit-identical results), a quarter of the DMMA chain per CTA.  A diagonal tile is then computed like any other
    // (its upper triangle is written too; nobody reads it).
    jb = origin;
    ib = part + tile_index / nstrip;
  }
  const int strip = (MODE == 0) ? 0 : tile_index % nstrip;
  const int rows_i = SY_BT / nstrip;
  const int i0 = ib * SY_BT + strip * rows_i, j0 = jb * SY_BT;
  const bool diag = (ib == jb) && nstrip == 1;
  const double* sc = (MODE == 0) ? scale + (size_t)c * scale_stride : nullptr;
  // operand sources (k-major: element (row, k) at base[row + ld * k]).  MODE 0 / 1: both operands are row blocks of
  // the same matrix.  MODE 2: the i operand is block column J of C itself (rows i0.., k = the 128 columns of the
  // panel), the j operand is the 128 x 128 inverse of the diagonal block (ld = 128, rows 0..127).
  const int jx = (MODE == 2) ? 0 : j0;
  const int ldi = (MODE == 0) ? SY_LDS : rows_i + 4;   // row pitch of the i operand in shared memory = its box width

  if (tid == 0) {
    for (int s = 0; s < SY_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();

  if (warp >= 8) {
    // ---------------- producer warpgroup: hands its registers to the consumers, one lane drives the TMA engine ----
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(SY_PRODUCER_REGS));
    if (warp == 8 && lane == 0) {
      // three requests per stage (two operand boxes + the 16 scales); the first version issued one 1 KB bulk copy per
      // k-row and operand -- 33 requests, ~1 us per stage at the TMA engine's ~30 ns per request, which bounded every
      // tile with less than ~1 us of DMMA work per stage (row strips, tiles of a short last row block)
      const unsigned bytes = SY_BK * SY_LDS * 8u + (diag ? 0u : SY_BK * (unsigned)ldi * 8u) + (MODE == 0 ? SY_BK * 8u : 0u);
      for (int kt = 0; kt < nk; ++kt) {
        const int stage = kt % SY_STAGES;
        const unsigned ph = (kt / SY_STAGES) & 1;
        mbar_wait(&empty[stage], ph ^ 1);
        double* sj = smem + (size_t)stage * SY_STAGE_DBL;
        double* si = sj + SY_BK * SY_LDS;
        mbar_expect_tx(&full[stage], bytes);
        tma_load_2d(sj, tmj, jx, jy0 + kt * SY_BK, &full[stage]);
        if (!diag) tma_load_2d(si, tmi, i0, iy0 + kt * SY_BK, &full[stage]);
        if (MODE == 0) bulk_g2s(si + SY_BK * SY_LDS, sc + kt * SY_BK, SY_BK * 8, &full[stage]);
      }
    }
    return;
  }

  // ---------------- consumers ----------------
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(SY_CONSUMER_REGS));
  const int lk = lane & 3, lr = lane >> 2;
  double* Cc = Cm + (size_t)c * c_chain_stride;

  if (diag) {
    switch (warp) {
      case 0: syrk_diag_tile<MODE, 0>(smem, full, empty, nk, lk, lr, lane, Cc, np, i0, diag_add); break;
      case 1: syrk_diag_tile<MODE, 1>(smem, full, empty, nk, lk, lr, lane, Cc, np, i0, diag_add); break;
      case 2: syrk_diag_tile<MODE, 2>(smem, full, empty, nk, lk, lr, lane, Cc, np, i0, diag_add); break;
      case 3: syrk_diag_tile<MODE, 3>(smem, full, empty, nk, lk, lr, lane, Cc, np, i0, diag_add); break;
      case 4: syrk_diag_tile<MODE, 4>(smem, full, empty, nk, lk, lr, lane, Cc, np, i0, diag_add); break;
      case 5: syrk_diag_tile<MODE, 5>(smem, full, empty, nk, lk, lr, lane, Cc, np, i0, diag_add); break;
      case 6: syrk_diag_tile<MODE, 6>(smem, full, empty, nk, lk, lr, lane, Cc, np, i0, diag_add); break;
      default: syrk_diag_tile<MODE, 7>(smem, full, empty, nk, lk, lr, lane, Cc, np, i0, diag_add); break;
    }
    return;
  }

  // strictly-lower tile: only the 8-row fragments of the i operand that hold a valid row are computed and stored.
  // Rows >= nvalid are zero padding: their entries of C are exactly zero, were zero-initialised at allocation and
  // are never written by any kernel, so skipping them changes nothing.
  int nfv = (nvalid - i0 + 7) / 8;
  nfv = nfv > rows_i / 8 ? rows_i / 8 : nfv;
  if (nfv <= 0) {
    // the whole row block is padding: keep the stage hand-shake alive and leave
    for (int kt = 0; kt < nk; ++kt) {
      mbar_wait(&full[kt % SY_STAGES], (kt / SY_STAGES) & 1);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[kt % SY_STAGES]);
    }
    return;
  }
  // (at least 4 row fragments: fewer template instances; the extra fragments are zero-padding rows of the last block)
  if (nfv < 4) nfv = 4;
  switch (nfv) {
#define BNR_STRIP_CASE(NF) case NF: syrk_strip_tile<MODE, NF>(smem, full, empty, nk, warp, lk, lr, lane, Cc, np, i0, j0, ldi); break;
    BNR_STRIP_CASE(4) BNR_STRIP_CASE(5) BNR_STRIP_CASE(6)
    BNR_STRIP_CASE(7) BNR_STRIP_CASE(8) BNR_STRIP_CASE(9) BNR_STRIP_CASE(10) BNR_STRIP_CASE(11) BNR_STRIP_CASE(12)
    BNR_STRIP_CASE(13) BNR_STRIP_CASE(14) BNR_STRIP_CASE(15)
#undef BNR_STRIP_CASE
    default: syrk_strip_tile<MODE, 16>(smem, full, empty, nk, warp, lk, lr, lane, Cc, np, i0, j0, ldi); break;
  }
}

// gridDim.z > 1 splits the contraction: split z handles k-steps [z * nk_split, ...) and writes its partial tile to
// ws[c][z - 1] (split 0 writes G itself, identity included); k_syrk_splitk_reduce adds them in a fixed order.  Used
// when chains x tiles cannot fill the SMs (few chains, large q: BASELINE config 4).
__global__ void __launch_bounds__(SY_THREADS, 1)
k_gram_syrk(const __grid_constant__ CUtensorMap tmX, const double* __restrict__ scale, size_t scale_stride,
            double* __restrict__ G, size_t g_chain_stride, int np, int nvalid, int nk, double diag_add,
            int nk_split, double* __restrict__ ws, int ws_cap) {
  // grid = (chains, k-splits, tiles): the hardware hands out CTAs x-fastest, z-slowest, so all splits of the expensive
  // tiles start before any cheap tile (with the split as the slowest index the last split's full-cost tiles started
  // last and the grid ended in a ~340 us tail of a few busy SMs)
  const int z = blockIdx.y, t = blockIdx.z;
  if (z == 0) {
    syrk_body<0>(&tmX, &tmX, 0, 0, scale, scale_stride, G, g_chain_stride, np, nvalid, nk < nk_split ? nk : nk_split, 0, diag_add,
                 0, 1, t);
  } else {
    const int kt0 = z * nk_split;
    const int nkl = (nk - kt0) < nk_split ? (nk - kt0) : nk_split;
    syrk_body<0>(&tmX, &tmX, kt0 * SY_BK, kt0 * SY_BK, scale + (size_t)kt0 * SY_BK, scale_stride,
                 ws + (size_t)(z - 1) * g_chain_stride, (size_t)ws_cap * g_chain_stride, np, nvalid, nkl, 0, 0.0, 0, 1, t);
  }
}

// G_c (lower tiles) += sum_z ws[c][z] (fixed order).  grid = (lower tiles * 8, C), block = 256: 2048 entries per block
__global__ void __launch_bounds__(256) k_syrk_splitk_reduce(double* __restrict__ G, size_t g_chain_stride, int np,
                                                            const double* __restrict__ ws, int ws_cap, int nz) {
  const int c = blockIdx.y, piece = blockIdx.x & 7;
  int t = blockIdx.x >> 3, ib = 0;
  while ((ib + 1) * (ib + 2) / 2 <= t) ++ib;
  const int jb = t - ib * (ib + 1) / 2;
  double* Gc = G + (size_t)c * g_chain_stride;
  const double* wc = ws + (size_t)c * ws_cap * g_chain_stride;
  for (int id = piece * 2048 + threadIdx.x; id < (piece + 1) * 2048; id += 256) {
    const int i = ib * SY_BT + (id & (SY_BT - 1)), j = jb * SY_BT + (id >> 7);
    const size_t o = (size_t)j * np + i;
    double v = Gc[o];
    for (int z = 0; z < nz; ++z) v += wc[(size_t)z * g_chain_stride + o];
    Gc[o] = v;
  }
}

// G[ib, jb] -= sum_k P[ib, k] P[jb, k]' for the row blocks ib = ib_first, ib_first + 1, ... (grid.y of them) of block
// column jb; P points at the first of the nk * 16 columns of the factor that contribute (the caller offsets it), so a
// launch applies any contiguous range of panels.
// (tmJ: the chain-stacked matrix {rows, columns x chains} with 132-row boxes; tmI: the same with boxes as wide as a row
//  strip + 4; kcol0: first contributing column)
__global__ void __launch_bounds__(SY_THREADS, 1)
k_chol_update(const __grid_constant__ CUtensorMap tmJ, const __grid_constant__ CUtensorMap tmI, int kcol0,
              double* __restrict__ G, size_t chain_stride, int np, int nvalid, int nk, int jb, int ib_first, int nstrip) {
  const int y0 = (int)blockIdx.x * np + kcol0;
  syrk_body<1>(&tmJ, &tmI, y0, y0, nullptr, 0, G, chain_stride, np, nvalid, nk, jb, 0.0, ib_first, nstrip, (int)blockIdx.y);
}

// panel solve on the tensor cores: G[I, J] <- G[I, J] Linv_J' for the row blocks I = ib_first, ... (in place: a CTA
// has consumed its whole tile through the ring before the first store).  tmL: the stacked inverses {128, 128 x panels x
// chains}; tmI as above.
__global__ void __launch_bounds__(SY_THREADS, 1)
k_trsm_dmma(const __grid_constant__ CUtensorMap tmL, const __grid_constant__ CUtensorMap tmI, double* __restrict__ G,
            size_t chain_stride, int np, int nvalid, int jb, int ib_first, int nstrip) {
  const int T = np / SY_BT;
  syrk_body<2>(&tmL, &tmI, ((int)blockIdx.x * T + jb) * SY_BT, (int)blockIdx.x * np + jb * SY_BT, nullptr, 0, G, chain_stride,
               np, nvalid, SY_BT / SY_BK, jb, 0.0, ib_first, nstrip, (int)blockIdx.y);
}

// ------------------------------------------------------------------------------------------------------------
// Blocked left-looking Cholesky, block size 128, of every chain's gdim x gdim matrix, with BOTH triangular solves
// organised around it:
//   * forward solve for free: the right-hand side r (scaled by a power of two to |r| ~ 1) is stored as row m (the first
//     padding row, m = n or q) of the matrix itself, with the diagonal entry d = 1 + |r|^2 / lmin (k_augment;
//     lmin <= lambda_min(G)).  The bordered
//     matrix [[G, r], [r', d]] is positive definite (r' G^-1 r <= |r|^2 / lambda_min < d), and row m of its Cholesky
//     factor IS w' = (L^-1 r)': the DMMA update / panel-solve kernels below carry the solve along as one more row of
//     the last row block.  (The corner entry sqrt(d - |w|^2) is never used.)
//   * for J = 0 .. T-1:
//       k_chol_update (DMMA): G[J.., J] -= L[J.., 0:J] L[J, 0:J]'
//       k_potf2_inv   one CTA per chain: the 128 x 128 diagonal block is factored in shared memory in 32-wide steps,
//                     software-pipelined around the pivot chain (one warp factors 32 x 32 in registers and publishes
//                     its columns; the rows below, the diagonal-block inverses, the trailing updates, the bordered
//                     inverse and the stores all run next to it, see the kernel) -> factor in place, Linv[c][J]
//       k_trsm_dmma   (DMMA): G[I, J] <- G[I, J] Linv_J' for I > J -- the panel solve is a GEMM
//   * backward solve L' x = w (+ z): k_bwd_stream, one CTA per chain streams the factor once (tensor-map boxes of
//     128 rows x 32 columns into a shared-memory ring), every step is a block mat-vec; the diagonal blocks use Linv.
//     Above BWD_STREAM_MAX_DIM k_bwd_cluster spreads the same solve over a cluster of BWC_K CTAs per chain.
// Index bound: N <= CHOL_MAX_DIM = 2^15, so N^2 = 2^30 and every in-matrix offset j * N + i fits an int; the kernels form
// them in size_t anyway.  A tensor-map coordinate c * N + k (chain c) is an int: it needs C * N < 2^31, far above any
// chain count whose factors fit in device memory (8.6 GB per chain at N = 32768).
// ------------------------------------------------------------------------------------------------------------
constexpr int PB = 128;            // panel / diagonal block size
constexpr int CHOL_MAX_DIM = 32768;        // largest factored dimension: N^2 fits an int, every grid fits its bound
constexpr int BWD_STREAM_MAX_DIM = 8192;   // the one-CTA back solve keeps all of x in shared memory

__device__ __forceinline__ void bulk_s2g(void* gdst, const void* ssrc, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// row m of every G_c <- (r_c, 1 + |r_c|^2 / lmin_c), lmin_c a lower bound of the smallest eigenvalue of G_c, so that
// the bordered matrix stays positive definite (r' G^-1 r <= |r|^2 / lambda_min):  n-form G = X D X' + I: lmin = 1;
// q-form P = (X'X + D^-1)/tau2: lmin = 1 / (tau2 max_j S_j)  (S, tau2 given).  grid = C, block = 256.
// The row holds r_c 2^-e with |r_c 2^-e| in [1/2, 1): the last pivot, 1 + |r|^2 / lmin - r' G^-1 r, is a difference of
// two terms of size |r|^2, and unscaled its rounding (eps |r|^2) made it negative from |r| ~ 1e8 on when r is nearly
// orthogonal to the range of X.  The row's arithmetic is linear in r, so the power-of-two scale is exact: k_bwd_stream
// multiplies w by 2^e, which k_augment leaves in r_c[m] (the first padding entry of the right-hand side).
__global__ void __launch_bounds__(256) k_augment(double* __restrict__ G, size_t chain_stride, int N, int m,
                                                 double* __restrict__ r, int r_stride,
                                                 const double* __restrict__ S, const double* __restrict__ tau2) {
  __shared__ double red[8], redm[8], scale;
  const int c = blockIdx.x, tid = threadIdx.x;
  double* Gc = G + (size_t)c * chain_stride;
  double* rc = r + (size_t)c * r_stride;
  double s = 0.0, mx = 0.0;
  for (int k = tid; k < m; k += 256) {
    const double v = rc[k];
    s += v * v;
    if (S) mx = fmax(mx, S[(size_t)c * r_stride + k]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((tid & 31) == 0) { red[tid >> 5] = s; redm[tid >> 5] = mx; }
  __syncthreads();
  if (tid == 0) {
    double t = 0.0, mm = 0.0;
    for (int w = 0; w < 8; ++w) { t += red[w]; mm = fmax(mm, redm[w]); }
    int e = 0;
    frexp(sqrt(t), &e);
    const double sc = ldexp(1.0, -e);
    const double inv_lmin = S ? tau2[c] * mm : 1.0;
    Gc[(size_t)m * N + m] = 1.0 + t * sc * sc * inv_lmin;
    rc[m] = ldexp(1.0, e);
    scale = sc;
  }
  __syncthreads();
  const double sc = scale;
  for (int k = tid; k < m; k += 256) Gc[(size_t)k * N + m] = rc[k] * sc;
}

// ---- warp-level 32 x 32 x 32 products on the FP64 tensor cores, operands column-major in shared memory ----
// One 8 x 8 output fragment of C = A B (A, B 32 x 32, leading dimensions lda / ldb == 4 mod 16 doubles -> conflict-free):
// the MMA runs on the transposed problem (M along the columns n of C, N along its rows m), so that the accumulator pair
// of a lane is rows m0 + 2 lk, + 1 of column n0 + lr -> one 16-byte store.   acc += A[m0.., :] B[:, n0..]
__device__ __forceinline__ void frag_mm32(double& c0, double& c1, const double* Aop, int lda, const double* Bop, int ldb,
                                          int m0, int n0, int lk, int lr) {
#pragma unroll
  for (int k4 = 0; k4 < 8; ++k4) {
    const int k = k4 * 4 + lk;
    const double bt = Bop[(n0 + lr) * ldb + k];       // "A" operand of the transposed problem: B'[n][k]
    const double at = Aop[k * lda + m0 + lr];         // "B" operand: A'[k][m]
    dmma884(c0, c1, bt, at);
  }
}

// NF independent fragments at once, k outermost: the NF accumulator chains interleave, so the warp is bound by the DMMA
// issue rate instead of the latency of one dependent chain (8 DMMAs back to back)
template <int NF>
__device__ __forceinline__ void frag_mm32_batch(double (&c)[NF][2], const double* const (&Aop)[NF], const int (&lda)[NF],
                                                const double* const (&Bop)[NF], const int (&ldb)[NF],
                                                const int (&m0)[NF], const int (&n0)[NF], int lk, int lr) {
#pragma unroll
  for (int k4 = 0; k4 < 8; ++k4) {
    const int k = k4 * 4 + lk;
#pragma unroll
    for (int i = 0; i < NF; ++i) {
      const double bt = Bop[i][(n0[i] + lr) * ldb[i] + k];
      const double at = Aop[i][k * lda[i] + m0[i] + lr];
      dmma884(c[i][0], c[i][1], bt, at);
    }
  }
}

constexpr int PLD = 132;           // column stride of the 128 x 128 working block (== 4 mod 16: conflict-free fragments)
constexpr int XD_LD = 36;          // column stride of the 32 x 32 scratch blocks (== 4 mod 16)
constexpr int XD_BLK = 32 * XD_LD;
// Optional in-kernel time stamps (lab builds only, -DBNR_POTF2_STAMPS): thread 0 of chain 0 records globaltimer at the
// phase boundaries of k_potf2_inv into bnr::g_potf2_stamps.
#ifdef BNR_POTF2_STAMPS
__device__ unsigned long long g_potf2_stamps[64];
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;\n" : "=l"(t));
  return t;
}
#define STAMP(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_potf2_stamps[i] = gtimer(); } while (0)
#else
#define STAMP(i) do { } while (0)
#endif

constexpr size_t POTF2_SMEM = sizeof(double) * ((size_t)PB * PLD + 8 * XD_BLK + PB) + 8 * (4 + PB);
#ifndef BNR_POTF2_PUBLISH
#define BNR_POTF2_PUBLISH 8
#endif
// the pivot warp publishes its columns in groups of this many: one release-arrive per column cost it ~0.25 us per 32
// columns more than one per 8 (measured: pivot block 4.2-4.9 / 4.0-4.1 / 3.9 us with 1 / 4 / 8)
constexpr int POTF2_PUBLISH = BNR_POTF2_PUBLISH;
constexpr int PU_ROWS = 32;        // k-rows of L(J, J-1) per staged chunk of the in-kernel diagonal update
static_assert(2 * PU_ROWS * PLD <= 8 * XD_BLK, "the update ring aliases the inverse scratch");

// One 32-k-row chunk of the diagonal-block update Delta += Lp Lp' (lower triangle by 8 x 8 fragments): warp W owns the
// fragment columns W and 15 - W (17 fragments, the same count for every warp) exactly like syrk_diag_tile.
template <int W>
__device__ __forceinline__ void potf2_update_chunk(const double* buf, int lk, int lr, double (&acc)[17][2]) {
  constexpr int NA = 16 - W;
#pragma unroll
  for (int k4 = 0; k4 < PU_ROWS / 4; ++k4) {
    const double* row = buf + (k4 * 4 + lk) * PLD + lr;
    const double a0 = row[W * 8], a1 = row[(15 - W) * 8];
    double bfr[NA];
#pragma unroll
    for (int i = 0; i < NA; ++i) bfr[i] = row[(W + i) * 8];
#pragma unroll
    for (int t = 0; t < NA; ++t) dmma884(acc[t][0], acc[t][1], a0, bfr[t]);
#pragma unroll
    for (int t = NA; t < 17; ++t) dmma884(acc[t][0], acc[t][1], a1, bfr[t - 1 - W]);
  }
}

template <int W>
__device__ __forceinline__ void potf2_update_apply(double* A, int lk, int lr, const double (&acc)[17][2]) {
  constexpr int NA = 16 - W;
#pragma unroll
  for (int t = 0; t < 17; ++t) {
    const int jf = (t < NA) ? W : 15 - W;
    const int ifr = (t < NA) ? W + t : t - 1;
    double2* p = reinterpret_cast<double2*>(A + (jf * 8 + lr) * PLD + ifr * 8 + 2 * lk);
    double2 v = *p;
    v.x -= acc[t][0];
    v.y -= acc[t][1];
    *p = v;
  }
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}

// Four 8 x 8 output fragments (rows m0.., columns 0..31) of a 32^3 block product on the FP64 tensor cores, operands
// column-major in shared memory:  c += A[m0.., :] B.   KIND 1: A is lower triangular (k <= m: the k-steps beyond the
// fragment's rows are skipped), KIND 2: B is lower triangular (k >= n: fragment i starts at k = 8 i), KIND 0: full.
// The skipped products are exact zeros, so the result does not depend on KIND.
template <int KIND>
__device__ __forceinline__ void quad_term(double (&c)[4][2], const double* Aop, int lda, const double* Bop, int ldb,
                                          int m0, int lk, int lr) {
  const int k4hi = (KIND == 1) ? (m0 >> 2) + 2 : 8;
#pragma unroll
  for (int k4 = 0; k4 < 8; ++k4) {
    if (k4 < k4hi) {
      const int k = k4 * 4 + lk;
      const double at = Aop[k * lda + m0 + lr];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (KIND != 2 || k4 >= 2 * i) dmma884(c[i][0], c[i][1], Bop[(8 * i + lr) * ldb + k], at);
    }
  }
}
__device__ __forceinline__ void quad_store(double* dst, int ldd, int m0, double sign, const double (&c)[4][2], int lk, int lr) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
    *reinterpret_cast<double2*>(dst + (8 * i + lr) * ldd + m0 + 2 * lk) = make_double2(sign * c[i][0], sign * c[i][1]);
}

// Panel kernel of the blocked Cholesky, one CTA per chain:
//   (late update)  D = G[J, J] - L[J, J-1] L[J, J-1]'   when `late` (the contributions of the panels before J-1 were
//                  applied earlier by k_chol_update; L[J, J-1] streams through a two-buffer TMA ring into DMMA fragments)
//   (factor)       D = L_JJ L_JJ'                       in shared memory, 32-wide steps
//   (inverse)      Linv_J = L_JJ^-1                     in place, 32^3 DMMA block products
__global__ void __launch_bounds__(256) k_potf2_inv(double* __restrict__ G, size_t chain_stride, int N, int J,
                                                   double* __restrict__ Linv, int T, int* status, int late) {
  extern __shared__ __align__(16) double sm[];
  double* A = sm;                          // column-major 128 x 128 working block: A[col * PLD + row]
  double* Xd = sm + PB * PLD;              // [4] inverses of the 32 x 32 diagonal blocks, column stride XD_LD
  double* Tm = Xd + 4 * XD_BLK;            // [4] intermediate products of the inverse
  double* dall = Tm + 4 * XD_BLK;          // [128] reciprocal diagonal of L
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(dall + PB);   // [0] block load, [1..2] update ring
  unsigned long long* colbar = bar + 4;    // [128] "column j of L is published" (one phase each, one arrival)
  const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lk = lane & 3, lr = lane >> 2;
  double* Gc = G + (size_t)c * chain_stride;
  double* D = Gc + (size_t)J * PB * N + (size_t)J * PB;
  STAMP(0);
  if (tid < PB) mbar_init(&colbar[tid], 1);
  if (tid == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); mbar_init(&bar[2], 1); }
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  __syncthreads();
  // the 128 x 128 block: 16-byte LDGSTS copies by all threads (a 1 KB column = one coalesced request of 64 threads;
  // 128 one-kilobyte bulk copies took 4.4 us here -- the TMA engine accepts ~1 such request per 30 ns)
  {
    const int chunk = tid & 63, c0 = tid >> 6;
#pragma unroll 8
    for (int i = 0; i < PB / 4; ++i) {
      const int col = c0 + 4 * i;
      cp_async16(A + col * PLD + chunk * 2, D + (size_t)col * N + chunk * 2);
    }
    cp_async_commit();
  }
  if (late && J > 0) {
    // L[J, J-1]: rows J*128.., columns (J-1)*128..: element (row, k) at Lp[row + N * k]
    const double* Lp = Gc + (size_t)(J - 1) * PB * N + (size_t)J * PB;
    double* ring = Xd;
    auto issue = [&](int chunk) {            // by warp 1: lane l loads k-row chunk * 32 + l
      double* buf = ring + (chunk & 1) * PU_ROWS * PLD;
      if (lane == 0) mbar_expect_tx(&bar[1 + (chunk & 1)], PU_ROWS * PB * 8);
      __syncwarp();
      bulk_g2s(buf + lane * PLD, Lp + (size_t)(chunk * PU_ROWS + lane) * N, PB * 8, &bar[1 + (chunk & 1)]);
    };
    if (warp == 1) { issue(0); issue(1); }
    double acc[17][2];
#pragma unroll
    for (int t = 0; t < 17; ++t) acc[t][0] = acc[t][1] = 0.0;
    constexpr int NCH = PB / PU_ROWS;
    for (int chunk = 0; chunk < NCH; ++chunk) {
      mbar_wait(&bar[1 + (chunk & 1)], (chunk >> 1) & 1);
      const double* buf = ring + (chunk & 1) * PU_ROWS * PLD;
      switch (warp) {
        case 0: potf2_update_chunk<0>(buf, lk, lr, acc); break;
        case 1: potf2_update_chunk<1>(buf, lk, lr, acc); break;
        case 2: potf2_update_chunk<2>(buf, lk, lr, acc); break;
        case 3: potf2_update_chunk<3>(buf, lk, lr, acc); break;
        case 4: potf2_update_chunk<4>(buf, lk, lr, acc); break;
        case 5: potf2_update_chunk<5>(buf, lk, lr, acc); break;
        case 6: potf2_update_chunk<6>(buf, lk, lr, acc); break;
        default: potf2_update_chunk<7>(buf, lk, lr, acc); break;
      }
      if (chunk + 2 < NCH) {
        __syncthreads();                     // every warp is done with this buffer before the TMA engine refills it
        if (warp == 1) issue(chunk + 2);
      }
    }
    cp_async_wait<0>();
    __syncthreads();
    switch (warp) {
      case 0: potf2_update_apply<0>(A, lk, lr, acc); break;
      case 1: potf2_update_apply<1>(A, lk, lr, acc); break;
      case 2: potf2_update_apply<2>(A, lk, lr, acc); break;
      case 3: potf2_update_apply<3>(A, lk, lr, acc); break;
      case 4: potf2_update_apply<4>(A, lk, lr, acc); break;
      case 5: potf2_update_apply<5>(A, lk, lr, acc); break;
      case 6: potf2_update_apply<6>(A, lk, lr, acc); break;
      default: potf2_update_apply<7>(A, lk, lr, acc); break;
    }
    __syncthreads();
  } else {
    cp_async_wait<0>();
    __syncthreads();
  }
  STAMP(1);
  // ---- factor + inverse, software-pipelined over the four 32-wide steps ----
  // Only the 32 x 32 pivot chain (128 dependent rsqrt steps of ~110 ns) is serial; everything else hangs off it:
  //   warp 0        pivot warp: factors the 32 x 32 diagonal block of step s in registers and PUBLISHES every finished
  //                 column of L (written in place + one mbarrier arrival per column).
  //   warps 1-3     rows below the diagonal block, one thread per row, eliminating column j as soon as it is published
  //                 (right-looking: the only inputs of column step j are that column of L_ss and its reciprocal pivot), so
  //                 the rows are complete one column behind the pivot warp instead of a phase after it.
  //   warp 7        the same elimination on the 32 unit rows e_j: x = e_j L_ss^-T is column j of L_ss^-1 -> Xd[s].
  //   warp 4        (the pivot warp's scheduler partition: no FP64) stores finished block columns of L and rows of Linv.
  //   warps 5, 6    + the row warps that have run out of rows: the inverse, bordered by block rows, on the tensor cores:
  //                   Y(i,j) = sum_{j<=k<i} L(i,k) X(k,j),  X(i,j) = -Xd_i Y(i,j),  X(i,i) = Xd_i = L_ii^-1
  //                 -- every product except the last block row is ready before the pivot chain ends.
  // Between steps only the 10 fragments of the NEXT diagonal block are updated by everybody (Tdiag); the rest of the
  // trailing update runs under the next pivot block (the lock-step rows simply start late and catch up).
  auto blkA = [&](int i, int j) { return A + (32 * j) * PLD + 32 * i; };        // block (i, j) of the working matrix
  auto trail = [&](int s, int f0, int f1, int slot, int nslots) {
    // A[r][cc] -= sum_p L[r][o+p] L[cc][o+p] for the 8 x 8 fragments f0 <= f < f1 of the lower triangle below step s
    // (fragment f = fr (fr + 1) / 2 + fc, fc <= fr; diagonal fragments are computed whole: what lands above the
    // diagonal is never read).  f < 10 is the next diagonal block.
    const int o = s * 32, base = o + 32;
    const double* P = A + o * PLD + base;             // panel: P[p * PLD + i] = L[base + i][o + p]
    for (int f = f0 + slot; f < f1; f += nslots) {
      int fr = 0;
      while ((fr + 1) * (fr + 2) / 2 <= f) ++fr;
      const int fc = f - fr * (fr + 1) / 2;
      double c0 = 0.0, c1 = 0.0;
#pragma unroll
      for (int k4 = 0; k4 < 8; ++k4) {
        const int k = k4 * 4 + lk;
        dmma884(c0, c1, P[k * PLD + fc * 8 + lr], P[k * PLD + fr * 8 + lr]);     // M along the column index cc
      }
      double2* dst = reinterpret_cast<double2*>(A + (base + fc * 8 + lr) * PLD + base + fr * 8 + 2 * lk);
      double2 v = *dst;
      v.x -= c0; v.y -= c1;
      *dst = v;
    }
  };
  bool bad = false;
  for (int s = 0; s < PB / 32; ++s) {
    const int o = s * 32;
    if (warp == 0) {
      // 32 x 32 Cholesky in registers: lane r holds row o+r (columns o .. o+31); entries above the diagonal are
      // whatever the block held there and never reach a valid entry.  Column j is broadcast through its final place in
      // shared memory, and the next pivot is updated and fetched FIRST so its rsqrt chain runs under the remaining
      // updates of column j.
      double a[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) a[j] = A[(o + j) * PLD + o + lane];
      double djj = __shfl_sync(0xffffffffu, a[0], 0);
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        if (!(djj > 0.0)) bad = true;
        const double inv = rsqrt(djj);
        const double lj = (lane == j) ? djj * inv : a[j] * inv;
        double* lc = A + (o + j) * PLD + o;
        if (lane >= j) lc[lane] = lj;
        if (lane == j) dall[o + j] = inv;
        if (j + 1 < 32) {
          // next pivot first, without the round trip through shared memory: for the lane that owns row j + 1 the
          // multiplier lc[j + 1] is its own lj (bit-identical to the generic update below)
          if (lane == j + 1) a[j + 1] = fma(-lj, lj, a[j + 1]);
          djj = __shfl_sync(0xffffffffu, a[j + 1], j + 1);
        }
        __syncwarp();
        if ((j % POTF2_PUBLISH) == POTF2_PUBLISH - 1 && lane == 0)
          mbar_arrive(&colbar[o + j]);                // release: columns <= j and their reciprocal pivots are visible
        if (j + 1 < 32 && lane != j + 1) a[j + 1] = fma(-lj, lc[j + 1], a[j + 1]);
#pragma unroll
        for (int cc = j + 2; cc < 32; ++cc) a[cc] -= lj * lc[cc];
      }
      STAMP(2 + 3 * s);
    } else {
      if (s > 0) {
        trail(s - 1, 10, (PB - o) / 8 * ((PB - o) / 8 + 1) / 2, warp - 1, 7);    // the rest of the previous step's update
        named_bar_sync(1, 224);
      }
      const int nrow_warps = 3 - s;                   // warps 1 .. nrow_warps own the rows below this step's block
      if (warp == 7 || warp <= nrow_warps) {
        const bool inv_row = (warp == 7);
        double* row = A + o * PLD + o + 32 + (warp - 1) * 32 + lane;
        double x[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) x[j] = inv_row ? ((j == lane) ? 1.0 : 0.0) : row[j * PLD];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if ((j % POTF2_PUBLISH) == 0) mbar_wait(&colbar[o + j + POTF2_PUBLISH - 1], 0);
          const double xj = x[j] * dall[o + j];
          x[j] = xj;
#pragma unroll
          for (int k = j + 1; k < 32; ++k) x[k] -= xj * A[(o + j) * PLD + o + k];
        }
        if (inv_row) {
#pragma unroll
          for (int j = 0; j < 32; ++j) Xd[s * XD_BLK + lane * XD_LD + j] = (j >= lane) ? x[j] : 0.0;
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) row[j * PLD] = x[j];
        }
      } else if (warp == 4) {
        // finished pieces go to global memory through the TMA engine (one bulk store per lane and column): direct
        // stores from this warp clogged the memory pipe it shares with the pivot warp (the following diagonal-block
        // update took 5 us instead of 1)
        fence_async_smem();                           // the pieces were written through the generic proxy
        if (s > 0) {
          // block column s-1 of the factor is final (rows from its diagonal block down)
          const int ob = o - 32;
          bulk_s2g(D + (size_t)(ob + lane) * N + ob, A + (ob + lane) * PLD + ob, (unsigned)(PB - ob) * 8u);
        }
        if (s == 3) {
          // rows 0..63 of the inverse are final: X(0,0) = Xd0, X(1,0), X(1,1) = Xd1 (zeros above the diagonal of the
          // diagonal blocks come from Xd; the zero blocks above them are never written: the buffer is zeroed at creation)
          double* dst = Linv + ((size_t)c * T + J) * PB * PB;
          bulk_s2g(dst + (size_t)lane * PB, Xd + lane * XD_LD, 256u);
          bulk_s2g(dst + (size_t)lane * PB + 32, A + lane * PLD + 32, 256u);
          bulk_s2g(dst + (size_t)(32 + lane) * PB + 32, Xd + XD_BLK + lane * XD_LD, 256u);
        }
        bulk_commit();
        bulk_wait_read0();                            // the sources may be overwritten after this step's barrier
      } else if (s > 0) {
        // the inverse, one block row behind the factorisation.  Slots: warps 5, 6, then the idle row warps 3, 2, 1.
        const int slot = (warp >= 5) ? warp - 5 : 5 - warp, nslots = 2 + s;
        double* Tm0 = Tm; double* Tm1 = Tm + XD_BLK; double* Tm2 = Tm + 2 * XD_BLK; double* Tm3 = Tm + 3 * XD_BLK;
        const double* X0 = Xd; const double* X1 = Xd + XD_BLK; const double* X2 = Xd + 2 * XD_BLK;
        if (s == 1) {
          for (int q = slot; q < 4; q += nslots) {                               // Y(1,0) = L(1,0) Xd0
            double cq[4][2] = {};
            quad_term<2>(cq, blkA(1, 0), PLD, X0, XD_LD, 8 * q, lk, lr);
            quad_store(Tm0, XD_LD, 8 * q, 1.0, cq, lk, lr);
          }
        } else if (s == 2) {
          for (int q = slot; q < 8; q += nslots) {
            const int m0 = 8 * (q & 3);
            double cq[4][2] = {};
            if (q < 4) {                                                         // X(1,0) = -Xd1 Y(1,0)   (in place of L(1,0))
              quad_term<1>(cq, X1, XD_LD, Tm0, XD_LD, m0, lk, lr);
              quad_store(blkA(1, 0), PLD, m0, -1.0, cq, lk, lr);
            } else {                                                             // Y(2,1) = L(2,1) Xd1
              quad_term<2>(cq, blkA(2, 1), PLD, X1, XD_LD, m0, lk, lr);
              quad_store(Tm2, XD_LD, m0, 1.0, cq, lk, lr);
            }
          }
          named_bar_sync(2, 32 * nslots);
          for (int q = slot; q < 4; q += nslots) {                               // Y(2,0) = L(2,0) Xd0 + L(2,1) X(1,0)
            double cq[4][2] = {};
            quad_term<2>(cq, blkA(2, 0), PLD, X0, XD_LD, 8 * q, lk, lr);
            quad_term<0>(cq, blkA(2, 1), PLD, blkA(1, 0), PLD, 8 * q, lk, lr);
            quad_store(Tm1, XD_LD, 8 * q, 1.0, cq, lk, lr);
          }
        } else {
          for (int q = slot; q < 12; q += nslots) {
            const int m0 = 8 * (q & 3);
            double cq[4][2] = {};
            if (q < 8) {                                                         // X(2,j) = -Xd2 Y(2,j), j = 0, 1
              quad_term<1>(cq, X2, XD_LD, q < 4 ? Tm1 : Tm2, XD_LD, m0, lk, lr);
              quad_store(blkA(2, q >> 2), PLD, m0, -1.0, cq, lk, lr);
            } else {                                                             // Y(3,2) = L(3,2) Xd2
              quad_term<2>(cq, blkA(3, 2), PLD, X2, XD_LD, m0, lk, lr);
              quad_store(Tm3, XD_LD, m0, 1.0, cq, lk, lr);
            }
          }
          named_bar_sync(2, 32 * nslots);
          for (int q = slot; q < 8; q += nslots) {
            const int m0 = 8 * (q & 3);
            double cq[4][2] = {};
            if (q < 4) {                                                         // Y(3,0) = L(3,0) Xd0 + L(3,1) X(1,0) + L(3,2) X(2,0)
              quad_term<2>(cq, blkA(3, 0), PLD, X0, XD_LD, m0, lk, lr);
              quad_term<0>(cq, blkA(3, 1), PLD, blkA(1, 0), PLD, m0, lk, lr);
              quad_term<0>(cq, blkA(3, 2), PLD, blkA(2, 0), PLD, m0, lk, lr);
              quad_store(Tm0, XD_LD, m0, 1.0, cq, lk, lr);
            } else {                                                             // Y(3,1) = L(3,1) Xd1 + L(3,2) X(2,1)
              quad_term<2>(cq, blkA(3, 1), PLD, X1, XD_LD, m0, lk, lr);
              quad_term<0>(cq, blkA(3, 2), PLD, blkA(2, 1), PLD, m0, lk, lr);
              quad_store(Tm1, XD_LD, m0, 1.0, cq, lk, lr);
            }
          }
        }
      }
    }
    fence_async_smem();                               // what this step wrote will be read by warp 4's bulk stores
    __syncthreads();                                  // step s: pivot block, rows below, Xd[s], side work all done
    STAMP(3 + 3 * s);
    if (s + 1 < PB / 32) {
      trail(s, 0, 10, warp, 8);                       // the next diagonal block
      __syncthreads();
    }
    STAMP(4 + 3 * s);
  }
  if (bad && lane == 0) atomicOr(&status[c], BNR_ST_G_NOTPD_);
  // ---- tail: the last block row of the inverse, X(3,j) = -Xd3 Y(3,j) (in place of L(3,j), which warp 4 has stored) ----
  for (int q = warp; q < 12; q += 8) {
    const int m0 = 8 * (q & 3), j = q >> 2;
    double cq[4][2] = {};
    quad_term<1>(cq, Xd + 3 * XD_BLK, XD_LD, Tm + (j == 2 ? 3 : j) * XD_BLK, XD_LD, m0, lk, lr);
    quad_store(blkA(3, j), PLD, m0, -1.0, cq, lk, lr);
  }
  {
    // the last diagonal block of the factor (32 x 32; rows 96..127 of columns 96..127)
    const int col = 96 + (tid >> 3), r = 96 + 4 * (tid & 7);
    *reinterpret_cast<double2*>(D + (size_t)col * N + r) = *reinterpret_cast<const double2*>(A + col * PLD + r);
    *reinterpret_cast<double2*>(D + (size_t)col * N + r + 2) = *reinterpret_cast<const double2*>(A + col * PLD + r + 2);
  }
  __syncthreads();
  STAMP(14);
  {
    // rows 64..127 of Linv_J: X(2,0..1), Xd2 | X(3,0..2), Xd3; the zero blocks above the diagonal are never written
    double* dst = Linv + ((size_t)c * T + J) * PB * PB;
    const int r = 64 + 2 * (tid & 31), c0 = tid >> 5;
#pragma unroll 4
    for (int i = 0; i < PB / 8; ++i) {
      const int cc = c0 + 8 * i;
      if ((cc >> 5) > (r >> 5)) continue;
      const double* src = ((r >> 5) == (cc >> 5)) ? Xd + (r >> 5) * XD_BLK + (cc & 31) * XD_LD + (r & 31) : A + cc * PLD + r;
      *reinterpret_cast<double2*>(dst + (size_t)cc * PB + r) = *reinterpret_cast<const double2*>(src);
    }
  }
  if (warp == 4) bulk_wait0();                        // this warp's bulk stores have landed
  STAMP(15);
  STAMP(16);
  STAMP(17);
}

// ------------------------------------------------------------------------------------------------------------
// Depth-128 tile kernels of the latency schedule, operands resident in shared memory.
//   MODE 2  panel solve     C[strip] = G[strip, J] Linv_J'                  (T1 / T2 of launch_cholesky)
//   MODE 1  late update     C[strip] -= L[strip, J] L[J+1, J]'              (Ulate)
// One CTA per (chain, row strip of 32 or 64 rows).  The ring-fed kernels above spend ~8 us per tile on their eight
// pipeline stages (32 one-kilobyte TMA requests each, ~30 ns per request) around 2-4 us of DMMA work; here the two
// operands arrive as 16-byte cp.async copies of all 256 threads (1.5-2 us for 160-200 KB), one barrier, then the same
// fragments in the same k order as syrk_strip_tile (bit-identical results), and a direct store.
// grid = (C, tiles * nstrip), block = 256.
// ------------------------------------------------------------------------------------------------------------
constexpr size_t small_tile_smem(int rows_i) { return sizeof(double) * ((size_t)PB * SY_LDS + (size_t)PB * (rows_i + 4)); }

template <int MODE, int NF>
__global__ void __launch_bounds__(256) k_small_tile(double* __restrict__ G, size_t chain_stride, int N, int jb, int ib_first,
                                                    int nstrip, const double* __restrict__ Bj, size_t bj_chain_stride,
                                                    int ldj, int kcol0, int tri) {
  extern __shared__ __align__(16) double sm[];
  constexpr int ROWS = NF * 8, LDI = ROWS + 4;       // LDI == 4 mod 16: conflict-free fragment loads
  double* sJ = sm;                                   // [128 k][132]  j operand: sJ[k * SY_LDS + row]
  double* sI = sm + PB * SY_LDS;                     // [128 k][LDI]  i operand (this CTA's row strip)
  const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lk = lane & 3, lr = lane >> 2;
  const int ib = ib_first + (int)blockIdx.y / nstrip, strip = (int)blockIdx.y % nstrip;
  const int i0 = ib * PB + strip * ROWS;
  double* Gc = G + (size_t)c * chain_stride;
  // sources (k-major: element (row, k) at base[row + ld * k]); kcol0 = first column of the contributing panel
  const double* srcJ = Bj + (size_t)c * bj_chain_stride;
  const double* srcI = Gc + (size_t)kcol0 * N + i0;
  // Only the part of the j operand that can reach an output is loaded.  MODE 2: Linv_J is lower triangular (entry
  // (col, k) with k <= col): k-row k is needed from its own 8-column fragment on.  MODE 1 on the diagonal tile (tri):
  // only the lower triangle of the tile is ever read, so the strip needs the columns up to its own last row.
  const int jmax = (MODE == 1 && tri) ? (strip + 1) * ROWS : PB;       // columns of the tile this CTA touches
  {
    const int chunk = tid & 63, r0 = tid >> 6;       // j operand: 128 k-rows of 64 16-byte chunks
#pragma unroll 8
    for (int i = 0; i < PB / 4; ++i) {
      const int k = r0 + 4 * i;
      const bool need = (MODE == 2) ? (chunk >= 4 * (k >> 3)) : (2 * chunk < jmax);
      if (need) cp_async16(sJ + k * SY_LDS + chunk * 2, srcJ + (size_t)k * ldj + chunk * 2);
    }
    constexpr int CPR = ROWS / 2;                    // 16-byte chunks per k-row of the i operand
    for (int id = tid; id < PB * CPR; id += 256) {
      const int k = id / CPR, ch = id % CPR;
      cp_async16(sI + k * LDI + ch * 2, srcI + (size_t)k * N + ch * 2);
    }
    cp_async_commit();
  }
  const int f0 = (MODE == 2) ? warp : 2 * warp, f1 = (MODE == 2) ? 15 - warp : 2 * warp + 1;
  const int lim0 = 2 * f0 + 2, lim1 = 2 * f1 + 2;    // MODE 2: k4-steps that can still reach the column fragment
  const int j0 = jb * PB;
  double acc[2][NF][2];
  const bool on0 = f0 * 8 < jmax, on1 = f1 * 8 < jmax;   // column fragments inside the needed part (always, unless tri)
  if (MODE == 1) {                                   // in place: start from the tile's current values
#pragma unroll
    for (int mf = 0; mf < 2; ++mf) {
      const int j = j0 + (mf == 0 ? f0 : f1) * 8 + lr;
      if (mf == 0 ? on0 : on1) {
#pragma unroll
        for (int nf = 0; nf < NF; ++nf) {
          const double2 v = *reinterpret_cast<const double2*>(Gc + (size_t)j * N + i0 + nf * 8 + 2 * lk);
          acc[mf][nf][0] = v.x; acc[mf][nf][1] = v.y;
        }
      }
    }
  } else {
#pragma unroll
    for (int mf = 0; mf < 2; ++mf)
#pragma unroll
      for (int nf = 0; nf < NF; ++nf) acc[mf][nf][0] = acc[mf][nf][1] = 0.0;
  }
  cp_async_wait<0>();
  __syncthreads();
  if (MODE == 1 && !on0) return;                     // (f0 < f1: nothing of this warp lies in the lower triangle)
#pragma unroll 4
  for (int k4 = 0; k4 < PB / 4; ++k4) {
    const int kr = k4 * 4 + lk;
    const double* rj = sJ + kr * SY_LDS + lr;
    const double* ri = sI + kr * LDI + lr;
    double af0 = 0.0, af1 = 0.0;
    if (MODE == 2) {                                 // (entries with k beyond the fragment's reach were not loaded)
      if (k4 < lim0) af0 = rj[f0 * 8];
      if (k4 < lim1) af1 = rj[f1 * 8];
    } else {
      af0 = neg_bits(rj[f0 * 8]);
      if (on1) af1 = neg_bits(rj[f1 * 8]);
    }
    double bf[NF];
#pragma unroll
    for (int nf = 0; nf < NF; ++nf) bf[nf] = ri[nf * 8];
    if (MODE == 2) {
      if (k4 < lim0) {
#pragma unroll
        for (int nf = 0; nf < NF; ++nf) dmma884(acc[0][nf][0], acc[0][nf][1], af0, bf[nf]);
      }
      if (k4 < lim1) {
#pragma unroll
        for (int nf = 0; nf < NF; ++nf) dmma884(acc[1][nf][0], acc[1][nf][1], af1, bf[nf]);
      }
    } else {
#pragma unroll
      for (int nf = 0; nf < NF; ++nf) {
        dmma884(acc[0][nf][0], acc[0][nf][1], af0, bf[nf]);
        if (on1) dmma884(acc[1][nf][0], acc[1][nf][1], af1, bf[nf]);
      }
    }
  }
#pragma unroll
  for (int mf = 0; mf < 2; ++mf) {
    const int j = j0 + (mf == 0 ? f0 : f1) * 8 + lr;
    if (mf == 1 && !on1) continue;
#pragma unroll
    for (int nf = 0; nf < NF; ++nf)
      *reinterpret_cast<double2*>(Gc + (size_t)j * N + i0 + nf * 8 + 2 * lk) = make_double2(acc[mf][nf][0], acc[mf][nf][1]);
  }
}

// ------------------------------------------------------------------------------------------------------------
// backward solve  L' x = b,  b = w (+ addz), w = row m of the factor (see above).  One CTA per chain streams the factor
// once, bottom-right to top-left, in parts of BW_COLS columns x 128 rows through a ring of TMA tensor-map boxes (one
// 32 KB request per part, full / empty mbarriers, a producer warp with one active lane).  History: 1 KB bulk copies from
// a producer warp (the TMA engine accepts ~one request per 30 ns: 157 us for a 1024 x 1024 factor), then 16-byte
// LDGSTS copies by all threads with a __syncthreads per part (118 us: ~500 of the ~1600 cycles per part were LDGSTS
// issue, the rest the per-part barrier chain), now box loads and barriers only at block-column boundaries.
// 8 consumer warps turn every part into BW_COLS dot products (warp per BW_COLS / 8 columns, lanes over the rows):
//   off-diagonal block (I, J): b_J -= L[I, J]' x_I          diagonal block J: x_J = Linv_J' b_J
// Within a block column every warp owns its entries of b_J, so the consumers only meet before and after the diagonal
// block.   grid = C, block = 288 (8 consumer warps + the producer warp).
// ------------------------------------------------------------------------------------------------------------
#ifndef BNR_BW_COLS
#define BNR_BW_COLS 32
#endif
constexpr int BW_COLS = BNR_BW_COLS;             // columns per staged part of a 128 x 128 block
constexpr int BW_NH = PB / BW_COLS;              // parts per block
constexpr int BW_CPW = BW_COLS / 8;              // columns per warp
constexpr int BW_MAX_STAGES = 6;
constexpr int BW_STAGE_DBL = BW_COLS * PB;
constexpr int BW_THREADS = 288;
static int bwd_stages(int N) {
  const size_t budget = 227 * 1024 - sizeof(double) * (size_t)N - 512;
  int ns = (int)(budget / (sizeof(double) * BW_STAGE_DBL));
  return ns > BW_MAX_STAGES ? BW_MAX_STAGES : ns;
}
static size_t bwd_smem(int N) { return sizeof(double) * ((size_t)bwd_stages(N) * BW_STAGE_DBL + N) + 256; }

// tmG: the chain-stacked factor {rows, columns x chains}, tmL: the stacked panel inverses {128, 128 x panels x chains};
// boxes of 128 rows x BW_COLS columns (dense in shared memory: part[col * 128 + row])
__global__ void __launch_bounds__(BW_THREADS) k_bwd_stream(const __grid_constant__ CUtensorMap tmG,
                                                           const __grid_constant__ CUtensorMap tmL,
                                                           const double* __restrict__ G, size_t chain_stride, int N, int m,
                                                           double* __restrict__ out, int out_stride,
                                                           const double* __restrict__ addz, int addz_stride, int nstages) {
  extern __shared__ __align__(128) double sm[];
  double* ring = sm;
  double* x = sm + (size_t)nstages * BW_STAGE_DBL;     // [N] right-hand side, overwritten block by block by x
  unsigned long long* full = reinterpret_cast<unsigned long long*>(x + N);
  unsigned long long* empty = full + BW_MAX_STAGES;
  const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = N / PB;
  const double* Gc = G + (size_t)c * chain_stride;
  const int total = T * (T + 1) / 2 * BW_NH;
  if (tid == 0) {
    for (int s = 0; s < nstages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();

  if (warp == 8) {
    // ---- producer: the parts in consumption order (J down, I from T-1 down to J, h up) ----
    if (lane == 0) {
      int pJ = T - 1, pI = T - 1, ph = 0;
      for (int p = 0; p < total; ++p) {
        const int stage = p % nstages;
        mbar_wait(&empty[stage], ((p / nstages) & 1) ^ 1);
        mbar_expect_tx(&full[stage], BW_STAGE_DBL * 8u);
        double* dst = ring + (size_t)stage * BW_STAGE_DBL;
        if (pI == pJ) tma_load_2d(dst, &tmL, 0, (c * T + pJ) * PB + ph * BW_COLS, &full[stage]);
        else tma_load_2d(dst, &tmG, pI * PB, c * N + pJ * PB + ph * BW_COLS, &full[stage]);
        if (++ph == BW_NH) { ph = 0; if (--pI < pJ) { --pJ; pI = T - 1; } }
      }
    }
    return;
  }

  const double unscale = out[(size_t)c * out_stride + m];       // 2^e of k_augment (out is its right-hand side)
  for (int k = tid; k < N; k += 256)
    x[k] = (k < m) ? Gc[(size_t)k * N + m] * unscale + (addz ? addz[(size_t)c * addz_stride + k] : 0.0) : 0.0;
  named_bar_sync(1, 256);

  int it = 0;
  for (int J = T - 1; J >= 0; --J) {
    for (int I = T - 1; I >= J; --I) {
      const bool dg = (I == J);
      if (dg) named_bar_sync(1, 256);                  // every warp's updates of b_J are in
      const double* v = x + I * PB;
      const double v0 = v[lane], v1 = v[lane + 32], v2 = v[lane + 64], v3 = v[lane + 96];
      double xn[BW_NH][BW_CPW];                        // diagonal block: this warp's entries of x_J
#pragma unroll
      for (int h = 0; h < BW_NH; ++h, ++it) {
        const int stage = it % nstages;
        mbar_wait(&full[stage], (it / nstages) & 1);
        const double* B = ring + (size_t)stage * BW_STAGE_DBL + (size_t)(warp * BW_CPW) * PB + lane;
        double acc[BW_CPW];
#pragma unroll
        for (int q = 0; q < BW_CPW; ++q)
          acc[q] = B[q * PB] * v0 + B[q * PB + 32] * v1 + B[q * PB + 64] * v2 + B[q * PB + 96] * v3;
#pragma unroll
        for (int q = 0; q < BW_CPW; ++q) {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
        }
        if (dg) {
#pragma unroll
          for (int q = 0; q < BW_CPW; ++q) xn[h][q] = acc[q];
        } else if (lane == 0) {
          double* bj = x + J * PB + h * BW_COLS + warp * BW_CPW;
#pragma unroll
          for (int q = 0; q < BW_CPW; ++q) bj[q] -= acc[q];
        }
        // Release the part only HERE, after the shuffles (and the update of b_J) have consumed every lane's loads.
        // An arrive right after the loads were ISSUED is not enough: it is not ordered behind shared-memory loads
        // that still wait in the memory pipe, the producer's next box then overwrote data that had not been read yet
        // -- chains differed from run to run under load (tools/determinism_check.py found it; the SASS showed the
        // DFMAs that consume the loads scheduled after the SYNCS.ARRIVE).
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
      }
      if (dg) {
        named_bar_sync(1, 256);                        // everybody has read b_J
        if (lane == 0) {
#pragma unroll
          for (int h = 0; h < BW_NH; ++h)
#pragma unroll
            for (int q = 0; q < BW_CPW; ++q) x[J * PB + h * BW_COLS + warp * BW_CPW + q] = xn[h][q];
        }
        named_bar_sync(1, 256);                        // x_J is visible
      }
    }
  }
  for (int k = tid; k < N; k += 256) out[(size_t)c * out_stride + k] = x[k];
}

// ------------------------------------------------------------------------------------------------------------
// backward solve above BWD_STREAM_MAX_DIM: one cluster of BWC_K CTAs per chain (the same solve as k_bwd_stream, over K
// SMs' share of L2 bandwidth instead of one, and with x spread over K shared memories instead of held by one).
//   ownership  CTA r owns the block rows I = r (mod K): it keeps b_I, overwritten by x_I, in its shared memory and
//              streams the tiles L[I, J], I > J, of its own rows (and Linv_J of its own columns) through its own ring
//              (tensor-map boxes, full / empty mbarriers, one producer lane: exactly k_bwd_stream's ring).
//   column J   every CTA forms p_r = sum_{own I > J, I descending} L[I, J]' x_I with k_bwd_stream's mat-vec (warp per
//              4 columns of a part, partial sums in registers).  A non-owner writes p_r into slot r of the owner's
//              current slot set (DSMEM stores by lane 0 of each warp, then one release-arrive per warp, cluster scope, on
//              the owner's "slot set full" mbarrier).  The owner waits for the K - 1 partials, forms
//              b_J - p_0 - p_1 - ... - p_{K-1} in rank order, releases the slot set (a remote arrive on a "slot free"
//              mbarrier in every other CTA) and computes x_J = Linv_J' b_J.  Only the owner waits: the x_I a CTA needs
//              are the ones it solved itself, so the others run ahead up to BWC_SLOTS columns per owner.
// K is a constant, so the summation order depends on N only: every chain count, chain grouping and device split adds
// in the same order.  grid = C * K (cluster K x 1 x 1), block = 288 (8 consumer warps + the producer warp).
// ------------------------------------------------------------------------------------------------------------
constexpr int BWC_K = 8;           // CTAs per chain (the portable cluster size)
constexpr int BWC_SLOTS = 2;       // slot sets per owner: a writer may run this many of the owner's columns ahead
static int bwc_own_blocks(int N) { return (N / PB + BWC_K - 1) / BWC_K; }
static size_t bwc_fixed_bytes(int N) {
  return sizeof(double) * ((size_t)bwc_own_blocks(N) * PB + (size_t)BWC_SLOTS * BWC_K * PB) +
         sizeof(unsigned long long) * (2 * BW_MAX_STAGES + BWC_SLOTS + BWC_K * BWC_SLOTS) + 128;
}
static int bwc_stages(int N) {
  const size_t budget = 227 * 1024 - bwc_fixed_bytes(N);
  const int ns = (int)(budget / (sizeof(double) * BW_STAGE_DBL));
  return ns > BW_MAX_STAGES ? BW_MAX_STAGES : ns;
}
static size_t bwc_smem(int N) { return sizeof(double) * (size_t)bwc_stages(N) * BW_STAGE_DBL + bwc_fixed_bytes(N); }

__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ unsigned mapa_rank(const void* p, unsigned rank) {
  unsigned a;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(a) : "r"(smem_u32(p)), "r"(rank));
  return a;
}
__device__ __forceinline__ void st_cluster_f64(unsigned addr, double v) {
  asm volatile("st.shared::cluster.f64 [%0], %1;\n" ::"r"(addr), "d"(v) : "memory");
}
// release at cluster scope: this thread's earlier (DSMEM) stores are visible to whoever acquires the phase
__device__ __forceinline__ void mbar_arrive_remote(unsigned addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];\n" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;\nbarrier.cluster.wait.acquire;\n" ::: "memory");
}

__global__ void __launch_bounds__(BW_THREADS) k_bwd_cluster(const __grid_constant__ CUtensorMap tmG,
                                                            const __grid_constant__ CUtensorMap tmL,
                                                            const double* __restrict__ G, size_t chain_stride, int N, int m,
                                                            double* __restrict__ out, int out_stride,
                                                            const double* __restrict__ addz, int addz_stride, int nstages) {
  extern __shared__ __align__(128) double sm[];
  const int T = N / PB, nown = (T + BWC_K - 1) / BWC_K;
  double* ring = sm;
  double* xo = sm + (size_t)nstages * BW_STAGE_DBL;               // [nown][128] b_I, then x_I, of the own blocks I = r + K li
  double* slot = xo + (size_t)nown * PB;                          // [BWC_SLOTS][BWC_K][128] partials of the other CTAs
  unsigned long long* full = reinterpret_cast<unsigned long long*>(slot + (size_t)BWC_SLOTS * BWC_K * PB);
  unsigned long long* empty = full + BW_MAX_STAGES;
  unsigned long long* sfull = empty + BW_MAX_STAGES;              // [BWC_SLOTS] the K - 1 partials of a slot set are in
  unsigned long long* sfree = sfull + BWC_SLOTS;                  // [owner][BWC_SLOTS] the owner has read that slot set
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = (int)cluster_ctarank(), c = (int)blockIdx.x / BWC_K;
  const int Itop = (T - 1) - (T - 1 - r) % BWC_K;                 // the last own block row (T > K: every rank owns one)
  const double* Gc = G + (size_t)c * chain_stride;
  if (tid == 0) {
    for (int s = 0; s < nstages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
    for (int s = 0; s < BWC_SLOTS; ++s) mbar_init(&sfull[s], 8 * (BWC_K - 1));
    for (int i = 0; i < BWC_K * BWC_SLOTS; ++i) mbar_init(&sfree[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  cluster_sync_all();                                             // every barrier of the cluster exists before a remote arrive

  if (warp == 8) {
    // ---- producer: the parts in consumption order (J down; own I from the top down to J + 1; Linv_J if J is own) ----
    if (lane == 0) {
      int p = 0;
      for (int J = T - 1; J >= 0; --J) {
        // own rows I > J of block column J, then (own column) the inverse of the diagonal block: I == J
        const int Ilast = (J % BWC_K == r) ? J : J + 1;
        for (int I = Itop; I >= Ilast; I -= BWC_K) {
          for (int h = 0; h < BW_NH; ++h, ++p) {
            const int stage = p % nstages;
            mbar_wait(&empty[stage], ((p / nstages) & 1) ^ 1);
            mbar_expect_tx(&full[stage], BW_STAGE_DBL * 8u);
            double* dst = ring + (size_t)stage * BW_STAGE_DBL;
            if (I == J) tma_load_2d(dst, &tmL, 0, (c * T + J) * PB + h * BW_COLS, &full[stage]);
            else tma_load_2d(dst, &tmG, I * PB, c * N + J * PB + h * BW_COLS, &full[stage]);
          }
        }
      }
    }
  } else {
    const double unscale = out[(size_t)c * out_stride + m];       // 2^e of k_augment (out is its right-hand side)
    for (int id = tid; id < nown * PB; id += 256) {
      const int I = r + BWC_K * (id / PB), k = I * PB + id % PB;
      xo[id] = (I < T && k < m) ? Gc[(size_t)k * N + m] * unscale + (addz ? addz[(size_t)c * addz_stride + k] : 0.0) : 0.0;
    }
    named_bar_sync(1, 256);

    int it = 0;
    for (int J = T - 1; J >= 0; --J) {
      const int o = J % BWC_K, u = (T - 1 - J) / BWC_K;            // owner of column J, and its use count of the slots
      const int s = u % BWC_SLOTS;
      const unsigned par = (u / BWC_SLOTS) & 1;
      double pr[BW_NH][BW_CPW];
#pragma unroll
      for (int h = 0; h < BW_NH; ++h)
#pragma unroll
        for (int q = 0; q < BW_CPW; ++q) pr[h][q] = 0.0;
      for (int I = Itop; I > J; I -= BWC_K) {
        const double* v = xo + (size_t)(I / BWC_K) * PB;
        const double v0 = v[lane], v1 = v[lane + 32], v2 = v[lane + 64], v3 = v[lane + 96];
#pragma unroll
        for (int h = 0; h < BW_NH; ++h, ++it) {
          const int stage = it % nstages;
          mbar_wait(&full[stage], (it / nstages) & 1);
          const double* B = ring + (size_t)stage * BW_STAGE_DBL + (size_t)(warp * BW_CPW) * PB + lane;
          double acc[BW_CPW];
#pragma unroll
          for (int q = 0; q < BW_CPW; ++q)
            acc[q] = B[q * PB] * v0 + B[q * PB + 32] * v1 + B[q * PB + 64] * v2 + B[q * PB + 96] * v3;
#pragma unroll
          for (int q = 0; q < BW_CPW; ++q) {
#pragma unroll
            for (int o2 = 16; o2 > 0; o2 >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o2);
            pr[h][q] += acc[q];
          }
          // released after the shuffles have consumed every lane's loads (DESIGN section 4, rule 4)
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[stage]);
        }
      }
      if (o != r) {
        if (lane == 0) {
          mbar_wait_cluster(&sfree[o * BWC_SLOTS + s], par ^ 1);   // the owner has read this slot set's previous use
          const unsigned dst = mapa_rank(slot + ((size_t)s * BWC_K + r) * PB, (unsigned)o);
#pragma unroll
          for (int h = 0; h < BW_NH; ++h)
#pragma unroll
            for (int q = 0; q < BW_CPW; ++q) st_cluster_f64(dst + 8u * (h * BW_COLS + warp * BW_CPW + q), pr[h][q]);
          mbar_arrive_remote(mapa_rank(&sfull[s], (unsigned)o));
        }
        __syncwarp();
        continue;
      }
      double* bJ = xo + (size_t)(J / BWC_K) * PB;
      if (lane == 0) {
        mbar_wait_cluster(&sfull[s], par);
        const double* sl = slot + (size_t)s * BWC_K * PB;
#pragma unroll
        for (int h = 0; h < BW_NH; ++h)
#pragma unroll
          for (int q = 0; q < BW_CPW; ++q) {
            const int col = h * BW_COLS + warp * BW_CPW + q;
            double t = bJ[col];
#pragma unroll
            for (int rr = 0; rr < BWC_K; ++rr) t -= (rr == r) ? pr[h][q] : sl[rr * PB + col];
            bJ[col] = t;
          }
      }
      __syncwarp();
      named_bar_sync(1, 256);                  // b_J is complete; every read of the slot set has gone into it
      if (tid == 0) {
        for (int rr = 0; rr < BWC_K; ++rr)
          if (rr != r) mbar_arrive_remote(mapa_rank(&sfree[r * BWC_SLOTS + s], (unsigned)rr));
      }
      const double v0 = bJ[lane], v1 = bJ[lane + 32], v2 = bJ[lane + 64], v3 = bJ[lane + 96];
      double xn[BW_NH][BW_CPW];
#pragma unroll
      for (int h = 0; h < BW_NH; ++h, ++it) {
        const int stage = it % nstages;
        mbar_wait(&full[stage], (it / nstages) & 1);
        const double* B = ring + (size_t)stage * BW_STAGE_DBL + (size_t)(warp * BW_CPW) * PB + lane;
        double acc[BW_CPW];
#pragma unroll
        for (int q = 0; q < BW_CPW; ++q)
          acc[q] = B[q * PB] * v0 + B[q * PB + 32] * v1 + B[q * PB + 64] * v2 + B[q * PB + 96] * v3;
#pragma unroll
        for (int q = 0; q < BW_CPW; ++q) {
#pragma unroll
          for (int o2 = 16; o2 > 0; o2 >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o2);
          xn[h][q] = acc[q];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
      }
      named_bar_sync(1, 256);                  // everybody has read b_J
      if (lane == 0) {
#pragma unroll
        for (int h = 0; h < BW_NH; ++h)
#pragma unroll
          for (int q = 0; q < BW_CPW; ++q) bJ[h * BW_COLS + warp * BW_CPW + q] = xn[h][q];
      }
      __syncwarp();
      named_bar_sync(1, 256);                  // x_J is visible
    }
    for (int id = tid; id < nown * PB; id += 256) {
      const int I = r + BWC_K * (id / PB);
      if (I < T) out[(size_t)c * out_stride + (size_t)I * PB + id % PB] = xo[id];
    }
  }
  cluster_sync_all();                          // no CTA leaves while another may still write its slots or barriers
}

// symmetric copy of G (lower -> full) into the aux buffer, for the parity tests.  grid = (np, C)
__global__ void k_copy_sym(const double* __restrict__ G, size_t chain_stride, int np, double* __restrict__ out) {
  const int c = blockIdx.y, j = blockIdx.x;
  const double* Gc = G + (size_t)c * chain_stride;
  double* o = out + (size_t)c * np * np;
  for (int i = threadIdx.x; i < np; i += blockDim.x) {
    const double v = (i >= j) ? Gc[(size_t)j * np + i] : Gc[(size_t)i * np + j];
    o[(size_t)j * np + i] = v;
  }
}

// ------------------------------------------------------------------------------------------------------------
// tall-skinny GEMM with X for all chains at once on the FP64 tensor cores: out[c][m] = sum_k A(m,k) in[c][k]
//   TRANS = 0: A(m,k) = X[m + np*k]  (M = np, K = qp)      TRANS = 1: A(m,k) = X[k + np*m]  (M = qp, K = np)
// CTA tile 128 (m) x 64 (chains), k-step 16, 3-stage cp.async pipeline, 8 warps as 4 (m) x 2 (chains), warp tile
// 32 x 32 = 4 x 4 DMMA m8n8k4 per k4-step.  K is split over gridDim.z (deterministic: partial sums go to a
// workspace and are added in a fixed order by k_splitk_reduce) so that ~2 waves of CTAs stream X exactly once.
// Shared tiles: X as [k][m] (ld 132) for TRANS 0 / [m][k] (ld 20) for TRANS 1, the vectors as [chain][k] (ld 20);
// both strides are == 4 mod 16 doubles, which makes the (row, k) fragment loads bank-conflict free.
// ------------------------------------------------------------------------------------------------------------
constexpr int XM_BM = 128, XM_BN = 64, XM_BK = 16, XM_STAGES = 3;
constexpr int XM_LDM = 132, XM_LDK = 20;
constexpr int XM_A_DBL = (XM_BK * XM_LDM > XM_BM * XM_LDK) ? XM_BK * XM_LDM : XM_BM * XM_LDK;   // 2560
constexpr int XM_STAGE_DBL = XM_A_DBL + XM_BN * XM_LDK;
constexpr size_t XMMA_SMEM = sizeof(double) * XM_STAGES * XM_STAGE_DBL;

__device__ __forceinline__ void cp_async16_zfill(void* smem, const void* gmem, bool valid) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(sa), "l"(gmem), "r"(sz));
}

template <int TRANS>
__global__ void __launch_bounds__(256) k_xmma(const double* __restrict__ X, int np, int M, int K, int N,
                                              const double* __restrict__ in, int ldin, double* __restrict__ out,
                                              int ldout, int k_per_split) {
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lk = lane & 3, lr = lane >> 2, wm = warp & 3, wn = warp >> 2;
  const int m0 = blockIdx.x * XM_BM, n0 = blockIdx.y * XM_BN;
  const int kbeg = blockIdx.z * k_per_split;
  const int kend = min(K, kbeg + k_per_split);
  const int nsteps = (kend - kbeg + XM_BK - 1) / XM_BK;
  double* o = out + (size_t)blockIdx.z * N * ldout;

  auto load_stage = [&](int step) {
    double* As = sm + (size_t)(step % XM_STAGES) * XM_STAGE_DBL;
    double* Vs = As + XM_A_DBL;
    const int k0 = kbeg + step * XM_BK;
    if (TRANS == 0) {
      // 16 k-rows of 128 contiguous m: 64 x 16-byte pieces per row
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int id = tid + 256 * r, kk = id >> 6, mm = (id & 63) * 2;
        cp_async16_zfill(As + kk * XM_LDM + mm, X + (size_t)(k0 + kk) * np + m0 + mm, m0 + mm < M);
      }
    } else {
      // 128 m-rows of 16 contiguous k: 8 x 16-byte pieces per row
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int id = tid + 256 * r, mm = id >> 3, kk = (id & 7) * 2;
        const bool ok = m0 + mm < M;
        cp_async16_zfill(As + mm * XM_LDK + kk, X + (size_t)(ok ? m0 + mm : 0) * np + k0 + kk, ok);
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int id = tid + 256 * r, nn = id >> 3, kk = (id & 7) * 2;
      const bool ok = n0 + nn < N;
      cp_async16_zfill(Vs + nn * XM_LDK + kk, in + (size_t)(ok ? n0 + nn : 0) * ldin + k0 + kk, ok);
    }
  };

  double acc[4][4][2];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
  // chain fragments of this warp that hold a real chain: with few chains (a chain group of 2-3, config 4's 8) the 64-chain
  // tile is mostly padding, and its DMMAs -- not the stream of X -- bounded the kernel (2 us per k-step for 16 KB)
  int nfv = (N - n0 - wn * 32 + 7) >> 3;
  nfv = nfv < 0 ? 0 : (nfv > 4 ? 4 : nfv);

  for (int s = 0; s < XM_STAGES - 1; ++s) {
    if (s < nsteps) load_stage(s);
    cp_async_commit();
  }
  for (int step = 0; step < nsteps; ++step) {
    cp_async_wait<XM_STAGES - 2>();
    __syncthreads();
    if (step + XM_STAGES - 1 < nsteps) load_stage(step + XM_STAGES - 1);
    cp_async_commit();
    const double* As = sm + (size_t)(step % XM_STAGES) * XM_STAGE_DBL;
    const double* Vs = As + XM_A_DBL;
    if (nfv == 0) continue;                          // (a warp without a real chain only keeps the barriers company)
#pragma unroll
    for (int k4 = 0; k4 < XM_BK / 4; ++k4) {
      const int kr = k4 * 4 + lk;
      double af[4], bf[4];
#pragma unroll
      for (int mf = 0; mf < 4; ++mf)
        af[mf] = (TRANS == 0) ? As[kr * XM_LDM + wm * 32 + mf * 8 + lr] : As[(wm * 32 + mf * 8 + lr) * XM_LDK + kr];
#pragma unroll
      for (int nf = 0; nf < 4; ++nf) bf[nf] = (nf < nfv) ? Vs[(wn * 32 + nf * 8 + lr) * XM_LDK + kr] : 0.0;
#pragma unroll
      for (int nf = 0; nf < 4; ++nf) {
        if (nf < nfv) {
#pragma unroll
          for (int mf = 0; mf < 4; ++mf) dmma884(acc[mf][nf][0], acc[mf][nf][1], af[mf], bf[nf]);
        }
      }
    }
  }
  cp_async_wait<0>();
#pragma unroll
  for (int mf = 0; mf < 4; ++mf) {
    const int mm = m0 + wm * 32 + mf * 8 + lr;
#pragma unroll
    for (int nf = 0; nf < 4; ++nf) {
      const int nn = n0 + wn * 32 + nf * 8 + 2 * lk;
      if (mm < M) {
        if (nn < N) o[(size_t)nn * ldout + mm] = acc[mf][nf][0];
        if (nn + 1 < N) o[(size_t)(nn + 1) * ldout + mm] = acc[mf][nf][1];
      }
    }
  }
}

__global__ void k_splitk_reduce(const double* __restrict__ ws, double* __restrict__ out, size_t count, int splits) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double s = 0.0;
  for (int z = 0; z < splits; ++z) s += ws[(size_t)z * count + i];
  out[i] = s;
}

// k-splits of X v, X' a4, X gamma and X_new gamma (M x K operand).  The split count sets the summation order, so it
// depends on the handle's chain count only: a chain group (a view with d.C < d.C_total) and an eager sweep over the whole
// handle add in the same order.
static int x_times_splits(int M, int K, int C_total) {
  const int tiles = ((M + XM_BM - 1) / XM_BM) * ((C_total + XM_BN - 1) / XM_BN);
  int ks = (2 * 148 + tiles - 1) / tiles;
  const int kmax = K / (4 * XM_BK) > 0 ? K / (4 * XM_BK) : 1;
  if (ks > kmax) ks = kmax;
  if (ks > 64) ks = 64;
  if (ks < 1) ks = 1;
  return ks;
}

// Every workspace (the handle's and each chain group's) holds splits x chains x rows partial sums for the handle's whole
// chain count.  A launch uses splits x d.C x rows with the same splits and d.C <= d.C_total, so it always fits.
size_t x_times_workspace_doubles(const Dims& d) {
  const int a = x_times_splits(d.np, d.qp, d.C_total), b = x_times_splits(d.qp, d.np, d.C_total);
  const size_t wa = (size_t)a * d.C_total * d.np, wb = (size_t)b * d.C_total * d.qp;
  return wa > wb ? wa : wb;
}

int pred_splits(const Dims& d, int mp) { return x_times_splits(mp, d.qp, d.C_total); }

void launch_x_times(const Dims& d, int trans, const double* A, int lda, int M, int K, const double* in, double* out,
                    double* ws, cudaStream_t s) {
  const int N = d.C, ldin = K, ldout = M;
  const int ks = x_times_splits(M, K, d.C_total);
  const int kper = ((K + ks - 1) / ks + XM_BK - 1) / XM_BK * XM_BK;
  dim3 grid((M + XM_BM - 1) / XM_BM, (N + XM_BN - 1) / XM_BN, ks);
  double* dst = (ks == 1 && out) ? out : ws;
  ++g_launches;
  if (trans) k_xmma<1><<<grid, 256, XMMA_SMEM, s>>>(A, lda, M, K, N, in, ldin, dst, ldout, kper);
  else k_xmma<0><<<grid, 256, XMMA_SMEM, s>>>(A, lda, M, K, N, in, ldin, dst, ldout, kper);
  if (ks > 1 && out) {
    const size_t count = (size_t)N * ldout;
    ++g_launches; k_splitk_reduce<<<(unsigned)((count + 255) / 256), 256, 0, s>>>(ws, out, count, ks);
  }
}

void launch_x_times(const Engine& e, int trans, const double* in, double* out, double* ws, cudaStream_t s) {
  const Dims& d = e.d;
  launch_x_times(d, trans, e.X, d.np, trans ? d.qp : d.np, trans ? d.np : d.qp, in, out, ws, s);
}

void launch_pred_product(const Engine& e, cudaStream_t s) {
  launch_x_times(e.d, 0, e.Xp, e.pred_mp, e.pred_mp, e.d.qp, e.gamma, nullptr, e.pred_ws, s);
}

__global__ void k_gram_i8(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                          const double* __restrict__ rscale, double* __restrict__ G, int np, int nvalid, int nkb);
extern const size_t GI_SMEM_BYTES;

void linalg_setup() {
  cudaFuncSetAttribute(k_xmma<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)XMMA_SMEM);
  cudaFuncSetAttribute(k_xmma<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)XMMA_SMEM);
  cudaFuncSetAttribute(k_gram_syrk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SYRK_SMEM);
  cudaFuncSetAttribute(k_gram_i8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GI_SMEM_BYTES);
  cudaFuncSetAttribute(k_chol_update, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SYRK_SMEM);
  cudaFuncSetAttribute(k_trsm_dmma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SYRK_SMEM);
  cudaFuncSetAttribute(k_potf2_inv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POTF2_SMEM);
  cudaFuncSetAttribute(k_bwd_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  cudaFuncSetAttribute(k_bwd_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  cudaFuncSetAttribute(k_small_tile<1, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_tile_smem(32));
  cudaFuncSetAttribute(k_small_tile<2, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_tile_smem(32));
  cudaFuncSetAttribute(k_small_tile<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_tile_smem(16));
  cudaFuncSetAttribute(k_small_tile<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_tile_smem(16));
  cudaFuncSetAttribute(k_small_tile<1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_tile_smem(64));
  cudaFuncSetAttribute(k_small_tile<2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_tile_smem(64));
}

// k-splits of the SYRK for a handle of C chains: when chains x tiles is below ~4 waves of CTAs, a CTA (one 128 x 128
// tile over the whole contraction: 0.7 ms at q = 5050, 2.7 ms at q = 20100) is too coarse a unit of work to balance over
// 148 SMs, so the contraction is cut into up to 8 pieces of at least 24 k-steps.  The count depends on the handle's chain
// count only (not on the chain groups, which each launch a part of the chains).
// ---- tensor maps (host): a k-major operand {rows (contiguous), k-rows} with boxes of box_rows x 16 ----
typedef CUresult (*TmapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TmapEncodeFn g_tmap_encode = nullptr;
bool tmap_setup() {
  if (g_tmap_encode) return true;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qr;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) != cudaSuccess ||
      qr != cudaDriverEntryPointSuccess || !fn)
    return false;
  g_tmap_encode = (TmapEncodeFn)fn;
  return true;
}
// rows beyond `rows` (the box is 4 rows wider than a tile) and k-rows beyond `krows` read as zeros
static CUresult encode_map(CUtensorMap* m, const double* base, uint64_t rows, uint64_t krows, uint64_t ld, uint32_t box_rows,
                           uint32_t box_k) {
  memset(m, 0, sizeof(*m));
  const cuuint64_t dims[2] = {rows, krows};
  const cuuint64_t strides[1] = {ld * sizeof(double)};
  const cuuint32_t box[2] = {box_rows, box_k};
  const cuuint32_t estr[2] = {1, 1};
  if (!tmap_setup()) return CUDA_ERROR_NOT_SUPPORTED;
  return g_tmap_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}
static CUtensorMap make_map(const double* base, uint64_t rows, uint64_t krows, uint64_t ld, uint32_t box_rows,
                            uint32_t box_k = SY_BK) {
  CUtensorMap m;
  const CUresult r = encode_map(&m, base, rows, krows, ld, box_rows, box_k);
  if (r != CUDA_SUCCESS) {
    // (bnr_create has already encoded every map of this handle's geometry, tmaps_check(): unreachable from the ABI)
    fprintf(stderr, "[bnr] cuTensorMapEncodeTiled failed (%d) for a %llu x %llu operand, box %u x %d\n", (int)r,
            (unsigned long long)rows, (unsigned long long)krows, box_rows, (int)box_k);
    abort();
  }
  return m;
}
// every tensor map the launchers will build for this handle, encoded once at creation so that a driver that refuses one
// is reported through the ABI (bnr_create -> BNR_ECUDA) instead of at the first sweep
bool tmaps_check(const Engine& e) {
  const Dims& d = e.d;
  const uint64_t N = d.gdim, C = d.C, T = d.gdim / SY_BT;
  CUtensorMap m;
  bool ok = true;
  if (d.gmode != 2) ok = ok && encode_map(&m, e.X, d.np, d.qp, d.np, SY_LDS, SY_BK) == CUDA_SUCCESS;
  for (uint32_t box : {(uint32_t)SY_LDS, (uint32_t)(SY_BT / 2 + 4), (uint32_t)(SY_BT / 4 + 4)})
    ok = ok && encode_map(&m, e.G, N, N * C, N, box, SY_BK) == CUDA_SUCCESS;
  ok = ok && encode_map(&m, e.Linv, SY_BT, SY_BT * T * C, SY_BT, SY_LDS, SY_BK) == CUDA_SUCCESS;
  ok = ok && encode_map(&m, e.G, N, N * C, N, SY_BT, BW_COLS) == CUDA_SUCCESS;       // back solve
  ok = ok && encode_map(&m, e.Linv, SY_BT, SY_BT * T * C, SY_BT, SY_BT, BW_COLS) == CUDA_SUCCESS;
  return ok;
}

int syrk_splits(const Dims& d, int C) {
  const int T = d.np / SY_BT, tiles = T * (T + 1) / 2, nk = d.qp / SY_BK;
  // (measured: once chains x tiles reaches one wave, splitting only removes the natural stagger between chain groups)
  if (tiles * C >= 148) return 1;
  int s = (4 * 148 + tiles * C - 1) / (tiles * C);
  if (s > nk / 24) s = nk / 24;
  if (s > SYRK_MAX_SPLITS) s = SYRK_MAX_SPLITS;
  return s < 1 ? 1 : s;
}

// ------------------------------------------------------------------------------------------------------------
// n-form Gram matrix on the INT8 tensor cores (Ozaki scheme): G_c = A_c A_c' + I with A_c = X diag(sqrt(S_c)).
//   k_gram_slice: row i of A_c is scaled by 2^p_i (row max in [2^53, 2^55)), rounded ONCE to an integer N (|N| < 2^55;
//     the entries near the row max are integers already: exact) and N is written as 7 balanced base-256 digits
//     N = sum_s D^(s) 2^(8(6-s)), s = 0 (top, |D| <= 127) .. 6 (each in [-128, 127]).  Planes [c][s][row][k] int8, k
//     contiguous (the k-major boxes the UMMA reads), plus rscale[c][row] = 2^-p_i.  Rounding the scaled value to the
//     nearest integer is unbiased, so the rounding errors of a row do not add up with one sign when X >= 0.
//   k_gram_i8: C_g = sum_{s+t=g} D^(s) D^(t)' for g = 0..6 (28 digit products, the pairs with s + t > 6 weigh at most
//     ~2^-56 of the row maxima and are dropped) in seven int32 TMEM accumulators of a 128 x 64 tile (448 of the 512
//     columns), then G = 2^96 rscale_i rscale_j sum_g 2^-8g C_g, added in a fixed order (Horner from g = 6), + I.
//     |D^(s) D^(t)| <= 2^14 and the largest group has 7 products per k, so int32 is exact while 7 qp 2^14 < 2^31:
//     qp <= GRAM_I8_QP_MAX.  Larger qp stays on the FP64 SYRK (gram_i8_selected).
// Warp roles of k_gram_i8 (192 threads, 1 CTA / SM): warp 4 lane 0 issues the TMA boxes (all 7 planes of the
// 128-row and of the 64-row operand per k-block: one 3-D box each) into a GI_STAGES ring; warp 5 lane 0 issues the
// tcgen05.mma and releases each stage with tcgen05.commit; warps 0-3 read the accumulators (TMEM lanes 32w..32w+31 =
// rows of the tile) and store G.  Tiles: 128-row block ib x 64-column block jb <= 2 ib + 1, chains slowest, so the
// CTAs of one chain run back to back while its planes are in L2.  The stored entries are exactly those the FP64 SYRK
// stores (same 8 x 8 fragment rule), so the matrix the factorisation sees is the same up to the rounding.
// GI_LAB_LOADS_ONLY / GI_LAB_MMA_ONLY are defined only by the diagnostic builds of tools/lab/gram_i8_lab.cu.
// ------------------------------------------------------------------------------------------------------------
#ifndef BNR_GI_BK
#define BNR_GI_BK 64
#endif
#ifndef BNR_GI_STAGES
#define BNR_GI_STAGES 2
#endif
constexpr int GI_S = 7;                   // digit planes (and digit-sum groups)
constexpr int GI_BM = 128, GI_BN = 64;    // tile
constexpr int GI_BK = BNR_GI_BK;          // k-block in bytes (int8 elements) = swizzle width
constexpr int GI_STAGES = BNR_GI_STAGES;
constexpr int GI_A_PLANE = GI_BM * GI_BK, GI_B_PLANE = GI_BN * GI_BK;
constexpr int GI_STAGE_BYTES = GI_S * (GI_A_PLANE + GI_B_PLANE);
constexpr size_t GI_SMEM = (size_t)GI_STAGES * GI_STAGE_BYTES + 1024 + 256;   // + alignment slack + barriers
const size_t GI_SMEM_BYTES = GI_SMEM;
constexpr int GI_THREADS = 192;
static_assert(GI_BK == 32 || GI_BK == 64 || GI_BK == 128, "k-block = swizzle width");
static_assert(GI_S * GI_BN <= 512, "accumulators exceed tensor memory");

// UMMA shared-memory descriptor of a K-major operand with GI_BK-byte swizzle: 8-row core groups GI_BK * 8 bytes apart
__device__ __forceinline__ unsigned long long gi_desc(unsigned saddr) {
  constexpr unsigned long long layout = GI_BK == 128 ? 2ull : (GI_BK == 64 ? 4ull : 6ull);
  return (unsigned long long)((saddr & 0x3FFFF) >> 4) | (1ull << 16) | ((unsigned long long)((GI_BK * 8) >> 4) << 32) |
         (1ull << 46) | (layout << 61);
}
// instruction descriptor: s32 accumulator, s8 x s8, both K-major, M = 128, N = n (n % 16 == 0, n <= 256)
__host__ __device__ constexpr unsigned gi_idesc(int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(n >> 3) << 17) | ((unsigned)(GI_BM >> 4) << 24);
}

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* tm, int x, int y, int z, unsigned long long* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(
                   smem_u32(smem_dst)), "l"((unsigned long long)tm), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_i8(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc, unsigned idesc,
                                        bool acc) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
               "l"(adesc), "l"(bdesc), "r"(idesc), "r"((int)acc));
}
__device__ __forceinline__ void umma_commit(unsigned long long* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld8(unsigned taddr, int (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
}

// k_gram_slice: a CTA takes GS_ROWS rows x GS_CB chains of the launch (the last chain block may be partial) over all k,
// so each X element it loads serves GS_CB chains, in both passes (row maximum, then the digits).  Lane l of a warp
// takes row l & 15 and the 16 k at 16 (l >> 4) of a 32-k block; the 8 warps take the 32-k blocks of a GS_TK-wide
// window in turn.  The roots sqrt(S_ck) of a window are taken once per CTA into shared memory (both passes: the roots of
// all k would not fit beside a resident k_gram_i8 CTA).  A thread's 16 k of one row are 16 contiguous bytes of each
// plane: the bytes of 4 elements are transposed into 4 words with __byte_perm and each plane is one 16-byte store, so a
// warp store covers 16 rows x 32 B, whole sectors.  Every element is computed as before, so the planes and rscale are
// the same bits for any GS_CB.  GS_LAB_NO_STORES / GS_LAB_NO_DIGITS are defined only by the diagnostic builds of
// tools/lab/gram_i8_lab.cu.
constexpr int GS_ROWS = 16, GS_CB = 4, GS_THREADS = 256, GS_TK = 512;
constexpr int GS_TKP = GS_TK + GS_TK / 8;   // 2 pad doubles per 16 k: the two half-warps read different banks
__device__ __forceinline__ int gs_tidx(int kk) { return kk + 2 * (kk >> 4); }

// sqrt(S_ck) for the window [t0, t0 + GS_TK) of the block's chains (0 for k >= q and for chains past the launch's)
__device__ __forceinline__ void gs_roots(double (*sq)[GS_TKP], const double* __restrict__ S, int qp, int q, int ncb, int t0) {
  for (int id = threadIdx.x; id < GS_CB * GS_TK; id += GS_THREADS) {
    const int cb = id / GS_TK, kk = id % GS_TK, k = t0 + kk;
    sq[cb][gs_tidx(kk)] = cb < ncb && k < q ? sqrt(S[(size_t)cb * qp + k]) : 0.0;
  }
}

// max(m, a) that keeps a NaN once it has met one (fmax drops it): a row with a non-finite entry must not slice as finite
__device__ __forceinline__ double gs_max(double m, double a) { return a > m || a != a ? a : m; }

__device__ __forceinline__ void gs_load_x(double (&x)[16], const double* __restrict__ X, int np, int q, int row, int k0) {
  const bool full = k0 + 16 <= q;
#pragma unroll
  for (int j = 0; j < 16; ++j) x[j] = full || k0 + j < q ? X[row + (size_t)np * (k0 + j)] : 0.0;
}

__global__ void __launch_bounds__(GS_THREADS, 2) k_gram_slice(const double* __restrict__ X, const double* __restrict__ S,
                                                            int np, int q, int qp, int C, signed char* __restrict__ planes,
                                                            double* __restrict__ rscale) {
  __shared__ __align__(16) double sq[GS_CB][GS_TKP];
  __shared__ double red[GS_THREADS / 32][GS_CB][GS_ROWS];
  __shared__ double2 scl[GS_CB][GS_ROWS];   // (2^p1, 2^(p - p1)) per chain and row
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, rr = lane & 15, h = lane >> 4;
  const int r0 = blockIdx.x * GS_ROWS, row = r0 + rr, c0 = blockIdx.y * GS_CB;
  const int ncb = C - c0 < GS_CB ? C - c0 : GS_CB;
  const double* Sb = S + (size_t)c0 * qp;
  constexpr int NW = GS_THREADS / 32, BPW = GS_TK / 32 / NW;   // warps, 32-k blocks per warp and window
  double x[16];

  // pass 1: row maxima of |A| over k < q
  double m[GS_CB];
#pragma unroll
  for (int cb = 0; cb < GS_CB; ++cb) m[cb] = 0.0;
  for (int t0 = 0; t0 < q; t0 += GS_TK) {
    __syncthreads();
    gs_roots(sq, Sb, qp, q, ncb, t0);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < BPW; ++i) {
      const int kk = 32 * (warp + NW * i) + 16 * h;
      if (t0 + kk >= q) continue;
      gs_load_x(x, X, np, q, row, t0 + kk);
#pragma unroll
      for (int cb = 0; cb < GS_CB; ++cb) {
        if (cb >= ncb) break;
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const double2 s2 = *reinterpret_cast<const double2*>(&sq[cb][gs_tidx(kk + j)]);
          m[cb] = gs_max(m[cb], fabs(x[j] * s2.x));
          m[cb] = gs_max(m[cb], fabs(x[j + 1] * s2.y));
        }
      }
    }
  }
#pragma unroll
  for (int cb = 0; cb < GS_CB; ++cb) {
    const double o = __shfl_xor_sync(0xffffffffu, m[cb], 16);
    if (h == 0) red[warp][cb][rr] = gs_max(m[cb], o);
  }
  __syncthreads();
  if (threadIdx.x < GS_CB * GS_ROWS) {
    const int cb = threadIdx.x / GS_ROWS, i = threadIdx.x % GS_ROWS;
    double mx = 0.0;
#pragma unroll
    for (int w = 0; w < NW; ++w) mx = gs_max(mx, red[w][cb][i]);
    // 2^p m in [2^53 * 126/64, 2^54) or [2^54, 2^54 * 126/64]: the top digit stays within [-127, 127].  A row with a
    // NaN or infinite entry (a NaN, infinite or negative S_k, a non-finite X) gets the scale NaN: its row and column of
    // G are NaN and the factorisation flags the chain, as the FP64 SYRK's G would (its digits are never used).
    const bool finite = mx <= 0x1.fffffffffffffp1023;
    int p = 0;
    if (finite && mx > 0.0) {
      p = 54 - ilogb(mx);
      if (ldexp(mx, p) > 126.0 * 0x1p48) --p;
    }
    if (cb < ncb) rscale[(size_t)(c0 + cb) * np + r0 + i] = finite ? ldexp(1.0, -p) : __longlong_as_double(0x7ff8000000000000ll);
    const int p1 = p > 1000 ? 1000 : p;
    scl[cb][i] = make_double2(ldexp(1.0, p1), ldexp(1.0, p - p1));
  }

  // pass 2: the digits.  With the bias B = 128 (1 + 2^8 + ... + 2^40), byte i of N + B is D^(6-i) + 128 for i < 6 and
  // byte 6 is the top digit D^(0); (N + B) ^ (128 (1 + ... + 2^40)) holds D^(6-i) in byte i.
#if defined(GS_LAB_NO_STORES)
  unsigned sink = 0;
#endif
  for (int t0 = 0; t0 < qp; t0 += GS_TK) {
    __syncthreads();
    gs_roots(sq, Sb, qp, q, ncb, t0);
    __syncthreads();
#pragma unroll 1
    for (int i = 0; i < BPW; ++i) {
      const int kk = 32 * (warp + NW * i) + 16 * h;
      if (t0 + kk >= qp) continue;
      gs_load_x(x, X, np, q, row, t0 + kk);
#pragma unroll 1
      for (int cb = 0; cb < ncb; ++cb) {
        const double2 sc = scl[cb][rr];
        uint4 w[GI_S];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          unsigned lo[4], hi[4];
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const int j = 4 * g + b;
#if defined(GS_LAB_NO_DIGITS)
            lo[b] = __double2loint(x[j]) + j; hi[b] = __double2hiint(x[j]) + cb;
#else
            const double sqk = sq[cb][gs_tidx(kk + j)];
            const unsigned long long M = (unsigned long long)__double2ll_rn(x[j] * sqk * sc.x * sc.y) + 0x808080808080ull;
            lo[b] = (unsigned)M; hi[b] = (unsigned)(M >> 32);
#endif
          }
          // 4 x 4 byte transpose: word s holds byte (6 - s) of the 4 elements, element b in byte b
          const unsigned a0 = __byte_perm(lo[0], lo[1], 0x5140), a1 = __byte_perm(lo[0], lo[1], 0x7362);
          const unsigned a2 = __byte_perm(lo[2], lo[3], 0x5140), a3 = __byte_perm(lo[2], lo[3], 0x7362);
          const unsigned b0 = __byte_perm(hi[0], hi[1], 0x5140), b1 = __byte_perm(hi[0], hi[1], 0x7362);
          const unsigned b2 = __byte_perm(hi[2], hi[3], 0x5140), b3 = __byte_perm(hi[2], hi[3], 0x7362);
          const unsigned v[GI_S] = {__byte_perm(b1, b3, 0x5410), __byte_perm(b0, b2, 0x7632) ^ 0x80808080u,
                                    __byte_perm(b0, b2, 0x5410) ^ 0x80808080u, __byte_perm(a1, a3, 0x7632) ^ 0x80808080u,
                                    __byte_perm(a1, a3, 0x5410) ^ 0x80808080u, __byte_perm(a0, a2, 0x7632) ^ 0x80808080u,
                                    __byte_perm(a0, a2, 0x5410) ^ 0x80808080u};
#pragma unroll
          for (int s = 0; s < GI_S; ++s) (&w[s].x)[g] = v[s];
        }
        signed char* out = planes + ((size_t)(c0 + cb) * GI_S * np + row) * qp + t0 + kk;
#pragma unroll
        for (int s = 0; s < GI_S; ++s) {
#if defined(GS_LAB_NO_STORES)
          sink ^= w[s].x ^ w[s].y ^ w[s].z ^ w[s].w;
#else
          *reinterpret_cast<uint4*>(out + (size_t)s * np * qp) = w[s];
#endif
        }
      }
    }
  }
#if defined(GS_LAB_NO_STORES)
  if (sink == 0x9e3779b9u) planes[0] = 1;   // keeps the digit math live
#endif
}

__global__ void __launch_bounds__(GI_THREADS, 1)
k_gram_i8(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
          const double* __restrict__ rscale, double* __restrict__ G, int np, int nvalid, int nkb) {
  extern __shared__ __align__(1024) unsigned char gsm_raw[];
  unsigned char* gsm = reinterpret_cast<unsigned char*>(((size_t)gsm_raw + 1023) & ~(size_t)1023);
  unsigned long long* full = reinterpret_cast<unsigned long long*>(gsm + (size_t)GI_STAGES * GI_STAGE_BYTES);
  unsigned long long* empty = full + GI_STAGES;
  unsigned long long* accf = empty + GI_STAGES;
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(accf + 1);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.y;
  int ib = 0;
  while (2 * (ib + 1) * (ib + 2) / 2 <= (int)blockIdx.x) ++ib;       // row block ib holds 64-column blocks 0..2ib+1
  const int jb = (int)blockIdx.x - ib * (ib + 1);
  const int i0 = ib * GI_BM, j0 = jb * GI_BN;
  const bool diag_block = (j0 / GI_BM) == ib;
  // rows the FP64 SYRK stores: all rows of the diagonal 128-block; in a strictly lower block the 8-row fragments that
  // hold a valid row, at least 4
  int rows_st = GI_BM;
  if (!diag_block) {
    int nfv = (nvalid - i0 + 7) / 8;
    if (nfv <= 0) return;                                             // block of padding rows only: nothing stored
    rows_st = (nfv < 4 ? 4 : nfv) * 8;
  }
  if (tid == 0) {
    for (int s = 0; s < GI_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(accf, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(smem_u32(tmem_slot)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const unsigned tmem = *tmem_slot;

  if (warp == 4 && lane == 0) {
#if defined(GI_LAB_MMA_ONLY)
    for (int kb = 0; kb < GI_STAGES && kb < nkb; ++kb) {
#else
    for (int kb = 0; kb < nkb; ++kb) {
#endif
      const int st = kb % GI_STAGES;
      mbar_wait(&empty[st], ((kb / GI_STAGES) & 1) ^ 1);
      unsigned char* sa = gsm + (size_t)st * GI_STAGE_BYTES;
      mbar_expect_tx(&full[st], GI_STAGE_BYTES);
      tma_load_3d(sa, &tmA, kb * GI_BK, i0, c * GI_S, &full[st]);
      tma_load_3d(sa + GI_S * GI_A_PLANE, &tmB, kb * GI_BK, j0, c * GI_S, &full[st]);
    }
  } else if (warp == 5 && lane == 0) {
    for (int kb = 0; kb < nkb; ++kb) {
      const int st = kb % GI_STAGES;
#if defined(GI_LAB_MMA_ONLY)
      if (kb < GI_STAGES) mbar_wait(&full[st], 0);
#else
      mbar_wait(&full[st], (kb / GI_STAGES) & 1);
#endif
      asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
#if defined(GI_LAB_LOADS_ONLY)
      umma_commit(&empty[st]);
      continue;
#endif
      const unsigned sa = smem_u32(gsm + (size_t)st * GI_STAGE_BYTES), sb = sa + GI_S * GI_A_PLANE;
      // A plane s times the B planes t = 0..6-s, which lie back to back in the stage (one K-major operand of 64 (7-s)
      // rows, the same 8-row group stride) and accumulate into the adjacent columns 64 (s+t): one MMA of N = 64 (7-s),
      // cut at N = 256.  10 instructions per 32-byte k-step; only the s = 0 pair of the first k-step (all 448
      // columns) overwrites.
#pragma unroll
      for (int kk = 0; kk < GI_BK / 32; ++kk) {
#pragma unroll
        for (int s = 0; s < GI_S; ++s) {
          const unsigned long long ad = gi_desc(sa + s * GI_A_PLANE + kk * 32);
#pragma unroll
          for (int t0 = 0; t0 < GI_S - s; t0 += 4) {
            const int nt = GI_S - s - t0 < 4 ? GI_S - s - t0 : 4;
            umma_i8(tmem + (unsigned)((s + t0) * GI_BN), ad, gi_desc(sb + t0 * GI_B_PLANE + kk * 32), gi_idesc(nt * GI_BN),
                    kb > 0 || kk > 0 || s > 0);
          }
        }
      }
      umma_commit(&empty[st]);
    }
    umma_commit(accf);
  } else if (warp < 4) {
    mbar_wait(accf, 0);
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const int r = warp * 32 + lane, i = i0 + r;
    const double ri = rscale[(size_t)c * np + i] * 0x1p96;
    double* Gc = G + (size_t)c * np * np;
    const unsigned trow = tmem + ((unsigned)(warp * 32) << 16);
    for (int j8 = 0; j8 < GI_BN; j8 += 8) {
      int acc[GI_S][8];
#pragma unroll
      for (int g = 0; g < GI_S; ++g) tmem_ld8(trow + (unsigned)(g * GI_BN + j8), acc[g]);
      asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const int j = j0 + j8 + jj;
        double v = (double)acc[GI_S - 1][jj];
#pragma unroll
        for (int g = GI_S - 2; g >= 0; --g) v = (double)acc[g][jj] + v * 0x1p-8;
        v = v * ri * rscale[(size_t)c * np + j];
        if (i == j) v += 1.0;
        if (r < rows_st && (i >> 3) >= (j >> 3)) Gc[(size_t)j * np + i] = v;
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" ::"r"(tmem));
  }
}

bool gram_i8_selected(const Dims& d) { return d.gmode == 1 && d.qp >= GRAM_I8_QP_MIN && d.qp <= GRAM_I8_QP_MAX; }

size_t gram_i8_plane_bytes(const Dims& d) { return (size_t)GI_S * d.np * d.qp; }

// planes [C][7][np rows][qp] as a 3-D map {qp, np, 7 C}; a box is all 7 planes of box_rows rows x GI_BK k
static CUresult encode_planes_map(CUtensorMap* m, const signed char* planes, const Dims& d, int C, uint32_t box_rows) {
  memset(m, 0, sizeof(*m));
  const cuuint64_t dims[3] = {(cuuint64_t)d.qp, (cuuint64_t)d.np, (cuuint64_t)GI_S * C};
  const cuuint64_t strides[2] = {(cuuint64_t)d.qp, (cuuint64_t)d.qp * d.np};
  const cuuint32_t box[3] = {(cuuint32_t)GI_BK, box_rows, (cuuint32_t)GI_S};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapSwizzle sw = GI_BK == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                             : (GI_BK == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  if (!tmap_setup()) return CUDA_ERROR_NOT_SUPPORTED;
  return g_tmap_encode(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<signed char*>(planes), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// k_gram_i8 alone (the digit planes of e's chains are in place)
static void launch_gram_i8_products(const Engine& e, cudaStream_t s) {
  const Dims& d = e.d;
  CUtensorMap tmA, tmB;
  if (encode_planes_map(&tmA, e.gram_planes, d, d.C, GI_BM) != CUDA_SUCCESS ||
      encode_planes_map(&tmB, e.gram_planes, d, d.C, GI_BN) != CUDA_SUCCESS) {
    fprintf(stderr, "[bnr] cuTensorMapEncodeTiled failed for the Gram digit planes (%d x %d)\n", d.np, d.qp);
    abort();
  }
  const int T = d.np / GI_BM;
  ++g_launches; k_gram_i8<<<dim3(T * (T + 1), d.C), GI_THREADS, GI_SMEM, s>>>(tmA, tmB, e.gram_rscale, e.G, d.np, d.n,
                                                                             (d.qp + GI_BK - 1) / GI_BK);
}

// k_gram_slice: the digit planes and row scales of e's chains
static void launch_gram_slice(const Engine& e, cudaStream_t s) {
  const Dims& d = e.d;
  ++g_launches; k_gram_slice<<<dim3(d.np / GS_ROWS, (d.C + GS_CB - 1) / GS_CB), GS_THREADS, 0, s>>>(
      e.X, e.S, d.np, d.q, d.qp, d.C, e.gram_planes, e.gram_rscale);
}

static void launch_gram_i8(const Engine& e, cudaStream_t s) {
  launch_gram_slice(e, s);
  launch_gram_i8_products(e, s);
}

void launch_syrk_G(const Engine& e, cudaStream_t s) {
  const Dims& d = e.d;
  if (gram_i8_selected(d)) {
    launch_gram_i8(e, s);
    if (e.aux.G_copy) {
      dim3 g2(d.np, d.C);
      ++g_launches; k_copy_sym<<<g2, 256, 0, s>>>(e.G, (size_t)d.np * d.np, d.np, e.aux.G_copy);
    }
    return;
  }
  const int T = d.np / SY_BT;
  const int nk = d.qp / SY_BK;
  const int ns = e.syrk_ws ? e.syrk_ws_cap + 1 : 1;   // fixed per handle: chain groups must not change the summation order
  const int nk_split = (nk + ns - 1) / ns;
#if defined(SYRK_LAB_ONLY_DIAG)
  dim3 grid(d.C, ns, T);
#elif defined(SYRK_LAB_ONLY_OFFDIAG)
  dim3 grid(d.C, ns, T * (T - 1) / 2);
#else
  dim3 grid(d.C, ns, T * (T + 1) / 2);
#endif
  const size_t gs = (size_t)d.np * d.np;
  const CUtensorMap tmX = make_map(e.X, d.np, d.qp, d.np, SY_LDS);
  ++g_launches; k_gram_syrk<<<grid, SY_THREADS, SYRK_SMEM, s>>>(tmX, e.S, (size_t)d.qp, e.G, gs, d.np, d.n, nk, 1.0,
                                                            nk_split, e.syrk_ws, e.syrk_ws_cap);
  if (ns > 1) {
    dim3 g2(T * (T + 1) / 2 * 8, d.C);
    ++g_launches; k_syrk_splitk_reduce<<<g2, 256, 0, s>>>(e.G, gs, d.np, e.syrk_ws, e.syrk_ws_cap, ns - 1);
  }
  if (e.aux.G_copy) {
    dim3 g2(d.np, d.C);
    ++g_launches; k_copy_sym<<<g2, 256, 0, s>>>(e.G, gs, d.np, e.aux.G_copy);
  }
}

// ------------------------------------------------------------------------------------------------------------
// q-form of the gamma draw: P_c = (X'X + diag(1/S_c)) / tau2_c  (q x q precision of gamma - W | rest).
// X'X is computed once per handle with the same DMMA SYRK (operand = X stored row-major, K = np, unit scales).
// ------------------------------------------------------------------------------------------------------------
// XtX (lower tiles of a qp x qp column-major matrix) from XT[i * qp + j] = X(i, j) (np rows, zero padded)
void launch_xtx(const Dims& d, const double* XT, const double* ones, double* XtX, cudaStream_t s) {
  const int T = d.qp / SY_BT;
  dim3 grid(1, 1, T * (T + 1) / 2);
  const CUtensorMap tmXT = make_map(XT, d.qp, d.np, d.qp, SY_LDS);
  ++g_launches; k_gram_syrk<<<grid, SY_THREADS, SYRK_SMEM, s>>>(tmXT, ones, 0, XtX, 0, d.qp, d.q, d.np / SY_BK, 0.0,
                                                            d.np / SY_BK, nullptr, 0);
}

// P_c lower triangle from XtX, S_c, tau2_c; padding rows/columns get the identity so the factorisation stays PD.
// grid = (qp/32, qp/32, C), block = (32, 8): tile (bi, bj) with bi >= bj only.
__global__ void __launch_bounds__(256) k_build_P(Engine e) {
  const Dims& d = e.d;
  if (blockIdx.x < blockIdx.y) return;
  const int c = blockIdx.z, N = d.qp;
  const int i = blockIdx.x * 32 + threadIdx.x;
  const double it2 = 1.0 / e.tau2[c];
  double* Gc = e.G + (size_t)c * N * N;
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    const int j = blockIdx.y * 32 + threadIdx.y * 4 + jj;
    if (i < j) continue;
    double v;
    if (i < d.q) {
      v = e.XtX[(size_t)j * N + i] * it2;
      if (i == j) v = (e.XtX[(size_t)j * N + i] + 1.0 / e.S[(size_t)c * d.qp + j]) * it2;
    } else {
      v = (i == j) ? 1.0 : 0.0;
    }
    Gc[(size_t)j * N + i] = v;
  }
}

void launch_build_P(const Engine& e, cudaStream_t s) {
  const Dims& d = e.d;
  dim3 grid(d.qp / 32, d.qp / 32, d.C), block(32, 8);
  ++g_launches; k_build_P<<<grid, block, 0, s>>>(e);
  if (e.aux.G_copy) {
    dim3 g2(d.qp, d.C);
    ++g_launches; k_copy_sym<<<g2, 256, 0, s>>>(e.G, (size_t)d.qp * d.qp, d.qp, e.aux.G_copy);
  }
}

// Factor every G_c (gdim x gdim) in place; the forward solve L w = rhs rides along as row m of the matrix.
// Two schedules of the same blocked algorithm, chosen from the handle's chain count (never from the chain grouping):
//
// (A) throughput schedule -- many chains, the SMs are busy anyway and total SM time is what counts.  Left-looking, one
//     deep update per block column; per panel J:
//       k_chol_update  tile (J, J) and, on `side`, tiles (i, J), i > J: all panels 0..J-1 at once (depth 128 J)
//       k_potf2_inv    factor + invert the diagonal block                                                  [main]
//       k_trsm_dmma    tiles (i, J), i > J                                                                 [main]
//
// (B) latency schedule -- few chains (chains x (T-1) <= 128; measured crossover between 16 and 32 chains at T = 8), the GPU is mostly idle and the length of the dependent
//     chain is what counts.  Left-looking with a one-panel look-ahead; per panel J, in program order (every tile sees its
//     updates in this order on any schedule):
//       PA(J)      k_potf2_inv    D_JJ -= L[J,J-1] L[J,J-1]' (late part, in the kernel), factor, invert       [main]
//       T1(J)      k_trsm_dmma    tile (J+1, J)                                                               [main]
//       T2(J)      k_trsm_dmma    tiles (i, J), i >= J+2                                                      [side]
//       Ulate(J)   k_chol_update  tiles (i, J+1), i >= J+2, contribution of panel J only (depth 128)          [side]
//       Uearly(J)  k_chol_update  tiles (i, J+2), i >= J+2 (diagonal included), panels 0..J (depth 128 (J+1)) [side]
//     i.e. block column j receives the panels 0..j-2 early (as soon as they exist, off the critical path) and panel j-1
//     late.  The critical path per panel is PA + T1; everything else runs on `side` next to the following panel
//     factorisation.  Tiles are cut into row strips (syrk_body) while the launch stays within one wave of CTAs.
//       dependencies across the two streams:  T2(J) after PA(J);  Ulate(J) after T1(J);
//                                             T1(J+1) after Ulate(J);  PA(J+2) after Uearly(J).
// `side` is a forked branch of the graph with the priority of the main stream.
void launch_cholesky(const Engine& e, double* rhs, const ForkJoin& fj, cudaStream_t s) {
  const Dims& d = e.d;
  const int N = d.gdim;
  const int m = d.gmode == 2 ? d.q : d.n;         // first padding row = the bordering row
  const size_t cs = (size_t)N * N;
  const int T = N / PB;
  const size_t ls = (size_t)T * PB * PB;
  const bool latency = (long long)d.C_total * (T - 1) <= 128;
  ++g_launches; k_augment<<<d.C, 256, 0, s>>>(e.G, cs, N, m, rhs, d.gmode == 2 ? d.qp : d.np, d.gmode == 2 ? e.S : nullptr, e.tau2);
  // operand maps of the ring-fed kernels: the chains' matrices stacked along the k axis (chain c, column k -> k-row
  // c N + k), boxes as wide as a tile / a half / a quarter tile (+ 4 rows of padding); the stacked panel inverses
  const CUtensorMap mG = make_map(e.G, N, (uint64_t)N * d.C, N, SY_LDS);
  const CUtensorMap mG2 = make_map(e.G, N, (uint64_t)N * d.C, N, SY_BT / 2 + 4);
  const CUtensorMap mG4 = make_map(e.G, N, (uint64_t)N * d.C, N, SY_BT / 4 + 4);
  const CUtensorMap mL = make_map(e.Linv, PB, (uint64_t)PB * T * d.C, PB, SY_LDS);
  auto mI = [&](int ns) -> const CUtensorMap& { return ns == 4 ? mG4 : (ns == 2 ? mG2 : mG); };

  if (!latency) {
    // ---- (A) ----
    // The forked updates run at the panel chain's priority.  With another chain group's SYRK resident (600 us CTAs that
    // give an SM back every ~4 us) every dependent kernel has to re-acquire its SMs one by one; on the SYRK's own
    // priority level they queued behind ALL its pending CTAs and the factorisation only ran in the SYRK's last wave
    // (timeline in profiles/r02_timeline_c3.txt: 1 ms per sweep without any SYRK CTA resident).
    cudaStream_t sideA = fj.side_hi;
    for (int J = 0; J < T; ++J) {
      const bool fork = J > 0 && J + 1 < T;
      if (J > 0) {
        const int nk = J * PB / SY_BK;
        if (fork) {
          cudaEventRecord(fj.fork, s);
          cudaStreamWaitEvent(sideA, fj.fork, 0);
          dim3 g2(d.C, T - J - 1);
          ++g_launches; k_chol_update<<<g2, SY_THREADS, SYRK_SMEM, sideA>>>(mG, mG, 0, e.G, cs, N, m + 1, nk, J, J + 1, 1);
          cudaEventRecord(fj.join, sideA);
          dim3 g1(d.C, 1);
          ++g_launches; k_chol_update<<<g1, SY_THREADS, SYRK_SMEM, s>>>(mG, mG, 0, e.G, cs, N, m + 1, nk, J, J, 1);
        } else {
          dim3 g2(d.C, T - J);
          ++g_launches; k_chol_update<<<g2, SY_THREADS, SYRK_SMEM, s>>>(mG, mG, 0, e.G, cs, N, m + 1, nk, J, J, 1);
        }
      }
      ++g_launches; k_potf2_inv<<<d.C, 256, POTF2_SMEM, s>>>(e.G, cs, N, J, e.Linv, T, e.status, 0);
      if (fork) cudaStreamWaitEvent(s, fj.join, 0);
      if (J + 1 < T) {
        dim3 g1(d.C, T - J - 1);
        ++g_launches; k_trsm_dmma<<<g1, SY_THREADS, SYRK_SMEM, s>>>(mL, mG, e.G, cs, N, m + 1, J, J + 1, 1);
      }
    }
    return;
  }

  // ---- (B) ----
  cudaStream_t side = fj.side_hi;
  cudaEvent_t* evP = fj.pool;                       // [T] each: after PA, after T1, after Ulate, after Uearly
  cudaEvent_t* evT = fj.pool + T;
  cudaEvent_t* evL = fj.pool + 2 * T;
  cudaEvent_t* evE = fj.pool + 3 * T;
  // row strips per tile (see syrk_body): as many as keep the launch within one wave of CTAs
  auto strips = [&](int tiles) {
    const int ctas = d.C_total * tiles;
    return ctas * 4 <= 148 ? 4 : (ctas * 2 <= 148 ? 2 : 1);
  };
  // panel solve of `rows` row blocks from ib_first of block column J: the shared-memory-resident kernel when the tiles
  // are cut into strips (few chains), else the ring-fed one
  auto launch_trsm = [&](int J, int ib_first, int rows, int ns, cudaStream_t st) {
    dim3 g(d.C, rows * ns);
    const double* Lj = e.Linv + (size_t)J * PB * PB;
    ++g_launches;
    if (ns == 8)
      k_small_tile<2, 2><<<g, 256, small_tile_smem(16), st>>>(e.G, cs, N, J, ib_first, 8, Lj, ls, PB, J * PB, 0);
    else if (ns == 4)
      k_small_tile<2, 4><<<g, 256, small_tile_smem(32), st>>>(e.G, cs, N, J, ib_first, 4, Lj, ls, PB, J * PB, 0);
    else if (ns == 2)
      k_small_tile<2, 8><<<g, 256, small_tile_smem(64), st>>>(e.G, cs, N, J, ib_first, 2, Lj, ls, PB, J * PB, 0);
    else
      k_trsm_dmma<<<g, SY_THREADS, SYRK_SMEM, st>>>(mL, mG, e.G, cs, N, m + 1, J, ib_first, 1);
  };
  // The late part of the diagonal tile (J+1, J+1) -- the contribution of panel J -- either runs inside k_potf2_inv
  // (one SM: ~12 us of DMMA) or, when the chains are few enough for 4-8 CTAs per tile, as its own strip kernel Ud(J)
  // right after T1(J) (~5 us), with T1 itself cut into as many strips.
  // (measured: config 2 0.320 -> 0.300 ms, config 4 1.684 -> 1.666 ms; with a chain group's SYRK competing for the SMs
  //  -- 8 / 16 chains of config 3 -- the extra CTAs wait for SMs and the in-kernel update stays ahead: 1.770 vs 1.782 ms)
  const bool quiet = d.gmode == 2 || e.syrk_ws != nullptr;          // no full-size SYRK CTAs of other groups around
  const int ud = quiet ? (d.C_total * 8 <= 148 ? 8 : (d.C_total * 4 <= 148 ? 4 : 0)) : 0;
  for (int J = 0; J < T; ++J) {
    const bool has_side = J + 2 < T;
    if (J >= 2 && !ud) cudaStreamWaitEvent(s, evE[J - 2], 0);
    ++g_launches; k_potf2_inv<<<d.C, 256, POTF2_SMEM, s>>>(e.G, cs, N, J, e.Linv, T, e.status, (J > 0 && !ud) ? 1 : 0);
    if (has_side) cudaEventRecord(evP[J], s);
    if (J + 1 < T) {
      if (J >= 1) cudaStreamWaitEvent(s, evL[J - 1], 0);
      const int ns1 = ud ? ud : strips(1);
      launch_trsm(J, J + 1, 1, ns1, s);
      if (has_side) cudaEventRecord(evT[J], s);
      if (ud) {
        // Ud(J): tile (J+1, J+1) -= L[J+1, J] L[J+1, J]' (lower triangle), after the early panels 0..J-1 (Uearly(J-1))
        if (J >= 1) cudaStreamWaitEvent(s, evE[J - 1], 0);
        dim3 gd(d.C, ud);
        const double* Lt = e.G + (size_t)J * PB * N + (size_t)(J + 1) * PB;
        ++g_launches;
        if (ud == 8) k_small_tile<1, 2><<<gd, 256, small_tile_smem(16), s>>>(e.G, cs, N, J + 1, J + 1, 8, Lt, cs, N, J * PB, 1);
        else k_small_tile<1, 4><<<gd, 256, small_tile_smem(32), s>>>(e.G, cs, N, J + 1, J + 1, 4, Lt, cs, N, J * PB, 1);
      }
    }
    if (has_side) {
      const int rows = T - J - 2;                   // row blocks J+2 .. T-1
      cudaStreamWaitEvent(side, evP[J], 0);
      const int ns2 = strips(rows);
      dim3 g2(d.C, rows * ns2);
      launch_trsm(J, J + 2, rows, ns2, side);
      cudaStreamWaitEvent(side, evT[J], 0);
      ++g_launches;
      if (ns2 == 4)
        k_small_tile<1, 4><<<g2, 256, small_tile_smem(32), side>>>(e.G, cs, N, J + 1, J + 2, 4, e.G + (size_t)J * PB * N + (size_t)(J + 1) * PB, cs, N, J * PB, 0);
      else if (ns2 == 2)
        k_small_tile<1, 8><<<g2, 256, small_tile_smem(64), side>>>(e.G, cs, N, J + 1, J + 2, 2, e.G + (size_t)J * PB * N + (size_t)(J + 1) * PB, cs, N, J * PB, 0);
      else
        k_chol_update<<<g2, SY_THREADS, SYRK_SMEM, side>>>(mG, mG, J * PB, e.G, cs, N, m + 1, PB / SY_BK, J + 1, J + 2, 1);
      cudaEventRecord(evL[J], side);
      ++g_launches; k_chol_update<<<g2, SY_THREADS, SYRK_SMEM, side>>>(mG, mI(ns2), 0, e.G, cs, N, m + 1, (J + 1) * PB / SY_BK,
                                                                   J + 2, J + 2, ns2);
      cudaEventRecord(evE[J], side);
    }
  }
}

// out_c <- L_c^-T (w_c + addz_c), w = L^-1 rhs = row m of the factor (launch_cholesky)
void launch_chol_solve(const Engine& e, double* out, const double* addz, cudaStream_t s) {
  const Dims& d = e.d;
  const int N = d.gdim;
  const int m = d.gmode == 2 ? d.q : d.n;
  const int stride = d.gmode == 2 ? d.qp : d.np;
  const CUtensorMap tmG = make_map(e.G, N, (uint64_t)N * d.C, N, PB, BW_COLS);
  const CUtensorMap tmL = make_map(e.Linv, PB, (uint64_t)PB * (N / PB) * d.C, PB, PB, BW_COLS);
  if (N <= BWD_STREAM_MAX_DIM) {
    ++g_launches; k_bwd_stream<<<d.C, BW_THREADS, bwd_smem(N), s>>>(tmG, tmL, e.G, (size_t)N * N, N, m, out, stride, addz,
                                                                 stride, bwd_stages(N));
    return;
  }
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = BWC_K; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.gridDim = dim3(d.C * BWC_K);
  cfg.blockDim = dim3(BW_THREADS);
  cfg.dynamicSmemBytes = bwc_smem(N);
  cfg.stream = s;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ++g_launches;
  cudaLaunchKernelEx(&cfg, k_bwd_cluster, tmG, tmL, (const double*)e.G, (size_t)N * N, N, m, out, stride, addz, stride,
                     bwc_stages(N));
}

// clusters of the back solve that can be resident at once for factored dimension N (0: the cluster cannot be placed,
// < 0: the query failed); N <= BWD_STREAM_MAX_DIM runs the one-CTA kernel, which needs no check
int bwd_cluster_capacity(int N) {
  if (N <= BWD_STREAM_MAX_DIM) return 1;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = BWC_K; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.gridDim = dim3(BWC_K);
  cfg.blockDim = dim3(BW_THREADS);
  cfg.dynamicSmemBytes = bwc_smem(N);
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, k_bwd_cluster, &cfg) != cudaSuccess) return -1;
  return n;
}

int chol_max_dim() { return CHOL_MAX_DIM; }
int bwd_stream_max_dim() { return BWD_STREAM_MAX_DIM; }

}  // namespace bnr
