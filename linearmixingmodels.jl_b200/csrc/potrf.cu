// Diagonal-tile factorisation: the panel step (dpotf2) of the blocked Cholesky (K6), fused with
// logdet accumulation (K7), non-PD detection and the triangular inverse W = inv(L_JJ) that turns
// every panel TRSM and every triangular vector solve into tensor-core GEMMs / plain GEMVs.
// One CTA (8 warps) per latent; the 128x128 tile lives in shared memory, column-major with
// ld = 132 (conflict-free DMMA fragment loads: column stride = 8 banks).
//
// potrf_tile_body (below): left-looking column updates inside the tile, reciprocal pivot chain, W built beside the panel
// steps.  Two kernels run it: potrf_tile_kernel2 (one launch per tile column) and chain_column_kernel, which fuses the
// whole per-column panel chain of a small-batch factorisation -- TRSM of column J, update of column J+1, diagonal tile
// J+1 -- into one launch whose CTAs hand tiles to each other through ready counters in global memory.
// Latency-bound by design (it sits on the critical path of each tile column; the host runs
// several latent groups on separate streams so the other SMs keep doing trailing updates).
#include "common.cuh"
#include "kernels.h"
#include "direct_gemm.cuh"

namespace lmm {

#ifdef LMM_POTRF_TIMING
__device__ long long g_potrf_clk[16];
__device__ long long g_potrf_acc[8];  // per-step sums: [0] column update, [1] panel (warp 0), [2] its wait at the step barrier, [3] W block row (warp 4)
#define PT(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_potrf_clk[k] = clock64(); } while (0)
#define ACC_DECL long long acc_t0 = 0
#define ACC_START(tidsel) do { if (blockIdx.x == 0 && threadIdx.x == (tidsel)) acc_t0 = clock64(); } while (0)
#define ACC_STOP(tidsel, k) do { if (blockIdx.x == 0 && threadIdx.x == (tidsel)) g_potrf_acc[k] += clock64() - acc_t0; } while (0)
#else
#define PT(k) do { } while (0)
#define ACC_DECL do { } while (0)
#define ACC_START(tidsel) do { } while (0)
#define ACC_STOP(tidsel, k) do { } while (0)
#endif

constexpr int LD = 132;
constexpr size_t POTRF_SMEM = (size_t)(TILE * LD + 2 * TILE + 32) * sizeof(double);

// 1/sqrt(x) for x > 0 in the normal range: MUFU.RSQ64H seed + two Newton-Raphson steps.  Measured on B200
// (tools/microbench/rsqrt_check.cu, max relative error over 2e7 arguments): seed 9.2e-7, one step 1.3e-12, two steps
// 2.7e-16, three steps 2.6e-16 -- the third step bought nothing and sat on the pivot chain (128 x 2 dependent FMAs).
// Non-positive / NaN pivots are reported separately by the caller: no special cases on the critical path.
__device__ __forceinline__ double fast_rsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double hx = 0.5 * x;
  double e = fma(-hx * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-hx * y, y, 0.5);
  y = fma(y, e, y);
  return y;
}

__device__ __forceinline__ void dmma884p(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1},{%2},{%3},{%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------------------------------------------
// The diagonal-tile factorisation.  Compared with a right-looking tile kernel with the inverse after the factor (round 1's
// first generation: 47 us) it needs about two thirds of the cycles:
//   * LEFT-looking inside the tile.  The first kernel's right-looking trailing update re-reads and re-writes every 8x8
//     block of the tile once per panel step (6 loads + 2 stores per pair of DMMAs: shared-memory-bandwidth bound, a third
//     of its cycles); here the column block about to be factored is brought up to date in one go,
//     C(bi, bj) -= sum_{k<bj} L(bi, k) L(bj, k)^T, accumulators in registers, 3 loads per pair of DMMAs, one
//     read-modify-write per block, by all 8 warps (two blocks of the column per warp sharing the B fragments);
//   * the pivot chain of each 8x8 diagonal block runs on reciprocals (LDL^T style): next pivot = fma(-u^2, 1/piv, d),
//     one MUFU.RCP64H + 3 dependent FMAs + 1 per column; the rsqrt that scales the stored column is computed beside the
//     chain, not on it.  The row owners of the diagonal block take the common path (no divergent branch on the critical
//     warp) and the non-positive-pivot report leaves the pivot loop;
//   * the two 64x64 diagonal halves of W are built one block row at a time, by warps 4-7, WHILE warps 0-3 run the
//     (row-owner, 128-thread) panel step of the next 8 columns:  W_ii = inv(L_ii),  W_ij = -W_ii * sum_{k=j}^{i-1} L_ik W_kj
//     needs only rows of L that are already final, and restricted to its own half a block row costs less than a panel
//     step.  W lives transposed in the free upper triangle of the tile (W(r,c) at S[r*LD+c], its diagonal in dinv[]),
//     so L stays intact underneath.  The off-diagonal half W21 = -W22 (L21 W11) follows the last panel step as two fully
//     unrolled DMMA stages on all 8 warps;
//   * tile load and both stores move 16 B per thread-access.
// Measured (tools/microbench/potrf_phases.cu, B200): 47.1 us -> 36.9 us per tile (profiles/r01_panel_chain.md).
__device__ __forceinline__ double fast_rcp(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double e = fma(-x, y, 1.0);  // seed is good to ~2^-20 (tools/microbench/rsqrt_check.cu); cubic step -> 2^-60
  return fma(y, fma(e, e, e), y);
}
__device__ __forceinline__ void named_bar(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// element (rr, cc) of the lower-triangular 8x8 block W_oo in the mirrored storage
__device__ __forceinline__ double wdiag(const double* S, const double* dinv, int o, int rr, int cc) {
  double v = 0.0;
  if (rr > cc) v = S[(o + rr) * LD + o + cc];
  if (rr == cc) v = dinv[o + rr];
  return v;
}

// Block row i of W restricted to the block columns [jmin, i), by `nw` warps (this warp = wl) sharing the named barrier
// `bar_id`.  Deliberately light on the FP64 pipe (one block at a time per warp, two accumulator chains): the pipe is
// shared with the panel warps, whose dependent chain is the critical path -- denser DMMA issue here was measured to slow
// the whole step down.
__device__ __forceinline__ void w_block_row(double* S, const double* dinv, int i, int jmin, int wl, int nw, int lane, int bar_id) {
  const int g = lane >> 2, t = lane & 3, o = 8 * i;
  if (wl == nw - 1 && lane < 8) {  // W_ii by substitution, one thread per column
    double Lb[8][8], w[8];
    const int col = lane;
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int k = 0; k < a; ++k) Lb[a][k] = S[(o + k) * LD + o + a];
#pragma unroll
    for (int rr = 0; rr < 8; ++rr) {
      double s = (rr == col) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < rr; ++k) s = fma(-Lb[rr][k], w[k], s);
      w[rr] = s * dinv[o + rr];
    }
#pragma unroll
    for (int rr = 1; rr < 8; ++rr)
      if (rr > col) S[(o + rr) * LD + o + col] = w[rr];
  }
  __syncwarp();
  // T_j = sum_{k=j}^{i-1} L_ik W_kj, parked where W_ij will live
  for (int j = jmin + wl; j < i; j += nw) {
    const int oj = 8 * j;
    double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0;
    {
      const double a0 = S[(oj + t) * LD + o + g];
      const double a1 = S[(oj + 4 + t) * LD + o + g];
      const double b0 = wdiag(S, dinv, oj, t, g);
      const double b1 = wdiag(S, dinv, oj, 4 + t, g);
      dmma884p(c0, c1, a0, b0);
      dmma884p(e0, e1, a1, b1);
    }
    for (int k = j + 1; k < i; ++k) {
      const int ok = 8 * k;
      const double a0 = S[(ok + t) * LD + o + g];
      const double a1 = S[(ok + 4 + t) * LD + o + g];
      const double b0 = S[(ok + t) * LD + oj + g];
      const double b1 = S[(ok + 4 + t) * LD + oj + g];
      dmma884p(c0, c1, a0, b0);
      dmma884p(e0, e1, a1, b1);
    }
    S[(o + g) * LD + oj + 2 * t] = c0 + e0;
    S[(o + g) * LD + oj + 2 * t + 1] = c1 + e1;
  }
  named_bar(bar_id, nw * 32);  // W_ii (and every T_j) visible to the warps of this group
  const double wa0 = wdiag(S, dinv, o, g, t);
  const double wa1 = wdiag(S, dinv, o, g, 4 + t);
  for (int j = jmin + wl; j < i; j += nw) {
    const int oj = 8 * j;
    double c0 = 0.0, c1 = 0.0;
    const double b0 = S[(o + t) * LD + oj + g];
    const double b1 = S[(o + 4 + t) * LD + oj + g];
    dmma884p(c0, c1, wa0, b0);
    dmma884p(c0, c1, wa1, b1);
    __syncwarp();  // every lane has read T_j before it is overwritten
    S[(o + g) * LD + oj + 2 * t] = -c0;
    S[(o + g) * LD + oj + 2 * t + 1] = -c1;
  }
}

// The off-diagonal half of W once both 64x64 diagonal halves are inverted: W21 = -W22 (L21 W11), 8 warps, everything
// unrolled (no branches between the loads and the DMMAs: this phase has the pipe to itself and is meant to fill it).
//   stage A: warp w owns block row i = 8 + w:    T_ij = sum_{k=j}^{7} L_ik W_kj      (A fragments shared along the row)
//   stage B: warp w owns block column j = w:     W_ij = -sum_{k=8}^{i} W_ik T_kj     (B fragments shared along the column)
__device__ __forceinline__ void w_lower_left(double* S, const double* dinv, int warp, int lane) {
  const int g = lane >> 2, t = lane & 3;
  {
    const int o = 64 + 8 * warp;
    double c0[8], c1[8], e0[8], e1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) c0[j] = c1[j] = e0[j] = e1[j] = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int ok = 8 * k;
      const double a0 = S[(ok + t) * LD + o + g];
      const double a1 = S[(ok + 4 + t) * LD + o + g];
#pragma unroll
      for (int j = 0; j <= k; ++j) {
        const int oj = 8 * j;
        double b0, b1;
        if (j == k) {
          b0 = wdiag(S, dinv, oj, t, g);
          b1 = wdiag(S, dinv, oj, 4 + t, g);
        } else {
          b0 = S[(ok + t) * LD + oj + g];
          b1 = S[(ok + 4 + t) * LD + oj + g];
        }
        dmma884p(c0[j], c1[j], a0, b0);
        dmma884p(e0[j], e1[j], a1, b1);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      S[(o + g) * LD + 8 * j + 2 * t] = c0[j] + e0[j];
      S[(o + g) * LD + 8 * j + 2 * t + 1] = c1[j] + e1[j];
    }
  }
  __syncthreads();
  {
    const int oj = 8 * warp;
    double c0[8], c1[8], e0[8], e1[8];
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) c0[ii] = c1[ii] = e0[ii] = e1[ii] = 0.0;
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      const int ok = 64 + 8 * kk;
      const double b0 = S[(ok + t) * LD + oj + g];
      const double b1 = S[(ok + 4 + t) * LD + oj + g];
#pragma unroll
      for (int ii = kk; ii < 8; ++ii) {
        const int o = 64 + 8 * ii;
        double a0, a1;
        if (ii == kk) {
          a0 = wdiag(S, dinv, o, g, t);
          a1 = wdiag(S, dinv, o, g, 4 + t);
        } else {
          a0 = S[(o + g) * LD + ok + t];
          a1 = S[(o + g) * LD + ok + 4 + t];
        }
        dmma884p(c0[ii], c1[ii], a0, b0);
        dmma884p(e0[ii], e1[ii], a1, b1);
      }
    }
    __syncthreads();  // every T block has been read by every warp that needs it
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      const int o = 64 + 8 * ii;
      S[(o + g) * LD + oj + 2 * t] = -(c0[ii] + e0[ii]);
      S[(o + g) * LD + oj + 2 * t + 1] = -(c1[ii] + e1[ii]);
    }
  }
}

// tile: diagonal tile (J,J) in HBM (factored in place); Wt: where W(J) goes; S: POTRF_SMEM bytes of dynamic shared memory;
// fail_col_p: one shared int.  logdet_b / info_b: this latent's accumulators.  The caller has made the tile's latest
// contents visible (stream order, griddepcontrol.wait or a ready counter) before calling.
__device__ __forceinline__ void potrf_tile_body(double* __restrict__ tile, double* __restrict__ Wt, int J, double* __restrict__ logdet_b,
                                                int* __restrict__ info_b, double* S, int* fail_col_p) {
  double* dinv = S + TILE * LD;               // 1 / L[r][r] = W[r][r];  S[c*LD + r]: L in the lower triangle, W^T strictly above
  double* red = dinv + TILE;
  int& fail_col = *fail_col_p;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;

  PT(0);
  if (tid == 0) fail_col = 0x7fffffff;
#pragma unroll 16
  for (int e2 = tid; e2 < TT / 2; e2 += 256) {
    const double2 v = __ldcg(reinterpret_cast<const double2*>(tile) + e2);  // L2: in the fused chain kernel other SMs wrote it in this launch
    int r, c;
    tile_rc(2 * e2, r, c);
    S[c * LD + r] = v.x;
    S[(c + 1) * LD + r] = v.y;
  }
  __syncthreads();

  PT(1);
  ACC_DECL;
  for (int j0 = 0; j0 < TILE; j0 += 8) {
    const int bj = j0 >> 3;
    ACC_START(0);
    if (bj > 0) {
      // left-looking update of column block bj: block rows bi0 = bj + warp and bi0 + 8.  A dependent DMMA costs ~100
      // cycles, so chain length is what matters: a warp with two blocks runs 4 chains of bj DMMAs; a warp with one block
      // (always the case once bj >= 8, when the chains are longest) splits k in two halves, 4 chains of bj/2.
      const int bi0 = bj + warp;
      if (bi0 < 16) {
        const bool two = bi0 + 8 < 16;
        const int R0 = 8 * bi0, R1 = two ? R0 + 64 : R0;
        const int trips = two ? bj : (bj + 1) >> 1;
        const int koff = two ? 0 : 8 * trips;  // column offset of the second pair of chains
        const int klast = 8 * (bj - 1);
        double p0 = 0.0, p1 = 0.0, q0 = 0.0, q1 = 0.0;  // block 0 (first half of k)
        double u0 = 0.0, u1 = 0.0, v0 = 0.0, v1 = 0.0;  // block 1, or block 0's second half of k
        // fragments of trip k + 1 are in flight while the DMMAs of trip k issue
        int c2 = koff < klast ? koff : klast;
        double bb0 = S[t * LD + j0 + g], bb1 = S[(4 + t) * LD + j0 + g];
        double a00 = S[t * LD + R0 + g], a01 = S[(4 + t) * LD + R0 + g];
        double bb2 = S[(c2 + t) * LD + j0 + g], bb3 = S[(c2 + 4 + t) * LD + j0 + g];
        double a10 = S[(c2 + t) * LD + R1 + g], a11 = S[(c2 + 4 + t) * LD + R1 + g];
        for (int k = 0; k < trips; ++k) {
          const int cn = 8 * (k + 1 < trips ? k + 1 : k);
          const int c2n = cn + koff < klast ? cn + koff : klast;
          const double nb0 = S[(cn + t) * LD + j0 + g];
          const double nb1 = S[(cn + 4 + t) * LD + j0 + g];
          const double n00 = S[(cn + t) * LD + R0 + g];
          const double n01 = S[(cn + 4 + t) * LD + R0 + g];
          const double nb2 = S[(c2n + t) * LD + j0 + g];
          const double nb3 = S[(c2n + 4 + t) * LD + j0 + g];
          const double n10 = S[(c2n + t) * LD + R1 + g];
          const double n11 = S[(c2n + 4 + t) * LD + R1 + g];
          dmma884p(p0, p1, a00, bb0);
          dmma884p(q0, q1, a01, bb1);
          if (two || 8 * k + koff <= klast) {  // warp-uniform; false only for the odd trip out of a split k range
            dmma884p(u0, u1, a10, bb2);
            dmma884p(v0, v1, a11, bb3);
          }
          bb0 = nb0; bb1 = nb1; a00 = n00; a01 = n01;
          bb2 = nb2; bb3 = nb3; a10 = n10; a11 = n11;
        }
        double* c0p = &S[(j0 + 2 * t) * LD + R0 + g];
        if (two) {
          c0p[0] -= p0 + q0;
          c0p[LD] -= p1 + q1;
          double* c1p = &S[(j0 + 2 * t) * LD + R1 + g];
          c1p[0] -= u0 + v0;
          c1p[LD] -= u1 + v1;
        } else {
          c0p[0] -= (p0 + q0) + (u0 + v0);
          c0p[LD] -= (p1 + q1) + (u1 + v1);
        }
      }
      __syncthreads();  // the column block is up to date for its row owners
    }
    ACC_STOP(0, 0);
    if (j0 == 8) PT(2);
    ACC_START(0);
    ACC_START(128);
    if (warp < 4) {
      const int r = tid;  // row owner
      double p[8];
      double d[8][8];
      const bool active = r >= j0;
      if (active) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int k = 0; k <= i; ++k) d[i][k] = S[(j0 + k) * LD + (j0 + i)];
#pragma unroll
        for (int k = 0; k < 8; ++k) p[k] = S[(j0 + k) * LD + r];
      }
      named_bar(1, 128);  // every row owner has read the diagonal block before its rows are overwritten
      if (active) {
        double dv[8], tm[8][8];
        int failj = 8;
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const double piv = d[jj][jj];
          if (!(piv > 0.0) && failj == 8) failj = jj;
          const double rc = fast_rcp(piv);
          dv[jj] = fast_rsqrt(piv);
#pragma unroll
          for (int j2 = jj + 1; j2 < 8; ++j2) {
            d[j2][j2] = fma(-(d[j2][jj] * d[j2][jj]), rc, d[j2][j2]);  // the pivot chain: one FMA behind the reciprocal
            tm[j2][jj] = d[j2][jj] * rc;
#pragma unroll
            for (int i = j2 + 1; i < 8; ++i) d[i][j2] = fma(-d[i][jj], tm[j2][jj], d[i][j2]);
          }
        }
        // every row, the 8 rows of the diagonal block included (their entries right of the diagonal are never stored):
        // u_j = a_j - sum_{k<j} u_k (u_jk / piv_k),  L_rj = u_j / sqrt(piv_j)
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          double v = p[jj];
#pragma unroll
          for (int k = 0; k < jj; ++k) v = fma(-p[k], tm[jj][k], v);
          p[jj] = v;
        }
        const int within = r - j0;  // >= 8 below the diagonal block
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k <= within) S[(j0 + k) * LD + r] = p[k] * dv[k];
        if (r == j0) {
#pragma unroll
          for (int k = 0; k < 8; ++k) dinv[j0 + k] = dv[k];
          if (failj < 8) atomicMin(&fail_col, j0 + failj);
        }
      }
    } else if (j0 > 0) {
      w_block_row(S, dinv, bj - 1, bj - 1 < 8 ? 0 : 8, warp - 4, 4, lane, 2);
    }
    ACC_STOP(0, 1);
    ACC_STOP(128, 3);
    ACC_START(0);
    __syncthreads();
    ACC_STOP(0, 2);
    if (j0 == 8) PT(3);
  }
  PT(4);
  w_block_row(S, dinv, 15, 8, warp, 8, lane, 0);  // ends the inversion of the lower-right 64x64 half
  w_lower_left(S, dinv, warp, lane);

  if (tid < TILE) {
    double v = log(S[tid * LD + tid]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp] = v;
  }
  __syncthreads();
  PT(5);
  if (tid == 0) {
    *logdet_b += 2.0 * (((red[0] + red[1]) + red[2]) + red[3]);
    if (fail_col != 0x7fffffff && *info_b == 0) *info_b = J * TILE + fail_col + 1;
  }
  PT(6);
  pdl_trigger();  // the column's TRSM may be scheduled while L and W are stored
  PT(7);
#pragma unroll 8
  for (int e2 = tid; e2 < TT / 2; e2 += 256) {
    int r, c;
    tile_rc(2 * e2, r, c);
    double2 l, w;
    l.x = (r >= c) ? S[c * LD + r] : 0.0;
    l.y = (r >= c + 1) ? S[(c + 1) * LD + r] : 0.0;
    const double2 wt = *reinterpret_cast<const double2*>(&S[r * LD + c]);  // 16-byte aligned: LD and c are even
    w.x = (r > c) ? wt.x : (r == c ? dinv[r] : 0.0);
    w.y = (r > c + 1) ? wt.y : (r == c + 1 ? dinv[r] : 0.0);
    reinterpret_cast<double2*>(tile)[e2] = l;
    reinterpret_cast<double2*>(Wt)[e2] = w;
  }
  PT(8);
  PT(9);
}

__global__ void __launch_bounds__(256, 1) potrf_tile_kernel2(TiledSym L, double* __restrict__ Wbase, size_t w_batch_stride, int J,
                                                             double* __restrict__ logdet, int* __restrict__ info) {
  extern __shared__ __align__(16) double S[];
  __shared__ int fail_col;
  const int b = blockIdx.x;
  pdl_wait();  // the tile was written by the previous kernel of the panel chain
  potrf_tile_body(L.tile(b, J, J), Wbase + (size_t)b * w_batch_stride + (size_t)J * TT, J, logdet + b, info + b, S, &fail_col);
}

cudaError_t launch_potrf_tile(cudaStream_t st, TiledSym L, double* W, size_t w_batch_stride, int J, int batch, double* logdet,
                              int* info) {
  static bool configured_dev[64] = {false};  // function attributes are per device
  int dev = 0;
  cudaGetDevice(&dev);
  bool& configured = configured_dev[dev & 63];
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(potrf_tile_kernel2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POTRF_SMEM);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  return launch_pdl(pdl_enabled(), potrf_tile_kernel2, dim3(batch), dim3(256), POTRF_SMEM, st, L, W, w_batch_stride, J, logdet, info);
}

// ---------------------------------------------------------------------------------------------------------------------
// The per-column panel chain of a small-batch factorisation in ONE launch (VERDICT r01 next #4).
// For tile column J (already factored: L(J,J), W(J) final), per latent b:
//     role T, CTA (I, s):     L(I,J)[slice s]    = C(I,J)[slice s] W(J)'                             I in (J, nt)
//     role U, CTA (I, c, s):  C(I,c)[slice s]   -= sum_{k in [k0, J]} L(I,k)[slice s] L(c,k)'        c in (J, c_end), I in [c, nt)
//     role P, one CTA:        factor C(J+1,J+1) -> L(J+1,J+1), W(J+1), logdet, info                  (do_potrf)
// instead of three (or more) dependent launches.  [k0, J] is the k-tile range the columns (J, c_end) still have to receive
// on the panel stream (k0 = first column of the current block; earlier columns were applied by the trailing updates);
// c_end = J + 2 inside a block (just the next column), the end of the NEXT block at a block boundary.
// Dependencies inside the launch run through counters in global memory (the 8 slice CTAs of a tile add 1 each): U(I, c, .)
// needs the tiles (I,J) and (c,J) of role T -- but only for its LAST k-tile, the k < J part runs before it looks at a
// counter --, P needs the 8 slices of U(J+1, J+1, .).  Block order = priority order = dependency order: the 8 slices of
// T(J+1), the 8 slices of U(J+1,J+1), P -- the critical path gets the first 17 block indices and P then keeps one SM for
// its ~30 us while everything else streams through the others --, then the T slices of the rows below, then the remaining U
// slices; the latent index is the FASTEST grid dimension, so that order holds across the batch.  Consumers only wait for
// CTAs with a lower linear block index, which are dispatched first; a bounded wait traps instead of hanging the GPU.
// What leaves the critical path: the launch boundaries potrf -> TRSM -> update -> potrf, and every TRSM / update tile below
// row J+1 (they now run beside the diagonal-tile factorisation instead of in front of it).
// Counters: cnt[b][J * nt + I] for role T, cnt[b][nt * nt + J + 1] for the diagonal tile of role U; zeroed once per
// factorisation (every column uses its own entries).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int ld_acquire_cnt(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void wait_count(const int* p, int target) {
  if (threadIdx.x == 0) {
    if (ld_acquire_cnt(p) < target) {
      unsigned long long t0, t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      unsigned ns = 32;
      while (ld_acquire_cnt(p) < target) {
        __nanosleep(ns);
        if (ns < 256) ns <<= 1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > 10000000000ull) __trap();
      }
    }
    __threadfence();
  }
  __syncthreads();
}
__device__ __forceinline__ void signal_count(int* p) {
  __syncthreads();  // every thread's stores of this slice are issued
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(p, 1);
  }
}

struct ChainArgs {
  TiledSym L;
  double* W;
  size_t w_batch_stride;
  double* logdet;
  int* info;
  int* cnt;           // [batch][nt * nt + nt + 1]
  int J, k0, c_end, do_potrf;
  const int* env;     // nullable: tile envelope [batch][nt] (tiles (I, k < env[I]) are exact zeros that may not be stored)
};

// grid (batch, 8 * (nT + nU) + (do_potrf ? 1 : 0)), 256 threads, POTRF_SMEM bytes of dynamic shared memory.
__global__ void __launch_bounds__(256, 1) chain_column_kernel(ChainArgs a) {
  extern __shared__ __align__(16) double S[];
  __shared__ int fail_col;
  const int nt = a.L.nt, J = a.J, b = blockIdx.x, warp = threadIdx.x >> 5;
  const int nT = nt - 1 - J;  // tiles of role T (rows J+1 .. nt-1)
  int* cnt = a.cnt + (size_t)b * ((size_t)nt * nt + nt + 1);
  const int np = a.do_potrf ? 1 : 0;
  const bool has_u = a.c_end > J + 1;
  int bid = blockIdx.y, role, I, c = J + 1, slice;  // role 0 = T, 1 = U, 2 = P
  if (bid < DIRECT_SPLIT) {
    role = 0; I = J + 1; slice = bid;
  } else if (has_u && bid < 2 * DIRECT_SPLIT) {
    role = 1; I = J + 1; slice = bid - DIRECT_SPLIT;
  } else if (bid < (has_u ? 2 : 1) * DIRECT_SPLIT + np) {
    role = 2; I = J + 1; slice = 0;
  } else {
    bid -= (has_u ? 2 : 1) * DIRECT_SPLIT + np;
    const int rest = (nT - 1) * DIRECT_SPLIT;
    if (bid < rest) {
      role = 0; I = J + 2 + bid / DIRECT_SPLIT; slice = bid % DIRECT_SPLIT;
    } else {
      role = 1;
      bid -= rest;
      int u = bid / DIRECT_SPLIT;
      slice = bid % DIRECT_SPLIT;
      int rows_c = nt - (J + 2);  // column J+1 without its diagonal tile
      while (u >= rows_c) {
        u -= rows_c;
        ++c;
        rows_c = nt - c;
      }
      I = (c == J + 1) ? J + 2 + u : c + u;
    }
  }
  pdl_wait();  // column J (and the trailing updates ordered before this launch) are complete and visible
  const int* eb = a.env ? a.env + (size_t)b * nt : nullptr;
  if (role == 0) {
    // ---- role T: TRSM of one slice of tile (I, J)
    if (eb && eb[I] > J) {  // a zero tile stays zero (and is not read: it may not be stored)
      signal_count(cnt + (size_t)J * nt + I);
      return;
    }
    double* Ctile = a.L.tile(b, I, J);
    int nb0, nb1, lim0, nsteps;
    direct_blocks<GEMM_TRSM>(warp, 1, nb0, nb1, lim0, nsteps);
    double acc[DIRECT_RB][2][2] = {};
    double2 cv[DIRECT_RB][2] = {};
    direct_accumulate<GEMM_TRSM>(Ctile, a.W + (size_t)b * a.w_batch_stride + (size_t)J * TT, slice, nb0, nb1, lim0, nsteps, acc);
    __syncthreads();  // every warp of this CTA has finished reading its rows of C(I,J)
    direct_store_c<GEMM_TRSM>(Ctile, slice, nb0, nb1, cv, acc);
    signal_count(cnt + (size_t)J * nt + I);
    return;
  }
  if (role == 1) {
    // ---- role U: update of one slice of tile (I, c) by the k-tiles [k0, J]
    // below max(env[I], env[c]) one operand is an exact zero (gemm_first_k): the sum starts there, bit for bit the full one
    const int kb = eb ? max(a.k0, max(eb[I], eb[c])) : a.k0;
    if (kb > J) {  // nothing to subtract: C(I,c) stays as it is
      if (I == J + 1 && c == J + 1) signal_count(cnt + (size_t)nt * nt + J + 1);
      return;
    }
    double* Ctile = a.L.tile(b, I, c);
    int nb0 = warp * 2, nb1 = warp * 2 + 1, lim0, nsteps;
    double acc[DIRECT_RB][2][2] = {};
    double2 cv[DIRECT_RB][2];
    direct_load_c(Ctile, slice, nb0, nb1, cv);
    if (kb < J) {  // the columns of this block before J: final before this launch
      direct_blocks<GEMM_UPDATE>(warp, J - kb, nb0, nb1, lim0, nsteps);
      direct_accumulate<GEMM_UPDATE>(a.L.tile(b, I, kb), a.L.tile(b, c, kb), slice, nb0, nb1, lim0, nsteps, acc);
    }
    // k = J: produced by role T of this launch -- all 8 slices of the B operand's tile (c, J) and of the A operand's tile (I, J)
    wait_count(cnt + (size_t)J * nt + c, DIRECT_SPLIT);
    if (I != c) wait_count(cnt + (size_t)J * nt + I, DIRECT_SPLIT);
    direct_blocks<GEMM_UPDATE>(warp, 1, nb0, nb1, lim0, nsteps);
    direct_accumulate<GEMM_UPDATE>(a.L.tile(b, I, J), a.L.tile(b, c, J), slice, nb0, nb1, lim0, nsteps, acc);
    direct_store_c<GEMM_UPDATE>(Ctile, slice, nb0, nb1, cv, acc);
    if (I == J + 1 && c == J + 1) signal_count(cnt + (size_t)nt * nt + J + 1);
    return;
  }
  // ---- role P: the next diagonal tile
  if (has_u) wait_count(cnt + (size_t)nt * nt + J + 1, DIRECT_SPLIT);
  potrf_tile_body(a.L.tile(b, J + 1, J + 1), a.W + (size_t)b * a.w_batch_stride + (size_t)(J + 1) * TT, J + 1, a.logdet + b, a.info + b, S,
                  &fail_col);
}

size_t chain_counter_ints(int nt) { return (size_t)nt * nt + nt + 1; }

// One launch for tile column J: TRSM of the column, update of the columns (J, c_end) by the k-tiles [k0, J], and (do_potrf)
// the factorisation of diagonal tile J+1.  c_end <= J + 1: no update (then do_potrf must be 0: the diagonal tile would not
// be up to date).
cudaError_t launch_chain_column(cudaStream_t st, TiledSym L, double* W, size_t w_batch_stride, int J, int k0, int c_end, int do_potrf,
                                int batch, double* logdet, int* info, int* counters, const int* env) {
  static bool configured_dev[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  bool& configured = configured_dev[dev & 63];
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(chain_column_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POTRF_SMEM);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  const int nt = L.nt, nT = nt - 1 - J;
  if (nT <= 0 || batch <= 0) return cudaSuccess;
  if (c_end > nt) c_end = nt;
  if (c_end <= J + 1) {
    c_end = J + 1;
    do_potrf = 0;
  }
  long long nU = 0;
  for (int c = J + 1; c < c_end; ++c) nU += nt - c;
  ChainArgs a{L, W, w_batch_stride, logdet, info, counters, J, k0, c_end, do_potrf, env};
  dim3 grid((unsigned)batch, (unsigned)((nT + nU) * DIRECT_SPLIT + (do_potrf ? 1 : 0)));
  return launch_pdl(pdl_enabled(), chain_column_kernel, grid, dim3(256), POTRF_SMEM, st, a);
}

}  // namespace lmm
