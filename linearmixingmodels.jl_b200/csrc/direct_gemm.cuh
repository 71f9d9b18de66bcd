// Latency-optimised "direct" tile GEMM for SMALL grids -- the panel chain of a batch-1 / partitioned / small-N factorisation:
// a handful of tiles whose 17 us per k-tile on one SM would sit on the critical path.  One 128x128 tile is split into
// DIRECT_SPLIT = 8 row slices of 16 rows, one CTA each (8 SMs per tile); no shared memory at all: in the k4-interleaved tile
// layout every m8n8k4 fragment is 32 contiguous doubles in lane order, so each warp loads its A / B fragments with coalesced
// 256-byte accesses straight from L2 (the 8 warps of a CTA share the A rows through L1) through a register ring that keeps
// the next DIRECT_PF k4-steps in flight.  UPDATE: warp w owns column blocks 2w, 2w+1.  TRSM: the zero blocks of the
// lower-triangular W(J) are skipped -- warp w owns column blocks w and 15-w, i.e. 2(w+1) + 2(16-w) = 34 of 64 block-steps.
// TRSM is in place: a CTA only reads its own rows of C(I,J), and a CTA barrier separates its last read from its first write.
//
// The pieces are device functions so that two kernels share them: gemm_direct2_kernel (one operation per launch, chained by
// programmatic dependent launch) and chain_column_kernel (potrf.cu: TRSM of a column + update of the next column + its
// diagonal-tile factorisation in ONE launch, tiles chained through ready counters in global memory).
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace lmm {

constexpr int DIRECT_RB = 2;                   // 8-row blocks per slice
constexpr int DIRECT_SPLIT = 16 / DIRECT_RB;   // slices (CTAs) per tile
constexpr int DIRECT_PF = 8;                   // k4-steps of operand fragments in flight

__device__ __forceinline__ void dmma884d(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1},{%2},{%3},{%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// First k-tile of the UPDATE of tile (I, J) of latent b: k0, or I (k_from_row: A(I,k) = 0 for k < I), or the later of the two
// rows' envelopes -- every product skipped below it has an all-zero operand, so the sums are those of the full range.
__device__ __forceinline__ int gemm_first_k(const GemmArgs& g, int I, int J, int b) {
  int kb = (g.k_from_row && I > g.k0) ? I : g.k0;
  if (g.env) {
    const int* e = g.env + (size_t)b * g.env_stride;
    kb = max(kb, max(e[I], e[J]));
  }
  return kb;
}

// Which column blocks a warp owns, and for how many k4-steps each is non-zero.
template <int MODE>
__device__ __forceinline__ void direct_blocks(int warp, int ktiles, int& nb0, int& nb1, int& lim0, int& nsteps) {
  if (MODE == GEMM_UPDATE) {
    nb0 = warp * 2;
    nb1 = warp * 2 + 1;
    nsteps = ktiles * 32;
    lim0 = nsteps;
  } else {
    nb0 = warp;  // W^T block (k8, nb) is zero for k8 > nb: column block nb needs the k4-steps q < 2 (nb + 1)
    nb1 = 15 - warp;
    lim0 = 2 * (nb0 + 1);
    nsteps = 2 * (nb1 + 1);
  }
}

// acc[i][j] += sum over `nsteps` k4-steps of A(slice rows, k) * B(column blocks nb0 / nb1, k)^T.  Asrc / Bsrc point at the
// first k-tile (consecutive k-tiles of a row panel are contiguous).  nsteps is even; lim0 <= nsteps bounds block nb0 (TRSM).
template <int MODE>
__device__ __forceinline__ void direct_accumulate(const double* __restrict__ Asrc, const double* __restrict__ Bsrc, int slice, int nb0, int nb1,
                                                  int lim0, int nsteps, double (&acc)[DIRECT_RB][2][2]) {
  constexpr int RB = DIRECT_RB, PF = DIRECT_PF;
  const int lane = threadIdx.x & 31;
  const double* pa = Asrc + (slice * RB) * 32 + lane;
  const double* pb0 = Bsrc + nb0 * 32 + lane;
  const double* pb1 = Bsrc + nb1 * 32 + lane;
  double ra[PF][RB], rb[PF][2];
#pragma unroll
  for (int u = 0; u < PF; ++u) {
    const int q = u < nsteps ? u : nsteps - 1;
#pragma unroll
    for (int i = 0; i < RB; ++i) ra[u][i] = pa[(size_t)q * 512 + i * 32];
    rb[u][0] = pb0[(size_t)q * 512];
    rb[u][1] = pb1[(size_t)q * 512];
  }
  for (int q0 = 0; q0 < nsteps; q0 += PF) {  // PF steps per trip, the tail of the last trip is predicated off
#pragma unroll
    for (int u = 0; u < PF; ++u) {
      const int q = q0 + u;
      double a[RB], bq[2];
#pragma unroll
      for (int i = 0; i < RB; ++i) a[i] = ra[u][i];
      bq[0] = rb[u][0];
      bq[1] = rb[u][1];
      const int qn = (q + PF < nsteps) ? q + PF : nsteps - 1;
#pragma unroll
      for (int i = 0; i < RB; ++i) ra[u][i] = pa[(size_t)qn * 512 + i * 32];
      rb[u][0] = pb0[(size_t)qn * 512];
      rb[u][1] = pb1[(size_t)qn * 512];
      if (q < nsteps) {
        if (MODE == GEMM_UPDATE || q < lim0) {
#pragma unroll
          for (int i = 0; i < RB; ++i) dmma884d(acc[i][0][0], acc[i][0][1], a[i], bq[0]);
        }
#pragma unroll
        for (int i = 0; i < RB; ++i) dmma884d(acc[i][1][0], acc[i][1][1], a[i], bq[1]);
      }
    }
  }
}

// Offset (in doubles) of this lane's 16-byte piece of the C fragment (row block slice*RB + i, column block nb).
__device__ __forceinline__ int direct_c_offset(int slice, int i, int nb) {
  const int lane = threadIdx.x & 31, g4 = lane >> 2, t4 = lane & 3;
  const int cg = nb * 2 + (t4 >> 1);
  return (cg << 9) + ((slice * DIRECT_RB + i) << 5) + (g4 << 2) + ((t4 & 1) << 1);
}

__device__ __forceinline__ void direct_load_c(const double* Ctile, int slice, int nb0, int nb1, double2 (&cv)[DIRECT_RB][2]) {
#pragma unroll
  for (int i = 0; i < DIRECT_RB; ++i) {
    cv[i][0] = *reinterpret_cast<const double2*>(Ctile + direct_c_offset(slice, i, nb0));
    cv[i][1] = *reinterpret_cast<const double2*>(Ctile + direct_c_offset(slice, i, nb1));
  }
}

// UPDATE: C = cv - acc;  TRSM: C = acc (callers put a CTA barrier between the last read of C(I,J) and this store).
template <int MODE>
__device__ __forceinline__ void direct_store_c(double* Ctile, int slice, int nb0, int nb1, const double2 (&cv)[DIRECT_RB][2],
                                               const double (&acc)[DIRECT_RB][2][2]) {
#pragma unroll
  for (int i = 0; i < DIRECT_RB; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      double2 v;
      if (MODE == GEMM_UPDATE) {
        v = cv[i][j];
        v.x -= acc[i][j][0];
        v.y -= acc[i][j][1];
      } else {
        v.x = acc[i][j][0];
        v.y = acc[i][j][1];
      }
      *reinterpret_cast<double2*>(Ctile + direct_c_offset(slice, i, j == 0 ? nb0 : nb1)) = v;
    }
}

// grid (ncols * DIRECT_SPLIT, nrows, batch), 256 threads, no shared memory.
template <int MODE>
__global__ void __launch_bounds__(256) gemm_direct2_kernel(GemmArgs g) {
  const int J = g.j0 + (int)(blockIdx.x / DIRECT_SPLIT), slice = (int)(blockIdx.x % DIRECT_SPLIT);
  const int I = g.i0 + blockIdx.y * (g.row_step > 0 ? g.row_step : 1), b = blockIdx.z;
  if (g.sym && I < J) return;
  if (g.upper && I > J) return;
  if (MODE == GEMM_TRSM && g.env && g.env[(size_t)b * g.env_stride + I] > J) return;  // a zero tile stays zero
  const int kb = gemm_first_k(g, I, J, b);
  if (MODE == GEMM_UPDATE && kb >= g.k1) return;
  double* Ctile = g.C.tile(b, I, J);
  const int warp = threadIdx.x >> 5;
  pdl_wait();  // everything below reads what the previous kernel of the panel chain wrote
  const double* Asrc = MODE == GEMM_UPDATE ? g.A.tile(b, I, kb) : Ctile;
  const double* Bsrc = MODE == GEMM_UPDATE ? g.B.tile(b, J, kb) : g.W + (size_t)b * g.w_batch_stride + (size_t)J * TT;
  int nb0, nb1, lim0, nsteps;
  direct_blocks<MODE>(warp, g.k1 - kb, nb0, nb1, lim0, nsteps);
  double acc[DIRECT_RB][2][2];
#pragma unroll
  for (int i = 0; i < DIRECT_RB; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  double2 cv[DIRECT_RB][2];  // UPDATE: the C fragments travel with the first operand fragments, not after the last DMMA
  if (MODE == GEMM_UPDATE) direct_load_c(Ctile, slice, nb0, nb1, cv);
  direct_accumulate<MODE>(Asrc, Bsrc, slice, nb0, nb1, lim0, nsteps, acc);
  pdl_trigger();  // the next kernel of the chain may be scheduled while this one stores
  if (MODE == GEMM_TRSM) __syncthreads();  // every warp of this CTA has finished reading its rows of C(I,J)
  direct_store_c<MODE>(Ctile, slice, nb0, nb1, cv, acc);
}

}  // namespace lmm
