// FP64 tensor-core (DMMA) tile GEMM: the trailing update / panel solve of the batched blocked
// Cholesky (K6) and of the posterior TRSM (K10).  Replaces the dsyrk/dgemm/dtrsm calls LAPACK
// dpotrf makes under `cholesky(Symmetric(C))` (reference call site src/oilmm.jl:90,128 via
// AbstractGPs).
//
//   UPDATE: C(I,J) -= sum_{k in [k0,k1)} A(I,k) * B(J,k)^T        (128x128 tiles, K = 128 per k)
//   TRSM  : C(I,J)  = C(I,J) * W(J)^T        with W(J) = inv(L(J,J)) (lower triangular)
//
// gemm_tile_kernel_v2: one CTA = one 128x128 output tile, 8 warps as 2(M) x 4(N), warp tile 64x32 = 8x4 m8n8k4 DMMA
// fragments (64 accumulator doubles / thread).  Operands arrive by TMA bulk copies (cp.async.bulk -> SASS UBLKCP): one
// elected thread issues two 32 KB copies per 32-column k-stage into a 3-stage / 192 KB ring; copies complete on `full`
// mbarriers, the consumer warps release stages through `empty` mbarriers -- no CTA-wide barrier in the main loop.  Chunks of
// consecutive k-tiles are contiguous in HBM (row-panel-major tile order) and the k4-interleaved tile layout makes every
// fragment load a conflict-free 256 B warp access (see common.cuh).
// gemm_direct2_kernel (direct_gemm.cuh): latency-optimised variant for the small grids of a panel chain -- no shared
// memory, a tile split into 8 row slices (8 SMs per tile), fragments straight from L2 through a register ring.
// Bound: FP64 tensor pipe (64 FMA/clk/SM): 2*128^3 flop per k-tile per CTA vs 256 KB of L2->SM
// traffic -> 16 flop/B, far above the L2 balance; HBM traffic is lower still (row panels are
// shared through L2 by the CTAs of one tile row / column).  ncu (profiles/r02_ncu_summary.json): DMMA pipe active 97 % of
// the cycles, 95.9 % of the FP64 tensor peak over elapsed time on the wide trailing update.
#include "common.cuh"
#include "kernels.h"
#include "direct_gemm.cuh"
#include "ozaki_slice.cuh"

namespace lmm {

constexpr int CHUNK = 2048;  // doubles per operand per 16 k-columns (128 rows x 16 k)

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1},{%2},{%3},{%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// ------------------------------------------------------------------------------------------------
// TMA bulk copies + full/empty mbarrier ring, no CTA-wide barrier in the main loop.
// One elected thread (warp 0, lane 0) is the producer on the side: per 16-column k-chunk it issues
// two 16 KB cp.async.bulk copies (SASS UBLKCP) that complete on the stage's `full` mbarrier; each
// of the 8 consumer warps waits on `full`, runs its 128 DMMAs and arrives on the stage's `empty`
// mbarrier.  Warps therefore drift apart by up to a few chunks, so one warp's chunk-boundary bubble
// (barrier wait + first LDS latency) is covered by the other warp of its SM sub-partition.
// ------------------------------------------------------------------------------------------------
// KC = k-columns per stage (16 or 32); the ring always holds 96 columns of A and of B (192 KB).
constexpr size_t GEMM_V2_SMEM = (size_t)6 * 2 * CHUNK * sizeof(double) + 2 * 6 * sizeof(uint64_t);

__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mb_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s_u32(bar)) : "memory");
}
__device__ __forceinline__ void mb_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  uint32_t spins = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(s_u32(bar)), "r"(parity)
        : "memory");
    if (!done && ++spins > (1u << 28)) __trap();  // never hang the GPU on a protocol bug
  }
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(s_u32(dst)), "l"(src),
               "r"(bytes), "r"(s_u32(bar))
               : "memory");
}

// SLICE (TRSM only): after storing the finished tile, the CTA copies it into the freed stage ring (128 of the 192 KB, tile layout)
// and writes its int8 digit planes from there (oz_slice_tile), for tile rows I >= sl.i0: one read of the tile from HBM and one
// launch per column fewer than a separate ozaki_slice_kernel pass.
template <int MODE, int KC, bool SLICE = false>
__global__ void __launch_bounds__(256, 1) gemm_tile_kernel_v2(GemmArgs g, TrsmSliceArgs sl) {
  constexpr int V2_STAGES = 96 / KC;
  constexpr int SCHUNK = 128 * KC;  // doubles per operand per stage
  extern __shared__ __align__(128) double smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)6 * 2 * CHUNK);
  uint64_t* empty = full + V2_STAGES;
  const int J = g.j0 + blockIdx.x, I = g.i0 + blockIdx.y * (g.row_step > 0 ? g.row_step : 1), b = blockIdx.z;
  if (g.sym && I < J) return;
  if (g.upper && I > J) return;
  if (MODE == GEMM_TRSM && g.env && g.env[(size_t)b * g.env_stride + I] > J) return;  // a zero tile stays zero
  const int kb = gemm_first_k(g, I, J, b);  // first k-tile of this CTA
  if (MODE == GEMM_UPDATE && kb >= g.k1) return;

  double* Ctile = g.C.tile(b, I, J);
  const double* Asrc;
  const double* Bsrc;
  int nchunks;
  if (MODE == GEMM_UPDATE) {
    Asrc = g.A.tile(b, I, kb);
    Bsrc = g.B.tile(b, J, kb);
    nchunks = (g.k1 - kb) * (128 / KC);
  } else {
    Asrc = Ctile;
    Bsrc = g.W + (size_t)b * g.w_batch_stride + (size_t)J * TT;
    nchunks = 128 / KC;
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp & 1, wn = warp >> 1;
  constexpr uint32_t CHUNK_BYTES = SCHUNK * sizeof(double);

  if (tid == 0) {
    for (int s = 0; s < V2_STAGES; ++s) {
      mb_init(&full[s], 1);
      mb_init(&empty[s], 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  auto produce = [&](int q) {
    const int s = q % V2_STAGES;
    double* sa = smem + (size_t)s * (2 * SCHUNK);
    mb_expect_tx(&full[s], 2 * CHUNK_BYTES);
    bulk_load(sa, Asrc + (size_t)q * SCHUNK, CHUNK_BYTES, &full[s]);
    bulk_load(sa + SCHUNK, Bsrc + (size_t)q * SCHUNK, CHUNK_BYTES, &full[s]);
  };
  if (tid == 0) {
    const int pre = nchunks < V2_STAGES ? nchunks : V2_STAGES;
    for (int q = 0; q < pre; ++q) produce(q);
  }

  // Accumulators: 64 doubles per thread in both modes.  UPDATE: warps 2(M) x 4(N), warp tile 64 x 32 = acc[8][4].  TRSM:
  // W(J) is LOWER triangular, so output column block nb only needs the k-blocks <= nb -- a 2 x 4 warp grid would leave the
  // warps of the low column groups idle, so the TRSM uses 8(M) x 1(N) warps, warp tile 16 x 128 = acc[2][16] (the same
  // storage, viewed differently), and every warp skips the same zero blocks: 120 of 256 block products.
  // UPDATE starts its accumulators from C(I,J) and feeds NEGATED B fragments (one sign flip per fragment, 4 per 32 DMMAs),
  // so the tile's read latency hides behind the first TMA stage and the epilogue is a store: the CTA retires -- and the
  // SM's next tile starts -- one L2/HBM round trip earlier than with a read-modify-write at the end.
  const int g4 = lane >> 2, t4 = lane & 3;
  double acc[8][4][2];
  if constexpr (MODE == GEMM_UPDATE) {
#pragma unroll
    for (int mb = 0; mb < 8; ++mb)
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) {
        const int cg = wn * 8 + nb * 2 + (t4 >> 1);
        const int off = (cg << 9) + ((wm * 8 + mb) << 5) + (g4 << 2) + ((t4 & 1) << 1);
        const double2 v = *reinterpret_cast<const double2*>(Ctile + off);
        acc[mb][nb][0] = v.x;
        acc[mb][nb][1] = v.y;
      }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  }
  double (*acct)[16][2] = reinterpret_cast<double (*)[16][2]>(&acc[0][0][0]);  // TRSM view: [2][16][2]

  for (int q = 0; q < nchunks; ++q) {
    const int s = q % V2_STAGES;
    mb_wait(&full[s], (uint32_t)((q / V2_STAGES) & 1));
    if constexpr (MODE == GEMM_TRSM) {
      const double* sa = smem + (size_t)s * (2 * SCHUNK) + (warp * 2) * 32 + lane;
      const double* sb = smem + (size_t)s * (2 * SCHUNK) + SCHUNK + lane;
#pragma unroll
      for (int ks = 0; ks < KC / 4; ++ks) {
        const int kb8 = (q * (KC / 4) + ks) >> 1;  // the 8-column block of W this k4-step belongs to
        const double a0 = sa[ks * 512], a1 = sa[ks * 512 + 32];
#pragma unroll
        for (int nb = 0; nb < 16; ++nb)
          if (nb >= kb8) {  // warp-uniform: W(n, k) = 0 for k > n
            const double bq = sb[ks * 512 + nb * 32];
            dmma884(acct[0][nb][0], acct[0][nb][1], a0, bq);
            dmma884(acct[1][nb][0], acct[1][nb][1], a1, bq);
          }
      }
    } else {
      const double* sa = smem + (size_t)s * (2 * SCHUNK) + (wm * 8) * 32 + lane;
      const double* sb = smem + (size_t)s * (2 * SCHUNK) + SCHUNK + (wn * 4) * 32 + lane;
#pragma unroll
      for (int ks = 0; ks < KC / 4; ++ks) {
        double a[8], bq[4];
#pragma unroll
        for (int mb = 0; mb < 8; ++mb) a[mb] = sa[ks * 512 + mb * 32];
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) bq[nb] = -sb[ks * 512 + nb * 32];
#pragma unroll
        for (int mb = 0; mb < 8; ++mb)
#pragma unroll
          for (int nb = 0; nb < 4; ++nb) dmma884(acc[mb][nb][0], acc[mb][nb][1], a[mb], bq[nb]);
      }
    }
    __syncwarp();
    if (lane == 0) mb_arrive(&empty[s]);
    // producer duty: refill the stage consumed one iteration ago (its readers had a whole chunk
    // of time to finish, so this wait is normally already satisfied)
    if (tid == 0 && q >= 1) {
      const int qn = q - 1 + V2_STAGES;
      if (qn < nchunks) {
        mb_wait(&empty[(q - 1) % V2_STAGES], (uint32_t)(((q - 1) / V2_STAGES) & 1));
        produce(qn);
      }
    }
  }

  if constexpr (MODE == GEMM_TRSM) {
    // in place: the whole tile C(I,J) went through the stage ring above (every chunk consumed by every warp), so a CTA
    // barrier is all that separates the last read from the first write
    __syncthreads();
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int nb = 0; nb < 16; ++nb) {
        const int cg = nb * 2 + (t4 >> 1);
        const int off = (cg << 9) + ((warp * 2 + mb) << 5) + (g4 << 2) + ((t4 & 1) << 1);
        double2 v;
        v.x = acct[mb][nb][0];
        v.y = acct[mb][nb][1];
        *reinterpret_cast<double2*>(Ctile + off) = v;
        if constexpr (SLICE) *reinterpret_cast<double2*>(smem + off) = v;
      }
    if constexpr (SLICE) {
      if (I >= sl.i0) {
        __syncthreads();
        oz_slice_tile(smem, sl.scale + (size_t)b * sl.scale_stride + (size_t)I * TILE,
                      sl.slices + (size_t)b * sl.slice_stride + sym_tile_index(I, J) * ((size_t)sl.S * 16384), sl.S, sl.bits,
                      sl.fp ? sl.fp + (size_t)b * sl.fp_stride + sym_tile_index(I, J) : nullptr);
      }
    }
  } else {
#pragma unroll
    for (int mb = 0; mb < 8; ++mb) {
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) {
        const int cg = wn * 8 + nb * 2 + (t4 >> 1);
        const int off = (cg << 9) + ((wm * 8 + mb) << 5) + (g4 << 2) + ((t4 & 1) << 1);
        double2 v;
        v.x = acc[mb][nb][0];
        v.y = acc[mb][nb][1];
        *reinterpret_cast<double2*>(Ctile + off) = v;
      }
    }
  }
}

static int g_gemm_small = 74;  // grids of at most this many tiles take the latency-optimised kernel (0 = never)
void set_gemm_small_threshold(int tiles) { g_gemm_small = tiles; }
bool gemm_takes_direct(long long tiles) { return tiles <= g_gemm_small; }

static bool g_pdl = true;   // programmatic dependent launch along the panel chain (direct kernels + diagonal-tile kernel)
void set_pdl(int v) { g_pdl = v != 0; }
bool pdl_enabled() { return g_pdl; }

static cudaError_t configure_v2() {
  static bool configured_dev[64] = {false};  // function attributes are per device
  int dev = 0;
  cudaGetDevice(&dev);
  bool& configured = configured_dev[dev & 63];
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tile_kernel_v2<GEMM_UPDATE, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_V2_SMEM);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(gemm_tile_kernel_v2<GEMM_TRSM, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_V2_SMEM);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(gemm_tile_kernel_v2<GEMM_TRSM, 32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_V2_SMEM);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  return cudaSuccess;
}

cudaError_t launch_gemm(cudaStream_t st, int mode, const GemmArgs& a, int ncols, int nrows, int batch, long long select_tiles) {
  if (ncols <= 0 || nrows <= 0 || batch <= 0) return cudaSuccess;
  cudaError_t e = configure_v2();
  if (e != cudaSuccess) return e;
  if (gemm_takes_direct(select_tiles > 0 ? select_tiles : (long long)ncols * nrows * batch)) {
    dim3 gs((unsigned)ncols * DIRECT_SPLIT, (unsigned)nrows, (unsigned)batch);
    if (mode == GEMM_UPDATE) return launch_pdl(g_pdl, gemm_direct2_kernel<GEMM_UPDATE>, gs, dim3(256), 0, st, a);
    return launch_pdl(g_pdl, gemm_direct2_kernel<GEMM_TRSM>, gs, dim3(256), 0, st, a);
  }
  dim3 grid((unsigned)ncols, (unsigned)nrows, (unsigned)batch);
  if (mode == GEMM_UPDATE)
    gemm_tile_kernel_v2<GEMM_UPDATE, 32><<<grid, 256, GEMM_V2_SMEM, st>>>(a, TrsmSliceArgs{});
  else
    gemm_tile_kernel_v2<GEMM_TRSM, 32><<<grid, 256, GEMM_V2_SMEM, st>>>(a, TrsmSliceArgs{});
  return cudaGetLastError();
}

cudaError_t launch_trsm_slice(cudaStream_t st, const GemmArgs& a, int nrows, int batch, const TrsmSliceArgs& s) {
  if (nrows <= 0 || batch <= 0) return cudaSuccess;
  cudaError_t e = configure_v2();
  if (e != cudaSuccess) return e;
  gemm_tile_kernel_v2<GEMM_TRSM, 32, true><<<dim3(1u, (unsigned)nrows, (unsigned)batch), 256, GEMM_V2_SMEM, st>>>(a, s);
  return cudaGetLastError();
}

}  // namespace lmm
