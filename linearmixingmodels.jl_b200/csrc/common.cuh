// Shared definitions for liblmm (sm_100a only).
//
// HBM layout of a symmetric / lower-triangular N x N matrix ("TiledSym"): N is padded to
// nt*128; only tiles (I, J) with I >= J are stored, row-panel-major: tile (I, J) lives at
// ((I*(I+1))/2 + J) * 16384 doubles, so the row panel L[I, 0:J] a trailing update streams is ONE
// contiguous run of HBM.  Inside a 128x128 tile elements are "k4-interleaved":
//     elem(r, c) = (c/4)*512 + (r/8)*32 + (r%8)*4 + (c%4)
// i.e. every (8 rows x 4 cols) block is 32 contiguous doubles in exactly the lane order of the
// FP64 tensor-core fragment of mma.m8n8k4 (lane = (r%8)*4 + c%4) for BOTH the A operand (rows of
// tile (I,k)) and the B operand (rows of tile (J,k), used transposed).  A 16-column k-chunk of a
// tile is one contiguous 16 KB run, fragment loads from shared memory are conflict-free 256 B
// warp accesses without any swizzle, and the accumulator fragment maps to 16 B stores.
// Rectangular operands ("TiledRect", e.g. K(x*, x) rows) use the same tiles, row-major by tile.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lmm {

constexpr int TILE = 128;
constexpr int TT = TILE * TILE;  // doubles per tile

__host__ __device__ __forceinline__ int tile_elem(int r, int c) {
  return ((c >> 2) << 9) + ((r >> 3) << 5) + ((r & 7) << 2) + (c & 3);
}
// inverse: offset e in [0, 16384) -> (r, c)
__host__ __device__ __forceinline__ void tile_rc(int e, int& r, int& c) {
  r = (((e >> 5) & 15) << 3) + ((e >> 2) & 7);
  c = ((e >> 9) << 2) + (e & 3);
}
__host__ __device__ __forceinline__ size_t sym_tile_index(int I, int J) {
  return (size_t)I * (size_t)(I + 1) / 2 + (size_t)J;
}
__host__ __device__ __forceinline__ size_t sym_tiles(int nt) { return (size_t)nt * (size_t)(nt + 1) / 2; }

// Tiles of the rows a rank owns in a row-cyclic partition (rank r of G owns the tile rows I = r, r + G, ...): row
// I = r + l*G holds its I + 1 tiles contiguously at l*(r+1) + G*l*(l-1)/2 (the rows before it hold r+1, r+G+1, ... tiles).
__host__ __device__ __forceinline__ size_t cyc_tile_index(int I, int J, int G, int r) {
  const size_t l = (size_t)((I - r) / G);
  return l * (size_t)(r + 1) + (size_t)G * (l * (l - 1) / 2) + (size_t)J;
}
__host__ __device__ __forceinline__ size_t cyc_tiles(int nrows, int G, int r) {  // tiles of the rows < nrows rank r owns
  if (nrows <= r) return 0;
  const int cnt = (nrows - 1 - r) / G + 1;
  return cyc_tile_index(r + cnt * G, 0, G, r);
}

struct TiledSym {
  double* base;
  int nt;
  size_t batch_stride;  // doubles
  // Two alternative tile addressings of the partitioned (distributed-storage) factorisation, batch 1; all 0 = packed lower:
  //   ntc > 0:   a rectangular WINDOW of the matrix, tile (I, J) at ((I - row0) * ntc + (J - col0)) -- the block column a
  //              panel is factored in; every kernel that takes a TiledSym (diagonal tile, fused chain) then works on it
  //   cyc_G > 0: only the tile rows I = cyc_r (mod cyc_G) exist, packed as cyc_tile_index says
  int ntc = 0, row0 = 0, col0 = 0;
  int cyc_G = 0, cyc_r = 0;
  __host__ __device__ __forceinline__ double* tile(int b, int I, int J) const {
    size_t idx;
    if (ntc) idx = (size_t)(I - row0) * (size_t)ntc + (size_t)(J - col0);
    else if (cyc_G) idx = cyc_tile_index(I, J, cyc_G, cyc_r);
    else idx = sym_tile_index(I, J);
    return base + (size_t)b * batch_stride + idx * TT;
  }
};

struct TiledRect {
  double* base;
  int ntr, ntc;
  size_t batch_stride;  // doubles
  __host__ __device__ __forceinline__ double* tile(int b, int R, int J) const {
    return base + (size_t)b * batch_stride + ((size_t)R * ntc + J) * TT;
  }
};

// Per-latent kernel parameters on the device.
constexpr int MAX_ARD = 8;    // == LMM_MAX_ARD of include/lmm.h
constexpr int MAX_TERMS = 4;  // == LMM_MAX_TERMS
// One further term of a composite (sum / product) kernel.
struct TermParams {
  int kind;
  int ard_dim;
  double variance;
  double inv_ls;
  double param;
  double ard[MAX_ARD];
};
struct LatentParams {
  int kind;
  int ard_dim;  // 0: isotropic ScaleTransform only; D (<= MAX_ARD): inputs are also multiplied by ard[0..D) (ARDTransform)
  double variance;
  double inv_ls;
  double noise;  // added on the diagonal (ΣT_i for OILMM, σ² for IndependentMOGP)
  double mean;
  double param;  // α of the RationalQuadraticKernel, r of the PeriodicKernel
  double ard[MAX_ARD];
  // composite kernels: nterms = 1 (plain kernel: everything above) .. MAX_TERMS; compose 1 = sum, 2 = product over term 0
  // (the fields above) and extra[0 .. nterms-2]; kdiag = k(x, x) of the whole kernel (= variance for a plain kernel)
  int nterms;
  int compose;
  double kdiag;
  TermParams extra[MAX_TERMS - 1];
};
// Multiplier of input dimension k: KernelFunctions `k ∘ ScaleTransform(s)` / `k ∘ ARDTransform(v)` scale the inputs
// BEFORE pairwise distances are taken.  p points at global memory (no dynamically indexed register copy).
__device__ __forceinline__ double input_scale(const LatentParams* p, int k) { return p->ard_dim ? p->inv_ls * p->ard[k] : p->inv_ls; }

// exp(x) for x <= 0, <= 1 ulp (checked against expl on 2e7 points, tools/microbench/exp_check.c): Cody-Waite
// reduction x = n ln2 + r with the round-to-nearest shift trick, degree-11 near-minimax polynomial on |r| <= ln2/2
// (Chebyshev-interpolated in 60-digit arithmetic, max relative error 2.4e-17), 2^n applied to the exponent field.
// 16 FP64-pipe instructions instead of the ~35 of the library exp(): the kernel-matrix builders evaluate one exp
// per stored element, and on B200 that -- not the 8-byte store -- was what bounded them.  Results below
// 2^-1021 (x < -708) are flushed to 0.
__device__ __forceinline__ double exp_nonpos(double x) {
  if (x < -708.0) return 0.0;
  const double t = fma(x, 1.4426950408889634074, 6755399441055744.0);  // low word of t = round(x log2 e)
  const int n = __double2loint(t);
  const double nf = t - 6755399441055744.0;
  double r = fma(nf, -6.93147180369123816490e-01, x);
  r = fma(nf, -1.90821492927058770002e-10, r);
  double p = 0x1.af4134720f354p-26;
  p = fma(p, r, 0x1.289876a2dbdc0p-22);
  p = fma(p, r, 0x1.71de0a0471800p-19);
  p = fma(p, r, 0x1.a019b31890abfp-16);
  p = fma(p, r, 0x1.a01a01a8ba744p-13);
  p = fma(p, r, 0x1.6c16c17a1c437p-10);
  p = fma(p, r, 0x1.1111111110871p-7);
  p = fma(p, r, 0x1.555555555394cp-5);
  p = fma(p, r, 0x1.5555555555556p-3);
  p = fma(p, r, 0x1.0000000000001p-1);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  return __hiloint2double(__double2hiint(p) + (n << 20), __double2loint(p));
}

// κ(d²)·variance -- KernelFunctions kappa for SE / Matern32 / Matern52 (SURVEY.md App. A.3).
__device__ __forceinline__ double kappa_eval(int kind, double variance, double d2, double param = 1.0) {
  // far-apart pairs (most of a kernel matrix whose inputs span many lengthscales) underflow to exactly 0.0
  double v;
  if (kind == 0) {
    v = exp_nonpos(-0.5 * d2);
  } else if (kind == 4) {
    v = pow(1.0 + d2 / (2.0 * param), -param);  // RationalQuadraticKernel(α)
  } else {
    double d = sqrt(d2);
    if (kind == 1) {
      double s = 1.7320508075688772 * d;  // sqrt(3)
      v = (1.0 + s) * exp_nonpos(-s);
    } else if (kind == 2) {
      double s = 2.23606797749979 * d;  // sqrt(5)
      v = (1.0 + s + (d * d) * 1.6666666666666667) * exp_nonpos(-s);
    } else {
      v = exp_nonpos(-d);  // ExponentialKernel = Matern12Kernel
    }
  }
  return variance * v;
}
// kappa_eval(kind, variance, d2) is exactly 0 for every d2 > kappa_zero_d2(kind) and finite variance: exp_nonpos flushes below
// -708, and the Matern prefactors stay finite.  The thresholds carry a 2^-40 relative guard for the rounded sqrt and the rounded
// products by sqrt(3) / sqrt(5) in front of the exp.  +inf for the kinds that never give an exact 0 (RationalQuadratic).
__host__ __device__ __forceinline__ double kappa_zero_d2(int kind) {
  const double g = 1.0 + 0x1p-40;
  switch (kind) {
    case 0: return 1416.0 * g;                                                          // SE: exp(-d²/2)
    case 1: return (708.0 / 1.7320508075688772) * (708.0 / 1.7320508075688772) * g;  // Matern32: exp(-√3 d)
    case 2: return (708.0 / 2.23606797749979) * (708.0 / 2.23606797749979) * g;      // Matern52: exp(-√5 d)
    case 3: return 708.0 * 708.0 * g;                                                   // Matern12: exp(-d)
    default: return __builtin_huge_val();
  }
}

// Squared distance of scaled points.  form 0: Distances.jl pairwise (|a|²+|b|² - 2 a·b, clamped at
// 0); form 1: direct differences.  a, b point at D scaled coordinates.
__device__ __forceinline__ double sqdist(const double* a, const double* b, int D, double sa, double sb, int form) {
  if (form == 0) {
    double dot = 0.0;
    for (int k = 0; k < D; ++k) dot = fma(a[k], b[k], dot);
    double t = sa + sb;
    double d2 = t - 2.0 * dot;
    return d2 > 0.0 ? d2 : 0.0;
  }
  double d2 = 0.0;
  for (int k = 0; k < D; ++k) {
    double df = a[k] - b[k];
    d2 = fma(df, df, d2);
  }
  return d2;
}

// Squared distance of one (Sq)Euclidean term on RAW points a, b: the term's own input scaling, then the Distances.jl form
// (form 0) or direct differences (form 1).  Shared by the value path (term_value) and the per-term gradient (grad.cu).
__device__ __forceinline__ double term_sqdist(int ard_dim, double inv_ls, const double* ard, const double* a, const double* b, int D,
                                              int form) {
  double d2;
  if (form == 0) {
    double sa = 0.0, sb = 0.0, dot = 0.0;
    for (int k = 0; k < D; ++k) {
      const double sc = ard_dim ? inv_ls * ard[k] : inv_ls;
      const double ak = sc * a[k], bk = sc * b[k];
      sa = fma(ak, ak, sa);
      sb = fma(bk, bk, sb);
      dot = (D == 1) ? ak * bk : fma(ak, bk, dot);  // D = 1: one rounded product, as the single-kernel fast path and a K = 1 GEMM do
    }
    d2 = fma(-2.0, dot, sa + sb);
    d2 = d2 > 0.0 ? d2 : 0.0;
  } else {
    d2 = 0.0;
    for (int k = 0; k < D; ++k) {
      const double sc = ard_dim ? inv_ls * ard[k] : inv_ls;
      const double df = sc * a[k] - sc * b[k];
      d2 = fma(df, df, d2);
    }
  }
  return d2;
}

// One term of a kernel on RAW (unscaled) points a, b (D coordinates each): the term's own input scaling, its own pairwise
// distance (Distances.jl form or direct differences; the PeriodicKernel's Sinus metric always works on differences), κ,
// variance.  This is what KernelFunctions evaluates per component of a KernelSum / KernelProduct.
__device__ __forceinline__ double term_value(int kind, int ard_dim, double variance, double inv_ls, double param, const double* ard,
                                             const double* a, const double* b, int D, int form, bool same_point) {
  if (same_point) return variance;  // d = 0 exactly on the diagonal (Distances.jl), κ(0) = 1 for every supported kernel
  if (kind == 5) {  // PeriodicKernel(r): Sinus(r) metric = Σ (sinpi(a_k - b_k) / r)², κ = exp(-d/2)
    double d = 0.0;
    for (int k = 0; k < D; ++k) {
      const double sc = ard_dim ? inv_ls * ard[k] : inv_ls;
      const double sn = sinpi(sc * a[k] - sc * b[k]) / param;
      d = fma(sn, sn, d);
    }
    return variance * exp_nonpos(-0.5 * d);
  }
  return kappa_eval(kind, variance, term_sqdist(ard_dim, inv_ls, ard, a, b, D, form), param);
}
// Value of a (possibly composite) latent kernel on raw points; gp points at global memory.
__device__ __forceinline__ double kernel_value_raw(const LatentParams* gp, const double* a, const double* b, int D, int form, bool same_point) {
  double v = term_value(gp->kind, gp->ard_dim, gp->variance, gp->inv_ls, gp->param, gp->ard, a, b, D, form, same_point);
  for (int t = 1; t < gp->nterms; ++t) {
    const TermParams* q = &gp->extra[t - 1];
    const double w = term_value(q->kind, q->ard_dim, q->variance, q->inv_ls, q->param, q->ard, a, b, D, form, same_point);
    v = (gp->compose == 2) ? v * w : v + w;
  }
  return v;
}
// true if the latent needs the raw-point path (composite, or a kernel whose metric is not (Sq)Euclidean)
__device__ __forceinline__ bool needs_raw_points(const LatentParams* gp) { return gp->nterms > 1 || gp->kind == 5; }

// Fixed-order sum over the 256 threads of a CTA (the result is valid in thread 0).
__device__ __forceinline__ double cta_sum256(double v, double* red) {
  const int t = threadIdx.x;
  red[t] = v;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  return red[0];
}

// Programmatic dependent launch (the panel chain of a batch-1 factorisation is three dependent small kernels per tile
// column): a kernel launched with launch_pdl() may be scheduled as soon as its predecessor in the stream executes
// pdl_trigger(); it must execute pdl_wait() before touching anything the predecessor wrote (pdl_wait returns when the
// predecessor grid has completed and its writes are visible).  Both are no-ops for a plain <<<>>> launch.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

}  // namespace lmm
