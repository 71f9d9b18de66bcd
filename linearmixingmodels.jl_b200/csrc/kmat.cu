// Fused kernel-matrix builders (K4/K5 of SURVEY.md §2.3; reference call site src/oilmm.jl:90 ->
// AbstractGPs mean_and_cov -> KernelFunctions kernelmatrix -> Distances pairwise + map(κ), then
// `+ Diagonal(ΣT_i)`).  One pass: scaled inputs -> pairwise squared distance -> κ -> variance
// scale -> (+ noise on the diagonal) written straight into the tiled factorisation workspace.
// The two 128-point input tiles are staged into shared memory with one TMA bulk copy each
// (cp.async.bulk + mbarrier).  HBM-write bound: 8 bytes per stored element, lower tiles only -- and on the OILMM / IndependentMOGP
// eval path only the tiles that kmat_bound_kernel cannot prove to be exact zeros.
#include "common.cuh"
#include "kernels.h"

namespace lmm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (!done && ++spins > (1u << 28)) __trap();  // never hang the GPU on a protocol bug (same bound as gemm.cu)
  }
}

// Stage the two point tiles (rows of xpad, D doubles per point) and scale them (ScaleTransform / ARDTransform).
// smem layout: xa[128*D] | xb[128*D] | sa[128] | sb[128]
__device__ __forceinline__ void stage_points(double* xa, double* xb, double* sa, double* sb, const double* ga, const double* gb,
                                             int D, const LatentParams* gp, uint64_t* bar) {
  const uint32_t bytes = (uint32_t)(TILE * D * sizeof(double));
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, 2 * bytes);
    bulk_g2s(xa, ga, bytes, bar);
    bulk_g2s(xb, gb, bytes, bar);
  }
  mbar_wait(bar, 0);
  if (needs_raw_points(gp)) return;  // composite / periodic latent: every term scales the raw points itself (kernel_value_raw)
  for (int i = threadIdx.x; i < TILE * D; i += blockDim.x) {
    const double s = input_scale(gp, i % D);
    xa[i] *= s;
    xb[i] *= s;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * TILE; i += blockDim.x) {
    const double* v = (i < TILE) ? xa + (size_t)i * D : xb + (size_t)(i - TILE) * D;
    double s = 0.0;
    for (int k = 0; k < D; ++k) s = fma(v[k], v[k], s);
    if (i < TILE) sa[i] = s; else sb[i - TILE] = s;
  }
  __syncthreads();
}

// Composite (KernelSum / KernelProduct) or periodic latent: xa / xb hold RAW points; each term applies its own input scaling,
// distance and κ (KernelFunctions evaluates the components separately and adds / multiplies the matrices).  Kept out of line
// so that the single-kernel tile body keeps its register allocation (it runs at 90 % of the HBM write bandwidth).
template <bool SYM>
__device__ __noinline__ bool kmat_tile_composite(double* __restrict__ tile, const double* xa, const double* xb, int dd, int r0, int c0, int Na,
                                                 int Nb, double noise, int form, const double* __restrict__ noise_vec, const LatentParams* gp) {
  const int t = threadIdx.x;
  const int r = (((2 * t) >> 5) & 15) * 8 + (((2 * t) >> 2) & 7);
  const int gr = r0 + r;
  bool nz = false;
  __syncthreads();  // stage_points returned right after the bulk copies landed
  for (int it = 0; it < 32; ++it) {
    const int c = 4 * it + ((2 * t) & 3);
    double2 v;
    double* vv = reinterpret_cast<double*>(&v);
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int gc = c0 + c + q;
      double val;
      if (gr >= Na || gc >= Nb) {
        val = (SYM && gr == gc) ? 1.0 : 0.0;
      } else {
        const bool same = SYM && gr == gc;
        val = kernel_value_raw(gp, xa + (size_t)r * dd, xb + (size_t)(c + q) * dd, dd, form, same);
        if (same) val += noise_vec ? noise_vec[gr] : noise;
      }
      vv[q] = val;
    }
    nz |= (v.x != 0.0) | (v.y != 0.0);
    *reinterpret_cast<double2*>(tile + it * 512 + 2 * t) = v;
  }
  return nz;
}

// One 128x128 tile of kernel values.  Thread t owns the fixed tile row r(t) and walks the columns
// c = 4*it + 2*(t&1) + {0,1}: its own scaled point / squared norm are hoisted into registers, the
// column points are shared-memory broadcasts, and each iteration ends in one coalesced 16-byte
// store at tile offset e = it*512 + 2*t (the k4-interleaved layout makes e linear in (it, t)).
// SYM: diagonal entries get d² = 0 exactly and + noise; padding is the identity (SYM) or zero.
// Returns whether this thread stored an entry that is not exactly 0 (NaN counts as nonzero).
template <bool SYM, int DS>
__device__ __forceinline__ bool kmat_tile_body(double* __restrict__ tile, const double* xa, const double* xb, const double* sa,
                                               const double* sb, int D, int r0, int c0, int Na, int Nb, const LatentParams& lp, int form,
                                               const double* __restrict__ noise_vec = nullptr, const LatentParams* gp = nullptr) {
  const int t = threadIdx.x;
  const int r = (((2 * t) >> 5) & 15) * 8 + (((2 * t) >> 2) & 7);
  const int gr = r0 + r;
  const int dd = DS > 0 ? DS : D;
  if (gp != nullptr && needs_raw_points(gp)) {  // composite (KernelSum / KernelProduct) or periodic latent: out-of-line slow path
    return kmat_tile_composite<SYM>(tile, xa, xb, dd, r0, c0, Na, Nb, lp.noise, form, noise_vec, gp);
  }
  const double* ar = xa + (size_t)r * dd;
  const double sar = sa[r];
  const double a0 = ar[0];
  bool nz = false;
  // interior off-diagonal tiles (almost all of them): no bounds / diagonal predicates in the element loop
  if (DS == 1 && form == 0 && r0 + TILE <= Na && c0 + TILE <= Nb && !(SYM && r0 == c0)) {
    const int cb = (2 * t) & 3;
#pragma unroll 4
    for (int it = 0; it < 32; ++it) {
      const int c = 4 * it + cb;
      const double2 xb2 = *reinterpret_cast<const double2*>(xb + c);
      const double2 sb2 = *reinterpret_cast<const double2*>(sb + c);
      // the same arithmetic as the general path: one rounded product (Distances.jl's K=1 GEMM), then |a|²+|b|² - 2ab
      double d0 = fma(-2.0, a0 * xb2.x, sar + sb2.x);
      double d1 = fma(-2.0, a0 * xb2.y, sar + sb2.y);
      d0 = d0 > 0.0 ? d0 : 0.0;
      d1 = d1 > 0.0 ? d1 : 0.0;
      double2 v;
      v.x = kappa_eval(lp.kind, lp.variance, d0, lp.param);
      v.y = kappa_eval(lp.kind, lp.variance, d1, lp.param);
      nz |= (v.x != 0.0) | (v.y != 0.0);
      *reinterpret_cast<double2*>(tile + it * 512 + 2 * t) = v;
    }
    return nz;
  }
  for (int it = 0; it < 32; ++it) {
    const int c = 4 * it + ((2 * t) & 3);
    double2 v;
    double* vv = reinterpret_cast<double*>(&v);
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int gc = c0 + c + q;
      double val;
      if (gr >= Na || gc >= Nb) {
        val = (SYM && gr == gc) ? 1.0 : 0.0;
      } else if (SYM && gr == gc) {
        val = kappa_eval(lp.kind, lp.variance, 0.0, lp.param) + (noise_vec ? noise_vec[gr] : lp.noise);
      } else {
        double d2;
        if (DS == 1 && form == 0) {
          const double tt = sar + sb[c + q];
          d2 = fma(-2.0, a0 * xb[c + q], tt);
          d2 = d2 > 0.0 ? d2 : 0.0;
        } else {
          d2 = sqdist(ar, xb + (size_t)(c + q) * dd, dd, sar, sb[c + q], form);
        }
        val = kappa_eval(lp.kind, lp.variance, d2, lp.param);
      }
      vv[q] = val;
    }
    nz |= (v.x != 0.0) | (v.y != 0.0);
    *reinterpret_cast<double2*>(tile + it * 512 + 2 * t) = v;
  }
  return nz;
}

// grid: (lower tiles, batch).  Writes K_b + noise_b*I (identity on the padding) into L tiles.
// env (nullable, [batch][nt], pre-filled with a value >= nt): env[b][I] = first tile column J of tile row I with an entry that is not
// exactly 0 -- taken from the values written, so it holds for every kernel, noise vector and point order.  The diagonal tile always
// counts.  atomicMin is order-independent: the result is deterministic.
template <int DS>
// (256, 4): 4 CTAs per SM as without the envelope test, which would otherwise take the single-kernel body from 64 to 76 registers
__global__ void __launch_bounds__(256, 4) kmat_sym_kernel(TiledSym out, const double* __restrict__ xpad, int N, int D,
                                                       const LatentParams* __restrict__ params, int form,
                                                       const double* __restrict__ noise_vec, size_t noise_stride, int tile0, int* env,
                                                       const int* __restrict__ rowoff, int batch) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* xa = reinterpret_cast<double*>(smem_raw);
  double* xb = xa + TILE * D;
  double* sa = xb + TILE * D;
  double* sb = sa + TILE;
  __shared__ __align__(8) uint64_t bar;

  int b, I, J;
  if (rowoff) {
    // grid (tiles inside the bound envelopes of the whole batch): the run of (latent, tile row) r that holds tile t,
    // rowoff[r] <= t < rowoff[r + 1], by a 256-way search -- two rounds for 8192 runs
    const int t = blockIdx.x;
    int r0 = 0, r1 = batch * out.nt;
    while (r1 - r0 > 1) {
      const int s = (r1 - r0 + (int)blockDim.x - 1) / (int)blockDim.x;
      const int i = r0 + (int)threadIdx.x * s;
      const int c = __syncthreads_count(i < r1 && rowoff[i] <= t);  // >= 1: rowoff[r0] <= t
      r0 += (c - 1) * s;
      r1 = min(r0 + s, r1);
    }
    b = r0 / out.nt;
    I = r0 - b * out.nt;
    J = I + 1 - (rowoff[r0 + 1] - rowoff[r0]) + (t - rowoff[r0]);  // the run is the tiles (I, fb .. I)
  } else {
    b = blockIdx.y;
    // linear lower-tile index -> (I, J); tile0 = first tile of the first row built (rows below a prefix that is already
    // factored: sequential conditioning extends a factor instead of rebuilding it)
    const int t = blockIdx.x + tile0;
    I = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
    while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)t) ++I;
    while ((size_t)I * (I + 1) / 2 > (size_t)t) --I;
    J = t - (int)((size_t)I * (I + 1) / 2);
  }
  const LatentParams lp = params[b];

  stage_points(xa, xb, sa, sb, xpad + (size_t)I * TILE * D, xpad + (size_t)J * TILE * D, D, params + b, &bar);
  const bool nz = kmat_tile_body<true, DS>(out.tile(b, I, J), xa, xb, sa, sb, D, I * TILE, J * TILE, N, N, lp, form,
                                           noise_vec ? noise_vec + (size_t)b * noise_stride : nullptr, params + b);
  if (env && (__syncthreads_or(nz) || I == J) && threadIdx.x == 0) atomicMin(env + (size_t)b * out.nt + I, J);
}

// grid: (ntr*ntc, batch).  Rows = points of xa_pad (e.g. x*), cols = points of xb_pad (train x).
// Padding rows/cols are zero.
template <int DS>
__global__ void __launch_bounds__(256) kmat_cross_kernel(TiledRect out, const double* __restrict__ xa_pad, int Na,
                                                         const double* __restrict__ xb_pad, int Nb, int D,
                                                         const LatentParams* __restrict__ params, int form) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* xa = reinterpret_cast<double*>(smem_raw);
  double* xb = xa + TILE * D;
  double* sa = xb + TILE * D;
  double* sb = sa + TILE;
  __shared__ __align__(8) uint64_t bar;

  const int b = blockIdx.y;
  const int R = blockIdx.x / out.ntc, J = blockIdx.x % out.ntc;
  const LatentParams lp = params[b];
  stage_points(xa, xb, sa, sb, xa_pad + (size_t)R * TILE * D, xb_pad + (size_t)J * TILE * D, D, params + b, &bar);
  kmat_tile_body<false, DS>(out.tile(b, R, J), xa, xb, sa, sb, D, R * TILE, J * TILE, Na, Nb, lp, form, nullptr, params + b);
}

// grid (batch), 256 threads, dynamic shared memory nt * (2D + 1) doubles: lo / hi [nt][D] and q [nt].
// The bound: for tile boxes A, B of the scaled points (the same products x * input_scale that stage_points forms), every pair
// (a, b) has |a - b|² >= g² = Σ_k gap_k², and the build's computed d² -- |a|²+|b|² - 2 a·b in either rounding order, or Σ (a_k -
// b_k)² -- differs from |a - b|² by less than (2D + 4) u (|a|² + |b|²) + u d² (u = 2^-53).  With q_T >= max |a|² over box T,
// lb = g² (1 - r) - r (q_A + q_B), r = 8 (D + 4) u, is below every computed d² of the tile; lb > kappa_zero_d2 proves it all-zero.
// Padding points are left out of the boxes: the build writes 0 for them off the diagonal.  A non-finite coordinate makes its box
// unbounded and its q infinite, so nothing involving that tile is skipped.
__global__ void __launch_bounds__(256) kmat_bound_kernel(const double* __restrict__ xpad, int N, int D, int nt,
                                                         const LatentParams* __restrict__ params, int* __restrict__ fb) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* lo = reinterpret_cast<double*>(smem_raw);
  double* hi = lo + (size_t)nt * D;
  double* q = hi + (size_t)nt * D;
  const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const LatentParams* gp = params + b;
  int* fbb = fb + (size_t)b * nt;
  const double thr = kappa_zero_d2(gp->kind);
  if (needs_raw_points(gp) || !(thr < __builtin_huge_val()) || !isfinite(gp->variance)) {  // ∞·0 = NaN counts as nonzero
    for (int I = threadIdx.x; I < nt; I += blockDim.x) fbb[I] = 0;
    return;
  }
  // one warp per (tile, dimension)
  for (int i = warp; i < nt * D; i += (int)blockDim.x / 32) {
    const int T = i / D, k = i - T * D;
    const double s = input_scale(gp, k);
    double l = __builtin_huge_val(), h = -__builtin_huge_val();
    bool bad = false;
    for (int r = T * TILE + lane; r < (T + 1) * TILE && r < N; r += 32) {
      const double v = xpad[(size_t)r * D + k] * s;
      bad |= !isfinite(v);
      l = fmin(l, v);
      h = fmax(h, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      l = fmin(l, __shfl_xor_sync(0xffffffffu, l, o));
      h = fmax(h, __shfl_xor_sync(0xffffffffu, h, o));
    }
    if (__any_sync(0xffffffffu, bad)) {
      l = -__builtin_huge_val();
      h = __builtin_huge_val();
    }
    if (lane == 0) {
      lo[i] = l;
      hi[i] = h;
    }
  }
  __syncthreads();
  for (int T = threadIdx.x; T < nt; T += blockDim.x) {
    double s = 0.0;
    for (int k = 0; k < D; ++k) s += fmax(lo[T * D + k] * lo[T * D + k], hi[T * D + k] * hi[T * D + k]);
    q[T] = s;
  }
  __syncthreads();
  const double rel = (double)(D + 4) * 0x1p-50;
  for (int I = threadIdx.x; I < nt; I += blockDim.x) {
    int f = 0;
    for (; f < I; ++f) {
      double g2 = 0.0;
      for (int k = 0; k < D; ++k) {
        const double g = fmax(0.0, fmax(lo[I * D + k] - hi[f * D + k], lo[f * D + k] - hi[I * D + k]));
        g2 = fma(g, g, g2);
      }
      const double lb = g2 * (1.0 - rel) - rel * (q[I] + q[f]);
      if (!(lb > thr)) break;
    }
    fbb[I] = f;
  }
}

// grid (nt, batch, KZ_SPLIT): the KZ_SPLIT CTAs of a tile row share the row's contiguous run of tiles (I, 0 .. env - 1).
constexpr int KZ_SPLIT = 8;
__global__ void __launch_bounds__(256) kmat_zero_kernel(TiledSym L, const int* __restrict__ env) {
  const int I = blockIdx.x, b = blockIdx.y;
  double2* p = reinterpret_cast<double2*>(L.tile(b, I, 0));
  const size_t n = (size_t)env[(size_t)b * L.nt + I] * (TT / 2);
  for (size_t i = (size_t)blockIdx.z * blockDim.x + threadIdx.x; i < n; i += (size_t)KZ_SPLIT * blockDim.x) p[i] = make_double2(0.0, 0.0);
}

static size_t kmat_smem(int D) { return (size_t)(2 * TILE * D + 2 * TILE) * sizeof(double); }

cudaError_t launch_kmat_sym(cudaStream_t st, TiledSym out, int batch, const double* xpad, int N, int D,
                            const LatentParams* params, int form, const double* noise_vec, size_t noise_stride, int row0, int* env,
                            const int* rowoff, long long ntiles) {
  size_t sm = kmat_smem(D);
  if (sm + 1024 > 48 * 1024) {  // static shared memory counts against the default limit too
    cudaError_t e = cudaFuncSetAttribute(kmat_sym_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return e;
  }
  const int tile0 = (int)sym_tiles(row0);  // row-panel-major order: the tiles of rows >= row0 are the tail of the list
  if (row0 >= out.nt) return cudaSuccess;
  if (rowoff && row0 != 0) return cudaErrorInvalidValue;
  if (env) {
    cudaError_t e = cudaMemsetAsync(env, 0x7f, (size_t)batch * out.nt * sizeof(int), st);
    if (e != cudaSuccess) return e;
  }
  if (rowoff && ntiles <= 0) return cudaSuccess;
  dim3 grid(rowoff ? (unsigned)ntiles : (unsigned)(sym_tiles(out.nt) - tile0), rowoff ? 1u : (unsigned)batch);
  if (D == 1)
    kmat_sym_kernel<1><<<grid, 256, sm, st>>>(out, xpad, N, D, params, form, noise_vec, noise_stride, tile0, env, rowoff, batch);
  else
    kmat_sym_kernel<0><<<grid, 256, sm, st>>>(out, xpad, N, D, params, form, noise_vec, noise_stride, tile0, env, rowoff, batch);
  return cudaGetLastError();
}

cudaError_t launch_kmat_bound(cudaStream_t st, int batch, const double* xpad, int N, int D, int nt, const LatentParams* params, int* fb) {
  if (batch <= 0) return cudaSuccess;
  const size_t sm = (size_t)nt * (2 * D + 1) * sizeof(double);
  if (sm > 200 * 1024)  // boxes too large for shared memory: no bound, every tile is built
    return cudaMemsetAsync(fb, 0, (size_t)batch * nt * sizeof(int), st);
  if (sm > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kmat_bound_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return e;
  }
  kmat_bound_kernel<<<batch, 256, sm, st>>>(xpad, N, D, nt, params, fb);
  return cudaGetLastError();
}

cudaError_t launch_kmat_zero(cudaStream_t st, TiledSym L, int batch, const int* env) {
  if (batch <= 0) return cudaSuccess;
  kmat_zero_kernel<<<dim3((unsigned)L.nt, (unsigned)batch, KZ_SPLIT), 256, 0, st>>>(L, env);
  return cudaGetLastError();
}

cudaError_t launch_kmat_cross(cudaStream_t st, TiledRect out, int batch, const double* xa_pad, int Na, const double* xb_pad,
                              int Nb, int D, const LatentParams* params, int form) {
  size_t sm = kmat_smem(D);
  if (sm + 1024 > 48 * 1024) {  // static shared memory counts against the default limit too
    cudaError_t e = cudaFuncSetAttribute(kmat_cross_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return e;
  }
  dim3 grid((unsigned)(out.ntr * out.ntc), (unsigned)batch);
  if (D == 1)
    kmat_cross_kernel<1><<<grid, 256, sm, st>>>(out, xa_pad, Na, xb_pad, Nb, D, params, form);
  else
    kmat_cross_kernel<0><<<grid, 256, sm, st>>>(out, xa_pad, Na, xb_pad, Nb, D, params, form);
  return cudaGetLastError();
}

}  // namespace lmm
