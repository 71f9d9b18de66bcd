// Fused kernel-gradient reduction for the logpdf rrule (SURVEY.md §8f-1; reference call sites
// test/oilmm.jl:31-32, test/ilmm.jl:31-32, test/independent_mogp.jl:65-66 `gradient(logpdf, fx, y)`).
// With G = d lml / dC = (αα' - C^{-1})/2 the hyper-parameter gradients of one latent are
//   d/d variance = <G, κ>,  d/d inv_lengthscale = <G, dK/ds>,  d/d noise = tr(G),
// contracted tile by tile: the kernel values and their lengthscale derivatives are recomputed in
// registers from the staged inputs (never stored), NegCinv = -C^{-1} comes from the batched
// `potri` (triangular TRSM sweep + SYRK on the DMMA kernel).  HBM-bound: one read of C^{-1}.
#include "common.cuh"
#include "kernels.h"

namespace lmm {

__device__ __forceinline__ uint32_t g_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// κ and dK/ds (both already multiplied by the variance where appropriate): returns κ (unscaled by variance)
__device__ __forceinline__ void kappa_and_ds(int kind, double d2, double rinv_ls, double& kap, double& dkds, double param = 1.0) {
  if (kind == 0) {
    kap = exp_nonpos(-0.5 * d2);
    dkds = -kap * d2 * rinv_ls;
  } else if (kind == 4) {  // (1 + d²/2α)^(-α);  d/ds = -(d²/s) (1 + d²/2α)^(-α-1)
    const double base = 1.0 + d2 / (2.0 * param);
    kap = pow(base, -param);
    dkds = -d2 * rinv_ls * kap / base;
  } else {
    const double d = sqrt(d2);
    if (kind == 1) {
      const double s = 1.7320508075688772 * d;
      const double e = exp_nonpos(-s);
      kap = (1.0 + s) * e;
      dkds = -3.0 * d2 * e * rinv_ls;
    } else if (kind == 2) {
      const double s = 2.23606797749979 * d;
      const double e = exp_nonpos(-s);
      kap = (1.0 + s + (d * d) * 1.6666666666666667) * e;
      dkds = -(5.0 / 3.0) * d2 * (1.0 + s) * e * rinv_ls;
    } else {  // exp(-d);  d/ds = -(d/s) exp(-d)
      kap = exp_nonpos(-d);
      dkds = -d * kap * rinv_ls;
    }
  }
}

// grid (lower tiles, batch).  partial[(b*ntiles + tile)*3 + {0,1,2}] = {<G,κ>, <G,dK/ds>/variance.., tr G}
__global__ void __launch_bounds__(256) kgrad_kernel(TiledSym negCinv, const double* __restrict__ xpad, int N, int D,
                                                    const LatentParams* __restrict__ params, const double* __restrict__ alpha,
                                                    size_t alpha_stride, int form, double* __restrict__ partial) {
  extern __shared__ __align__(16) double sm[];
  double* xa = sm;                 // [128*D] scaled
  double* xb = xa + TILE * D;
  double* sa = xb + TILE * D;
  double* sb = sa + TILE;
  double* aa = sb + TILE;          // alpha rows
  double* ab = aa + TILE;          // alpha cols
  __shared__ double red[3][256];

  const int b = blockIdx.y, tl = blockIdx.x, t = threadIdx.x;
  int I = (int)((sqrt(8.0 * (double)tl + 1.0) - 1.0) * 0.5);
  while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tl) ++I;
  while ((size_t)I * (I + 1) / 2 > (size_t)tl) --I;
  const int J = tl - (int)((size_t)I * (I + 1) / 2);
  const LatentParams lp = params[b];
  const double rinv_ls = 1.0 / lp.inv_ls;
  for (int i = t; i < TILE * D; i += 256) {
    const double s = input_scale(params + b, i % D);
    xa[i] = xpad[(size_t)I * TILE * D + i] * s;
    xb[i] = xpad[(size_t)J * TILE * D + i] * s;
  }
  if (t < TILE) {
    aa[t] = alpha[(size_t)b * alpha_stride + I * TILE + t];
    ab[t] = alpha[(size_t)b * alpha_stride + J * TILE + t];
  }
  __syncthreads();
  for (int i = t; i < 2 * TILE; i += 256) {
    const double* v = (i < TILE) ? xa + (size_t)i * D : xb + (size_t)(i - TILE) * D;
    double s = 0.0;
    for (int k = 0; k < D; ++k) s = fma(v[k], v[k], s);
    if (i < TILE) sa[i] = s; else sb[i - TILE] = s;
  }
  __syncthreads();

  const double* tile = negCinv.tile(b, I, J);
  const int r = (((2 * t) >> 5) & 15) * 8 + (((2 * t) >> 2) & 7);
  const int gr = I * TILE + r;
  double gv = 0.0, gs = 0.0, gn = 0.0;
  for (int it = 0; it < 32; ++it) {
    const int c = 4 * it + ((2 * t) & 3);
    const double2 nc = *reinterpret_cast<const double2*>(tile + it * 512 + 2 * t);
    const double ncv[2] = {nc.x, nc.y};
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int cc = c + q, gc = J * TILE + cc;
      if (gr >= N || gc >= N) continue;
      if (I == J && cc > r) continue;  // lower triangle only; off-diagonal entries count twice
      const double G = 0.5 * (aa[r] * ab[cc] + ncv[q]);
      if (gr == gc) {
        gn += G;
        gv = fma(G, 1.0, gv);  // κ(0) = 1, dK/ds = 0 on the diagonal
      } else {
        const double d2 = sqdist(xa + (size_t)r * D, xb + (size_t)cc * D, D, sa[r], sb[cc], form);
        double kap, dk;
        kappa_and_ds(lp.kind, d2, rinv_ls, kap, dk, lp.param);
        gv = fma(2.0 * G, kap, gv);
        gs = fma(2.0 * G, dk, gs);
      }
    }
  }
  red[0][t] = gv; red[1][t] = gs; red[2][t] = gn;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) {
      red[0][t] += red[0][t + w];
      red[1][t] += red[1][t + w];
      red[2][t] += red[2][t + w];
    }
    __syncthreads();
  }
  if (t == 0) {
    double* out = partial + ((size_t)b * gridDim.x + tl) * 3;
    out[0] = red[0][0];
    out[1] = red[1][0] * lp.variance;  // dK/ds carries the variance
    out[2] = red[2][0];
  }
}

cudaError_t launch_kgrad(cudaStream_t st, TiledSym negCinv, int batch, const double* xpad, int N, int D, const LatentParams* params,
                         const double* alpha, size_t alpha_stride, int form, double* partial) {
  const size_t smem = (size_t)(2 * TILE * D + 4 * TILE) * sizeof(double);
  if (smem + 1024 > 48 * 1024) {  // static shared memory counts against the default limit too
    cudaError_t e = cudaFuncSetAttribute(kgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  dim3 grid((unsigned)sym_tiles(negCinv.nt), (unsigned)batch);
  kgrad_kernel<<<grid, 256, smem, st>>>(negCinv, xpad, N, D, params, alpha, alpha_stride, form, partial);
  return cudaGetLastError();
}

// out[b*4 + {0,1,2}] = fixed-order sums of the tile partials; out[b*4+3] = sum(alpha_b) (d/d mean)
__global__ void __launch_bounds__(256) kgrad_finish_kernel(const double* __restrict__ partial, int ntiles_, const double* __restrict__ alpha,
                                                           size_t alpha_stride, int N, double* __restrict__ out) {
  __shared__ double red[4][256];
  const int b = blockIdx.x, t = threadIdx.x;
  double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
  for (int i = t; i < ntiles_; i += 256) {
    const double* p = partial + ((size_t)b * ntiles_ + i) * 3;
    s0 += p[0]; s1 += p[1]; s2 += p[2];
  }
  for (int i = t; i < N; i += 256) s3 += alpha[(size_t)b * alpha_stride + i];
  red[0][t] = s0; red[1][t] = s1; red[2][t] = s2; red[3][t] = s3;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w)
      for (int k = 0; k < 4; ++k) red[k][t] += red[k][t + w];
    __syncthreads();
  }
  if (t < 4) out[(size_t)b * 4 + t] = red[t][0];
}
cudaError_t launch_kgrad_finish(cudaStream_t st, const double* partial, int ntiles_, int batch, const double* alpha, size_t alpha_stride,
                                int N, double* out) {
  kgrad_finish_kernel<<<batch, 256, 0, st>>>(partial, ntiles_, alpha, alpha_stride, N, out);
  return cudaGetLastError();
}

// X (rectangular tiles, nt x nt per latent) <- identity
__global__ void __launch_bounds__(256) rect_identity_kernel(TiledRect X) {
  const int b = blockIdx.y, R = blockIdx.x / X.ntc, J = blockIdx.x % X.ntc;
  double* tile = X.tile(b, R, J);
  for (int e = threadIdx.x; e < TT; e += 256) {
    int r, c;
    tile_rc(e, r, c);
    tile[e] = (R == J && r == c) ? 1.0 : 0.0;
  }
}
cudaError_t launch_rect_identity(cudaStream_t st, TiledRect X, int batch) {
  dim3 grid((unsigned)(X.ntr * X.ntc), (unsigned)batch);
  rect_identity_kernel<<<grid, 256, 0, st>>>(X);
  return cudaGetLastError();
}


// ---- general-ILMM gradient: the joint (mN x mN) matrix C = blockdiag(K_a) + ΣT ⊗ I -----------------
// Latent blocks start at multiples of N, not of the tile size, so elements are addressed one by one.
__device__ __forceinline__ double sym_get(const double* __restrict__ base, int r, int c) {  // r >= c
  return base[sym_tile_index(r / TILE, c / TILE) * TT + tile_elem(r % TILE, c % TILE)];
}

// grid (chunks of the lower triangle of one N x N latent block, m).  x is [N][D] (unpadded), alpha the
// joint vector (latent a at a*N).  partial[(a*nchunks + chunk)*2 + {0,1}] = {<G_aa, κ>, <G_aa, dK_a/ds>}.
__global__ void __launch_bounds__(256) kgrad_block_kernel(TiledSym negCinv, const double* __restrict__ x, int N, int D,
                                                          const LatentParams* __restrict__ params, const double* __restrict__ alpha,
                                                          int form, double* __restrict__ partial) {
  extern __shared__ __align__(16) double sm[];
  double* xa = sm;
  double* xb = xa + TILE * D;
  double* sa = xb + TILE * D;
  double* sb = sa + TILE;
  double* aa = sb + TILE;
  double* ab = aa + TILE;
  __shared__ double red[2][256];
  const int a = blockIdx.y, tl = blockIdx.x, t = threadIdx.x;
  int I = (int)((sqrt(8.0 * (double)tl + 1.0) - 1.0) * 0.5);
  while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tl) ++I;
  while ((size_t)I * (I + 1) / 2 > (size_t)tl) --I;
  const int J = tl - (int)((size_t)I * (I + 1) / 2);
  const LatentParams lp = params[a];
  const double rinv_ls = 1.0 / lp.inv_ls;
  for (int i = t; i < TILE * D; i += 256) {
    const int ra = I * TILE + i / D, rb = J * TILE + i / D;
    const double s = input_scale(params + a, i % D);
    xa[i] = ra < N ? x[(size_t)ra * D + i % D] * s : 0.0;
    xb[i] = rb < N ? x[(size_t)rb * D + i % D] * s : 0.0;
  }
  if (t < TILE) {
    aa[t] = (I * TILE + t < N) ? alpha[(size_t)a * N + I * TILE + t] : 0.0;
    ab[t] = (J * TILE + t < N) ? alpha[(size_t)a * N + J * TILE + t] : 0.0;
  }
  __syncthreads();
  for (int i = t; i < 2 * TILE; i += 256) {
    const double* v = (i < TILE) ? xa + (size_t)i * D : xb + (size_t)(i - TILE) * D;
    double s = 0.0;
    for (int k = 0; k < D; ++k) s = fma(v[k], v[k], s);
    if (i < TILE) sa[i] = s; else sb[i - TILE] = s;
  }
  __syncthreads();
  const double* base = negCinv.base;
  double gv = 0.0, gs = 0.0;
  for (int e = t; e < TT; e += 256) {
    const int c = ((e >> 9) << 2) + (e & 3), r = (e >> 2) & 127;
    const int gr = I * TILE + r, gc = J * TILE + c;
    if (gr >= N || gc >= N || gc > gr) continue;
    const double G = 0.5 * (aa[r] * ab[c] + sym_get(base, a * N + gr, a * N + gc));
    if (gr == gc) {
      gv += G;
    } else {
      const double d2 = sqdist(xa + (size_t)r * D, xb + (size_t)c * D, D, sa[r], sb[c], form);
      double kap, dk;
      kappa_and_ds(lp.kind, d2, rinv_ls, kap, dk, lp.param);
      gv = fma(2.0 * G, kap, gv);
      gs = fma(2.0 * G, dk, gs);
    }
  }
  red[0][t] = gv; red[1][t] = gs;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) {
      red[0][t] += red[0][t + w];
      red[1][t] += red[1][t + w];
    }
    __syncthreads();
  }
  if (t == 0) {
    double* out = partial + ((size_t)a * gridDim.x + tl) * 2;
    out[0] = red[0][0];
    out[1] = red[1][0] * lp.variance;
  }
}

// out[a*3 + {0,1,2}] = {Σ chunks <G,κ>, Σ chunks <G,dK/ds>, Σ_n α[a*N+n]} in a fixed order.
__global__ void __launch_bounds__(256) kgrad_block_finish_kernel(const double* __restrict__ partial, int nchunks,
                                                                 const double* __restrict__ alpha, int N, double* __restrict__ out) {
  __shared__ double red[3][256];
  const int a = blockIdx.x, t = threadIdx.x;
  double s0 = 0, s1 = 0, s2 = 0;
  for (int i = t; i < nchunks; i += 256) {
    s0 += partial[((size_t)a * nchunks + i) * 2];
    s1 += partial[((size_t)a * nchunks + i) * 2 + 1];
  }
  for (int i = t; i < N; i += 256) s2 += alpha[(size_t)a * N + i];
  red[0][t] = s0; red[1][t] = s1; red[2][t] = s2;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w)
      for (int k = 0; k < 3; ++k) red[k][t] += red[k][t + w];
    __syncthreads();
  }
  if (t < 3) out[(size_t)a * 3 + t] = red[t][0];
}

// B[a,b] = Σ_n G[(a,n),(b,n)] = Σ_n (α_a[n] α_b[n] - C^{-1}[(a,n),(b,n)])/2  (m x m, symmetric): d lml / dΣT.
__global__ void __launch_bounds__(256) block_trace_kernel(TiledSym negCinv, const double* __restrict__ alpha, int N, int m,
                                                          double* __restrict__ B) {
  __shared__ double red[256];
  const int a = blockIdx.x, b = blockIdx.y, t = threadIdx.x;
  if (b > a) return;
  double s = 0.0;
  for (int n = t; n < N; n += 256) s += 0.5 * (alpha[(size_t)a * N + n] * alpha[(size_t)b * N + n] + sym_get(negCinv.base, a * N + n, b * N + n));
  red[t] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  if (t == 0) {
    B[(size_t)b * m + a] = red[0];
    B[(size_t)a * m + b] = red[0];
  }
}

cudaError_t launch_kgrad_joint(cudaStream_t st, TiledSym negCinv, const double* x, int N, int D, const LatentParams* params, int m,
                               const double* alpha, int form, double* partial, double* out3, double* B) {
  const size_t smem = (size_t)(2 * TILE * D + 4 * TILE) * sizeof(double);
  if (smem + 1024 > 48 * 1024) {  // static shared memory counts against the default limit too
    cudaError_t e = cudaFuncSetAttribute(kgrad_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const int ntn = (N + TILE - 1) / TILE;
  const int nchunks = (int)sym_tiles(ntn);
  dim3 grid((unsigned)nchunks, (unsigned)m);
  kgrad_block_kernel<<<grid, 256, smem, st>>>(negCinv, x, N, D, params, alpha, form, partial);
  kgrad_block_finish_kernel<<<m, 256, 0, st>>>(partial, nchunks, alpha, N, out3);
  dim3 g2((unsigned)m, (unsigned)m);
  block_trace_kernel<<<g2, 256, 0, st>>>(negCinv, alpha, N, m, B);
  return cudaGetLastError();
}

cudaError_t launch_block_trace(cudaStream_t st, TiledSym negCinv, const double* alpha, int N, int m, double* B) {
  dim3 g2((unsigned)m, (unsigned)m);
  block_trace_kernel<<<g2, 256, 0, st>>>(negCinv, alpha, N, m, B);
  return cudaGetLastError();
}

// ---- gradient w.r.t. the ARD multipliers (only launched when a latent has an ARDTransform and the caller asks) ------
// dK/d a_k = variance κ'(d²) 2 u_k² / a_k with u = scaled coordinate difference; κ'(d²) 2 = (dK/ds per unit variance) s / d².
// One generic kernel for both storages: per-latent factors (mat_batch_stride = tile storage of one latent, off_per_lat = 0)
// and the joint ILMM matrix (mat_batch_stride = 0, off_per_lat = N).  grid (chunks of the lower triangle, latents).
__global__ void __launch_bounds__(256) kgrad_ard_kernel(const double* __restrict__ mat_base, size_t mat_batch_stride, int off_per_lat,
                                                        const double* __restrict__ x, int N, int D,
                                                        const LatentParams* __restrict__ params, const double* __restrict__ alpha,
                                                        size_t alpha_stride, int form, double* __restrict__ partial) {
  extern __shared__ __align__(16) double sm[];
  double* xa = sm;
  double* xb = xa + TILE * D;
  double* sa = xb + TILE * D;
  double* sb = sa + TILE;
  double* aa = sb + TILE;
  double* ab = aa + TILE;
  __shared__ double red[MAX_ARD][256];
  const int lat = blockIdx.y, tl = blockIdx.x, t = threadIdx.x;
  double ga[MAX_ARD];
#pragma unroll
  for (int k = 0; k < MAX_ARD; ++k) ga[k] = 0.0;
  const LatentParams lp = params[lat];
  if (lp.ard_dim > 0) {  // block-uniform
    int I = (int)((sqrt(8.0 * (double)tl + 1.0) - 1.0) * 0.5);
    while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tl) ++I;
    while ((size_t)I * (I + 1) / 2 > (size_t)tl) --I;
    const int J = tl - (int)((size_t)I * (I + 1) / 2);
    const double* base = mat_base + (size_t)lat * mat_batch_stride;
    const int off = lat * off_per_lat;
    const double* al = alpha + (size_t)lat * alpha_stride;
    const double rinv_ls = 1.0 / lp.inv_ls;
    for (int i = t; i < TILE * D; i += 256) {
      const int ra = I * TILE + i / D, rb = J * TILE + i / D;
      const double s = input_scale(params + lat, i % D);
      xa[i] = ra < N ? x[(size_t)ra * D + i % D] * s : 0.0;
      xb[i] = rb < N ? x[(size_t)rb * D + i % D] * s : 0.0;
    }
    if (t < TILE) {
      aa[t] = (I * TILE + t < N) ? al[I * TILE + t] : 0.0;
      ab[t] = (J * TILE + t < N) ? al[J * TILE + t] : 0.0;
    }
    __syncthreads();
    for (int i = t; i < 2 * TILE; i += 256) {
      const double* v = (i < TILE) ? xa + (size_t)i * D : xb + (size_t)(i - TILE) * D;
      double s = 0.0;
      for (int k = 0; k < D; ++k) s = fma(v[k], v[k], s);
      if (i < TILE) sa[i] = s; else sb[i - TILE] = s;
    }
    __syncthreads();
    for (int e = t; e < TT; e += 256) {
      const int c = ((e >> 9) << 2) + (e & 3), r = (e >> 2) & 127;
      const int gr = I * TILE + r, gc = J * TILE + c;
      if (gr >= N || gc >= N || gc >= gr) continue;  // strictly lower: the diagonal does not depend on the inputs
      const double d2 = sqdist(xa + (size_t)r * D, xb + (size_t)c * D, D, sa[r], sb[c], form);
      if (!(d2 > 0.0)) continue;
      const double G = 0.5 * (aa[r] * ab[c] + sym_get(base, off + gr, off + gc));
      double kap, dk;
      kappa_and_ds(lp.kind, d2, rinv_ls, kap, dk, lp.param);
      const double w = 2.0 * G * dk * lp.inv_ls / d2;
#pragma unroll
      for (int k = 0; k < MAX_ARD; ++k)
        if (k < D) {
          const double u = xa[(size_t)r * D + k] - xb[(size_t)c * D + k];
          ga[k] = fma(w, u * u, ga[k]);
        }
    }
  }
#pragma unroll
  for (int k = 0; k < MAX_ARD; ++k) red[k][t] = ga[k];
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w)
#pragma unroll
      for (int k = 0; k < MAX_ARD; ++k) red[k][t] += red[k][t + w];
    __syncthreads();
  }
  if (t < MAX_ARD) partial[((size_t)lat * gridDim.x + tl) * MAX_ARD + t] = red[t][0] * lp.variance / (lp.ard_dim > 0 ? params[lat].ard[t] : 1.0);
}
// out[lat*MAX_ARD + k] = Σ chunks (fixed order)
__global__ void __launch_bounds__(256) kgrad_ard_finish_kernel(const double* __restrict__ partial, int nchunks, double* __restrict__ out) {
  __shared__ double red[256];
  const int lat = blockIdx.x, k = blockIdx.y, t = threadIdx.x;
  double s = 0.0;
  for (int i = t; i < nchunks; i += 256) s += partial[((size_t)lat * nchunks + i) * MAX_ARD + k];
  red[t] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  if (t == 0) out[(size_t)lat * MAX_ARD + k] = red[0];
}
cudaError_t launch_kgrad_ard(cudaStream_t st, const double* mat_base, size_t mat_batch_stride, int off_per_lat, const double* x, int N, int D,
                             const LatentParams* params, int nlat, const double* alpha, size_t alpha_stride, int form, double* partial,
                             double* out) {
  const size_t smem = (size_t)(2 * TILE * D + 4 * TILE) * sizeof(double);
  const int ntn = (N + TILE - 1) / TILE;
  const int nchunks = (int)sym_tiles(ntn);
  dim3 grid((unsigned)nchunks, (unsigned)nlat);
  kgrad_ard_kernel<<<grid, 256, smem, st>>>(mat_base, mat_batch_stride, off_per_lat, x, N, D, params, alpha, alpha_stride, form, partial);
  dim3 g2((unsigned)nlat, (unsigned)MAX_ARD);
  kgrad_ard_finish_kernel<<<g2, 256, 0, st>>>(partial, nchunks, out);
  return cudaGetLastError();
}

// ---- per-term gradient: every hyper-parameter of every term of a (possibly composite) latent --------------------------
// Term t of a latent is the LatentParams' own fields (t = 0) or extra[t - 1].  For each term the kernel accumulates
// <G, ∂K/∂θ> for θ = variance, inv_lengthscale s, param (α / r) and ard[k], over the lower triangle with off-diagonal
// entries counted twice (as kgrad_kernel).  Points are staged RAW: every term applies its own scaling, as kernel_value_raw.

// Per unit variance: κ, ∂κ/∂s, ∂κ/∂param and the ARD factor wa with ∂κ/∂ard_k = wa · ard_factor(k) / ard_k.
// (Sq)Euclidean kinds: the d² of the value path (term_sqdist), ∂κ/∂s of kappa_and_ds, wa = (∂κ/∂s) s / d² (kgrad_ard_kernel).
// PeriodicKernel(r), q = Σ_k sin²(π u_k) / r², κ = e^{-q/2}: ∂κ/∂s = wa Σ_k u_k sin(2π u_k) / s, ∂κ/∂r = κ q / r,
// wa = -κ π / (2 r²).
__device__ __forceinline__ void term_grad(const TermParams& q, const double* a, const double* b, int D, int form, double& kap,
                                          double& ds, double& dp, double& wa) {
  if (q.kind == 5) {
    double qs = 0.0, us = 0.0;
    for (int k = 0; k < D; ++k) {
      const double sc = q.ard_dim ? q.inv_ls * q.ard[k] : q.inv_ls;
      const double u = sc * a[k] - sc * b[k];
      const double sn = sinpi(u) / q.param;
      qs = fma(sn, sn, qs);
      us = fma(u, sinpi(2.0 * u), us);
    }
    kap = exp_nonpos(-0.5 * qs);
    wa = -kap * 1.5707963267948966 / (q.param * q.param);
    ds = wa * us / q.inv_ls;
    dp = kap * qs / q.param;
    return;
  }
  const double d2 = term_sqdist(q.ard_dim, q.inv_ls, q.ard, a, b, D, form);
  kappa_and_ds(q.kind, d2, 1.0 / q.inv_ls, kap, ds, q.param);
  wa = d2 > 0.0 ? ds * q.inv_ls / d2 : 0.0;
  dp = 0.0;
  if (q.kind == 4) {  // RationalQuadraticKernel: ∂κ/∂α = κ (d² / (2α base) - log(base)), base = 1 + d²/(2α)
    const double base = 1.0 + d2 / (2.0 * q.param);
    dp = kap * (d2 / (2.0 * q.param * base) - log(base));
  }
}
// u_k² ((Sq)Euclidean kinds) or u_k sin(2π u_k) (PeriodicKernel), u_k = s ard_k (a_k - b_k)
__device__ __forceinline__ double ard_factor(const TermParams& q, const double* a, const double* b, int k) {
  const double sc = q.inv_ls * q.ard[k];
  const double u = sc * a[k] - sc * b[k];
  return q.kind == 5 ? u * sinpi(2.0 * u) : u * u;
}

constexpr int GRAD_TERM_STRIDE = 3 + MAX_ARD;            // == LMM_GRAD_TERM_STRIDE
constexpr int GRAD_TERM_SLOTS = MAX_TERMS * GRAD_TERM_STRIDE;

// Adds w2 ∂K/∂θ at one element to the per-term sums acc (variance, s, param) and aca (ARD).  kap / ds / dp / wa are the
// terms' per-unit-variance values of term_grad.  Weight of term u: w2 for a sum; w2 Π_{v≠u} k_v for a product, from prefix /
// suffix products (a term far from its own centre underflows to exactly 0, so K / k_u is no option).
template <int NT, bool ARD>
__device__ __forceinline__ void accumulate_terms(const TermParams* tp, bool product, double w2, const double* kap, const double* ds,
                                                 const double* dp, const double* wa, const double* pa, const double* pb, int D,
                                                 double (*acc)[3], double (*aca)[MAX_ARD]) {
  double suf[NT + 1];
  suf[NT] = 1.0;
  if (product) {
#pragma unroll
    for (int u = NT - 1; u >= 0; --u) suf[u] = suf[u + 1] * (tp[u].variance * kap[u]);
  }
  double pre = 1.0;
#pragma unroll
  for (int u = 0; u < NT; ++u) {
    const double w = product ? w2 * pre * suf[u + 1] : w2;
    if (product) pre *= tp[u].variance * kap[u];
    acc[u][0] = fma(w, kap[u], acc[u][0]);
    acc[u][1] = fma(w, ds[u], acc[u][1]);
    acc[u][2] = fma(w, dp[u], acc[u][2]);
    if (ARD && tp[u].ard_dim && wa[u] != 0.0) {
      const double wk = w * wa[u];
#pragma unroll
      for (int k = 0; k < MAX_ARD; ++k)
        if (k < D) aca[ARD ? u : 0][k] = fma(wk, ard_factor(tp[u], pa, pb, k), aca[ARD ? u : 0][k]);
    }
  }
}

// Per-thread term sums -> wsum[slot][warp] by warp shuffles (fixed order, no atomics).
template <int NT, bool ARD>
__device__ __forceinline__ void warp_term_sums(double (*acc)[3], double (*aca)[MAX_ARD], double (*wsum)[8]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int u = 0; u < NT; ++u) {
#pragma unroll
    for (int j = 0; j < (ARD ? GRAD_TERM_STRIDE : 3); ++j) {
      double v = j < 3 ? acc[u][j] : aca[ARD ? u : 0][j - 3];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
      if (lane == 0) wsum[u * GRAD_TERM_STRIDE + j][warp] = v;
    }
  }
}

// One lower-triangle chunk of one latent with NT terms; ARD: some term has an ARDTransform.  The per-thread sums are
// reduced across each warp by shuffles and written to wsum[slot][warp] (fixed order, no atomics).
template <int NT, bool ARD>
__device__ __forceinline__ void kgrad_terms_body(const TermParams* tp, bool product, const double* __restrict__ base, int off,
                                                 const double* xa, const double* xb, const double* aa, const double* ab, int I, int J,
                                                 int N, int D, int form, double (*wsum)[8]) {
  const int t = threadIdx.x;
  double acc[NT][3], aca[ARD ? NT : 1][MAX_ARD];
#pragma unroll
  for (int u = 0; u < NT; ++u) {
    acc[u][0] = acc[u][1] = acc[u][2] = 0.0;
#pragma unroll
    for (int k = 0; k < MAX_ARD; ++k) aca[ARD ? u : 0][k] = 0.0;
  }
  for (int e = t; e < TT; e += 256) {
    const int c = ((e >> 9) << 2) + (e & 3), r = (e >> 2) & 127;
    const int gr = I * TILE + r, gc = J * TILE + c;
    if (gr >= N || gc >= N || gc > gr) continue;
    const double G = 0.5 * (aa[r] * ab[c] + sym_get(base, off + gr, off + gc));
    const double* pa = xa + (size_t)r * D;
    const double* pb = xb + (size_t)c * D;
    double kap[NT], ds[NT], dp[NT], wa[NT];
    double w2;
    if (gr == gc) {  // κ(0) = 1: only the variances have a derivative on the diagonal
#pragma unroll
      for (int u = 0; u < NT; ++u) { kap[u] = 1.0; ds[u] = dp[u] = wa[u] = 0.0; }
      w2 = G;
    } else {
#pragma unroll
      for (int u = 0; u < NT; ++u) term_grad(tp[u], pa, pb, D, form, kap[u], ds[u], dp[u], wa[u]);
      w2 = 2.0 * G;
    }
    accumulate_terms<NT, ARD>(tp, product, w2, kap, ds, dp, wa, pa, pb, D, acc, aca);
  }
  warp_term_sums<NT, ARD>(acc, aca, wsum);
}

// Term 0 (the LatentParams' own fields) and the extra terms of a latent -> tp[0 .. MAX_TERMS) (threads 0 .. MAX_TERMS-1).
__device__ __forceinline__ void stage_terms(const LatentParams* lp, TermParams* tp) {
  const int t = threadIdx.x;
  if (t == 0) {
    tp[0].kind = lp->kind; tp[0].ard_dim = lp->ard_dim; tp[0].variance = lp->variance; tp[0].inv_ls = lp->inv_ls; tp[0].param = lp->param;
    for (int k = 0; k < MAX_ARD; ++k) tp[0].ard[k] = lp->ard[k];
  } else if (t < MAX_TERMS) {
    tp[t] = lp->extra[t - 1];
  }
}

// Threads t < GRAD_TERM_SLOTS: the CTA's sum of slot t (fixed order over the warps), scaled as a gradient: ∂K/∂θ carries the
// term's variance (∂K/∂variance does not) and ∂/∂ard_k the 1 / ard_k of ard_factor.  Absent slots are 0.
__device__ __forceinline__ double cta_slot_sum(const TermParams* tp, int nterms, bool ard, int D, double (*wsum)[8]) {
  const int t = threadIdx.x, u = t / GRAD_TERM_STRIDE, j = t % GRAD_TERM_STRIDE;
  double s = 0.0;
  if (u < nterms && (j < 3 || (ard && tp[u].ard_dim && j - 3 < D))) {
    for (int w = 0; w < 8; ++w) s += wsum[t][w];
    if (j >= 1) s *= tp[u].variance;
    if (j >= 3) s /= tp[u].ard[j - 3];
  }
  return s;
}

// grid (chunks of the lower triangle, latents), storage as kgrad_ard_kernel.  partial[(lat*nchunks + chunk)*GRAD_TERM_SLOTS
// + t*GRAD_TERM_STRIDE + {0, 1, 2, 3 + k}] = <G, ∂K/∂{variance_t, s_t, param_t, ard_t[k]}> of the chunk; unused slots 0.
// NTMAX / ARDANY bound the terms and ARD use of the batch, so a batch of small kernels gets the registers it needs only.
template <int NTMAX, bool ARDANY>
__global__ void __launch_bounds__(256, (NTMAX <= 2 && !ARDANY) ? 2 : 1) kgrad_terms_kernel(const double* __restrict__ mat_base, size_t mat_batch_stride, int off_per_lat,
                                                          const double* __restrict__ x, int N, int D,
                                                          const LatentParams* __restrict__ params, const double* __restrict__ alpha,
                                                          size_t alpha_stride, int form, double* __restrict__ partial) {
  extern __shared__ __align__(16) double sm[];
  double* xa = sm;  // raw points
  double* xb = xa + TILE * D;
  double* aa = xb + TILE * D;
  double* ab = aa + TILE;
  __shared__ TermParams tp[MAX_TERMS];
  __shared__ double wsum[GRAD_TERM_SLOTS][8];
  const int lat = blockIdx.y, tl = blockIdx.x, t = threadIdx.x;
  const LatentParams* lp = params + lat;
  int I = (int)((sqrt(8.0 * (double)tl + 1.0) - 1.0) * 0.5);
  while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tl) ++I;
  while ((size_t)I * (I + 1) / 2 > (size_t)tl) --I;
  const int J = tl - (int)((size_t)I * (I + 1) / 2);
  const double* al = alpha + (size_t)lat * alpha_stride;
  stage_terms(lp, tp);
  for (int i = t; i < TILE * D; i += 256) {
    const int ra = I * TILE + i / D, rb = J * TILE + i / D;
    xa[i] = ra < N ? x[(size_t)ra * D + i % D] : 0.0;
    xb[i] = rb < N ? x[(size_t)rb * D + i % D] : 0.0;
  }
  if (t < TILE) {
    aa[t] = (I * TILE + t < N) ? al[I * TILE + t] : 0.0;
    ab[t] = (J * TILE + t < N) ? al[J * TILE + t] : 0.0;
  }
  __syncthreads();
  const int nterms = lp->nterms;
  const bool product = lp->compose == 2;
  bool ard = false;
  for (int u = 0; u < nterms; ++u) ard |= tp[u].ard_dim > 0;
  const double* base = mat_base + (size_t)lat * mat_batch_stride;
  const int off = lat * off_per_lat;
#define LMM_TERMS_CASE(n, a)                                                                           \
  if constexpr (n <= NTMAX && (ARDANY || !a))                                                          \
    if (nterms == n && ard == a) kgrad_terms_body<n, a>(tp, product, base, off, xa, xb, aa, ab, I, J, N, D, form, wsum);
  LMM_TERMS_CASE(1, false) LMM_TERMS_CASE(1, true) LMM_TERMS_CASE(2, false) LMM_TERMS_CASE(2, true)
  LMM_TERMS_CASE(3, false) LMM_TERMS_CASE(3, true) LMM_TERMS_CASE(4, false) LMM_TERMS_CASE(4, true)
#undef LMM_TERMS_CASE
  __syncthreads();
  if (t < GRAD_TERM_SLOTS) partial[((size_t)lat * gridDim.x + tl) * GRAD_TERM_SLOTS + t] = cta_slot_sum(tp, nterms, ard, D, wsum);
}
// out[lat*GRAD_TERM_SLOTS + slot] = Σ chunks (fixed order)
__global__ void __launch_bounds__(256) kgrad_terms_finish_kernel(const double* __restrict__ partial, int nchunks, double* __restrict__ out) {
  __shared__ double red[256];
  const int lat = blockIdx.x, slot = blockIdx.y, t = threadIdx.x;
  double s = 0.0;
  for (int i = t; i < nchunks; i += 256) s += partial[((size_t)lat * nchunks + i) * GRAD_TERM_SLOTS + slot];
  red[t] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  if (t == 0) out[(size_t)lat * GRAD_TERM_SLOTS + slot] = red[0];
}
cudaError_t launch_kgrad_terms(cudaStream_t st, const double* mat_base, size_t mat_batch_stride, int off_per_lat, const double* x, int N,
                               int D, const LatentParams* params, int nlat, int max_terms, bool any_ard, const double* alpha, size_t alpha_stride,
                               int form, double* partial, double* out) {
  const size_t smem = (size_t)(2 * TILE * D + 2 * TILE) * sizeof(double);
  const int ntn = (N + TILE - 1) / TILE;
  const int nchunks = (int)sym_tiles(ntn);
  dim3 grid((unsigned)nchunks, (unsigned)nlat);
  auto kern = any_ard ? (max_terms <= 1 ? kgrad_terms_kernel<1, true> : max_terms == 2 ? kgrad_terms_kernel<2, true>
                                          : max_terms == 3 ? kgrad_terms_kernel<3, true> : kgrad_terms_kernel<4, true>)
                      : (max_terms <= 1 ? kgrad_terms_kernel<1, false> : max_terms == 2 ? kgrad_terms_kernel<2, false>
                                          : max_terms == 3 ? kgrad_terms_kernel<3, false> : kgrad_terms_kernel<4, false>);
  if (smem + 4096 > 48 * 1024) {  // static shared memory counts against the default limit too
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<grid, 256, smem, st>>>(mat_base, mat_batch_stride, off_per_lat, x, N, D, params, alpha, alpha_stride, form, partial);
  dim3 g2((unsigned)nlat, (unsigned)GRAD_TERM_SLOTS);
  kgrad_terms_finish_kernel<<<g2, 256, 0, st>>>(partial, nchunks, out);
  return cudaGetLastError();
}

// ---- posterior-predictive gradient: the rectangular cross block K(x, x*) ----------------------------------------------
// The posterior-predictive logpdf depends on K(x, x*) through the predictive mean and covariance; its derivative w.r.t.
// that block is Gc = G + u v' (N x N*, rows: training points, columns: test points).  Every element counts once: the block
// has no diagonal, so point identity plays no role (two equal points have d = 0 like any other pair).
template <int NT, bool ARD>
__device__ __forceinline__ void kgrad_cross_body(const TermParams* tp, bool product, const double* __restrict__ tile, const double* xa,
                                                 const double* xb, const double* ua, const double* vb, int R, int J, int Na, int Nb, int D,
                                                 int form, double (*wsum)[8]) {
  double acc[NT][3], aca[ARD ? NT : 1][MAX_ARD];
#pragma unroll
  for (int u = 0; u < NT; ++u) {
    acc[u][0] = acc[u][1] = acc[u][2] = 0.0;
#pragma unroll
    for (int k = 0; k < MAX_ARD; ++k) aca[ARD ? u : 0][k] = 0.0;
  }
  for (int e = threadIdx.x; e < TT; e += 256) {
    const int c = ((e >> 9) << 2) + (e & 3), r = (e >> 2) & 127;  // tile_rc: coalesced reads of the tile
    if (R * TILE + r >= Na || J * TILE + c >= Nb) continue;
    const double w = tile[e] + ua[r] * vb[c];
    const double* pa = xa + (size_t)r * D;
    const double* pb = xb + (size_t)c * D;
    double kap[NT], ds[NT], dp[NT], wa[NT];
#pragma unroll
    for (int u = 0; u < NT; ++u) term_grad(tp[u], pa, pb, D, form, kap[u], ds[u], dp[u], wa[u]);
    accumulate_terms<NT, ARD>(tp, product, w, kap, ds, dp, wa, pa, pb, D, acc, aca);
  }
  warp_term_sums<NT, ARD>(acc, aca, wsum);
}

// grid (tiles of G, latents).  partial[(lat*ntiles + tile)*GRAD_TERM_SLOTS + slot] as kgrad_terms_kernel; points RAW
// ([Na][D] rows, [Nb][D] columns).  NTMAX / ARDANY as kgrad_terms_kernel.
template <int NTMAX, bool ARDANY>
__global__ void __launch_bounds__(256, (NTMAX <= 2 && !ARDANY) ? 2 : 1) kgrad_cross_terms_kernel(TiledRect G, const double* __restrict__ xa_raw, int Na,
                                                                                               const double* __restrict__ xb_raw, int Nb, int D,
                                                                                               const LatentParams* __restrict__ params,
                                                                                               const double* __restrict__ u, size_t u_stride,
                                                                                               const double* __restrict__ v, size_t v_stride, int form,
                                                                                               double* __restrict__ partial) {
  extern __shared__ __align__(16) double sm[];
  double* xa = sm;
  double* xb = xa + TILE * D;
  double* ua = xb + TILE * D;
  double* vb = ua + TILE;
  __shared__ TermParams tp[MAX_TERMS];
  __shared__ double wsum[GRAD_TERM_SLOTS][8];
  const int lat = blockIdx.y, tl = blockIdx.x, t = threadIdx.x;
  const int R = tl / G.ntc, J = tl % G.ntc;
  const LatentParams* lp = params + lat;
  stage_terms(lp, tp);
  for (int i = t; i < TILE * D; i += 256) {
    const int ra = R * TILE + i / D, rb = J * TILE + i / D;
    xa[i] = ra < Na ? xa_raw[(size_t)ra * D + i % D] : 0.0;
    xb[i] = rb < Nb ? xb_raw[(size_t)rb * D + i % D] : 0.0;
  }
  if (t < TILE) {
    ua[t] = R * TILE + t < Na ? u[(size_t)lat * u_stride + R * TILE + t] : 0.0;
    vb[t] = J * TILE + t < Nb ? v[(size_t)lat * v_stride + J * TILE + t] : 0.0;
  }
  __syncthreads();
  const int nterms = lp->nterms;
  const bool product = lp->compose == 2;
  bool ard = false;
  for (int q = 0; q < nterms; ++q) ard |= tp[q].ard_dim > 0;
  const double* tile = G.tile(lat, R, J);
#define LMM_CROSS_CASE(n, a)                                                                           \
  if constexpr (n <= NTMAX && (ARDANY || !a))                                                          \
    if (nterms == n && ard == a) kgrad_cross_body<n, a>(tp, product, tile, xa, xb, ua, vb, R, J, Na, Nb, D, form, wsum);
  LMM_CROSS_CASE(1, false) LMM_CROSS_CASE(1, true) LMM_CROSS_CASE(2, false) LMM_CROSS_CASE(2, true)
  LMM_CROSS_CASE(3, false) LMM_CROSS_CASE(3, true) LMM_CROSS_CASE(4, false) LMM_CROSS_CASE(4, true)
#undef LMM_CROSS_CASE
  __syncthreads();
  if (t < GRAD_TERM_SLOTS) partial[((size_t)lat * gridDim.x + tl) * GRAD_TERM_SLOTS + t] = cta_slot_sum(tp, nterms, ard, D, wsum);
}

cudaError_t launch_kgrad_cross_terms(cudaStream_t st, TiledRect G, const double* xa, int Na, const double* xb, int Nb, int D,
                                     const LatentParams* params, int nlat, int max_terms, bool any_ard, const double* u, size_t u_stride,
                                     const double* v, size_t v_stride, int form, double* partial, double* out) {
  const size_t smem = (size_t)(2 * TILE * D + 2 * TILE) * sizeof(double);
  const int ntiles_ = G.ntr * G.ntc;
  dim3 grid((unsigned)ntiles_, (unsigned)nlat);
  auto kern = any_ard ? (max_terms <= 1 ? kgrad_cross_terms_kernel<1, true> : max_terms == 2 ? kgrad_cross_terms_kernel<2, true>
                                          : max_terms == 3 ? kgrad_cross_terms_kernel<3, true> : kgrad_cross_terms_kernel<4, true>)
                      : (max_terms <= 1 ? kgrad_cross_terms_kernel<1, false> : max_terms == 2 ? kgrad_cross_terms_kernel<2, false>
                                          : max_terms == 3 ? kgrad_cross_terms_kernel<3, false> : kgrad_cross_terms_kernel<4, false>);
  if (smem + 4096 > 48 * 1024) {  // static shared memory counts against the default limit too
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<grid, 256, smem, st>>>(G, xa, Na, xb, Nb, D, params, u, u_stride, v, v_stride, form, partial);
  dim3 g2((unsigned)nlat, (unsigned)GRAD_TERM_SLOTS);
  kgrad_terms_finish_kernel<<<g2, 256, 0, st>>>(partial, ntiles_, out);
  return cudaGetLastError();
}

// M(r, c) += s v_r v_c on the stored (lower) tiles of a batch of packed-lower matrices; grid (tiles, batch).
__global__ void __launch_bounds__(256) sym_rank1_kernel(TiledSym M, const double* __restrict__ v, size_t v_stride, double s) {
  const int b = blockIdx.y, tl = blockIdx.x;
  int I = (int)((sqrt(8.0 * (double)tl + 1.0) - 1.0) * 0.5);
  while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tl) ++I;
  while ((size_t)I * (I + 1) / 2 > (size_t)tl) --I;
  const int J = tl - (int)((size_t)I * (I + 1) / 2);
  double* tile = M.tile(b, I, J);
  const double* vb = v + (size_t)b * v_stride;
  for (int e = threadIdx.x; e < TT; e += 256) {
    int r, c;
    tile_rc(e, r, c);
    tile[e] = fma(s * vb[I * TILE + r], vb[J * TILE + c], tile[e]);
  }
}
cudaError_t launch_sym_rank1(cudaStream_t st, TiledSym M, int batch, const double* v, size_t v_stride, double s) {
  dim3 grid((unsigned)sym_tiles(M.nt), (unsigned)batch);
  sym_rank1_kernel<<<grid, 256, 0, st>>>(M, v, v_stride, s);
  return cudaGetLastError();
}

// ---- missing-data (heterotopic) dense model: contraction over the observed-entry matrix ----------------------------------
// Rows and columns a of the (nobs x nobs) matrix are the observed entries obs[a] = j_a*N + i_a (output j_a at input i_a),
// C_ab = Σ_l H[j_a,l] H[j_b,l] k_l(x_{i_a}, x_{i_b}) + σ² [a = b].  Per latent l and term t the hyper-parameter gradient is
// Σ_ab G_ab H[j_a,l] H[j_b,l] ∂k_l/∂θ_t; d/dH needs the row sums v_l(a) = Σ_b G_ab H[j_b,l] k_l(a,b).  Every entry pair
// couples every latent, so one CTA per lower tile reads its block of -C⁻¹ ONCE -- a 32-row strip at a time, into
// registers -- and loops over all latents and terms on it.  The kernel diagonal is decided by point identity
// (i_a == i_b: κ = 1, no derivative but d/d variance, as kernel_pair in the value path); the factor 2 of the off-diagonal
// lower triangle by entry identity (a != b).
constexpr int MSTRIP = 32;  // rows of a strip: 16 elements per thread

// One latent on one strip.  Thread t = (warp w, lane) holds rows 8gi + lane/4 (gi < 4) and columns 16w + 4h + lane%4 (h < 4)
// of the strip; sg[4gi + h][t] is G there (0 outside the lower triangle and past nobs: padding rows hold the identity).  The
// row sums Σ_h G H[j_b,l] k_l are reduced over the 4 lanes of a row and written to rowred[w][row]; the column sums
// Σ_gi G H[j_a,l] k_l (entry-diagonal elements excluded: they count once, in the row sums) are left in scs[h][t]; the per-slot
// sums are warp-reduced into wsum[slot][warp] as in kgrad_terms_body.  The 16 elements are a loop, not unrolled: one copy of
// the term derivatives per instantiation.
template <int NT, bool ARD>
__device__ __forceinline__ void kgrad_masked_body(const TermParams* tp, bool product, double (*sg)[256], const double* xa, const double* xb,
                                                  const int* pta, const int* ptb, const int* ja, const int* jb,
                                                  const double* __restrict__ Hl, int D, int form, int rbase, int cbase, bool diag_tile,
                                                  double (*rowred)[MSTRIP], double (*scs)[256], double (*wsum)[8]) {
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  double acc[NT][3], aca[ARD ? NT : 1][MAX_ARD];
#pragma unroll
  for (int u = 0; u < NT; ++u) {
    acc[u][0] = acc[u][1] = acc[u][2] = 0.0;
#pragma unroll
    for (int k = 0; k < MAX_ARD; ++k) aca[ARD ? u : 0][k] = 0.0;
  }
#pragma unroll
  for (int h = 0; h < 4; ++h) scs[h][t] = 0.0;
  double rsum = 0.0, hr = 0.0;
#pragma unroll 1
  for (int e = 0; e < 16; ++e) {
    const int gi = e >> 2, h = e & 3;
    const int r = rbase + 8 * gi, c = cbase + 4 * h;
    if (h == 0) hr = Hl[ja[r]];
    const double G = sg[e][t];
    if (G != 0.0) {  // every contribution carries G: outside the triangle, padding, or an exact zero
      const bool same_entry = diag_tile && r == c;
      const double* pa = xa + (size_t)r * D;
      const double* pb = xb + (size_t)c * D;
      double kap[NT], ds[NT], dp[NT], wa[NT];
      if (pta[r] == ptb[c]) {  // same input point: κ(0) = 1, only the variances have a derivative
#pragma unroll
        for (int u = 0; u < NT; ++u) { kap[u] = 1.0; ds[u] = dp[u] = wa[u] = 0.0; }
      } else {
#pragma unroll
        for (int u = 0; u < NT; ++u) term_grad(tp[u], pa, pb, D, form, kap[u], ds[u], dp[u], wa[u]);
      }
      const double hc = Hl[jb[c]];
      const double w2 = (same_entry ? G : 2.0 * G) * (hr * hc);
      double suf[NT + 1];
      suf[NT] = 1.0;
      double kval = 0.0;  // k_l(a, b) of the whole latent kernel
      if (product) {
#pragma unroll
        for (int u = NT - 1; u >= 0; --u) suf[u] = suf[u + 1] * (tp[u].variance * kap[u]);
        kval = suf[0];
      } else {
#pragma unroll
        for (int u = 0; u < NT; ++u) kval = fma(tp[u].variance, kap[u], kval);
      }
      double pre = 1.0;
#pragma unroll
      for (int u = 0; u < NT; ++u) {
        const double w = product ? w2 * pre * suf[u + 1] : w2;
        if (product) pre *= tp[u].variance * kap[u];
        acc[u][0] = fma(w, kap[u], acc[u][0]);
        acc[u][1] = fma(w, ds[u], acc[u][1]);
        acc[u][2] = fma(w, dp[u], acc[u][2]);
        if (ARD && tp[u].ard_dim && wa[u] != 0.0) {
          const double wk = w * wa[u];
#pragma unroll
          for (int k = 0; k < MAX_ARD; ++k)
            if (k < D) aca[ARD ? u : 0][k] = fma(wk, ard_factor(tp[u], pa, pb, k), aca[ARD ? u : 0][k]);
        }
      }
      rsum = fma(G * hc, kval, rsum);
      if (!same_entry) scs[h][t] = fma(G * hr, kval, scs[h][t]);
    }
    if (h == 3) {  // row 8gi + lane/4 done on this thread: the 4 lanes sharing it hold the warp's 16 columns
      rsum += __shfl_xor_sync(0xffffffffu, rsum, 1);
      rsum += __shfl_xor_sync(0xffffffffu, rsum, 2);
      if ((lane & 3) == 0) rowred[warp][8 * gi + (lane >> 2)] = rsum;
      rsum = 0.0;
    }
  }
#pragma unroll
  for (int u = 0; u < NT; ++u) {
#pragma unroll
    for (int j = 0; j < (ARD ? GRAD_TERM_STRIDE : 3); ++j) {
      double v = j < 3 ? acc[u][j] : aca[ARD ? u : 0][j - 3];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
      if (lane == 0) wsum[u * GRAD_TERM_STRIDE + j][warp] = v;
    }
  }
}

// grid (lower tiles of the nobs x nobs matrix).  Per latent l and tile tl (all in fixed order, no atomics):
//   tpart[(l*ntl + tl)*GRAD_TERM_SLOTS + slot]  per-term slots as kgrad_terms_kernel (summed over the tile's 4 strips),
//   rowpart[(l*ntl + tl)*TILE + r]  Σ_c G_rc H[j_c,l] k_l(r,c) over the tile's lower-triangle columns,
//   colpart[(l*ntl + tl)*TILE + c]  Σ_r G_rc H[j_r,l] k_l(r,c) over its rows, the entry diagonal excluded.
// NTMAX / ARDANY bound the terms and ARD use of all latents (register budget as kgrad_terms_kernel).
template <int NTMAX, bool ARDANY>
__global__ void __launch_bounds__(256, (NTMAX <= 2 && !ARDANY) ? 2 : 1) kgrad_masked_kernel(TiledSym negCinv, const int* __restrict__ obs, int nobs,
                                                                                          const double* __restrict__ x, int N, int D,
                                                                                          const LatentParams* __restrict__ params, int m, int p,
                                                                                          const double* __restrict__ Hm, const double* __restrict__ alpha,
                                                                                          int form, double* __restrict__ tpart,
                                                                                          double* __restrict__ rowpart, double* __restrict__ colpart) {
  extern __shared__ __align__(16) double sm[];
  double* xa = sm;  // raw points of the tile's row entries
  double* xb = xa + TILE * D;
  double* aa = xb + TILE * D;
  double* ab = aa + TILE;
  double(*sg)[256] = reinterpret_cast<double(*)[256]>(ab + TILE);  // the strip's G, one column per thread
  double(*scs)[256] = sg + 16;                                      // the thread's column sums
  __shared__ int pta[TILE], ptb[TILE], ja[TILE], jb[TILE];  // input point and output of the row / column entries
  __shared__ TermParams tp[MAX_TERMS];
  __shared__ double wsum[GRAD_TERM_SLOTS][8];
  __shared__ double rowred[8][MSTRIP];
  const int tl = blockIdx.x, ntl = gridDim.x, t = threadIdx.x, w = t >> 5, lane = t & 31;
  int I = (int)((sqrt(8.0 * (double)tl + 1.0) - 1.0) * 0.5);
  while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tl) ++I;
  while ((size_t)I * (I + 1) / 2 > (size_t)tl) --I;
  const int J = tl - (int)((size_t)I * (I + 1) / 2);
  const bool diag_tile = I == J;
  if (t < TILE) {
    const int gr = I * TILE + t, gc = J * TILE + t;
    const int oa = gr < nobs ? obs[gr] : 0, ob = gc < nobs ? obs[gc] : 0;
    ja[t] = oa / N; pta[t] = oa % N;
    jb[t] = ob / N; ptb[t] = ob % N;
    aa[t] = gr < nobs ? alpha[gr] : 0.0;
    ab[t] = gc < nobs ? alpha[gc] : 0.0;
  }
  __syncthreads();
  for (int i = t; i < TILE * D; i += 256) {
    const int r = i / D, k = i % D;
    xa[i] = x[(size_t)pta[r] * D + k];
    xb[i] = x[(size_t)ptb[r] * D + k];
  }
  const double* tile = negCinv.tile(0, I, J);
  const int cbase = 16 * w + (lane & 3);
  for (int s = 0; s < TILE / MSTRIP; ++s) {
    const int rbase = MSTRIP * s + (lane >> 2);
    // the strip's 32 x 128 block of -C⁻¹, read once for all latents (only thread t reads sg[.][t] back)
#pragma unroll
    for (int gi = 0; gi < 4; ++gi)
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int r = rbase + 8 * gi, c = cbase + 4 * h;
        const double nc = tile[(4 * w + h) * 512 + (4 * s + gi) * 32 + lane];  // = tile_elem(r, c): 256 B per warp
        const bool in = I * TILE + r < nobs && J * TILE + c < nobs && (!diag_tile || c <= r);
        sg[4 * gi + h][t] = in ? 0.5 * (aa[r] * ab[c] + nc) : 0.0;
      }
    for (int l = 0; l < m; ++l) {
      const LatentParams* lp = params + l;
      if (t == 0) {
        tp[0].kind = lp->kind; tp[0].ard_dim = lp->ard_dim; tp[0].variance = lp->variance; tp[0].inv_ls = lp->inv_ls; tp[0].param = lp->param;
        for (int k = 0; k < MAX_ARD; ++k) tp[0].ard[k] = lp->ard[k];
      } else if (t < MAX_TERMS) {
        tp[t] = lp->extra[t - 1];
      }
      __syncthreads();  // also orders the staged points (first pass) and the previous latent's reads of wsum / rowred
      const int nterms = lp->nterms;
      const bool product = lp->compose == 2;
      bool ard = false;
      for (int u = 0; u < nterms; ++u) ard |= tp[u].ard_dim > 0;
      const double* Hl = Hm + (size_t)l * p;
#define LMM_MASKED_CASE(n, a)                                                                                                  \
  if constexpr (n <= NTMAX && (ARDANY || !a))                                                                                \
    if (nterms == n && ard == a)                                                                                             \
      kgrad_masked_body<n, a>(tp, product, sg, xa, xb, pta, ptb, ja, jb, Hl, D, form, rbase, cbase, diag_tile, rowred, scs, wsum);
      LMM_MASKED_CASE(1, false) LMM_MASKED_CASE(1, true) LMM_MASKED_CASE(2, false) LMM_MASKED_CASE(2, true)
      LMM_MASKED_CASE(3, false) LMM_MASKED_CASE(3, true) LMM_MASKED_CASE(4, false) LMM_MASKED_CASE(4, true)
#undef LMM_MASKED_CASE
      // columns: the 8 lanes sharing lane % 4 hold one column's 32 rows of the strip; the column belongs to this warp only
      double cv = 0.0;
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        double v = scs[h][t];
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        v += __shfl_xor_sync(0xffffffffu, v, 8);
        v += __shfl_xor_sync(0xffffffffu, v, 16);
        if ((lane >> 2) == h) cv = v;
      }
      __syncthreads();
      const size_t lt = (size_t)l * ntl + tl;
      if (lane < 16) {
        double* dst = colpart + lt * TILE + cbase + 4 * (lane >> 2);
        *dst = s == 0 ? cv : *dst + cv;  // the same thread adds the strips in order
      }
      if (t < MSTRIP) {
        double v = 0.0;
        for (int k = 0; k < 8; ++k) v += rowred[k][t];
        rowpart[lt * TILE + MSTRIP * s + t] = v;
      }
      if (t < GRAD_TERM_SLOTS) {
        const int u = t / GRAD_TERM_STRIDE, j = t % GRAD_TERM_STRIDE;
        double v = 0.0;
        if (u < nterms && (j < 3 || (ard && tp[u].ard_dim && j - 3 < D))) {
          for (int k = 0; k < 8; ++k) v += wsum[t][k];
          if (j >= 1) v *= tp[u].variance;  // ∂K/∂θ carries the term's variance (∂K/∂variance does not)
          if (j >= 3) v /= tp[u].ard[j - 3];
        }
        double* dst = tpart + lt * GRAD_TERM_SLOTS + t;
        *dst = s == 0 ? v : *dst + v;
      }
      __syncthreads();
    }
  }
}

// v[l*nobs + a] = Σ_{J <= A} rowpart[(A,J)] + Σ_{I >= A} colpart[(I,A)] (A = a / 128), in that order: grid (ceil(nobs/256), m)
__global__ void __launch_bounds__(256) kgrad_masked_rows_kernel(const double* __restrict__ rowpart, const double* __restrict__ colpart, int nobs,
                                                                int nt, double* __restrict__ v) {
  const int a = blockIdx.x * 256 + threadIdx.x, l = blockIdx.y;
  if (a >= nobs) return;
  const size_t ntl = sym_tiles(nt);
  const int A = a / TILE, r = a % TILE;
  const double* rp = rowpart + (size_t)l * ntl * TILE;
  const double* cp = colpart + (size_t)l * ntl * TILE;
  double s = 0.0;
  for (int J = 0; J <= A; ++J) s += rp[sym_tile_index(A, J) * TILE + r];
  for (int I = A; I < nt; ++I) s += cp[sym_tile_index(I, A) * TILE + r];
  v[(size_t)l * nobs + a] = s;
}

// gH[l*p + j] = 2 Σ_{a in [seg[j], seg[j+1])} v[l*nobs + a] (obs is sorted by outputs); grid (p, m).  An output with no
// observed entry gets exactly 0.
__global__ void __launch_bounds__(256) kgrad_masked_outputs_kernel(const double* __restrict__ v, const int* __restrict__ seg, int nobs, int p,
                                                                   double* __restrict__ gH) {
  __shared__ double red[256];
  const int j = blockIdx.x, l = blockIdx.y, t = threadIdx.x;
  double s = 0.0;
  for (int a = seg[j] + t; a < seg[j + 1]; a += 256) s += v[(size_t)l * nobs + a];
  red[t] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  if (t == 0) gH[(size_t)l * p + j] = 2.0 * red[0];
}

// out[0] = Σ_a (-C⁻¹)_aa over the nobs observed entries (fixed order, one block)
__global__ void __launch_bounds__(256) sym_diag_sum_kernel(TiledSym M, int n, double* __restrict__ out) {
  __shared__ double red[256];
  const int t = threadIdx.x;
  double s = 0.0;
  for (int a = t; a < n; a += 256) s += M.tile(0, a / TILE, a / TILE)[tile_elem(a % TILE, a % TILE)];
  red[t] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  if (t == 0) out[0] = red[0];
}

cudaError_t launch_kgrad_masked(cudaStream_t st, TiledSym negCinv, const int* obs, int nobs, const double* x, int N, int D, const LatentParams* params,
                                int m, int p, const double* Hm, const double* alpha, int max_terms, bool any_ard, int form, const int* seg,
                                double* tpart, double* rowpart, double* colpart, double* v, double* out_terms, double* out_H, double* out_diag) {
  const size_t smem = (size_t)(2 * TILE * D + 2 * TILE + 20 * 256) * sizeof(double);
  const int nt = negCinv.nt;
  const int ntl = (int)sym_tiles(nt);
  auto kern = any_ard ? (max_terms <= 1 ? kgrad_masked_kernel<1, true> : max_terms == 2 ? kgrad_masked_kernel<2, true>
                                          : max_terms == 3 ? kgrad_masked_kernel<3, true> : kgrad_masked_kernel<4, true>)
                      : (max_terms <= 1 ? kgrad_masked_kernel<1, false> : max_terms == 2 ? kgrad_masked_kernel<2, false>
                                          : max_terms == 3 ? kgrad_masked_kernel<3, false> : kgrad_masked_kernel<4, false>);
  if (smem + 8192 > 48 * 1024) {  // static shared memory counts against the default limit too
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<(unsigned)ntl, 256, smem, st>>>(negCinv, obs, nobs, x, N, D, params, m, p, Hm, alpha, form, tpart, rowpart, colpart);
  dim3 g2((unsigned)m, (unsigned)GRAD_TERM_SLOTS);
  kgrad_terms_finish_kernel<<<g2, 256, 0, st>>>(tpart, ntl, out_terms);
  dim3 g3((unsigned)((nobs + 255) / 256), (unsigned)m);
  kgrad_masked_rows_kernel<<<g3, 256, 0, st>>>(rowpart, colpart, nobs, nt, v);
  dim3 g4((unsigned)p, (unsigned)m);
  kgrad_masked_outputs_kernel<<<g4, 256, 0, st>>>(v, seg, nobs, p, out_H);
  sym_diag_sum_kernel<<<1, 256, 0, st>>>(negCinv, nobs, out_diag);
  return cudaGetLastError();
}

// v[i] = a[i] * sa - b[i]
__global__ void scale_sub_kernel(double* __restrict__ v, const double* __restrict__ a, double sa, const double* __restrict__ b, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = a[i] * sa - b[i];
}
cudaError_t launch_scale_sub(cudaStream_t st, double* v, const double* a, double sa, const double* b, size_t n) {
  scale_sub_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(v, a, sa, b, n);
  return cudaGetLastError();
}

}  // namespace lmm
