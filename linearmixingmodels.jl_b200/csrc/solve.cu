// Triangular vector solves, quadratic form and prediction reductions on the tiled factor
// (K8/K9/K10 of SURVEY.md §2.3; reference: AbstractGPs `C.U' \ δ`, `C \ δ`, posterior mean / var
// reached from src/oilmm.jl:90,128,61).  All of these read each 128 KB tile exactly once:
// HBM-bound GEMV-shaped work.  With W(J) = inv(L_JJ) from the panel kernel a solve is a chain of
// nt column steps:  z_J = W_J r_J ;  r_I -= L(I,J) z_J  (I > J)   -- one launch per step, all
// tiles of the column (and all latents) in parallel.
#include "common.cuh"
#include "kernels.h"

namespace lmm {

// Per-thread partial products of y = T x over one tile (interleaved layout), 256 threads.
// Thread t, iteration it touches element e = it*256 + t:  row = ((it&1)*8 + warp)*8 + (t>>2)&7,
// col = (it>>1)*4 + (t&3).  acc0 collects even it (row rlo), acc1 odd it (row rlo + 64).
__device__ __forceinline__ void tile_gemv_n_acc(const double* __restrict__ tile, const double* xs, double& acc0, double& acc1) {
  const int t = threadIdx.x;
#pragma unroll 8
  for (int it = 0; it < 64; it += 2) {
    const double x = xs[(it >> 1) * 4 + (t & 3)];
    acc0 = fma(tile[it * 256 + t], x, acc0);
    acc1 = fma(tile[(it + 1) * 256 + t], x, acc1);
  }
}
// Finish: quad-reduce and scatter to ys[128] (shared).  Caller syncs afterwards.
__device__ __forceinline__ void tile_gemv_n_finish(double acc0, double acc1, double* ys) {
  const int t = threadIdx.x;
  acc0 += __shfl_xor_sync(0xffffffffu, acc0, 1);
  acc0 += __shfl_xor_sync(0xffffffffu, acc0, 2);
  acc1 += __shfl_xor_sync(0xffffffffu, acc1, 1);
  acc1 += __shfl_xor_sync(0xffffffffu, acc1, 2);
  if ((t & 3) == 0) {
    const int rlo = (t >> 5) * 8 + ((t >> 2) & 7);
    ys[rlo] = acc0;
    ys[rlo + 64] = acc1;
  }
}
// y = T^T x over one tile: ys[c] = sum_r T(r,c) xs[r].  part: 8*128 doubles of shared scratch.
// Ends with a __syncthreads(); ys valid for all threads afterwards.
__device__ __forceinline__ void tile_gemv_t(const double* __restrict__ tile, const double* xs, double* ys, double* part) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int rlo = warp * 8 + ((t >> 2) & 7);
  const double x0 = xs[rlo], x1 = xs[rlo + 64];
#pragma unroll 8
  for (int it = 0; it < 64; it += 2) {
    double v = tile[it * 256 + t] * x0;
    v = fma(tile[(it + 1) * 256 + t], x1, v);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    if (lane < 4) part[warp * TILE + (it >> 1) * 4 + lane] = v;
  }
  __syncthreads();
  if (t < TILE) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += part[w * TILE + t];
    ys[t] = s;
  }
  __syncthreads();
}

// grid (nt - J, batch).  rvec: running right-hand side (destroyed), zvec: solution.
// env (nullable): tiles (I, J) with env[b][I] > J are exact zeros that are skipped (they need not be stored).
__global__ void __launch_bounds__(256) fwd_step_kernel(TiledSym L, const double* __restrict__ W, size_t w_batch_stride,
                                                       double* __restrict__ rvec, double* __restrict__ zvec, size_t vec_stride, int J,
                                                       const int* __restrict__ env) {
  __shared__ double xs[TILE], zs[TILE], ys[TILE];
  const int b = blockIdx.y, i = blockIdx.x, t = threadIdx.x;
  if (i > 0 && env && env[(size_t)b * L.nt + J + i] > J) return;  // r_I -= 0
  double* r = rvec + (size_t)b * vec_stride;
  if (t < TILE) xs[t] = r[J * TILE + t];
  __syncthreads();
  double a0 = 0.0, a1 = 0.0;
  tile_gemv_n_acc(W + (size_t)b * w_batch_stride + (size_t)J * TT, xs, a0, a1);
  tile_gemv_n_finish(a0, a1, zs);
  __syncthreads();
  if (i == 0) {
    if (t < TILE) zvec[(size_t)b * vec_stride + J * TILE + t] = zs[t];
    return;
  }
  const int I = J + i;
  a0 = a1 = 0.0;
  tile_gemv_n_acc(L.tile(b, I, J), zs, a0, a1);
  tile_gemv_n_finish(a0, a1, ys);
  __syncthreads();
  if (t < TILE) r[I * TILE + t] -= ys[t];
}

// grid (J + 1, batch).  rvec: running rhs (destroyed), avec: solution of L^T a = r.  env: as fwd_step_kernel.
__global__ void __launch_bounds__(256) bwd_step_kernel(TiledSym L, const double* __restrict__ W, size_t w_batch_stride,
                                                       double* __restrict__ rvec, double* __restrict__ avec, size_t vec_stride, int J,
                                                       const int* __restrict__ env) {
  __shared__ double xs[TILE], as[TILE], ys[TILE];
  __shared__ double part[8 * TILE];
  const int b = blockIdx.y, k = blockIdx.x, t = threadIdx.x;
  if (k < J && env && env[(size_t)b * L.nt + J] > k) return;  // r_k -= 0
  double* r = rvec + (size_t)b * vec_stride;
  if (t < TILE) xs[t] = r[J * TILE + t];
  __syncthreads();
  tile_gemv_t(W + (size_t)b * w_batch_stride + (size_t)J * TT, xs, as, part);
  if (k == J) {
    if (t < TILE) avec[(size_t)b * vec_stride + J * TILE + t] = as[t];
    return;
  }
  tile_gemv_t(L.tile(b, J, k), as, ys, part);
  if (t < TILE) r[k * TILE + t] -= ys[t];
}

// ------------------------------------------------------------------------------------------------
// Persistent sweeps: ONE launch per direction instead of nt dependent launches (VERDICT r01 weak #5: at 8 latents per
// GPU the 128 launches per direction were launch-latency bound, 41 % of HBM peak).
//
// Forward, left-looking by tile ROW: CTA (I, b) owns z_I of latent b,
//     z_I = W_I (rhs_I - sum_{K<I} L(I,K) z_K),
// streams its row panel L(I, 0:I) -- one contiguous run of HBM, each tile read exactly once -- and consumes z_K as soon
// as CTA (K, b) has published it (a per-(b, K) ready flag in global memory: st.release.gpu by the producer after its
// CTA barrier + fence, ld.acquire.gpu by one polling lane of the consumer).  Backward, by tile COLUMN: CTA (J, b) owns
//     a_J = W_J^T (rhs_J - sum_{I>J} L(I,J)^T a_I),   I = nt-1 ... J+1 (the order in which the a_I appear).
// Dependencies only point to CTAs with a LOWER linear block index (rows ascending / columns descending, latent index
// fastest), which the hardware dispatches first, so a resident CTA never waits for one that cannot be scheduled; a
// bounded wait (10 s on %globaltimer) traps instead of hanging the GPU should that ever be violated.
// The tile loads do not depend on the flags: they are issued one 16-value chunk ahead (register double buffer) so a
// CTA that is waiting for z_K already has the first part of tile (I, K) in flight.  Summation order is fixed (per
// thread: K ascending; then lane / warp reduction trees) -> bit-reproducible run to run.
// With the tile envelope (env[b][I]: L(I,K) = 0 for K < env[b][I]) row I starts at K = env[b][I] and column J visits only the rows
// with env[b][I] <= J: the skipped terms are exact zeros, so the sums -- and the solutions -- are those of the full sweep, without
// the loads of the zero tiles or the waits for the blocks they would multiply.  The envelope need not be monotone (unsorted x).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) { asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void wait_ready(const int* flag) {
  if (ld_acquire_gpu(flag) != 0) return;
  const unsigned long long t0 = globaltimer_ns();
  unsigned ns = 32;
  while (ld_acquire_gpu(flag) == 0) {
    __nanosleep(ns);
    if (ns < 512) ns <<= 1;
    if (globaltimer_ns() - t0 > 10000000000ull) __trap();  // never hang the GPU on a scheduling assumption
  }
}
// Warp 0 of the CTA: wait for vector block `blk` of latent-vector `v` and stage it (128 doubles) into xs.
__device__ __forceinline__ void stage_ready_block(const int* flag, const double* __restrict__ v, double* xs, int lane) {
  if (lane == 0) wait_ready(flag);
  __syncwarp();
  const double2* src = reinterpret_cast<const double2*>(v) + lane * 2;
  const double2 p0 = __ldcg(src), p1 = __ldcg(src + 1);  // L2: written by another SM during this kernel
  reinterpret_cast<double2*>(xs)[lane * 2] = p0;
  reinterpret_cast<double2*>(xs)[lane * 2 + 1] = p1;
}
// All threads stored their part of the solution block; publish it.
__device__ __forceinline__ void publish_block(int* flag) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    st_release_gpu(flag, 1);
  }
}

constexpr int SW_CH = 16;  // tile elements per thread per chunk (a 128x128 tile = 4 chunks of 16 for 256 threads)

// grid nt*batch (linear index = I*batch + b), 256 threads.
__global__ void __launch_bounds__(256, 3) fwd_sweep_kernel(TiledSym L, const double* __restrict__ W, size_t w_batch_stride,
                                                           const double* __restrict__ rhs, double* __restrict__ sol, size_t vec_stride,
                                                           int* __restrict__ flags, int batch, const int* __restrict__ env) {
  __shared__ __align__(16) double xs[2][TILE];
  __shared__ double ys[TILE];
  const int I = blockIdx.x / batch, b = blockIdx.x % batch, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int nt = L.nt;
  const int K0 = env ? min(env[(size_t)b * nt + I], I) : 0;  // first tile column of the row that is not zero
  const double* row = L.tile(b, I, K0);  // tiles (I, K0..I-1) are contiguous
  double* zb = sol + (size_t)b * vec_stride;
  int* fl = flags + (size_t)b * nt;
  double a0 = 0.0, a1 = 0.0;
  double buf[SW_CH];
  if (I > K0) {
#pragma unroll
    for (int u = 0; u < SW_CH; ++u) buf[u] = row[u * 256 + t];
  }
  for (int K = K0; K < I; ++K) {
    if (warp == 0) stage_ready_block(fl + K, zb + (size_t)K * TILE, xs[K & 1], lane);
    __syncthreads();
    const double* xk = xs[K & 1];
    const double* tile = row + (size_t)(K - K0) * TT;
#pragma unroll
    for (int c = 0; c < 64 / SW_CH; ++c) {
      double nxt[SW_CH];
      const bool more = (c + 1 < 64 / SW_CH) || (K + 1 < I);
      const double* np = tile + (c + 1) * SW_CH * 256 + t;  // chunk c+1 of this tile == chunk 0 of the next one when c = 3
      if (more) {
#pragma unroll
        for (int u = 0; u < SW_CH; ++u) nxt[u] = np[u * 256];
      }
#pragma unroll
      for (int u = 0; u < SW_CH; u += 2) {
        const double x = xk[((c * SW_CH + u) >> 1) * 4 + (t & 3)];
        a0 = fma(buf[u], x, a0);
        a1 = fma(buf[u + 1], x, a1);
      }
      if (more) {
#pragma unroll
        for (int u = 0; u < SW_CH; ++u) buf[u] = nxt[u];
      }
    }
  }
  // r_I = rhs_I - (row sums) ;  z_I = W_I r_I
  tile_gemv_n_finish(a0, a1, ys);
  __syncthreads();
  double* rs = xs[0];
  if (t < TILE) rs[t] = rhs[(size_t)b * vec_stride + (size_t)I * TILE + t] - ys[t];
  __syncthreads();
  a0 = a1 = 0.0;
  tile_gemv_n_acc(W + (size_t)b * w_batch_stride + (size_t)I * TT, rs, a0, a1);
  tile_gemv_n_finish(a0, a1, ys);
  __syncthreads();
  if (t < TILE) zb[(size_t)I * TILE + t] = ys[t];
  publish_block(fl + I);
}

// Per-thread partial sums of y = T^T x over one tile: thread t holds, for j = 0..31, the column c = 4j + (t&3) restricted
// to its rows rlo = warp*8 + (t>>2)&7 and rlo + 64.  acc[j] += T(rlo, c) x[rlo] + T(rlo+64, c) x[rlo+64].
__device__ __forceinline__ void gemv_t_reduce_store(const double (&acc)[32], double* part, double* ys) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    double v = acc[j];
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    if (lane < 4) part[warp * TILE + j * 4 + lane] = v;
  }
  __syncthreads();
  if (t < TILE) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += part[w * TILE + t];
    ys[t] = s;
  }
  __syncthreads();
}

constexpr int SW_CHB = 8;  // the backward sweep carries 32 accumulators per thread: a shallower prefetch keeps it at 128 registers without spills
// grid nt*batch (linear index = (nt-1-J)*batch + b), 256 threads.
__global__ void __launch_bounds__(256, 2) bwd_sweep_kernel(TiledSym L, const double* __restrict__ W, size_t w_batch_stride,
                                                           const double* __restrict__ rhs, double* __restrict__ sol, size_t vec_stride,
                                                           int* __restrict__ flags, int batch, const int* __restrict__ env) {
  __shared__ __align__(16) double xs[2][TILE];
  __shared__ double ys[TILE];
  __shared__ double part[8 * TILE];
  const int nt = L.nt;
  const int J = nt - 1 - (int)(blockIdx.x / batch), b = blockIdx.x % batch, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int rlo = warp * 8 + ((t >> 2) & 7);
  double* ab = sol + (size_t)b * vec_stride;
  int* fl = flags + (size_t)b * nt;
  const int* eb = env ? env + (size_t)b * nt : nullptr;
  // the next row above I whose tile in column J is inside the envelope; J when there is none
  auto next_row = [&](int r) {
    --r;
    if (eb)
      while (r > J && __ldg(eb + r) > J) --r;
    return r;
  };
  double acc[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) acc[j] = 0.0;
  double buf[SW_CHB];
  int I = next_row(nt);
  if (I > J) {
    const double* tile = L.tile(b, I, J);
#pragma unroll
    for (int u = 0; u < SW_CHB; ++u) buf[u] = tile[u * 256 + t];
  }
  int par = 0;
  for (; I > J; par ^= 1) {
    const int In = next_row(I);
    if (warp == 0) stage_ready_block(fl + I, ab + (size_t)I * TILE, xs[par], lane);
    __syncthreads();
    const double x0 = xs[par][rlo], x1 = xs[par][rlo + 64];
    const double* tile = L.tile(b, I, J);
    const double* tnext = (In > J) ? L.tile(b, In, J) : tile;
#pragma unroll
    for (int c = 0; c < 64 / SW_CHB; ++c) {
      double nxt[SW_CHB];
      const bool more = (c + 1 < 64 / SW_CHB) || (In > J);
      const double* np = (c + 1 < 64 / SW_CHB) ? tile + (c + 1) * SW_CHB * 256 + t : tnext + t;
      if (more) {
#pragma unroll
        for (int u = 0; u < SW_CHB; ++u) nxt[u] = np[u * 256];
      }
#pragma unroll
      for (int u = 0; u < SW_CHB; u += 2) {
        const int j = (c * SW_CHB + u) >> 1;
        acc[j] = fma(buf[u], x0, acc[j]);
        acc[j] = fma(buf[u + 1], x1, acc[j]);
      }
      if (more) {
#pragma unroll
        for (int u = 0; u < SW_CHB; ++u) buf[u] = nxt[u];
      }
    }
    I = In;
  }
  gemv_t_reduce_store(acc, part, ys);
  // r_J = rhs_J - (column sums) ;  a_J = W_J^T r_J
  double* rs = xs[0];
  if (t < TILE) rs[t] = rhs[(size_t)b * vec_stride + (size_t)J * TILE + t] - ys[t];
  __syncthreads();
  tile_gemv_t(W + (size_t)b * w_batch_stride + (size_t)J * TT, rs, ys, part);
  if (t < TILE) ab[(size_t)J * TILE + t] = ys[t];
  publish_block(fl + J);
}

static int g_solve_impl = 1;  // 1: persistent sweeps (default); 0: one launch per tile column
void set_solve_impl(int v) { g_solve_impl = v; }

static cudaError_t sweep_flags(cudaStream_t st, int n, int** out) {
  cudaError_t e = cudaMallocAsync((void**)out, (size_t)n * sizeof(int), st);
  if (e != cudaSuccess) return e;
  return cudaMemsetAsync(*out, 0, (size_t)n * sizeof(int), st);
}

// rvec is the right-hand side; it is left untouched by the persistent sweeps (the stepwise kernels consume it).
cudaError_t launch_fwd_solve(cudaStream_t st, TiledSym L, const double* W, size_t w_batch_stride, double* rvec, double* zvec,
                             size_t vec_stride, int batch, int64_t* launches, const int* env) {
  if (g_solve_impl == 1) {
    int* flags = nullptr;
    cudaError_t e = sweep_flags(st, L.nt * batch, &flags);
    if (e != cudaSuccess) return e;
    fwd_sweep_kernel<<<(unsigned)(L.nt * batch), 256, 0, st>>>(L, W, w_batch_stride, rvec, zvec, vec_stride, flags, batch, env);
    if (launches) ++*launches;
    e = cudaGetLastError();
    cudaFreeAsync(flags, st);
    return e;
  }
  for (int J = 0; J < L.nt; ++J) {
    dim3 grid((unsigned)(L.nt - J), (unsigned)batch);
    fwd_step_kernel<<<grid, 256, 0, st>>>(L, W, w_batch_stride, rvec, zvec, vec_stride, J, env);
    if (launches) ++*launches;
  }
  return cudaGetLastError();
}

cudaError_t launch_bwd_solve(cudaStream_t st, TiledSym L, const double* W, size_t w_batch_stride, double* rvec, double* avec,
                             size_t vec_stride, int batch, int64_t* launches, const int* env) {
  if (g_solve_impl == 1) {
    int* flags = nullptr;
    cudaError_t e = sweep_flags(st, L.nt * batch, &flags);
    if (e != cudaSuccess) return e;
    bwd_sweep_kernel<<<(unsigned)(L.nt * batch), 256, 0, st>>>(L, W, w_batch_stride, rvec, avec, vec_stride, flags, batch, env);
    if (launches) ++*launches;
    e = cudaGetLastError();
    cudaFreeAsync(flags, st);
    return e;
  }
  for (int J = L.nt - 1; J >= 0; --J) {
    dim3 grid((unsigned)(J + 1), (unsigned)batch);
    bwd_step_kernel<<<grid, 256, 0, st>>>(L, W, w_batch_stride, rvec, avec, vec_stride, J, env);
    if (launches) ++*launches;
  }
  return cudaGetLastError();
}

// out[b] = sum v^2, one CTA per latent, fixed summation order.
__global__ void __launch_bounds__(256) sumsq_kernel(const double* __restrict__ v, size_t stride, int n, double* __restrict__ out) {
  __shared__ double red[256];
  const double* p = v + (size_t)blockIdx.x * stride;
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) s = fma(p[i], p[i], s);
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = red[0];
}
cudaError_t launch_sumsq(cudaStream_t st, const double* v, size_t stride, int n, int batch, double* out) {
  sumsq_kernel<<<batch, 256, 0, st>>>(v, stride, n, out);
  return cudaGetLastError();
}

// grid (ntr, batch): y[b][R*128 + r] = (add_mean ? mean_b : 0) + sum_J T(R,J) x[b][J*128 + :]
__global__ void __launch_bounds__(256) rect_gemv_kernel(TiledRect A, const double* __restrict__ x, size_t x_stride,
                                                        double* __restrict__ y, size_t y_stride,
                                                        const LatentParams* __restrict__ params, int add_mean) {
  __shared__ double xs[2][TILE], ys[TILE];
  const int b = blockIdx.y, R = blockIdx.x, t = threadIdx.x;
  const double* xb = x + (size_t)b * x_stride;
  double a0 = 0.0, a1 = 0.0;
  for (int J = 0; J < A.ntc; ++J) {
    if (t < TILE) xs[J & 1][t] = xb[J * TILE + t];
    __syncthreads();
    tile_gemv_n_acc(A.tile(b, R, J), xs[J & 1], a0, a1);
  }
  tile_gemv_n_finish(a0, a1, ys);
  __syncthreads();
  if (t < TILE) y[(size_t)b * y_stride + R * TILE + t] = ys[t] + (add_mean ? params[b].mean : 0.0);
}
cudaError_t launch_rect_gemv(cudaStream_t st, TiledRect A, const double* x, size_t x_stride, double* y, size_t y_stride,
                             const LatentParams* params, int add_mean, int batch) {
  dim3 grid((unsigned)A.ntr, (unsigned)batch);
  rect_gemv_kernel<<<grid, 256, 0, st>>>(A, x, x_stride, y, y_stride, params, add_mean);
  return cudaGetLastError();
}

// grid (ntr, batch): y[b][R*128 + r] = variance_b - sum_J sum_c T(R,J)(r,c)^2   (params == null: the row sums of squares)
__global__ void __launch_bounds__(256) rect_rowsumsq_kernel(TiledRect A, double* __restrict__ y, size_t y_stride,
                                                            const LatentParams* __restrict__ params) {
  __shared__ double ys[TILE];
  const int b = blockIdx.y, R = blockIdx.x, t = threadIdx.x;
  double a0 = 0.0, a1 = 0.0;
  for (int J = 0; J < A.ntc; ++J) {
    const double* tile = A.tile(b, R, J);
#pragma unroll 8
    for (int it = 0; it < 64; it += 2) {
      const double v0 = tile[it * 256 + t], v1 = tile[(it + 1) * 256 + t];
      a0 = fma(v0, v0, a0);
      a1 = fma(v1, v1, a1);
    }
  }
  tile_gemv_n_finish(a0, a1, ys);
  __syncthreads();
  if (t < TILE) y[(size_t)b * y_stride + R * TILE + t] = params ? params[b].kdiag - ys[t] : ys[t];
}
cudaError_t launch_rect_rowsumsq(cudaStream_t st, TiledRect A, double* y, size_t y_stride, const LatentParams* params, int batch) {
  dim3 grid((unsigned)A.ntr, (unsigned)batch);
  rect_rowsumsq_kernel<<<grid, 256, 0, st>>>(A, y, y_stride, params);
  return cudaGetLastError();
}

// grid (nt, batch): y_I = sum_{J <= I} L(I,J) z_J   (diagonal tiles have a zero upper part)
__global__ void __launch_bounds__(256) lower_gemv_kernel(TiledSym L, const double* __restrict__ z, size_t z_stride,
                                                         double* __restrict__ y, size_t y_stride) {
  __shared__ double xs[2][TILE], ys[TILE];
  const int b = blockIdx.y, I = blockIdx.x, t = threadIdx.x;
  const double* zb = z + (size_t)b * z_stride;
  double a0 = 0.0, a1 = 0.0;
  for (int J = 0; J <= I; ++J) {
    if (t < TILE) xs[J & 1][t] = zb[J * TILE + t];
    __syncthreads();
    tile_gemv_n_acc(L.tile(b, I, J), xs[J & 1], a0, a1);
  }
  tile_gemv_n_finish(a0, a1, ys);
  __syncthreads();
  if (t < TILE) y[(size_t)b * y_stride + I * TILE + t] = ys[t];
}
cudaError_t launch_lower_gemv(cudaStream_t st, TiledSym L, const double* z, size_t z_stride, double* y, size_t y_stride, int batch) {
  dim3 grid((unsigned)L.nt, (unsigned)batch);
  lower_gemv_kernel<<<grid, 256, 0, st>>>(L, z, z_stride, y, y_stride);
  return cudaGetLastError();
}

// grid (lower tiles): dense[c*N + r] = L(r, c) for r >= c (dense pre-zeroed by the caller)
__global__ void __launch_bounds__(256) untile_lower_kernel(TiledSym L, int b, double* __restrict__ dense, int N) {
  const int tl = blockIdx.x;
  int I = (int)((sqrt(8.0 * (double)tl + 1.0) - 1.0) * 0.5);
  while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tl) ++I;
  while ((size_t)I * (I + 1) / 2 > (size_t)tl) --I;
  const int J = tl - (int)((size_t)I * (I + 1) / 2);
  const double* tile = L.tile(b, I, J);
  for (int idx = threadIdx.x; idx < TT; idx += 256) {
    const int r = idx & 127, c = idx >> 7;  // coalesced dense writes
    const int gr = I * TILE + r, gc = J * TILE + c;
    if (gr < N && gc < N && gr >= gc) dense[(size_t)gc * N + gr] = tile[tile_elem(r, c)];
  }
}
cudaError_t launch_untile_lower(cudaStream_t st, TiledSym L, int b, double* dense, int N) {
  untile_lower_kernel<<<(unsigned)sym_tiles(L.nt), 256, 0, st>>>(L, b, dense, N);
  return cudaGetLastError();
}

// grid (lower tiles, batch): tiles <- dense symmetric (lower triangle read), identity padding
__global__ void __launch_bounds__(256) tile_from_dense_kernel(TiledSym L, const double* __restrict__ dense, int N) {
  const int tl = blockIdx.x, b = blockIdx.y;
  int I = (int)((sqrt(8.0 * (double)tl + 1.0) - 1.0) * 0.5);
  while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tl) ++I;
  while ((size_t)I * (I + 1) / 2 > (size_t)tl) --I;
  const int J = tl - (int)((size_t)I * (I + 1) / 2);
  double* tile = L.tile(b, I, J);
  const double* A = dense + (size_t)b * N * N;
  for (int idx = threadIdx.x; idx < TT; idx += 256) {
    const int r = idx & 127, c = idx >> 7;
    const int gr = I * TILE + r, gc = J * TILE + c;
    double v;
    if (gr >= N || gc >= N) v = (gr == gc) ? 1.0 : 0.0;
    else v = (gr >= gc) ? A[(size_t)gc * N + gr] : A[(size_t)gr * N + gc];
    tile[tile_elem(r, c)] = v;
  }
}
cudaError_t launch_tile_from_dense(cudaStream_t st, TiledSym L, int batch, const double* dense, int N) {
  dim3 grid((unsigned)sym_tiles(L.nt), (unsigned)batch);
  tile_from_dense_kernel<<<grid, 256, 0, st>>>(L, dense, N);
  return cudaGetLastError();
}

// grid (ntr*ntc, batch): dense block-diagonal scatter of rectangular tiled matrices:
// dense[(b*Na + r) + (b*Nb + c) * ld] = A_b(r, c)   for r < Na, c < Nb   (dense pre-zeroed)
__global__ void __launch_bounds__(256) untile_rect_blockdiag_kernel(TiledRect A, int Na, int Nb, double* __restrict__ dense, size_t ld) {
  const int b = blockIdx.y, R = blockIdx.x / A.ntc, J = blockIdx.x % A.ntc;
  const double* tile = A.tile(b, R, J);
  for (int idx = threadIdx.x; idx < TT; idx += 256) {
    const int r = idx & 127, c = idx >> 7;
    const int gr = R * TILE + r, gc = J * TILE + c;
    if (gr < Na && gc < Nb) dense[((size_t)b * Nb + gc) * ld + (size_t)b * Na + gr] = tile[tile_elem(r, c)];
  }
}
cudaError_t launch_untile_rect_blockdiag(cudaStream_t st, TiledRect A, int batch, int Na, int Nb, double* dense, size_t ld) {
  dim3 grid((unsigned)(A.ntr * A.ntc), (unsigned)batch);
  untile_rect_blockdiag_kernel<<<grid, 256, 0, st>>>(A, Na, Nb, dense, ld);
  return cudaGetLastError();
}


// ---- row-cyclic block-column exchange (multi-GPU Cholesky of one large factor) ---------------------
// Tile rows [ra, rb) of block column [s0, s1); rank r owns the rows I = r (mod G).  Slot q of rank r is its q-th
// own row >= ra.  grid (slots, ob): one CTA copies one tile (16384 doubles, 128-bit accesses).
__global__ void __launch_bounds__(256) rowcyclic_copy_kernel(TiledSym L, int s0, int s1, int ra, int rb, int G, int rank_lo, int rank_hi,
                                                             int skip_rank, int slots, double* __restrict__ buf, int to_buf) {
  const int ob = s1 - s0, q = blockIdx.x, c = blockIdx.y;
  for (int r = rank_lo; r < rank_hi; ++r) {
    if (r == skip_rank) continue;
    const int first = ra + ((r - ra % G) % G + G) % G;  // first tile row >= ra owned by rank r
    const int I = first + q * G;
    if (I >= rb) continue;
    const int J = s0 + c;
    if (J > I) continue;  // above the diagonal inside the block
    double2* t = reinterpret_cast<double2*>(L.tile(0, I, J));
    double2* bslot = reinterpret_cast<double2*>(buf + (((size_t)(to_buf ? 0 : r) * slots + q) * ob + c) * TT);
    for (int e = threadIdx.x; e < TT / 2; e += 256) {
      if (to_buf) bslot[e] = t[e];
      else t[e] = bslot[e];
    }
  }
}
cudaError_t launch_rowcyclic_pack(cudaStream_t st, TiledSym L, int s0, int s1, int ra, int rb, int G, int rank, int slots, double* buf) {
  dim3 grid((unsigned)slots, (unsigned)(s1 - s0));
  rowcyclic_copy_kernel<<<grid, 256, 0, st>>>(L, s0, s1, ra, rb, G, rank, rank + 1, -1, slots, buf, 1);
  return cudaGetLastError();
}
cudaError_t launch_rowcyclic_unpack(cudaStream_t st, TiledSym L, int s0, int s1, int ra, int rb, int G, int rank, int slots,
                                    const double* all) {
  dim3 grid((unsigned)slots, (unsigned)(s1 - s0));
  rowcyclic_copy_kernel<<<grid, 256, 0, st>>>(L, s0, s1, ra, rb, G, 0, G, rank, slots, const_cast<double*>(all), 0);
  return cudaGetLastError();
}


// ---- distributed-storage row-cyclic factorisation (host_chol.cu: chol_factor_rowcyclic_dist) ----
// dst(I, J) = src(I, J) for the tile rows I = first, first + step, ... < rows_end and the tile columns [s0, s1), J <= I:
// the finished panel window -> the owner's packed rows.
__global__ void __launch_bounds__(256) tile_rows_copy_kernel(TiledSym dst, TiledSym src, int s0, int first, int step, int rows_end) {
  const int I = first + blockIdx.x * step, J = s0 + blockIdx.y;
  if (I >= rows_end || J > I) return;
  const double2* a = reinterpret_cast<const double2*>(src.tile(0, I, J));
  double2* d = reinterpret_cast<double2*>(dst.tile(0, I, J));
  for (int e = threadIdx.x; e < TT / 2; e += 256) d[e] = a[e];
}
cudaError_t launch_tile_rows_copy(cudaStream_t st, TiledSym dst, TiledSym src, int s0, int s1, int first, int step, int rows_end) {
  if (first >= rows_end || s1 <= s0) return cudaSuccess;
  dim3 grid((unsigned)((rows_end - 1 - first) / step + 1), (unsigned)(s1 - s0));
  tile_rows_copy_kernel<<<grid, 256, 0, st>>>(dst, src, s0, first, step, rows_end);
  return cudaGetLastError();
}
// The right-hand side as ONE extra tile row under the matrix: tile (I, J), J < I, holds rhs[J*128 ..] in its row 0 and zeros
// below; the factorisation then leaves z = L^{-1} rhs in that row (the forward solve rides on the panel TRSMs).
__global__ void __launch_bounds__(256) rhs_row_kernel(TiledSym L, int I, const double* __restrict__ rhs) {
  const int J = blockIdx.x;
  double* t = L.tile(0, I, J);
  for (int e = threadIdx.x; e < TT; e += 256) {
    int r, c;
    tile_rc(e, r, c);
    t[e] = (r == 0 && J < I) ? rhs[(size_t)J * TILE + c] : 0.0;
  }
}
cudaError_t launch_rhs_row(cudaStream_t st, TiledSym L, int I, const double* rhs) {
  rhs_row_kernel<<<(unsigned)(I + 1), 256, 0, st>>>(L, I, rhs);
  return cudaGetLastError();
}
// z[J*128 + c] = row 0 of tile (I, J), J in [s0, s1)
__global__ void __launch_bounds__(128) rhs_row_extract_kernel(TiledSym L, int I, int s0, double* __restrict__ z) {
  const int J = s0 + blockIdx.x, c = threadIdx.x;
  z[(size_t)J * TILE + c] = L.tile(0, I, J)[tile_elem(0, c)];
}
cudaError_t launch_rhs_row_extract(cudaStream_t st, TiledSym L, int I, int s0, int s1, double* z) {
  if (s1 <= s0) return cudaSuccess;
  rhs_row_extract_kernel<<<(unsigned)(s1 - s0), 128, 0, st>>>(L, I, s0, z);
  return cudaGetLastError();
}

}  // namespace lmm
