// Sparse variational (VFE, Titsias 2009) bound of a batch of latent GPs with M inducing inputs z shared by the latents:
//   Kz = K(z, z) + jitter I = Lz Lz',  B' = K(x, z) Lz^{-T} (N x M),  Ψ = B B',  b = B δ,  Σ = I + Ψ/ν = L_Σ L_Σ',  c = L_Σ^{-1} b
//   ELBO = -½ [N log 2π + N log ν + log|Σ| + δ'δ/ν - c'c/ν² + (Σ_i k_ii - tr Ψ)/ν]
// vfe_gram_kernel forms Ψ, b and δ'δ in one pass over B' (the hot path: M² N flop against 8 M N bytes); the rest is O(M²).
#include "common.cuh"
#include "kernels.h"

namespace lmm {

__device__ __forceinline__ void vfe_dmma(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1},{%2},{%3},{%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
__device__ __forceinline__ uint32_t vfe_s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void vfe_mb_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(vfe_s32(bar)), "r"(count));
}
__device__ __forceinline__ void vfe_mb_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(vfe_s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void vfe_mb_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(vfe_s32(bar)) : "memory");
}
__device__ __forceinline__ void vfe_mb_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (!done) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done)
                 : "r"(vfe_s32(bar)), "r"(parity)
                 : "memory");
    if (!done && ++spins > (1u << 28)) __trap();  // never hang the GPU on a protocol bug
  }
}
__device__ __forceinline__ void vfe_bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(vfe_s32(dst)), "l"(src),
               "r"(bytes), "r"(vfe_s32(bar))
               : "memory");
}

// A stage holds 32 rows (the contraction index) of the two column tiles I and J of B'.  In the k4-interleaved tile layout
// (common.cuh) rows [r0, r0 + 32) of a 4-column group are one contiguous run of 128 doubles, so a stage is 32 bulk copies per
// operand, one per lane of the producer warp.  The runs are stored VG_RUN = 132 doubles apart: the fragments below read 16
// consecutive doubles per half-warp wherever the runs sit, and the padding spreads the b = B δ reads (one column per thread,
// eight 4-column groups per warp) over all banks.
constexpr int VG_ROWS = 32;
constexpr int VG_RUN = 132;
constexpr int VG_OP = 32 * VG_RUN;
constexpr int VG_STAGE = 2 * VG_OP + VG_ROWS;  // A | B | δ
constexpr int VG_STAGES = 3;
constexpr size_t VG_SMEM = (size_t)VG_STAGES * VG_STAGE * sizeof(double) + 2 * VG_STAGES * sizeof(uint64_t);

// grid (sym_tiles(mt), splits, batch), 256 threads.  CTA (tile (I, J), split s, latent b): the Gram tile
//   part[s][b][(I, J)] = Σ_{row tiles R of split s} B'(R, I)' B'(R, J)
// with 8 warps as 2 x 4, warp tile 64 x 32 = 8 x 4 m8n8k4 fragments.  The contraction runs over the ROWS of the stored tiles, so
// both operands need the fragment transposed against the storage: lane l takes (row 4 ks + l%4, column 8 nb + l/4).  The
// diagonal CTAs (I = J) load one operand and also form bpart[s][b][I*128 + c] = Σ_r B'(r, c) δ_r (c in tile I); the CTA of
// tile (0, 0) forms ddpart[s][b] = Σ_r δ_r².  Every sum runs in a fixed order: the results do not depend on the schedule.
__global__ void __launch_bounds__(256, 1) vfe_gram_kernel(TiledRect X, const double* __restrict__ delta, size_t delta_stride, int splits,
                                                          double* __restrict__ part, double* __restrict__ bpart, double* __restrict__ ddpart) {
  extern __shared__ __align__(128) double smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)VG_STAGES * VG_STAGE);
  uint64_t* empty = full + VG_STAGES;
  const int t = blockIdx.x, s = blockIdx.y, b = blockIdx.z;
  int I = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((I + 1) * (I + 2) / 2 <= t) ++I;
  while (I * (I + 1) / 2 > t) --I;
  const int J = t - I * (I + 1) / 2;
  const bool diag = I == J;
  const int R0 = (int)((long long)s * X.ntr / splits), R1 = (int)((long long)(s + 1) * X.ntr / splits);
  const int nchunks = (R1 - R0) * (TILE / VG_ROWS);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double* dl = delta + (size_t)b * delta_stride;

  if (tid == 0) {
    for (int q = 0; q < VG_STAGES; ++q) {
      vfe_mb_init(&full[q], 1);
      vfe_mb_init(&empty[q], 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // warp 0 produces: lane l copies the run of 4-column group l of each operand
  auto produce = [&](int q) {
    const int st = q % VG_STAGES;
    double* sa = smem + (size_t)st * VG_STAGE;
    const int R = R0 + q / (TILE / VG_ROWS), rq = q % (TILE / VG_ROWS);
    if (lane == 0) vfe_mb_expect_tx(&full[st], (diag ? 1u : 2u) * 32u * 128u * 8u + (diag ? VG_ROWS * 8u : 0u));
    __syncwarp();
    const size_t off = (size_t)lane * 512 + (size_t)rq * 128;
    vfe_bulk_load(sa + lane * VG_RUN, X.tile(b, R, I) + off, 128 * 8, &full[st]);
    if (!diag) vfe_bulk_load(sa + VG_OP + lane * VG_RUN, X.tile(b, R, J) + off, 128 * 8, &full[st]);
    if (diag && lane == 0) vfe_bulk_load(sa + 2 * VG_OP, dl + (size_t)R * TILE + rq * VG_ROWS, VG_ROWS * 8, &full[st]);
  };
  if (warp == 0) {
    const int pre = nchunks < VG_STAGES ? nchunks : VG_STAGES;
    for (int q = 0; q < pre; ++q) produce(q);
  }

  const int wm = warp & 1, wn = warp >> 1, g4 = lane >> 2, t4 = lane & 3;
  const int lo = (lane >> 4) * VG_RUN + t4 * 4 + (g4 & 3);  // this lane's fragment element inside a k4-step of a column block
  double acc[8][4][2];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  const int bc = tid & 127, bh = tid >> 7;  // b = B δ: column bc of tile I over rows [16 bh, 16 bh + 16) of each stage
  double bacc = 0.0, ddacc = 0.0;

  for (int q = 0; q < nchunks; ++q) {
    const int st = q % VG_STAGES;
    vfe_mb_wait(&full[st], (uint32_t)((q / VG_STAGES) & 1));
    const double* sa = smem + (size_t)st * VG_STAGE;
    const double* sb = diag ? sa : sa + VG_OP;
    const double* pa = sa + (wm * 16) * VG_RUN + lo;
    const double* pb = sb + (wn * 8) * VG_RUN + lo;
#pragma unroll
    for (int ks = 0; ks < VG_ROWS / 4; ++ks) {
      const int ko = (ks >> 1) * 32 + (ks & 1) * 16;
      double a[8], bq[4];
#pragma unroll
      for (int mb = 0; mb < 8; ++mb) a[mb] = pa[mb * 2 * VG_RUN + ko];
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) bq[nb] = pb[nb * 2 * VG_RUN + ko];
#pragma unroll
      for (int mb = 0; mb < 8; ++mb)
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) vfe_dmma(acc[mb][nb][0], acc[mb][nb][1], a[mb], bq[nb]);
    }
    if (diag) {
      const double* sd = sa + 2 * VG_OP;
      const double* col = sa + (bc >> 2) * VG_RUN + (bc & 3);
#pragma unroll
      for (int r = 16 * bh; r < 16 * bh + 16; ++r) bacc = fma(col[(r >> 3) * 32 + (r & 7) * 4], sd[r], bacc);
      if (I == 0 && tid < VG_ROWS) ddacc = fma(sd[tid], sd[tid], ddacc);
    }
    __syncwarp();
    if (lane == 0) vfe_mb_arrive(&empty[st]);
    if (warp == 0 && q >= 1) {  // refill the stage consumed one iteration ago
      const int qn = q - 1 + VG_STAGES;
      if (qn < nchunks) {
        vfe_mb_wait(&empty[(q - 1) % VG_STAGES], (uint32_t)(((q - 1) / VG_STAGES) & 1));
        produce(qn);
      }
    }
  }

  double* Ct = part + (((size_t)s * gridDim.z + b) * gridDim.x + t) * TT;
#pragma unroll
  for (int mb = 0; mb < 8; ++mb)
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
      const int cg = wn * 8 + nb * 2 + (t4 >> 1);
      const int off = (cg << 9) + ((wm * 8 + mb) << 5) + (g4 << 2) + ((t4 & 1) << 1);
      *reinterpret_cast<double2*>(Ct + off) = make_double2(acc[mb][nb][0], acc[mb][nb][1]);
    }
  if (diag) {
    __syncthreads();  // every stage has been consumed: reuse stage 0 for the two row halves of b
    double* red = smem;
    if (bh == 1) red[bc] = bacc;
    __syncthreads();
    const size_t mpad = (size_t)X.ntc * TILE;
    if (bh == 0) bpart[((size_t)s * gridDim.z + b) * mpad + (size_t)I * TILE + bc] = bacc + red[bc];
    if (I == 0 && warp == 0) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) ddacc += __shfl_xor_sync(0xffffffffu, ddacc, o);
      if (lane == 0) ddpart[(size_t)s * gridDim.z + b] = ddacc;
    }
  }
}

// grid (sym_tiles(mt), batch): psi (+)= Σ_s part[s] in split order; the CTA of tile 0 does the same for b and δ'δ.
__global__ void __launch_bounds__(256) vfe_gram_reduce_kernel(TiledSym psi, double* __restrict__ bvec, double* __restrict__ dd, int splits,
                                                              const double* __restrict__ part, const double* __restrict__ bpart,
                                                              const double* __restrict__ ddpart, int accumulate) {
  const int t = blockIdx.x, b = blockIdx.y, batch = gridDim.y, ntl = gridDim.x;
  double* dst = psi.base + (size_t)b * psi.batch_stride + (size_t)t * TT;
  for (int e = threadIdx.x; e < TT; e += 256) {
    double v = accumulate ? dst[e] : 0.0;
    for (int s = 0; s < splits; ++s) v += part[(((size_t)s * batch + b) * ntl + t) * TT + e];
    dst[e] = v;
  }
  if (t != 0) return;
  const size_t mpad = (size_t)psi.nt * TILE;
  for (size_t i = threadIdx.x; i < mpad; i += 256) {
    double v = accumulate ? bvec[(size_t)b * mpad + i] : 0.0;
    for (int s = 0; s < splits; ++s) v += bpart[((size_t)s * batch + b) * mpad + i];
    bvec[(size_t)b * mpad + i] = v;
  }
  if (threadIdx.x == 0) {
    double v = accumulate ? dd[b] : 0.0;
    for (int s = 0; s < splits; ++s) v += ddpart[(size_t)s * batch + b];
    dd[b] = v;
  }
}

// grid (sym_tiles(mt), batch): Σ = I + Ψ/ν tile by tile (Ψ is 0 on the padding, so Σ is the identity there).
__global__ void __launch_bounds__(256) vfe_sigma_kernel(TiledSym psi, TiledSym sig, const LatentParams* __restrict__ params) {
  const int t = blockIdx.x, b = blockIdx.y;
  int I = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((I + 1) * (I + 2) / 2 <= t) ++I;
  while (I * (I + 1) / 2 > t) --I;
  const bool diag = t - I * (I + 1) / 2 == I;
  const double inv_nu = 1.0 / params[b].noise;
  const double* src = psi.base + (size_t)b * psi.batch_stride + (size_t)t * TT;
  double* dst = sig.base + (size_t)b * sig.batch_stride + (size_t)t * TT;
  for (int e = threadIdx.x; e < TT; e += 256) {
    int r, c;
    tile_rc(e, r, c);
    dst[e] = src[e] * inv_nu + ((diag && r == c) ? 1.0 : 0.0);
  }
}

// grid (batch), one CTA per latent: elbo[b] from tr Ψ (diagonal of psi), log|Σ|, c = L_Σ^{-1} b, δ'δ, N, ν and k_ii = kdiag
// (κ(0) = 1 for every supported kernel), fixed order; cnu (nullable) = c / ν, the right-hand side of the posterior's weights.
__global__ void __launch_bounds__(256) vfe_terms_kernel(TiledSym psi, const double* __restrict__ logdet, const double* __restrict__ c,
                                                        const double* __restrict__ dd, int N, const LatentParams* __restrict__ params,
                                                        double log2pi, double* __restrict__ cnu, double* __restrict__ elbo) {
  __shared__ double red[256];
  const int b = blockIdx.x, t = threadIdx.x;
  const size_t mpad = (size_t)psi.nt * TILE;
  const double nu = params[b].noise;
  double tr = 0.0, cc = 0.0;
  for (int i = t; i < (int)mpad; i += 256) {
    tr += psi.tile(b, i / TILE, i / TILE)[tile_elem(i % TILE, i % TILE)];
    const double ci = c[(size_t)b * mpad + i];
    cc = fma(ci, ci, cc);
    if (cnu) cnu[(size_t)b * mpad + i] = ci / nu;
  }
  tr = cta_sum256(tr, red);
  __syncthreads();
  cc = cta_sum256(cc, red);
  if (t == 0) {
    const double n = (double)N;
    elbo[b] = -0.5 * (n * log2pi + n * log(nu) + logdet[b] + dd[b] / nu - cc / (nu * nu) + (n * params[b].kdiag - tr) / nu);
  }
}

// grid (mt * mt, batch): the two bracket matrices of the gradient as full square tiles, from the packed-lower negSinv = -Σ⁻¹ and
// Ψ (tile (J, I) read transposed above the diagonal), with q = β_w / ν = Σ⁻¹ b / ν:
//   A = ((I - Σ⁻¹) - q q') / ν          (contracted with K(x, z) through B' A Lz⁻¹)
//   P = I - Σ⁻¹ - Ψ/ν - q q'            (= 2I - Σ⁻¹ - Σ - β_w β_w'/ν²; contracted with K(z, z) through ½ Lz⁻ᵀ P Lz⁻¹)
// The CTA of tile (0, 0) also writes v = w / ν (w = Lz⁻ᵀ q: v = β / ν², the rank-1 factor of the K(x, z) cotangent).
__global__ void __launch_bounds__(256) vfe_brackets_kernel(TiledSym negSinv, TiledSym psi, const double* __restrict__ q,
                                                           const double* __restrict__ w, const LatentParams* __restrict__ params,
                                                           TiledRect A, TiledRect P, double* __restrict__ v) {
  const int b = blockIdx.y, I = blockIdx.x / A.ntc, J = blockIdx.x % A.ntc;
  const size_t mpad = (size_t)A.ntc * TILE;
  const double nu = params[b].noise, inv_nu = 1.0 / nu;
  const double* qb = q + (size_t)b * mpad;
  const double* sn = I >= J ? negSinv.tile(b, I, J) : negSinv.tile(b, J, I);
  const double* sp = I >= J ? psi.tile(b, I, J) : psi.tile(b, J, I);
  double* da = A.tile(b, I, J);
  double* dp = P.tile(b, I, J);
  for (int e = threadIdx.x; e < TT; e += 256) {
    int r, c;
    tile_rc(e, r, c);
    const int se = I >= J ? e : tile_elem(c, r);
    const double id = (I == J && r == c) ? 1.0 : 0.0;
    const double qq = qb[I * TILE + r] * qb[J * TILE + c];
    const double a = id + sn[se] - qq;
    da[e] = a * inv_nu;
    dp[e] = a - sp[se] * inv_nu;
  }
  if (blockIdx.x == 0)
    for (size_t i = threadIdx.x; i < mpad; i += 256) v[(size_t)b * mpad + i] = w[(size_t)b * mpad + i] * inv_nu;
}

// grid (batch), one CTA per latent, fixed order.  y holds B'q on entry and a = (δ - B'q)/ν = -dELBO/dδ on exit (0 on padding);
// out4[b*4 + 2] = dELBO/dν, out4[b*4 + 3] = Σ a, dot[b] = a·δ;
// gterms[b][slot] = gz + gx (the K(z, z) and K(x, z) contractions) and, in every term's variance slot, -N/(2ν) ∂(Σ_i k_ii)/∂variance.
__global__ void __launch_bounds__(256) vfe_grad_kernel(TiledSym negSinv, TiledSym psi, const double* __restrict__ q,
                                                       const double* __restrict__ c, const double* __restrict__ dd, const double* __restrict__ delta,
                                                       size_t npad, int N, const LatentParams* __restrict__ params, double* __restrict__ y,
                                                       double* __restrict__ out4, double* __restrict__ dot, const double* __restrict__ gz,
                                                       const double* __restrict__ gx, double* __restrict__ gterms) {
  __shared__ double red[256];
  const int b = blockIdx.x, t = threadIdx.x;
  const LatentParams* lp = params + b;
  const double nu = lp->noise;
  const int mt = psi.nt;
  const size_t mpad = (size_t)mt * TILE;
  const double* qb = q + (size_t)b * mpad;
  double sa = 0.0, ad = 0.0;
  for (int i = t; i < (int)npad; i += 256) {
    const size_t k = (size_t)b * npad + i;
    const double a = i < N ? (delta[k] - y[k]) / nu : 0.0;
    y[k] = a;
    sa += a;
    ad = fma(a, delta[k], ad);
  }
  // tr(Σ⁻¹Ψ), q'Ψq, tr Ψ over the stored tiles (off-diagonal tiles twice, diagonal tiles hold the whole symmetric block)
  double tsp = 0.0, qpq = 0.0, tr = 0.0, cc = 0.0;
  const size_t ntl = sym_tiles(mt);
  for (size_t tl = 0; tl < ntl; ++tl) {
    int I = 0;
    while ((size_t)(I + 1) * (I + 2) / 2 <= tl) ++I;
    const int J = (int)(tl - (size_t)I * (I + 1) / 2);
    const double wgt = I == J ? 1.0 : 2.0;
    const double* ps = psi.tile(b, I, J);
    const double* ns = negSinv.tile(b, I, J);
    for (int e = t; e < TT; e += 256) {
      int r, cc2;
      tile_rc(e, r, cc2);
      const double pv = ps[e];
      tsp = fma(-wgt * ns[e], pv, tsp);
      qpq = fma(wgt * pv * qb[I * TILE + r], qb[J * TILE + cc2], qpq);
      if (I == J && r == cc2) tr += pv;
    }
  }
  for (int i = t; i < (int)mpad; i += 256) cc = fma(c[(size_t)b * mpad + i], c[(size_t)b * mpad + i], cc);
  sa = cta_sum256(sa, red);
  __syncthreads();
  ad = cta_sum256(ad, red);
  __syncthreads();
  tsp = cta_sum256(tsp, red);
  __syncthreads();
  qpq = cta_sum256(qpq, red);
  __syncthreads();
  tr = cta_sum256(tr, red);
  __syncthreads();
  cc = cta_sum256(cc, red);
  if (t == 0) {
    const double n = (double)N;
    // b'β_w = |c|², β_w'Ψβ_w = ν² q'Ψq
    out4[(size_t)b * 4 + 2] = -0.5 * (n / nu - tsp / (nu * nu) - dd[b] / (nu * nu) + 2.0 * cc / (nu * nu * nu) - qpq / (nu * nu)
                                      - (n * lp->kdiag - tr) / (nu * nu));
    out4[(size_t)b * 4 + 3] = sa;
    dot[b] = ad;
  }
  constexpr int SLOTS = MAX_TERMS * (3 + MAX_ARD);
  if (t < SLOTS) {
    const int term = t / (3 + MAX_ARD), slot = t % (3 + MAX_ARD);
    double g = gz[(size_t)b * SLOTS + t] + gx[(size_t)b * SLOTS + t];
    if (slot == 0 && term < lp->nterms) {
      double dk = 1.0;  // ∂ k(x, x) / ∂ variance of the term: 1 for a sum, the other terms' variances for a product
      if (lp->compose == 2)
        for (int u = 0; u < lp->nterms; ++u)
          if (u != term) dk *= u == 0 ? lp->variance : lp->extra[u - 1].variance;
      g -= 0.5 * (double)N / nu * dk;
    }
    gterms[(size_t)b * SLOTS + t] = g;
  }
}

cudaError_t launch_vfe_brackets(cudaStream_t st, TiledSym negSinv, TiledSym psi, const double* q, const double* w, const LatentParams* params,
                                TiledRect A, TiledRect P, double* v, int batch) {
  if (batch <= 0) return cudaSuccess;
  vfe_brackets_kernel<<<dim3((unsigned)(A.ntr * A.ntc), (unsigned)batch), 256, 0, st>>>(negSinv, psi, q, w, params, A, P, v);
  return cudaGetLastError();
}

cudaError_t launch_vfe_grad(cudaStream_t st, TiledSym negSinv, TiledSym psi, const double* q, const double* c, const double* dd,
                            const double* delta, size_t npad, int N, const LatentParams* params, int batch, double* y, double* out4,
                            double* dot, const double* gz, const double* gx, double* gterms) {
  if (batch <= 0) return cudaSuccess;
  vfe_grad_kernel<<<batch, 256, 0, st>>>(negSinv, psi, q, c, dd, delta, npad, N, params, y, out4, dot, gz, gx, gterms);
  return cudaGetLastError();
}

int vfe_gram_splits(int mt, int batch, int ntr) {
  const int ntiles_out = (int)sym_tiles(mt) * batch;
  const int sp = (2 * 148 + ntiles_out - 1) / ntiles_out;  // about two CTAs per SM over the whole grid
  return sp < 1 ? 1 : (sp > ntr ? ntr : sp);
}

cudaError_t launch_vfe_gram(cudaStream_t st, TiledRect X, const double* delta, size_t delta_stride, int batch, TiledSym psi, double* bvec,
                            double* dd, int accumulate, int splits, double* part, double* bpart, double* ddpart) {
  if (batch <= 0 || X.ntr <= 0) return cudaSuccess;
  if (splits < 1) return cudaErrorInvalidValue;  // splits past the row tiles of a short last chunk sum empty ranges (zeros)
  static bool configured[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(vfe_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VG_SMEM);
    if (e != cudaSuccess) return e;
    configured[dev & 63] = true;
  }
  const int ntl = (int)sym_tiles(X.ntc);
  vfe_gram_kernel<<<dim3((unsigned)ntl, (unsigned)splits, (unsigned)batch), 256, VG_SMEM, st>>>(X, delta, delta_stride, splits, part, bpart,
                                                                                                 ddpart);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  vfe_gram_reduce_kernel<<<dim3((unsigned)ntl, (unsigned)batch), 256, 0, st>>>(psi, bvec, dd, splits, part, bpart, ddpart, accumulate);
  return cudaGetLastError();
}

cudaError_t launch_vfe_sigma(cudaStream_t st, TiledSym psi, TiledSym sig, const LatentParams* params, int batch) {
  if (batch <= 0) return cudaSuccess;
  vfe_sigma_kernel<<<dim3((unsigned)sym_tiles(psi.nt), (unsigned)batch), 256, 0, st>>>(psi, sig, params);
  return cudaGetLastError();
}

cudaError_t launch_vfe_terms(cudaStream_t st, TiledSym psi, const double* logdet, const double* c, const double* dd, int N,
                             const LatentParams* params, int batch, double log2pi, double* cnu, double* elbo) {
  if (batch <= 0) return cudaSuccess;
  vfe_terms_kernel<<<batch, 256, 0, st>>>(psi, logdet, c, dd, N, params, log2pi, cnu, elbo);
  return cudaGetLastError();
}

}  // namespace lmm
