// Leave-one-input-out (LOO) cross-validation of one latent GP (Rasmussen & Williams §5.4.2), C = K + νI, δ = ỹ - m:
//   A = C⁻¹, α = Aδ, d_i = A_ii, q_i = α_i / d_i, r_i = (1 + α_i q_i) / (2 d_i), w = A q,
//   LOO = Σ_{i<N} (-½ log 2π + ½ log d_i - ½ α_i q_i);  the LOO predictive of ỹ_i has mean ỹ_i - q_i, variance 1/d_i;
//   dLOO/dC = G = ½(αw' + wα') - A R A = ½(uu' + M),  u = α + w,  M = -αα' - ww' - 2 A R A;  dLOO/dδ = -w.
// Padding rows i >= N carry the identity in the factor (A_ii = 1, α_i = 0) and are given q = r = 0.
#include "common.cuh"
#include "kernels.h"

namespace lmm {

// grid (batch), one CTA per latent.  d_i = -negA(i,i) (negA.base != null) or dvec[b][i].  Outputs per latent b, i < npad
// (each nullable): q, sc = sqrt(2 r) and v = q / sc (0 on padding: B = A diag(sc) gives -B B' = -2 A R A and w = B v = A q),
// lmean = ỹ_i - q_i = δ_i + mean - q_i and lvar = 1/d_i - ν (0 on padding); loo[b] = LOO of the latent.
__global__ void __launch_bounds__(256) loo_terms_kernel(TiledSym negA, const double* __restrict__ dvec, const double* __restrict__ alpha,
                                                        const double* __restrict__ delta, size_t stride, int N,
                                                        const LatentParams* __restrict__ params, double log2pi, double* __restrict__ q,
                                                        double* __restrict__ sc, double* __restrict__ v, double* __restrict__ lmean,
                                                        double* __restrict__ lvar, double* __restrict__ loo) {
  __shared__ double red[256];
  const int b = blockIdx.x, t = threadIdx.x;
  const size_t off = (size_t)b * stride;
  const double nu = params[b].noise, mean = params[b].mean;
  double s = 0.0;
  for (int i = t; i < (int)stride; i += 256) {
    double qi = 0.0, sci = 0.0, vi = 0.0, mi = 0.0, vari = 0.0;
    if (i < N) {
      const double d = negA.base ? -negA.tile(b, i / TILE, i / TILE)[tile_elem(i % TILE, i % TILE)] : dvec[off + i];
      const double a = alpha[off + i];
      qi = a / d;
      sci = sqrt((1.0 + a * qi) / d);
      vi = qi / sci;
      mi = delta[off + i] + mean - qi;
      vari = 1.0 / d - nu;
      s += -0.5 * log2pi + 0.5 * log(d) - 0.5 * a * qi;
    }
    if (q) q[off + i] = qi;
    if (sc) sc[off + i] = sci;
    if (v) v[off + i] = vi;
    if (lmean) lmean[off + i] = mi;
    if (lvar) lvar[off + i] = vari;
  }
  s = cta_sum256(s, red);
  if (t == 0) loo[b] = s;
}
cudaError_t launch_loo_terms(cudaStream_t st, TiledSym negA, const double* dvec, const double* alpha, const double* delta, size_t stride,
                             int N, const LatentParams* params, int batch, double log2pi, double* q, double* sc, double* v, double* lmean,
                             double* lvar, double* loo) {
  loo_terms_kernel<<<batch, 256, 0, st>>>(negA, dvec, alpha, delta, stride, N, params, log2pi, q, sc, v, lmean, lvar, loo);
  return cudaGetLastError();
}

// grid (nt * nt, batch): B(I,J) = A(I,J) diag(sc_J) as full square tiles from the packed-lower -A (tile (J,I) transposed above
// the diagonal; the lower half of a diagonal tile is read for both halves).
__global__ void __launch_bounds__(256) sym_expand_scale_kernel(TiledSym negA, const double* __restrict__ sc, size_t sc_stride,
                                                               TiledRect B) {
  const int b = blockIdx.y, I = blockIdx.x / B.ntc, J = blockIdx.x % B.ntc;
  const double* src = I >= J ? negA.tile(b, I, J) : negA.tile(b, J, I);
  double* dst = B.tile(b, I, J);
  const double* s = sc + (size_t)b * sc_stride + (size_t)J * TILE;
  for (int e = threadIdx.x; e < TT; e += 256) {
    int r, c;
    tile_rc(e, r, c);
    const double a = (I > J || (I == J && r >= c)) ? src[e] : src[tile_elem(c, r)];
    dst[e] = -a * s[c];
  }
}
cudaError_t launch_sym_expand_scale(cudaStream_t st, TiledSym negA, const double* sc, size_t sc_stride, TiledRect B, int batch) {
  dim3 grid((unsigned)(B.ntr * B.ntc), (unsigned)batch);
  sym_expand_scale_kernel<<<grid, 256, 0, st>>>(negA, sc, sc_stride, B);
  return cudaGetLastError();
}

// grid (batch): u = α + w (0 on padding) and out[b*4 + {2, 3}] = {tr G = ½ Σ_{i<N} (u_i² + M_ii), Σ_{i<N} w_i}, dot[b] = w·δ,
// fixed order.  M is the packed-lower -αα' - ww' - 2ARA.
__global__ void __launch_bounds__(256) loo_grad_vectors_kernel(TiledSym M, const double* __restrict__ alpha, const double* __restrict__ w,
                                                               const double* __restrict__ delta, size_t stride, int N,
                                                               double* __restrict__ u, double* __restrict__ out, double* __restrict__ dot) {
  __shared__ double red[256];
  const int b = blockIdx.x, t = threadIdx.x;
  const size_t off = (size_t)b * stride;
  double tr = 0.0, sw = 0.0, wd = 0.0;
  for (int i = t; i < (int)stride; i += 256) {
    double ui = 0.0;
    if (i < N) {
      const double wi = w[off + i];
      ui = alpha[off + i] + wi;
      tr += ui * ui + M.tile(b, i / TILE, i / TILE)[tile_elem(i % TILE, i % TILE)];
      sw += wi;
      wd += wi * delta[off + i];
    }
    u[off + i] = ui;
  }
  tr = cta_sum256(tr, red);
  if (t == 0) out[(size_t)b * 4 + 2] = 0.5 * tr;
  __syncthreads();
  sw = cta_sum256(sw, red);
  if (t == 0) out[(size_t)b * 4 + 3] = sw;
  __syncthreads();
  wd = cta_sum256(wd, red);
  if (t == 0) dot[b] = wd;
}
cudaError_t launch_loo_grad_vectors(cudaStream_t st, TiledSym M, const double* alpha, const double* w, const double* delta, size_t stride,
                                    int N, int batch, double* u, double* out, double* dot) {
  loo_grad_vectors_kernel<<<batch, 256, 0, st>>>(M, alpha, w, delta, stride, N, u, out, dot);
  return cudaGetLastError();
}

}  // namespace lmm
