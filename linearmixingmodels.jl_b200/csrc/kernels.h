// Host-callable launchers of the liblmm kernels (internal header).
#pragma once
#include <cuda_runtime.h>
#include "common.cuh"

namespace lmm {

// ---- kmat.cu
// noise_vec (nullable): per-point diagonal noise [batch][noise_stride] overriding params[b].noise
// row0: only the tile rows I >= row0 are built (the rows above belong to a factor that is being extended)
// env (nullable, [batch][nt] ints, row0 = 0): the tile envelope -- env[b][I] = first tile column of tile row I with an entry != 0.
// The Cholesky factor keeps it (L(I,k) = 0 for k < env[b][I]), so the factorisation and the solves may skip those tiles.
// rowoff (nullable, row0 = 0, [batch * nt + 1] ints): build only the tiles (I, k >= fb[b][I]) of launch_kmat_bound's envelope;
// rowoff[b * nt + I] = number of such tiles in the rows before (b, I), ntiles = rowoff[batch * nt].  The tiles left out are NOT
// written: only code that takes env may read the matrix (launch_kmat_zero writes the zeros).
cudaError_t launch_kmat_sym(cudaStream_t st, TiledSym out, int batch, const double* xpad, int N, int D,
                            const LatentParams* params, int form, const double* noise_vec = nullptr, size_t noise_stride = 0, int row0 = 0,
                            int* env = nullptr, const int* rowoff = nullptr, long long ntiles = 0);
// fb[b][I] (<= I): a tile column below which every tile (I, k) of launch_kmat_sym's matrix is provably exactly 0 -- from per-tile
// bounding boxes of the scaled points, a lower bound of the squared distance the build computes, and kappa_zero_d2.  0 (nothing
// provable) for composite, periodic and rational-quadratic latents and for a non-finite variance.  fb <= env holds for every row.
cudaError_t launch_kmat_bound(cudaStream_t st, int batch, const double* xpad, int N, int D, int nt, const LatentParams* params, int* fb);
// Writes the exact zeros of the tiles (I, k < env[b][I]) that a launch_kmat_sym with rowoff may have left out.
cudaError_t launch_kmat_zero(cudaStream_t st, TiledSym L, int batch, const int* env);
cudaError_t launch_kmat_cross(cudaStream_t st, TiledRect out, int batch, const double* xa_pad, int Na, const double* xb_pad,
                              int Nb, int D, const LatentParams* params, int form);

// ---- gemm.cu : C(I,J) -= sum_k X(I,k) L(J,k)^T   |   C(I,J) = C(I,J) W(J)^T
struct TileOperand {
  double* base;
  size_t batch_stride;  // doubles
  int rect;             // 0: packed-lower tiles, 1: rectangular (row-major by tile, ntc tiles per row; window origin row0 / col0),
                        // 2: the rows one rank of a row-cyclic partition owns (cyc_tile_index)
  int ntc;
  int row0 = 0, col0 = 0;
  int cyc_G = 0, cyc_r = 0;
  __host__ __device__ __forceinline__ double* tile(int b, int I, int k) const {
    size_t idx;
    if (rect == 1) idx = (size_t)(I - row0) * (size_t)ntc + (size_t)(k - col0);
    else if (rect == 2) idx = cyc_tile_index(I, k, cyc_G, cyc_r);
    else idx = sym_tile_index(I, k);
    return base + (size_t)b * batch_stride + idx * TT;
  }
};
inline TileOperand operand(const TiledSym& s) {
  if (s.ntc) return TileOperand{s.base, s.batch_stride, 1, s.ntc, s.row0, s.col0, 0, 0};
  if (s.cyc_G) return TileOperand{s.base, s.batch_stride, 2, s.nt, 0, 0, s.cyc_G, s.cyc_r};
  return TileOperand{s.base, s.batch_stride, 0, s.nt};
}
inline TileOperand operand(const TiledRect& r) { return TileOperand{r.base, r.batch_stride, 1, r.ntc}; }
struct GemmArgs {
  TileOperand A;          // rows I of the left operand (UPDATE only)
  TileOperand B;          // rows J of the right operand, used transposed (UPDATE only)
  TileOperand C;          // output tiles (I, J); TRSM reads its left operand from C
  const double* W;        // inverse diagonal tiles [batch][nt] (TRSM only)
  size_t w_batch_stride;
  int i0, j0;             // tile (I, J) = (i0 + blockIdx.y, j0 + blockIdx.x)
  int k0, k1;             // UPDATE: k-tile range
  int sym;                // skip tiles with I < J
  int upper;              // skip tiles with I > J (upper-triangular X, e.g. L^{-T})
  int k_from_row;         // UPDATE: k range starts at max(k0, I) (A(I,k) = 0 for k < I)
  int row_step;           // tile row I = i0 + blockIdx.y * row_step (0 or 1: consecutive rows; G: the rows one rank of a
                          // row-cyclic partition owns)
  const int* env;         // nullable: tile envelope [batch][env_stride] of a packed-lower factor (launch_kmat_sym).  UPDATE: the k range
  int env_stride;         // starts at max(k0, env[b][I], env[b][J]); TRSM: tiles with env[b][I] > J are zero and are skipped
};
enum { GEMM_UPDATE = 0, GEMM_TRSM = 1 };
// select_tiles > 0: choose between the direct and the TMA-pipelined kernel as for a grid of that many tiles (the two sum in different
// orders; a grid trimmed to the envelope keeps the kernel, and so the bits, of the full grid)
cudaError_t launch_gemm(cudaStream_t st, int mode, const GemmArgs& a, int ncols, int nrows, int batch, long long select_tiles = 0);
void set_gemm_small_threshold(int tiles);  // grids of <= tiles tiles use the latency-optimised direct kernel (default 74; 0 = off)
bool gemm_takes_direct(long long tiles);  // a grid of that many tiles takes the direct kernel (launch_gemm's choice)
// Digit planes written by the panel TRSM of the int8 Cholesky: the finished tiles (I, J) with I >= i0 are sliced as launch_ozaki_slice
// slices them (same digits, first-plane bytes, planes skipped for all-zero tiles)
struct TrsmSliceArgs {
  const double* scale;  // [batch][scale_stride]: row scales 2^(E - 6)
  size_t scale_stride;
  uint8_t* slices;      // [batch][slice_stride] bytes, packed-lower tile order, S * 16 KB per tile
  size_t slice_stride;
  uint8_t* fp;          // nullable: first plane with a nonzero digit per tile [batch][fp_stride]
  size_t fp_stride;
  int S, bits, i0;
};
// TRSM of column a.j0, tile rows [a.i0, a.i0 + nrows), on the TMA-pipelined kernel whatever the grid size, with the digit planes
cudaError_t launch_trsm_slice(cudaStream_t st, const GemmArgs& a, int nrows, int batch, const TrsmSliceArgs& s);
void set_pdl(int v);       // 1: programmatic dependent launch along the batch-1 panel chain (default 1)
bool pdl_enabled();

// ---- potrf.cu : factor diagonal tile (J,J) in place, W(J) = inv(L_JJ), logdet += 2*sum(log diag)
cudaError_t launch_potrf_tile(cudaStream_t st, TiledSym L, double* W, size_t w_batch_stride, int J, int batch, double* logdet,
                              int* info);

// Fused panel chain of one tile column (small batches): TRSM of column J, update of the columns (J, c_end) by the k-tiles
// [k0, J], and (do_potrf) the factorisation of diagonal tile J+1 in ONE launch (potrf.cu: chain_column_kernel).
// counters: batch * chain_counter_ints(nt) ints, zeroed once per factorisation.
// env (nullable, [batch][nt]): tile envelope of the factor; the tiles (I, k < env[b][I]) are neither read nor solved.
size_t chain_counter_ints(int nt);
cudaError_t launch_chain_column(cudaStream_t st, TiledSym L, double* W, size_t w_batch_stride, int J, int k0, int c_end, int do_potrf,
                                int batch, double* logdet, int* info, int* counters, const int* env = nullptr);

// ---- solve.cu
// forward: z = L^{-1} r; backward: a = L^{-T} r.  rvec[batch][nt*128] is consumed (destroyed).
// env (nullable, [batch][nt]): tile envelope of the factor (launch_kmat_sym); both solve_impl variants skip the tiles outside it
// (they need not be stored).
cudaError_t launch_fwd_solve(cudaStream_t st, TiledSym L, const double* W, size_t w_batch_stride, double* rvec, double* zvec,
                             size_t vec_stride, int batch, int64_t* launches, const int* env = nullptr);
cudaError_t launch_bwd_solve(cudaStream_t st, TiledSym L, const double* W, size_t w_batch_stride, double* rvec, double* avec,
                             size_t vec_stride, int batch, int64_t* launches, const int* env = nullptr);
void set_solve_impl(int v);  // 1: persistent sweep kernels, one launch per direction (default); 0: one launch per tile column
// out[b] = sum_i v[b][i]^2 (fixed order)
cudaError_t launch_sumsq(cudaStream_t st, const double* v, size_t stride, int n, int batch, double* out);
// y[b][R*128 + r] = add[b] + sum_J T(R,J) x[b][J*128 + :]   over a rectangular tiled matrix
cudaError_t launch_rect_gemv(cudaStream_t st, TiledRect A, const double* x, size_t x_stride, double* y, size_t y_stride,
                             const LatentParams* params, int add_mean, int batch);
// y[b][R*128 + r] = base[b] - sum_J sum_c T(R,J)(r,c)^2     (posterior variance; params == null: base = 0, sign +)
cudaError_t launch_rect_rowsumsq(cudaStream_t st, TiledRect A, double* y, size_t y_stride, const LatentParams* params, int batch);
// y = L * z for a packed-lower factor (rand): y[b][I] = sum_{J<=I} L(I,J) z[b][J]
cudaError_t launch_lower_gemv(cudaStream_t st, TiledSym L, const double* z, size_t z_stride, double* y, size_t y_stride, int batch);
// untile: copy factor b to a dense N x N column-major matrix (lower, zero upper)
cudaError_t launch_untile_lower(cudaStream_t st, TiledSym L, int b, double* dense, int N);
// tile: dense N x N col-major (lower read, mirrored) -> tiles (identity on padding)
cudaError_t launch_tile_from_dense(cudaStream_t st, TiledSym L, int batch, const double* dense, int N);
// Row-cyclic exchange of tile rows [ra, rb) of one block column [s0, s1) of a packed-lower matrix (batch 1): rank r
// owns tile rows I = r (mod G).  pack: own rows -> buf[q][ob tiles] (q = index among the own rows >= ra); unpack: every
// other rank's rows from an all-gathered buffer [G][slots][ob tiles] back into the matrix.
cudaError_t launch_rowcyclic_pack(cudaStream_t st, TiledSym L, int s0, int s1, int ra, int rb, int G, int rank, int slots, double* buf);
cudaError_t launch_rowcyclic_unpack(cudaStream_t st, TiledSym L, int s0, int s1, int ra, int rb, int G, int rank, int slots,
                                    const double* all);
// distributed-storage variant (tiles addressed through the TiledSym window / cyclic views)
cudaError_t launch_tile_rows_copy(cudaStream_t st, TiledSym dst, TiledSym src, int s0, int s1, int first, int step, int rows_end);
cudaError_t launch_rhs_row(cudaStream_t st, TiledSym L, int I, const double* rhs);
cudaError_t launch_rhs_row_extract(cudaStream_t st, TiledSym L, int I, int s0, int s1, double* z);

// ---- ozaki.cu : integer-slice (Ozaki) FP64 trailing update on the int8 tensor cores (tcgen05 / TMEM); optional
// scale[b][row] = 2^(E_row - 6) from the diagonal of the matrix about to be factored (2^E > sqrt(A_ii))
cudaError_t launch_ozaki_scales(cudaStream_t st, TiledSym L, int batch, double* scale, size_t scale_batch_stride);
// slice the finished tiles (I, k), I in [i0, i0 + nrows), k in [k0, k0 + ncols), into S int8 digit planes (S * 16 KB per tile)
// env (nullable, [batch][L.nt]): tiles with k < env[b][I] are zero, are never read, and are not sliced
// first_plane (nullable, [batch][fp_stride], packed-lower tile order): per sliced tile the first plane with a nonzero digit, S when
// every digit is zero (such a tile's planes are then not written)
cudaError_t launch_ozaki_slice(cudaStream_t st, TiledSym L, const double* scale, size_t scale_batch_stride, uint8_t* slices,
                               size_t slice_batch_stride, int i0, int nrows, int k0, int ncols, int batch, int S, int bits,
                               const int* env = nullptr, uint8_t* first_plane = nullptr, size_t fp_stride = 0);
// C(I,J) -= sum_{k < k1} L(I,k) L(J,k)' for I in [i0, i0 + nrows), J in [j0, j0 + ncols), I >= J, from the sliced factor;
// env (nullable, [batch][L.nt]): the k range of tile (I, J) starts at max(env[b][I], env[b][J]);
// first_plane (nullable, as written by launch_ozaki_slice): k-tiles whose digit products are all exactly zero are skipped
cudaError_t launch_ozaki_update(cudaStream_t st, TiledSym L, const uint8_t* slices, size_t slice_batch_stride, const double* scale,
                                size_t scale_batch_stride, int i0, int nrows, int j0, int ncols, int k1, int batch, int S, int bits,
                                const int* env = nullptr, const uint8_t* first_plane = nullptr, size_t fp_stride = 0);
// the prediction sweep X <- X L^{-T} on the same path: row scales of a FINISHED factor (row 2-norms) and of X (prior variance bound),
// digit planes of rectangular tiles, wide update with the left operand from the sliced X
cudaError_t launch_ozaki_factor_scales(cudaStream_t st, TiledSym L, int batch, double* scale, size_t scale_batch_stride);
cudaError_t launch_ozaki_const_scales(cudaStream_t st, const LatentParams* params, int ntr, int batch, double* scale, size_t scale_batch_stride);
cudaError_t launch_ozaki_slice_rect(cudaStream_t st, TiledRect X, const double* scale, size_t scale_batch_stride, uint8_t* slices,
                                    size_t slice_batch_stride, int k0, int ncols, int batch, int S, int bits);
cudaError_t launch_ozaki_update_rect(cudaStream_t st, TiledRect X, const uint8_t* xslices, size_t xslice_batch_stride, const double* xscale,
                                     size_t xscale_stride, const uint8_t* lslices, size_t lslice_batch_stride, const double* lscale,
                                     size_t lscale_stride, int j0, int ncols, int k1, int batch, int S, int bits);

// ---- proj.cu
// Ty[i][n] = sum_j T[i + lat0][j] Y[j][n] - mean_i  (i < mloc), written to ty[i*ty_stride + n], zero padding to ty_stride
// resid_partial[blk] = sum over the block's columns of |Y - Q (P Y)|^2
void set_project_impl(int v);      // 1: DMMA projection kernel (default); 0: register-tiled scalar-FMA kernel
int project_max_partials(int N);  // size of the resid_partial buffer launch_project may write (callers zero it and sum that many)
cudaError_t launch_project(cudaStream_t st, const double* y, int N, int p, const double* T, int m, int lat0, int mloc,
                           const double* means, double* ty, size_t ty_stride, const double* P, const double* Q,
                           double* resid_partial, int* nblocks_out, double* resid_out = nullptr, double* z_out = nullptr);
// out (ra x rb, column-major) += scale * A B'  with A: ra x N, B: rb x N stored row by row (strides lda, ldb)
cudaError_t launch_abt(cudaStream_t st, const double* A, size_t lda, int ra, const double* B, size_t ldb, int rb, int N, double scale,
                       double* out);
cudaError_t launch_sum_partials(cudaStream_t st, const double* partial, int n, double* out);
// back-projection: mean[j*Ns+n] = sum_i H[j, lat0+i] ML[i][n]; var = sum_i H^2 (VL + jitter) (+ sigma2 if add_noise)
cudaError_t launch_backproject(cudaStream_t st, const double* H, int p, int m, int lat0, int mloc, const double* ML,
                               const double* VL, size_t lat_stride, int Ns, double jitter, double sigma2, int add_noise,
                               double* mean, double* var);

}  // namespace lmm

namespace lmm {
// ---- assemble.cu
cudaError_t launch_assemble_ilmm(cudaStream_t st, TiledSym out, const double* x, int N, int D, const LatentParams* params, int m,
                                 int q, const double* E, const double* Hm, int mode, int form);
cudaError_t launch_assemble_cross_blockdiag(cudaStream_t st, TiledRect out, const double* xs, int Ns, const double* x, int N, int D,
                                            const LatentParams* params, int m, int form);
cudaError_t launch_ilmm_predict(cudaStream_t st, TiledRect V, int Ns, int m, int p, const double* H, const LatentParams* params,
                                const double* mlat, double sigma2, double* mean, double* var);
cudaError_t launch_gather_rows(cudaStream_t st, double* dst, const double* src, const int* idx, size_t stride, int n);
// heterotopic / missing-data dense model over the observed entries obs[k] = j*N + i
cudaError_t launch_assemble_masked(cudaStream_t st, TiledSym out, const int* obs, int nobs, const double* x, int N, int D,
                                   const LatentParams* params, int m, int p, const double* Hm, double sigma2, int form);
cudaError_t launch_assemble_masked_cross(cudaStream_t st, TiledRect out, const double* xs, int Ns, const int* obs, int nobs, const double* x,
                                         int N, int D, const LatentParams* params, int m, int p, const double* Hm, int form);
}  // namespace lmm

namespace lmm {
cudaError_t launch_mix_cov(cudaStream_t st, TiledSym C, int nloc, int lat0, const double* H, int p, int Ns, double* out);
cudaError_t launch_mix_cov_joint(cudaStream_t st, TiledSym Cl, int m, const double* H, int p, int Ns, double* out);
cudaError_t launch_add_diag(cudaStream_t st, double* out, int dim, double s);
}  // namespace lmm

namespace lmm {
// ---- grad.cu
cudaError_t launch_kgrad(cudaStream_t st, TiledSym negCinv, int batch, const double* xpad, int N, int D, const LatentParams* params,
                         const double* alpha, size_t alpha_stride, int form, double* partial);
cudaError_t launch_kgrad_finish(cudaStream_t st, const double* partial, int ntiles_, int batch, const double* alpha, size_t alpha_stride,
                                int N, double* out);
cudaError_t launch_rect_identity(cudaStream_t st, TiledRect X, int batch);
// general ILMM: contraction of G = (αα' - C^{-1})/2 over the joint (mN) matrix (batch 1, negCinv = -C^{-1}):
// out3[a*3+{0,1,2}] = {<G_aa,κ_a>, <G_aa,dK_a/ds>, Σ_n α_a}; B (m x m) = block traces (d lml / dΣT).
// partial: m * sym_tiles(ceil(N/128)) * 2 doubles of scratch.  x is [N][D] unpadded.
cudaError_t launch_kgrad_joint(cudaStream_t st, TiledSym negCinv, const double* x, int N, int D, const LatentParams* params, int m,
                               const double* alpha, int form, double* partial, double* out3, double* B);
// B (m x m) = block traces of G over a joint (m*N) matrix whose latent blocks start at multiples of N
cudaError_t launch_block_trace(cudaStream_t st, TiledSym negCinv, const double* alpha, int N, int m, double* B);
// gradient w.r.t. the ARD multipliers: out[lat*8 + k]; partial: nlat * sym_tiles(ceil(N/128)) * 8 doubles of scratch.
// Per-latent factors: mat_batch_stride = doubles per latent, off_per_lat = 0; joint ILMM matrix: 0 and N.  D <= 8.
cudaError_t launch_kgrad_ard(cudaStream_t st, const double* mat_base, size_t mat_batch_stride, int off_per_lat, const double* x, int N, int D,
                             const LatentParams* params, int nlat, const double* alpha, size_t alpha_stride, int form, double* partial,
                             double* out);
// gradient w.r.t. every hyper-parameter of every term of a (possibly composite) latent, storage as launch_kgrad_ard; x holds
// RAW points.  out[lat*44 + t*11 + {0, 1, 2, 3 + k}] = d/d {variance, inv_lengthscale, param, ard[k]} of term t (the
// LMM_GRAD_TERM_STRIDE layout of lmm.h), zeros where a term, shape parameter or ARD slot is absent.
// partial: nlat * sym_tiles(ceil(N/128)) * 44 doubles of scratch.  D <= 8 when a term has an ARDTransform.  max_terms /
// any_ard: the most terms of a latent of the batch, and whether a term of any latent has an ARDTransform.
cudaError_t launch_kgrad_terms(cudaStream_t st, const double* mat_base, size_t mat_batch_stride, int off_per_lat, const double* x, int N,
                               int D, const LatentParams* params, int nlat, int max_terms, bool any_ard, const double* alpha,
                               size_t alpha_stride, int form, double* partial, double* out);
// Posterior-predictive gradient, rectangular cross block: contraction of Gc = G + u v' (G: N x N* TiledRect per latent, rows the
// training points xa, columns the test points xb, both RAW [n][D]; u [nlat][u_stride], v [nlat][v_stride]) with ∂k(xa_r, xb_c)/∂θ
// for every term, every element once.  out[lat*44 + ...] as launch_kgrad_terms; partial: nlat * G.ntr * G.ntc * 44 doubles.
cudaError_t launch_kgrad_cross_terms(cudaStream_t st, TiledRect G, const double* xa, int Na, const double* xb, int Nb, int D,
                                     const LatentParams* params, int nlat, int max_terms, bool any_ard, const double* u, size_t u_stride,
                                     const double* v, size_t v_stride, int form, double* partial, double* out);
// M += s v v' on the stored tiles of a batch of packed-lower matrices (v [batch][v_stride], zero past the matrix size)
cudaError_t launch_sym_rank1(cudaStream_t st, TiledSym M, int batch, const double* v, size_t v_stride, double s);
// Missing-data dense model: contraction of G = (αα' - C^{-1})/2 over the (nobs x nobs) observed-entry matrix (negCinv = -C^{-1},
// batch 1; obs sorted by outputs, seg[j] = first entry of output j, seg[p] = nobs; x [N][D] raw points, Hm p x m col-major).
// out_terms[l*44 + ...] as launch_kgrad_terms with the weight H[j_a,l] H[j_b,l]; out_H[l*p + j] = 2 Σ_{a: j_a = j} Σ_b G_ab
// H[j_b,l] k_l(a,b); out_diag[0] = tr(-C^{-1}).  Scratch (ntl = sym_tiles(negCinv.nt)): tpart m*ntl*44, rowpart and colpart
// m*ntl*128 each, v m*nobs doubles.
cudaError_t launch_kgrad_masked(cudaStream_t st, TiledSym negCinv, const int* obs, int nobs, const double* x, int N, int D, const LatentParams* params,
                                int m, int p, const double* Hm, const double* alpha, int max_terms, bool any_ard, int form, const int* seg,
                                double* tpart, double* rowpart, double* colpart, double* v, double* out_terms, double* out_H, double* out_diag);
cudaError_t launch_scale_sub(cudaStream_t st, double* v, const double* a, double sa, const double* b, size_t n);
}  // namespace lmm

namespace lmm {
// ---- loo.cu : leave-one-input-out cross-validation of a batch of latent GPs (C = K + νI, A = C⁻¹, α = Aδ)
// d_i = A_ii from the diagonal of negA = -A (negA.base != null) or from dvec; per latent b, i < stride (each output nullable):
// q = α/d, sc = sqrt((1 + α q)/d), v = q/sc, lmean = δ + mean - q, lvar = 1/d - ν (all 0 for i >= N); loo[b] = LOO value.
cudaError_t launch_loo_terms(cudaStream_t st, TiledSym negA, const double* dvec, const double* alpha, const double* delta, size_t stride,
                             int N, const LatentParams* params, int batch, double log2pi, double* q, double* sc, double* v, double* lmean,
                             double* lvar, double* loo);
// B = A diag(sc) (full square tiles) from the packed-lower negA = -A
cudaError_t launch_sym_expand_scale(cudaStream_t st, TiledSym negA, const double* sc, size_t sc_stride, TiledRect B, int batch);
// u = α + w; out[b*4 + 2] = tr G = ½ Σ (u_i² + M_ii), out[b*4 + 3] = Σ w_i, dot[b] = w·δ  (i < N; M = -αα' - ww' - 2ARA)
cudaError_t launch_loo_grad_vectors(cudaStream_t st, TiledSym M, const double* alpha, const double* w, const double* delta, size_t stride,
                                    int N, int batch, double* u, double* out, double* dot);
}  // namespace lmm

namespace lmm {
cudaError_t launch_untile_rect_blockdiag(cudaStream_t st, TiledRect A, int batch, int Na, int Nb, double* dense, size_t ld);
}  // namespace lmm

namespace lmm {
// ---- misc.cu : small elementwise / bookkeeping kernels of the host drivers
cudaError_t launch_lml_terms(cudaStream_t st, double* terms, int slot0, int nb, const double* logdet, const double* quad, int n, double log2pi);
cudaError_t launch_regulariser(cudaStream_t st, double* slot, double c0, const double* resid, double sigma2);
cudaError_t launch_add_scalar(cudaStream_t st, double* v, size_t n, double s);
cudaError_t launch_copy_add(cudaStream_t st, int nlat, double* out, size_t stride_out, const double* in, size_t stride_in, int n, double s);
cudaError_t launch_add_mean(cudaStream_t st, int nlat, double* v, size_t stride, int n, const LatentParams* params);
cudaError_t launch_axpy(cudaStream_t st, double* y, const double* x, size_t n, double a);
cudaError_t launch_fill_noise(cudaStream_t st, int nlat, double* nv, size_t stride, int n_old, int n_new, const double* old_vec, size_t old_stride,
                              const LatentParams* old_params, const double* new_noise);
cudaError_t launch_repeat_block(cudaStream_t st, double* dst, const double* E, int mm, size_t total);
}  // namespace lmm
