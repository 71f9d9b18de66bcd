// Leave-one-input-out (LOO) cross-validation of an OILMM / IndependentMOGP: value, LOO predictive marginals and gradient.
// Leaving out one input (all p outputs at x_i) keeps the OILMM structure -- T = S^{-1/2}U' acts input by input and the
// orthogonal-complement regulariser is a sum over inputs -- so exactly
//   Σ_i log p(y_i | y_{-i}) = Σ_l LOO_l(ỹ_l; ν_l) + regulariser(U, S, σ², Y)
// with the per-latent GP LOO of loo.cu on ỹ_l = (TY)_l, ν_l = σ²/S_l (IndependentMOGP: T = I, ν = σ², no regulariser).
// Per latent the value costs the factorisation plus X = L^{-T} (TRSM on an identity, N³/3): d = rowsumsq(X).  The gradient
// adds -A = -XX' (SYRK, N³/3), B = A R^{1/2} and -2BB' (SYRK, N³) for M = -αα' - ww' - 2ARA, contracted as G = ½(uu' + M)
// with u = α + w by kgrad_terms.  dLOO/dδ = -w takes the place of the logpdf's -α in the chain to U, S, σ², y and the means,
// which is the logpdf gradient's own (grad_run_setup / grad_run_finish).
#include "host_internal.h"

namespace lmm_host {
namespace {

int loo_run(lmm_ctx* ctx, bool orth, const lmm_gp_desc* latents, int m, const double* x, int N, int D, int p, double sigma2,
            const double* y, const Projection& pr, const double* Shost, const std::vector<double>& Hhost, GradOut out, double* loo_mean,
            double* loo_var) {
  const bool grad = out.grad_latents || out.grad_ard || out.grad_sigma2 || out.grad_y || out.grad_U || out.grad_S || out.grad_terms;
  const bool marg = loo_mean || loo_var;
  GradRun s;
  int rc = grad_run_setup(ctx, orth, latents, m, x, N, D, p, y, pr, out, s);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  const int lo = s.lo, mloc = s.mloc, nt = s.nt, nl = s.nl;
  const size_t npad = s.npad;
  double* d_vec = s.b_vec.as<double>();
  if (grad && !s.b_gterms.p) {  // the per-term contraction supplies grad_latents[:, 0:2] and grad_ard too
    terms_shape(latents, lo, s.hi, s.max_terms, s.terms_ard);
    CU(s.b_gterms.alloc(ctx, (size_t)m * TERM_SLOTS * sizeof(double)));
    CU(cudaMemsetAsync(s.b_gterms.p, 0, (size_t)m * TERM_SLOTS * sizeof(double), st));
  }
  DevBuf b_L, b_W, b_X, b_alpha, b_w, b_r, b_z, b_logdet, b_info, b_d, b_sc, b_v, b_u, b_lm, b_lv, b_g4, b_dot, b_tpart;
  std::vector<int> hinfo(nl, 0);
  std::vector<double> hg4((size_t)nl * 4, 0.0), hdot(nl, 0.0);
  if (mloc > 0) {
    const size_t per_lat = factor_bytes_per_latent(nt) + (size_t)nt * nt * TT * sizeof(double) + 9 * npad * sizeof(double);
    int chunk = 0;
    CU(mem_fit(ctx, per_lat, mloc, &chunk));
    const int ntl = (int)sym_tiles(nt);
    CU(b_L.alloc(ctx, (size_t)chunk * sym_tiles(nt) * TT * sizeof(double)));
    CU(b_W.alloc(ctx, (size_t)chunk * nt * TT * sizeof(double)));
    CU(b_X.alloc(ctx, (size_t)chunk * nt * nt * TT * sizeof(double)));
    CU(b_alpha.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    CU(b_r.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    CU(b_z.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    CU(b_logdet.alloc(ctx, (size_t)mloc * sizeof(double)));
    CU(b_info.alloc(ctx, (size_t)mloc * sizeof(int)));
    if (grad) {
      CU(b_w.alloc(ctx, (size_t)mloc * npad * sizeof(double)));
      CU(b_sc.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
      CU(b_v.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
      CU(b_u.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
      CU(b_g4.alloc(ctx, (size_t)mloc * 4 * sizeof(double)));
      CU(b_dot.alloc(ctx, (size_t)mloc * sizeof(double)));
      CU(b_tpart.alloc(ctx, (size_t)chunk * ntl * TERM_SLOTS * sizeof(double)));
    } else {
      CU(b_d.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    }
    if (marg) {
      CU(b_lm.alloc(ctx, (size_t)mloc * npad * sizeof(double)));
      CU(b_lv.alloc(ctx, (size_t)mloc * npad * sizeof(double)));
    }
    CU(cudaMemsetAsync(b_logdet.p, 0, (size_t)mloc * sizeof(double), st));
    CU(cudaMemsetAsync(b_info.p, 0, (size_t)mloc * sizeof(int), st));
    for (int c0 = 0; c0 < mloc; c0 += chunk) {
      const int nb = (c0 + chunk <= mloc) ? chunk : mloc - c0;
      TiledSym L{b_L.as<double>(), nt, sym_tiles(nt) * TT};
      TiledRect X{b_X.as<double>(), nt, nt, (size_t)nt * nt * TT};
      double* W = b_W.as<double>();
      const size_t wstride = (size_t)nt * TT;
      const LatentParams* dp = s.b_params.as<LatentParams>() + c0;
      const double* delta = s.b_ty.as<double>() + (size_t)c0 * npad;
      double* alpha = b_alpha.as<double>();
      double* lm = marg ? b_lm.as<double>() + (size_t)c0 * npad : nullptr;
      double* lv = marg ? b_lv.as<double>() + (size_t)c0 * npad : nullptr;
      CU(launch_kmat_sym(st, L, nb, s.b_x.as<double>(), N, D, dp, ctx->distance_form));
      CU(chol_factor(ctx, L, W, wstride, nb, b_logdet.as<double>() + c0, b_info.as<int>() + c0));
      CU(cudaMemcpyAsync(b_r.p, delta, (size_t)nb * npad * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_fwd_solve(st, L, W, wstride, b_r.as<double>(), b_z.as<double>(), npad, nb, &ctx->launches));
      CU(cudaMemcpyAsync(b_r.p, b_z.p, (size_t)nb * npad * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_bwd_solve(st, L, W, wstride, b_r.as<double>(), alpha, npad, nb, &ctx->launches));
      // X = L^{-T}: row i of X is column i of L^{-1}, so d_i = A_ii = |X(i, :)|²
      CU(launch_rect_identity(st, X, nb));
      CU(trsm_right_lt_upper(ctx, st, X, L, W, wstride, nb));
      ctx->launches += 2;
      if (!grad) {
        CU(launch_rect_rowsumsq(st, X, b_d.as<double>(), npad, nullptr, nb));
        CU(launch_loo_terms(st, TiledSym{nullptr, nt, 0}, b_d.as<double>(), alpha, delta, npad, N, dp, nb, LOG2PI, nullptr, nullptr,
                            nullptr, lm, lv, d_vec + lo + c0));
        ctx->launches += 2;
        continue;
      }
      double* w = b_w.as<double>() + (size_t)c0 * npad;
      // -A = -X X' into the (no longer needed) factor tiles
      CU(cudaMemsetAsync(b_L.p, 0, (size_t)nb * sym_tiles(nt) * TT * sizeof(double), st));
      GemmArgs g{};
      g.A = operand(X); g.B = operand(X); g.C = operand(L);
      g.i0 = 0; g.j0 = 0; g.k0 = 0; g.k1 = nt; g.sym = 1; g.k_from_row = 1;
      CU(launch_gemm(st, GEMM_UPDATE, g, nt, nt, nb));
      CU(launch_loo_terms(st, L, nullptr, alpha, delta, npad, N, dp, nb, LOG2PI, nullptr, b_sc.as<double>(), b_v.as<double>(), lm, lv,
                          d_vec + lo + c0));
      // B = A diag(sqrt(2r)) into X (free now): w = B (q / sqrt(2r)) = A q, and -B B' = -2 A R A into the tiles of -A
      CU(launch_sym_expand_scale(st, L, b_sc.as<double>(), npad, X, nb));
      CU(launch_rect_gemv(st, X, b_v.as<double>(), npad, w, npad, dp, 0, nb));
      CU(cudaMemsetAsync(b_L.p, 0, (size_t)nb * sym_tiles(nt) * TT * sizeof(double), st));
      g.k_from_row = 0;
      CU(launch_gemm(st, GEMM_UPDATE, g, nt, nt, nb));
      CU(launch_sym_rank1(st, L, nb, alpha, npad, -1.0));
      CU(launch_sym_rank1(st, L, nb, w, npad, -1.0));
      CU(launch_loo_grad_vectors(st, L, alpha, w, delta, npad, N, nb, b_u.as<double>(), b_g4.as<double>() + (size_t)c0 * 4,
                                 b_dot.as<double>() + c0));
      CU(launch_kgrad_terms(st, L.base, L.batch_stride, 0, s.b_x.as<double>(), N, D, dp, nb, s.max_terms, s.terms_ard, b_u.as<double>(), npad,
                            ctx->distance_form, b_tpart.as<double>(), s.b_gterms.as<double>() + (size_t)(lo + c0) * TERM_SLOTS));
      ctx->launches += 10;
      // term 0's variance / inv_lengthscale and ARD slots are the single-kernel outputs of the shared chain
      double* gt = s.b_gterms.as<double>() + (size_t)(lo + c0) * TERM_SLOTS;
      CU(cudaMemcpy2DAsync(b_g4.as<double>() + (size_t)c0 * 4, 4 * sizeof(double), gt, TERM_SLOTS * sizeof(double), 2 * sizeof(double),
                           (size_t)nb, cudaMemcpyDeviceToDevice, st));
      if (s.want_ard)
        CU(cudaMemcpy2DAsync(s.b_gard.as<double>() + (size_t)(lo + c0) * MAX_ARD, MAX_ARD * sizeof(double), gt + 3, TERM_SLOTS * sizeof(double),
                             MAX_ARD * sizeof(double), (size_t)nb, cudaMemcpyDeviceToDevice, st));
    }
    CU(copy_out(ctx, hinfo.data(), b_info.p, (size_t)mloc * sizeof(int)));
    if (grad) {
      CU(copy_out(ctx, hg4.data(), b_g4.p, (size_t)mloc * 4 * sizeof(double)));
      CU(copy_out(ctx, hdot.data(), b_dot.p, (size_t)mloc * sizeof(double)));
    }
    CU(cudaStreamSynchronize(st));
  }
  if (marg) {
    // observation space: mean = H (ỹ - q), var = H∘H (1/d - ν) + σ²  (H = U√S, or I for an IndependentMOGP)
    const size_t nout = (size_t)p * N;
    const bool multi = s.multi;
    DevBuf b_H, b_out;
    CU(b_H.alloc(ctx, Hhost.size() * sizeof(double)));
    CU(copy_in(ctx, b_H.as<double>(), Hhost.data(), Hhost.size()));
    CU(b_out.alloc(ctx, 2 * nout * sizeof(double)));
    CU(cudaMemsetAsync(b_out.p, 0, 2 * nout * sizeof(double), st));
    if (mloc > 0) {
      CU(launch_backproject(st, b_H.as<double>(), p, m, lo, mloc, b_lm.as<double>(), b_lv.as<double>(), npad, N, 0.0, sigma2, multi ? 0 : 1,
                            b_out.as<double>(), b_out.as<double>() + nout));
      ++ctx->launches;
    }
    if (multi) {
      int r = nccl_api().AllReduce(b_out.p, b_out.p, 2 * nout, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
      if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
      CU(launch_add_scalar(st, b_out.as<double>() + nout, nout, sigma2));
      ++ctx->launches;
    }
    if (loo_mean) CU(copy_out(ctx, loo_mean, b_out.p, nout * sizeof(double)));
    if (loo_var) CU(copy_out(ctx, loo_var, b_out.as<double>() + nout, nout * sizeof(double)));
    CU(cudaStreamSynchronize(st));
  }
  return grad_run_finish(ctx, orth, latents, m, N, D, p, sigma2, pr, Shost, out, s, b_w.as<double>(), hinfo, hg4, hdot);
}

// LMM_E_ARG for a NaN in y (host or device pointer): LOO of partially observed data is not defined here.
int reject_nan(lmm_ctx* ctx, const double* y, size_t n) {
  std::vector<double> h;
  const double* v = y;
  if (is_device_ptr(y)) {
    h.resize(n);
    CU(cudaMemcpyAsync(h.data(), y, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    v = h.data();
  }
  for (size_t i = 0; i < n; ++i)
    if (v[i] != v[i]) return ctx->fail(LMM_E_ARG, "y has a NaN entry: leave-one-out needs fully observed data");
  return LMM_OK;
}

}  // namespace
}  // namespace lmm_host

extern "C" int lmm_oilmm_loo(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U, const double* S,
                             int p, double sigma2, const double* y, int out_dim, double* out_loo, double* loo_mean, double* loo_var,
                             double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_U, double* grad_S,
                             double* grad_terms, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!U || !S || !y) return ctx->fail(LMM_E_ARG, "null pointer");
  if (m > p) return ctx->fail(LMM_E_ARG, "more latents than outputs");
  CU(cudaSetDevice(ctx->device));
  if ((rc = reject_nan(ctx, y, (size_t)p * N))) return rc;
  Projection pr;
  std::vector<double> H;
  if ((rc = oilmm_projection(ctx, U, S, p, m, sigma2, N, pr, H))) return rc;
  GradOut out{out_loo, grad_latents, grad_sigma2, grad_y, info_latent};
  out.grad_U = grad_U;
  out.grad_S = grad_S;
  out.grad_ard = grad_ard;
  out.grad_terms = grad_terms;
  return loo_run(ctx, true, latents, m, x, N, D, p, sigma2, y, pr, S, H, out, loo_mean, loo_var);
}

extern "C" int lmm_imogp_loo(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, double sigma2, const double* y,
                             int out_dim, double* out_loo, double* loo_mean, double* loo_var, double* grad_latents, double* grad_ard,
                             double* grad_sigma2, double* grad_y, double* grad_terms, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, fs, m, x, N, D, m, out_dim);
  if (rc) return rc;
  if (!y) return ctx->fail(LMM_E_ARG, "null pointer");
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  CU(cudaSetDevice(ctx->device));
  if ((rc = reject_nan(ctx, y, (size_t)m * N))) return rc;
  Projection pr;
  pr.T.assign((size_t)m * m, 0.0);
  for (int i = 0; i < m; ++i) pr.T[(size_t)i * m + i] = 1.0;
  pr.noise.assign(m, sigma2);
  pr.has_reg = false;
  GradOut out{out_loo, grad_latents, grad_sigma2, grad_y, info_latent};
  out.grad_ard = grad_ard;
  out.grad_terms = grad_terms;
  return loo_run(ctx, false, fs, m, x, N, D, m, sigma2, y, pr, nullptr, pr.T, out, loo_mean, loo_var);
}
