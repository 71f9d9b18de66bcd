// Sparse variational (VFE) inference of an OILMM / IndependentMOGP: Titsias' collapsed bound with M inducing inputs z shared by
// the latents (u_l = f_l(z)), and the approximate posterior's marginals.  After the projection the likelihood factorises exactly
// as for the logpdf and LOO (host_loo.cu), so
//   ELBO = Σ_l ELBO_l(ỹ_l = (TY)_l; ν_l = σ²/S_l) + regulariser(U, S, σ², Y)     (IndependentMOGP: T = I, ν = σ², no regulariser)
// with the per-latent bound of vfe.cu.  Per latent: Kz = K(z, z) + jitter I is factored, and the training points are streamed in
// chunks of whole tile rows: K(x_c, z) (launch_kmat_cross), B'_c = K(x_c, z) Lz^{-T} (trsm_right_lt) and the Gram of [B'_c | δ_c]
// (vfe_gram_kernel) accumulated in chunk order -- about 2 M² N flop instead of the exact path's N³/3, and no N x N matrix.  Then
// Σ = I + Ψ/ν is factored (chol_factor) and c = L_Σ^{-1} b (forward solve) gives b'Σ^{-1}b = |c|².
// The posterior keeps Lz, L_Σ and the weights w = Lz^{-T} Σ^{-1} b / ν: at x*, with V = K(x*, z) Lz^{-T},
//   mean = μ + K(x*, z) w,   latent var = k(x*, x*) - |V|²_rows + |V L_Σ^{-T}|²_rows
// which post_latent_marginals evaluates with the exact posterior's kernels plus one more TRSM sweep.
#include "host_internal.h"

namespace lmm_host {
namespace {

int vfe_run(lmm_ctx* ctx, bool orth, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* z, int M, double jitter,
            int p, double sigma2, const double* y, const Projection& pr, const double* Shost, const std::vector<double>& Hhost, GradOut out,
            lmm_post** out_post) {
  const bool grad = out.grad_latents || out.grad_ard || out.grad_sigma2 || out.grad_y || out.grad_U || out.grad_S || out.grad_terms;
  GradRun s;
  int rc = grad_run_setup(ctx, orth, latents, m, x, N, D, p, y, pr, out, s);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  const int lo = s.lo, hi = s.hi, mloc = s.mloc, nt = s.nt, nl = s.nl;
  const size_t npad = s.npad;
  const int mt = ntiles(M);
  const size_t mpad = (size_t)mt * TILE, symd = sym_tiles(mt) * TT, rectd = (size_t)mt * mt * TT, wst = (size_t)mt * TT;
  DevBuf b_z, b_zp, b_Lz, b_Wz, b_LS, b_WS, b_psi, b_b, b_dd, b_r, b_c, b_w, b_q, b_tmp, b_ldz, b_lds, b_iz, b_is, b_X, b_part, b_bpart,
      b_ddpart;
  DevBuf b_G, b_Xz, b_XS, b_nS, b_Af, b_Pf, b_OA, b_OP, b_Mz, b_v, b_zero, b_a, b_gz, b_gx, b_gc, b_tp, b_g4, b_dot;
  if ((rc = stage_xpad(ctx, b_z, z, M, D))) return rc;
  std::vector<double> jit(m, jitter);
  if ((rc = upload_params(ctx, b_zp, latents, jit.data(), lo, hi, D))) return rc;
  std::vector<int> hinfo(nl, 0);
  std::vector<double> hg4((size_t)nl * 4, 0.0), hdot(nl, 0.0);
  if (grad && !s.b_gterms.p) {  // the per-term contraction supplies grad_latents[:, 0:2] and grad_ard too
    terms_shape(latents, lo, hi, s.max_terms, s.terms_ard);
    CU(s.b_gterms.alloc(ctx, (size_t)m * TERM_SLOTS * sizeof(double)));
    CU(cudaMemsetAsync(s.b_gterms.p, 0, (size_t)m * TERM_SLOTS * sizeof(double), st));
  }
  if (mloc > 0) {
    // per latent: the M x M factors, Gram and vectors (+ the gradient's square matrices); per tile row of training points: B'
    // (+ the K(x, z) cotangent)
    const size_t fixed = (3 * symd + 2 * wst + 7 * mpad + (grad ? 6 * rectd + 2 * symd + symd / TT * TERM_SLOTS : 0)) * sizeof(double);
    const size_t row_bytes = (size_t)mt * TT * sizeof(double) * (grad ? 2 : 1) + (grad ? (size_t)mt * TERM_SLOTS * sizeof(double) : 0);
    int chunk = mloc;
    if (!out_post) CU(mem_fit(ctx, fixed + (size_t)(nt < 64 ? nt : 64) * row_bytes, mloc, &chunk));
    auto alloc_d = [&](DevBuf& bf, size_t n) { return bf.alloc(ctx, n * sizeof(double)); };
    CU(alloc_d(b_Lz, chunk * symd));
    CU(alloc_d(b_Wz, chunk * wst));
    CU(alloc_d(b_LS, chunk * symd));
    CU(alloc_d(b_WS, chunk * wst));
    CU(alloc_d(b_psi, chunk * symd));
    CU(alloc_d(b_b, chunk * mpad));
    CU(alloc_d(b_r, chunk * mpad));
    CU(alloc_d(b_c, chunk * mpad));
    CU(alloc_d(b_w, chunk * mpad));
    CU(alloc_d(b_q, chunk * mpad));
    CU(alloc_d(b_tmp, chunk * mpad));
    CU(alloc_d(b_dd, chunk));
    CU(alloc_d(b_ldz, chunk));
    CU(alloc_d(b_lds, chunk));
    CU(b_iz.alloc(ctx, (size_t)mloc * sizeof(int)));
    CU(b_is.alloc(ctx, (size_t)mloc * sizeof(int)));
    CU(cudaMemsetAsync(b_iz.p, 0, (size_t)mloc * sizeof(int), st));
    CU(cudaMemsetAsync(b_is.p, 0, (size_t)mloc * sizeof(int), st));
    // tile rows of training points per chunk: the option, or as many as fit
    int ct = ctx->vfe_chunk;
    if (ct <= 0) CU(mem_fit(ctx, (size_t)chunk * row_bytes, nt, &ct));
    if (ct > nt) ct = nt;
    // one split for every launch of the call: the scratch below holds splits x chunk partial Grams, and no batch exceeds chunk
    const int splits = vfe_gram_splits(mt, chunk, ct);
    CU(alloc_d(b_X, (size_t)chunk * ct * mt * TT));
    CU(alloc_d(b_part, (size_t)splits * chunk * symd));
    CU(alloc_d(b_bpart, (size_t)splits * chunk * mpad));
    CU(alloc_d(b_ddpart, (size_t)splits * chunk));
    if (grad) {
      CU(alloc_d(b_G, (size_t)chunk * ct * mt * TT));
      for (DevBuf* bf : {&b_Xz, &b_XS, &b_Af, &b_Pf, &b_OA, &b_OP}) CU(alloc_d(*bf, chunk * rectd));
      CU(alloc_d(b_nS, chunk * symd));
      CU(alloc_d(b_Mz, chunk * symd));
      CU(alloc_d(b_v, chunk * mpad));
      CU(alloc_d(b_zero, chunk * mpad));
      CU(cudaMemsetAsync(b_zero.p, 0, chunk * mpad * sizeof(double), st));
      CU(alloc_d(b_a, (size_t)mloc * npad));
      CU(alloc_d(b_gz, (size_t)chunk * TERM_SLOTS));
      CU(alloc_d(b_gx, (size_t)chunk * TERM_SLOTS));
      CU(alloc_d(b_gc, (size_t)chunk * TERM_SLOTS));
      const size_t tpn = std::max(sym_tiles(mt), (size_t)ct * mt) * TERM_SLOTS;
      CU(alloc_d(b_tp, chunk * tpn));
      CU(alloc_d(b_g4, (size_t)mloc * 4));
      CU(alloc_d(b_dot, (size_t)mloc));
      CU(cudaMemsetAsync(b_g4.p, 0, (size_t)mloc * 4 * sizeof(double), st));
    }
    double* d_vec = s.b_vec.as<double>();
    const double* dx = s.b_x.as<double>();
    for (int c0 = 0; c0 < mloc; c0 += chunk) {
      const int nb = (c0 + chunk <= mloc) ? chunk : mloc - c0;
      const TiledSym Lz{b_Lz.as<double>(), mt, symd}, LS{b_LS.as<double>(), mt, symd}, Psi{b_psi.as<double>(), mt, symd};
      const LatentParams* dp = s.b_params.as<LatentParams>() + c0;  // noise = ν_l
      const LatentParams* zp = b_zp.as<LatentParams>() + c0;        // noise = jitter
      const double* delta = s.b_ty.as<double>() + (size_t)c0 * npad;
      // B'_c = K(x_c, z) Lz^{-T} for the row chunk [r0, r0 + nr)
      auto build_rows = [&](int r0, const TiledRect& X) -> int {
        CU(launch_kmat_cross(st, X, nb, dx + (size_t)r0 * TILE * D, N - r0 * TILE, b_z.as<double>(), M, D, dp, ctx->distance_form));
        CU(trsm_right_lt(ctx, X, Lz, b_Wz.as<double>(), wst, nb, dp));  // |B'(i, :)|² = Q_ii <= k_ii bounds the rows
        ctx->launches += 2;
        return LMM_OK;
      };
      CU(launch_kmat_sym(st, Lz, nb, b_z.as<double>(), M, D, zp, ctx->distance_form));
      CU(chol_factor(ctx, Lz, b_Wz.as<double>(), wst, nb, b_ldz.as<double>(), b_iz.as<int>() + c0));
      ++ctx->launches;
      for (int r0 = 0; r0 < nt; r0 += ct) {
        const int nr = (r0 + ct <= nt) ? ct : nt - r0;
        const TiledRect X{b_X.as<double>(), nr, mt, (size_t)nr * mt * TT};
        if ((rc = build_rows(r0, X))) return rc;
        CU(launch_vfe_gram(st, X, delta + (size_t)r0 * TILE, npad, nb, Psi, b_b.as<double>(), b_dd.as<double>(), r0 > 0, splits,
                           b_part.as<double>(), b_bpart.as<double>(), b_ddpart.as<double>()));
        ++ctx->launches;
      }
      CU(launch_vfe_sigma(st, Psi, LS, dp, nb));
      CU(cudaMemsetAsync(b_lds.p, 0, (size_t)nb * sizeof(double), st));
      CU(chol_factor(ctx, LS, b_WS.as<double>(), wst, nb, b_lds.as<double>(), b_is.as<int>() + c0));
      CU(cudaMemcpyAsync(b_r.p, b_b.p, (size_t)nb * mpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_fwd_solve(st, LS, b_WS.as<double>(), wst, b_r.as<double>(), b_c.as<double>(), mpad, nb, &ctx->launches));
      CU(launch_vfe_terms(st, Psi, b_lds.as<double>(), b_c.as<double>(), b_dd.as<double>(), N, dp, nb, LOG2PI,
                          (out_post || grad) ? b_r.as<double>() : nullptr, d_vec + lo + c0));
      ctx->launches += 3;
      if (!out_post && !grad) continue;
      // q = Σ⁻¹ b / ν = L_Σ^{-T} c / ν and w = Lz^{-T} q (the solves consume their right-hand sides)
      CU(launch_bwd_solve(st, LS, b_WS.as<double>(), wst, b_r.as<double>(), b_q.as<double>(), mpad, nb, &ctx->launches));
      CU(cudaMemcpyAsync(b_tmp.p, b_q.p, (size_t)nb * mpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_bwd_solve(st, Lz, b_Wz.as<double>(), wst, b_tmp.as<double>(), b_w.as<double>(), mpad, nb, &ctx->launches));
      if (!grad) continue;
      // ---- gradient.  Xz = Lz^{-T}, -Σ⁻¹ = -XS XS' (XS = L_Σ^{-T}), the brackets A and P (full tiles), then
      //   OA = -Xz A, OP = -Xz P,  Mz = -OP Xz' = Lz^{-T} P Lz⁻¹ (= 2 Ḡz),  G_c = -B'_c OA' = B'_c A Lz⁻¹ (Ḡxz without δβ'/ν²)
      const TiledRect Xz{b_Xz.as<double>(), mt, mt, rectd}, XS{b_XS.as<double>(), mt, mt, rectd};
      const TiledRect Af{b_Af.as<double>(), mt, mt, rectd}, Pf{b_Pf.as<double>(), mt, mt, rectd};
      const TiledRect OA{b_OA.as<double>(), mt, mt, rectd}, OP{b_OP.as<double>(), mt, mt, rectd};
      const TiledSym nS{b_nS.as<double>(), mt, symd}, Mz{b_Mz.as<double>(), mt, symd};
      CU(launch_rect_identity(st, Xz, nb));
      CU(trsm_right_lt_upper(ctx, st, Xz, Lz, b_Wz.as<double>(), wst, nb));
      CU(launch_rect_identity(st, XS, nb));
      CU(trsm_right_lt_upper(ctx, st, XS, LS, b_WS.as<double>(), wst, nb));
      CU(cudaMemsetAsync(b_nS.p, 0, (size_t)nb * symd * sizeof(double), st));
      GemmArgs g{};
      g.A = operand(XS); g.B = operand(XS); g.C = operand(nS);
      g.k0 = 0; g.k1 = mt; g.sym = 1; g.k_from_row = 1;
      CU(launch_gemm(st, GEMM_UPDATE, g, mt, mt, nb));
      CU(launch_vfe_brackets(st, nS, Psi, b_q.as<double>(), b_w.as<double>(), dp, Af, Pf, b_v.as<double>(), nb));
      CU(cudaMemsetAsync(b_OA.p, 0, (size_t)nb * rectd * sizeof(double), st));
      CU(cudaMemsetAsync(b_OP.p, 0, (size_t)nb * rectd * sizeof(double), st));
      g = GemmArgs{};
      g.A = operand(Xz); g.B = operand(Af); g.C = operand(OA);
      g.k0 = 0; g.k1 = mt; g.k_from_row = 1;  // Xz is upper triangular
      CU(launch_gemm(st, GEMM_UPDATE, g, mt, mt, nb));
      g.B = operand(Pf); g.C = operand(OP);
      CU(launch_gemm(st, GEMM_UPDATE, g, mt, mt, nb));
      CU(cudaMemsetAsync(b_Mz.p, 0, (size_t)nb * symd * sizeof(double), st));
      g = GemmArgs{};
      g.A = operand(OP); g.B = operand(Xz); g.C = operand(Mz);
      g.k0 = 0; g.k1 = mt; g.sym = 1;
      CU(launch_gemm(st, GEMM_UPDATE, g, mt, mt, nb));
      // K(z, z): G = ½ Mz
      CU(launch_kgrad_terms(st, Mz.base, Mz.batch_stride, 0, b_z.as<double>(), M, D, zp, nb, s.max_terms, s.terms_ard, b_zero.as<double>(),
                            mpad, ctx->distance_form, b_tp.as<double>(), b_gz.as<double>()));
      ctx->launches += 12;
      // K(x, z), chunk by chunk: G_c + δ_c (β/ν²)', accumulated in chunk order; B'_c q into a (finished by vfe_grad)
      CU(cudaMemsetAsync(b_gx.p, 0, (size_t)nb * TERM_SLOTS * sizeof(double), st));
      double* a = b_a.as<double>() + (size_t)c0 * npad;
      CU(cudaMemsetAsync(a, 0, (size_t)nb * npad * sizeof(double), st));
      for (int r0 = 0; r0 < nt; r0 += ct) {
        const int nr = (r0 + ct <= nt) ? ct : nt - r0;
        const TiledRect X{b_X.as<double>(), nr, mt, (size_t)nr * mt * TT}, G{b_G.as<double>(), nr, mt, (size_t)nr * mt * TT};
        if ((rc = build_rows(r0, X))) return rc;
        CU(launch_rect_gemv(st, X, b_q.as<double>(), mpad, a + (size_t)r0 * TILE, npad, dp, 0, nb));
        CU(cudaMemsetAsync(b_G.p, 0, (size_t)nb * nr * mt * TT * sizeof(double), st));
        g = GemmArgs{};
        g.A = operand(X); g.B = operand(OA); g.C = operand(G);
        g.k0 = 0; g.k1 = mt;
        CU(launch_gemm(st, GEMM_UPDATE, g, mt, nr, nb));
        CU(launch_kgrad_cross_terms(st, G, dx + (size_t)r0 * TILE * D, N - r0 * TILE, b_z.as<double>(), M, D, dp, nb, s.max_terms,
                                    s.terms_ard, delta + (size_t)r0 * TILE, npad, b_v.as<double>(), mpad, ctx->distance_form,
                                    b_tp.as<double>(), b_gc.as<double>()));
        CU(launch_axpy(st, b_gx.as<double>(), b_gc.as<double>(), (size_t)nb * TERM_SLOTS, 1.0));
        ctx->launches += 4;
      }
      double* gt = s.b_gterms.as<double>() + (size_t)(lo + c0) * TERM_SLOTS;
      CU(launch_vfe_grad(st, nS, Psi, b_q.as<double>(), b_c.as<double>(), b_dd.as<double>(), delta, npad, N, dp, nb, a,
                         b_g4.as<double>() + (size_t)c0 * 4, b_dot.as<double>() + c0, b_gz.as<double>(), b_gx.as<double>(), gt));
      ++ctx->launches;
      // term 0's variance / inv_lengthscale and ARD slots are the single-kernel outputs of the shared chain
      CU(cudaMemcpy2DAsync(b_g4.as<double>() + (size_t)c0 * 4, 4 * sizeof(double), gt, TERM_SLOTS * sizeof(double), 2 * sizeof(double),
                           (size_t)nb, cudaMemcpyDeviceToDevice, st));
      if (s.want_ard)
        CU(cudaMemcpy2DAsync(s.b_gard.as<double>() + (size_t)(lo + c0) * MAX_ARD, MAX_ARD * sizeof(double), gt + 3, TERM_SLOTS * sizeof(double),
                             MAX_ARD * sizeof(double), (size_t)nb, cudaMemcpyDeviceToDevice, st));
    }
    std::vector<int> hz(mloc), hs(mloc);
    CU(copy_out(ctx, hz.data(), b_iz.p, (size_t)mloc * sizeof(int)));
    CU(copy_out(ctx, hs.data(), b_is.p, (size_t)mloc * sizeof(int)));
    if (grad) {
      CU(copy_out(ctx, hg4.data(), b_g4.p, (size_t)mloc * 4 * sizeof(double)));
      CU(copy_out(ctx, hdot.data(), b_dot.p, (size_t)mloc * sizeof(double)));
    }
    CU(cudaStreamSynchronize(st));
    for (int i = 0; i < mloc; ++i) hinfo[i] = hz[i] ? hz[i] : hs[i];
  }
  if ((rc = grad_run_finish(ctx, orth, latents, m, N, D, p, sigma2, pr, Shost, out, s, b_a.as<double>(), hinfo, hg4, hdot))) return rc;
  if (!out_post) return LMM_OK;
  DevBuf b_H;
  CU(b_H.alloc(ctx, Hhost.size() * sizeof(double)));
  CU(copy_in(ctx, b_H.as<double>(), Hhost.data(), Hhost.size()));
  CU(cudaStreamSynchronize(st));
  lmm_post* P = new lmm_post();  // nothing below can fail: ownership of the device buffers moves to P
  P->ctx = ctx; P->kind = POST_VFE; P->vfe_oilmm = orth;
  P->m = m; P->p = p; P->N = M; P->D = D; P->nt = mt; P->lo = lo; P->hi = hi;
  P->adopt_descs(latents, m, D);
  P->noise = pr.noise;
  P->H = Hhost;
  P->sigma2 = sigma2;
  P->bytes = (size_t)mloc * (2 * symd + 2 * (size_t)mt * TT + mpad) * sizeof(double) + mpad * D * sizeof(double);
  P->d_xpad = (double*)b_z.detach();
  P->d_L = (double*)b_Lz.detach();
  P->d_W = (double*)b_Wz.detach();
  P->d_L2 = (double*)b_LS.detach();
  P->d_W2 = (double*)b_WS.detach();
  P->d_alpha = (double*)b_w.detach();
  P->d_params = (LatentParams*)s.b_params.detach();
  P->d_H = (double*)b_H.detach();
  *out_post = P;
  return LMM_OK;
}

// Arguments every VFE entry point shares: inducing inputs, jitter, fully observed y.
int check_vfe(lmm_ctx* ctx, const double* z, int M, double jitter, double sigma2, const double* y, size_t ny) {
  if (!z || !y) return ctx->fail(LMM_E_ARG, "null pointer");
  if (M < 1) return ctx->fail(LMM_E_ARG, "VFE needs at least one inducing input (M >= 1)");
  if (!(jitter >= 0.0) || !std::isfinite(jitter)) return ctx->fail(LMM_E_ARG, "the inducing-point jitter must be finite and >= 0");
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  CU(cudaSetDevice(ctx->device));
  std::vector<double> h;
  const double* v = y;
  if (is_device_ptr(y)) {
    h.resize(ny);
    CU(cudaMemcpyAsync(h.data(), y, ny * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    v = h.data();
  }
  for (size_t i = 0; i < ny; ++i)
    if (v[i] != v[i]) return ctx->fail(LMM_E_ARG, "y has a NaN entry: the VFE bound needs fully observed data");
  return LMM_OK;
}

int oilmm_vfe(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* z, int M, double jitter,
              const double* U, const double* S, int p, double sigma2, const double* y, int out_dim, GradOut out, lmm_post** out_post) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (out_post) *out_post = nullptr;
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!U || !S) return ctx->fail(LMM_E_ARG, "null pointer");
  if (m > p) return ctx->fail(LMM_E_ARG, "more latents than outputs");
  if ((rc = check_vfe(ctx, z, M, jitter, sigma2, y, (size_t)p * N))) return rc;
  Projection pr;
  std::vector<double> H;
  if ((rc = oilmm_projection(ctx, U, S, p, m, sigma2, N, pr, H))) return rc;
  return vfe_run(ctx, true, latents, m, x, N, D, z, M, jitter, p, sigma2, y, pr, S, H, out, out_post);
}

int imogp_vfe(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, const double* z, int M, double jitter, double sigma2,
              const double* y, int out_dim, GradOut out, lmm_post** out_post) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (out_post) *out_post = nullptr;
  int rc = check_common(ctx, fs, m, x, N, D, m, out_dim);
  if (rc) return rc;
  if ((rc = check_vfe(ctx, z, M, jitter, sigma2, y, (size_t)m * N))) return rc;
  Projection pr;
  pr.T.assign((size_t)m * m, 0.0);
  for (int i = 0; i < m; ++i) pr.T[(size_t)i * m + i] = 1.0;
  pr.noise.assign(m, sigma2);
  pr.has_reg = false;
  return vfe_run(ctx, false, fs, m, x, N, D, z, M, jitter, m, sigma2, y, pr, nullptr, pr.T, out, out_post);
}

}  // namespace
}  // namespace lmm_host

extern "C" int lmm_oilmm_vfe(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* z, int M,
                             double jitter, const double* U, const double* S, int p, double sigma2, const double* y, int out_dim,
                             double* out_elbo, double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_U,
                             double* grad_S, double* grad_terms, int* info_latent) {
  GradOut out{out_elbo, grad_latents, grad_sigma2, grad_y, info_latent};
  out.grad_U = grad_U;
  out.grad_S = grad_S;
  out.grad_ard = grad_ard;
  out.grad_terms = grad_terms;
  return oilmm_vfe(ctx, latents, m, x, N, D, z, M, jitter, U, S, p, sigma2, y, out_dim, out, nullptr);
}

extern "C" int lmm_imogp_vfe(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, const double* z, int M, double jitter,
                             double sigma2, const double* y, int out_dim, double* out_elbo, double* grad_latents, double* grad_ard,
                             double* grad_sigma2, double* grad_y, double* grad_terms, int* info_latent) {
  GradOut out{out_elbo, grad_latents, grad_sigma2, grad_y, info_latent};
  out.grad_ard = grad_ard;
  out.grad_terms = grad_terms;
  return imogp_vfe(ctx, fs, m, x, N, D, z, M, jitter, sigma2, y, out_dim, out, nullptr);
}

extern "C" int lmm_oilmm_vfe_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* z,
                                       int M, double jitter, const double* U, const double* S, int p, double sigma2, const double* y,
                                       int out_dim, lmm_post** out_post, double* out_elbo, int* info_latent) {
  if (ctx && !out_post) return ctx->fail(LMM_E_ARG, "null pointer");
  return oilmm_vfe(ctx, latents, m, x, N, D, z, M, jitter, U, S, p, sigma2, y, out_dim, GradOut{out_elbo, nullptr, nullptr, nullptr, info_latent},
                   out_post);
}

extern "C" int lmm_imogp_vfe_posterior(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, const double* z, int M,
                                       double jitter, double sigma2, const double* y, int out_dim, lmm_post** out_post, double* out_elbo,
                                       int* info_latent) {
  if (ctx && !out_post) return ctx->fail(LMM_E_ARG, "null pointer");
  return imogp_vfe(ctx, fs, m, x, N, D, z, M, jitter, sigma2, y, out_dim, GradOut{out_elbo, nullptr, nullptr, nullptr, info_latent}, out_post);
}
