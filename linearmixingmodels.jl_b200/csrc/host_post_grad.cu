// Gradient of the posterior-predictive logpdf through the conditioning: logpdf(posterior(f(x, σ²), y)(x*, σ*²), y*) w.r.t.
// the latents' hyper-parameters and means, σ², σ*², y, y*, U and S (per-latent posteriors: OILMM, IndependentMOGP).
//
// Per latent (T = S^{-1/2} U', ν = σ²/S_i, ν* = σ*²/S_i; T = I, ν = σ² for an IndependentMOGP):
//   C = K(x,x) + ν I, α = C⁻¹ δ, W = C⁻¹ K(x,x*), Σ* = K(x*,x*) - K(x*,x) W + ν* I = L* L*', P = Σ*⁻¹,
//   β = P (ỹ* - m - K(x*,x) α), γ = W β, Φ = W L*⁻ᵀ, X* = L*⁻ᵀ.
// The derivative w.r.t. the three kernel blocks is
//   K(x*,x*): G** = (ββ' - P)/2                        (launch_kgrad_terms with -P = -X* X*', β)
//   K(x,x*):  Gc  = (α - γ)β' + Φ X*'  (N x N*)         (launch_kgrad_cross_terms with Φ X*', u = α - γ, v = β)
//   K(x,x):   Gx  = ((γ-α)(γ-α)' - αα' - ΦΦ')/2          (launch_kgrad_terms with -(ΦΦ' + αα'), α - γ)
// and d/dỹ = γ, d/dỹ* = -β, d/dm = Σβ - Σγ, d/dν = tr(Gx), d/dν* = tr(G**).  W comes from the handle's factor without
// touching it: X = L⁻ᵀ (potri TRSM into scratch), V = K(x*,x) L⁻ᵀ, W = X V'.
#include <algorithm>

#include "host_internal.h"

namespace lmm_host {
namespace {

// Sums n doubles of device memory over the ranks of the communicator (no-op without one).
int allreduce_dev(lmm_ctx* ctx, double* d, size_t n) {
  if (!(ctx->comm && ctx->nranks > 1) || n == 0) return LMM_OK;
  if (nccl_api().AllReduce(d, d, n, NCCL_DOUBLE, NCCL_SUM, ctx->comm, ctx->stream) != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
  return LMM_OK;
}

// Same for a host vector (through a device buffer).
int allreduce_host(lmm_ctx* ctx, std::vector<double>& h) {
  if (!(ctx->comm && ctx->nranks > 1) || h.empty()) return LMM_OK;
  DevBuf b;
  CU(b.alloc(ctx, h.size() * sizeof(double)));
  CU(copy_in(ctx, b.as<double>(), h.data(), h.size()));
  int rc = allreduce_dev(ctx, b.as<double>(), h.size());
  if (rc) return rc;
  CU(copy_out(ctx, h.data(), b.p, h.size() * sizeof(double)));
  CU(cudaStreamSynchronize(ctx->stream));
  return LMM_OK;
}

const double* device_view(lmm_ctx* ctx, DevBuf& buf, const double* src, size_t n, int* rc) {
  *rc = LMM_OK;
  if (is_device_ptr(src)) return src;
  cudaError_t e = buf.alloc(ctx, n * sizeof(double));
  if (e == cudaSuccess) e = copy_in(ctx, buf.as<double>(), src, n);
  if (e != cudaSuccess) {
    *rc = ctx->fail_cuda(e, "staging an input", __LINE__, __FILE__);
    return nullptr;
  }
  return buf.as<double>();
}

}  // namespace
}  // namespace lmm_host

extern "C" int lmm_post_logpdf_grad_full(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, const double* y_train,
                                         double* out_logpdf, double* grad_sigma2, double* grad_y, double* grad_latents, double* grad_ard,
                                         double* grad_terms, double* grad_train_sigma2, double* grad_train_y, double* grad_U, double* grad_S,
                                         int* info_latent) {
  if (!post || !xs || Ns <= 0 || !ys) return LMM_E_ARG;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (post->kind == POST_VFE) return ctx->fail(LMM_E_UNSUPPORTED, VFE_POST_ONLY);
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  if (post->joint())
    return ctx->fail(LMM_E_UNSUPPORTED, "the posterior-predictive gradient through the conditioning is built for per-latent posteriors "
                                        "(OILMM, IndependentMOGP); joint posteriors (general ILMM, dense Σy, missing data): σ² and y* only");
  if (post->d_noise_vec)
    return ctx->fail(LMM_E_UNSUPPORTED, "the posterior-predictive gradient through the conditioning is not built for a sequentially "
                                        "conditioned posterior: σ² and y* only");
  if (!y_train) return ctx->fail(LMM_E_ARG, "y_train (the data the posterior was conditioned on) is required");
  const bool orth = post->kind == POST_OILMM;
  if (!orth && (grad_U || grad_S)) return ctx->fail(LMM_E_ARG, "grad_U / grad_S are for OILMM posteriors only");
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p, N = post->N, D = post->D, lo = post->lo, nloc = post->nloc(), nt = post->nt, nl = nloc > 0 ? nloc : 1;
  const size_t npad = post->npad();
  const double s2t = post->sigma2;  // training noise
  int rc;

  // ---- y_train must be the data of the handle: T y_train - m == δ to 1e-12 (norm-relative, over all ranks)
  Projection pr;
  std::vector<double> Hm;
  if (orth) {
    if ((rc = oilmm_projection(ctx, post->U.data(), post->S.data(), p, m, s2t, N, pr, Hm))) return rc;
  } else {
    pr.T.assign((size_t)m * m, 0.0);
    for (int i = 0; i < m; ++i) pr.T[(size_t)i * m + i] = 1.0;
  }
  DevBuf b_ytr, b_ys, b_T, b_means, b_ty, b_part, b_chk;
  const double* d_ytr = device_view(ctx, b_ytr, y_train, (size_t)p * N, &rc);
  if (rc) return rc;
  const double* d_ys = device_view(ctx, b_ys, ys, (size_t)p * Ns, &rc);
  if (rc) return rc;
  CU(b_T.alloc(ctx, pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, b_T.as<double>(), pr.T.data(), pr.T.size()));
  {
    std::vector<double> hmeans(nl, 0.0), chk(2, 0.0);
    for (int i = lo; i < post->hi; ++i) hmeans[i - lo] = post->descs[i].mean_const;
    CU(b_means.alloc(ctx, (size_t)nl * sizeof(double)));
    CU(copy_in(ctx, b_means.as<double>(), hmeans.data(), (size_t)nl));
    if (nloc > 0) {
      const size_t tot = (size_t)nloc * npad;
      CU(b_ty.alloc(ctx, tot * sizeof(double)));
      CU(cudaMemsetAsync(b_ty.p, 0, tot * sizeof(double), st));
      CU(b_part.alloc(ctx, (size_t)project_max_partials(N) * sizeof(double)));
      CU(launch_project(st, d_ytr, N, p, b_T.as<double>(), m, lo, nloc, b_means.as<double>(), b_ty.as<double>(), npad, nullptr, nullptr,
                        b_part.as<double>(), nullptr));
      CU(launch_scale_sub(st, b_ty.as<double>(), b_ty.as<double>(), 1.0, post->d_delta, tot));
      CU(b_chk.alloc(ctx, 2 * (size_t)nloc * sizeof(double)));
      CU(launch_sumsq(st, b_ty.as<double>(), npad, (int)npad, nloc, b_chk.as<double>()));
      CU(launch_sumsq(st, post->d_delta, npad, (int)npad, nloc, b_chk.as<double>() + nloc));
      ctx->launches += 4;
      std::vector<double> h(2 * (size_t)nloc);
      CU(copy_out(ctx, h.data(), b_chk.p, h.size() * sizeof(double)));
      CU(cudaStreamSynchronize(st));
      for (int i = 0; i < nloc; ++i) {
        chk[0] += h[i];
        chk[1] += h[(size_t)nloc + i];
      }
    }
    if ((rc = allreduce_host(ctx, chk))) return rc;  // collective: every rank takes part
    if (!(std::sqrt(chk[0]) <= 1e-12 * std::sqrt(chk[1])))
      return ctx->fail(LMM_E_ARG, "y_train does not match the data the posterior was conditioned on");
  }

  // ---- value, σ*² and y* gradients: the code of lmm_post_logpdf_grad, keeping its predictive factors and β
  PredictiveKeep keep;
  double gs2 = 0.0;
  if ((rc = post_logpdf_impl(post, xs, Ns, sigma2, ys, out_logpdf, &gs2, grad_y, info_latent, &keep))) return rc;
  if (grad_sigma2) *grad_sigma2 = gs2;
  const Predictive& P = keep.P;
  const int nts = P.nts;
  const size_t nspad = P.nspad;

  int max_terms = 1;
  bool any_ard = false;
  terms_shape(post->descs.data(), lo, post->hi, max_terms, any_ard);
  DevBuf b_gt, b_u, b_g, b_sq, b_sb, b_sg;
  const size_t ngt = (size_t)3 * m * TERM_SLOTS;  // [K(x*,x*) | K(x,x) | K(x,x*)] contributions
  CU(b_gt.alloc(ctx, ngt * sizeof(double)));
  CU(cudaMemsetAsync(b_gt.p, 0, ngt * sizeof(double), st));
  CU(b_u.alloc(ctx, (size_t)nl * npad * sizeof(double)));  // α - γ
  CU(b_g.alloc(ctx, (size_t)nl * npad * sizeof(double)));  // -γ
  CU(cudaMemsetAsync(b_g.p, 0, (size_t)nl * npad * sizeof(double), st));
  CU(b_sq.alloc(ctx, (size_t)3 * nl * sizeof(double)));    // |α - γ|², |α|², |Φ|_F²
  CU(b_sb.alloc(ctx, (size_t)4 * nl * sizeof(double)));    // Σβ in slot 3 (launch_kgrad_finish)
  CU(b_sg.alloc(ctx, (size_t)4 * nl * sizeof(double)));    // Σ(-γ) in slot 3
  double* gt_ss = b_gt.as<double>();
  double* gt_x = gt_ss + (size_t)m * TERM_SLOTS;
  double* gt_c = gt_x + (size_t)m * TERM_SLOTS;
  const int form = ctx->distance_form;
  if (nloc > 0) {
    const size_t sq_t = (size_t)nt * nt * TT, rect_t = (size_t)nt * nts * TT, sqs_t = (size_t)nts * nts * TT, syms_t = sym_tiles(nts) * TT;
    const size_t npart = std::max({sym_tiles(nt), (size_t)nt * nts, sym_tiles(nts)}) * TERM_SLOTS;
    const size_t per_lat = (sq_t + 2 * rect_t + sqs_t + syms_t + npart) * sizeof(double);
    int chunk = 0;
    CU(mem_fit(ctx, per_lat, nloc, &chunk));
    DevBuf b_X, b_V, b_Wn, b_Xs, b_Ms, b_tp;
    CU(b_X.alloc(ctx, (size_t)chunk * sq_t * sizeof(double)));
    CU(b_V.alloc(ctx, (size_t)chunk * rect_t * sizeof(double)));
    CU(b_Wn.alloc(ctx, (size_t)chunk * rect_t * sizeof(double)));
    CU(b_Xs.alloc(ctx, (size_t)chunk * sqs_t * sizeof(double)));
    CU(b_Ms.alloc(ctx, (size_t)chunk * syms_t * sizeof(double)));
    CU(b_tp.alloc(ctx, (size_t)chunk * npart * sizeof(double)));
    const TiledSym L = post->Lsym();
    const size_t wst = post->wstride(), wsts = (size_t)nts * TT;
    const size_t syml = sym_tiles(nt) * TT;
    for (int c0 = 0; c0 < nloc; c0 += chunk) {
      const int nb = (c0 + chunk <= nloc) ? chunk : nloc - c0;
      const TiledSym Lc{L.base + (size_t)c0 * L.batch_stride, nt, L.batch_stride};
      const double* Wc = post->d_W + (size_t)c0 * wst;
      const TiledSym Lsc{P.C.as<double>() + (size_t)c0 * syms_t, nts, syms_t};
      const double* Wsc = P.W.as<double>() + (size_t)c0 * wsts;
      const LatentParams* trp = post->d_params + c0;               // training noise (kernel terms are the same)
      const LatentParams* tsp = P.params.as<LatentParams>() + c0;  // test noise
      const double* alpha = post->d_alpha + (size_t)c0 * npad;
      const double* beta = keep.beta.as<double>() + (size_t)c0 * nspad;
      double* u = b_u.as<double>() + (size_t)c0 * npad;
      double* g = b_g.as<double>() + (size_t)c0 * npad;
      TiledRect X{b_X.as<double>(), nt, nt, sq_t};
      TiledRect V{b_V.as<double>(), nts, nt, rect_t};
      TiledRect Wn{b_Wn.as<double>(), nt, nts, rect_t};
      TiledRect Xs{b_Xs.as<double>(), nts, nts, sqs_t};
      TiledSym Ms{b_Ms.as<double>(), nts, syms_t};
      // X = L⁻ᵀ (scratch: the handle's factor stays as it is) and V = K(x*,x) L⁻ᵀ
      CU(launch_rect_identity(st, X, nb));
      CU(trsm_right_lt_upper(ctx, st, X, Lc, Wc, wst, nb));
      CU(launch_kmat_cross(st, V, nb, P.xs.as<double>(), Ns, post->d_xpad, N, D, tsp, form));
      CU(trsm_right_lt(ctx, V, Lc, Wc, wst, nb));
      // -W = -X V' (X is upper triangular: the k range of tile row I starts at I)
      CU(cudaMemsetAsync(b_Wn.p, 0, (size_t)nb * rect_t * sizeof(double), st));
      GemmArgs gw{};
      gw.A = operand(X); gw.B = operand(V); gw.C = operand(Wn);
      gw.k0 = 0; gw.k1 = nt; gw.k_from_row = 1;
      CU(launch_gemm(st, GEMM_UPDATE, gw, nts, nt, nb));
      // -γ = (-W) β,  u = α - γ
      CU(launch_rect_gemv(st, Wn, beta, nspad, g, npad, tsp, 0, nb));
      CU(cudaMemcpyAsync(u, alpha, (size_t)nb * npad * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_axpy(st, u, g, (size_t)nb * npad, 1.0));
      // -Φ = -W L*⁻ᵀ in place
      CU(trsm_right_lt(ctx, Wn, Lsc, Wsc, wsts, nb));
      // X* = L*⁻ᵀ, -P = -X* X*'
      CU(launch_rect_identity(st, Xs, nb));
      CU(trsm_right_lt_upper(ctx, st, Xs, Lsc, Wsc, wsts, nb));
      CU(cudaMemsetAsync(b_Ms.p, 0, (size_t)nb * syms_t * sizeof(double), st));
      GemmArgs gp{};
      gp.A = operand(Xs); gp.B = operand(Xs); gp.C = operand(Ms);
      gp.k0 = 0; gp.k1 = nts; gp.sym = 1; gp.k_from_row = 1;
      CU(launch_gemm(st, GEMM_UPDATE, gp, nts, nts, nb));
      // Φ X*' into V's storage (V is consumed); the rank-1 part (α - γ)β' is added inside the contraction
      TiledRect Gc{b_V.as<double>(), nt, nts, rect_t};
      CU(cudaMemsetAsync(b_V.p, 0, (size_t)nb * rect_t * sizeof(double), st));
      GemmArgs gc{};
      gc.A = operand(Wn); gc.B = operand(Xs); gc.C = operand(Gc);
      gc.k0 = 0; gc.k1 = nts;
      CU(launch_gemm(st, GEMM_UPDATE, gc, nts, nt, nb));
      // -(ΦΦ' + αα') into X's storage, packed lower (X is consumed)
      TiledSym Mx{b_X.as<double>(), nt, syml};
      CU(cudaMemsetAsync(b_X.p, 0, (size_t)nb * syml * sizeof(double), st));
      GemmArgs gx{};
      gx.A = operand(Wn); gx.B = operand(Wn); gx.C = operand(Mx);
      gx.k0 = 0; gx.k1 = nts; gx.sym = 1;
      CU(launch_gemm(st, GEMM_UPDATE, gx, nt, nt, nb));
      CU(launch_sym_rank1(st, Mx, nb, alpha, npad, -1.0));
      ctx->launches += 9;
      // the three contractions
      const size_t go = (size_t)(lo + c0) * TERM_SLOTS;
      CU(launch_kgrad_terms(st, Ms.base, Ms.batch_stride, 0, P.xs.as<double>(), Ns, D, tsp, nb, max_terms, any_ard, beta, nspad, form,
                            b_tp.as<double>(), gt_ss + go));
      CU(launch_kgrad_terms(st, Mx.base, Mx.batch_stride, 0, post->d_xpad, N, D, trp, nb, max_terms, any_ard, u, npad, form,
                            b_tp.as<double>(), gt_x + go));
      CU(launch_kgrad_cross_terms(st, Gc, post->d_xpad, N, P.xs.as<double>(), Ns, D, trp, nb, max_terms, any_ard, u, npad, beta, nspad,
                                  form, b_tp.as<double>(), gt_c + go));
      // traces of Gx and the mean gradient
      CU(launch_sumsq(st, u, npad, (int)npad, nb, b_sq.as<double>() + c0));
      CU(launch_sumsq(st, alpha, npad, (int)npad, nb, b_sq.as<double>() + nloc + c0));
      CU(launch_sumsq(st, b_Wn.as<double>(), rect_t, (int)rect_t, nb, b_sq.as<double>() + 2 * (size_t)nloc + c0));
      CU(launch_kgrad_finish(st, nullptr, 0, nb, beta, nspad, Ns, b_sb.as<double>() + (size_t)c0 * 4));
      CU(launch_kgrad_finish(st, nullptr, 0, nb, g, npad, N, b_sg.as<double>() + (size_t)c0 * 4));
      ctx->launches += 11;
    }
  }
  // per-latent scalars: [tr(Gx) (m) | d/d mean (m)]
  std::vector<double> hv((size_t)2 * m, 0.0);
  if (nloc > 0) {
    std::vector<double> hsq((size_t)3 * nloc), hsb((size_t)4 * nloc), hsg((size_t)4 * nloc);
    CU(copy_out(ctx, hsq.data(), b_sq.p, hsq.size() * sizeof(double)));
    CU(copy_out(ctx, hsb.data(), b_sb.p, hsb.size() * sizeof(double)));
    CU(copy_out(ctx, hsg.data(), b_sg.p, hsg.size() * sizeof(double)));
    CU(cudaStreamSynchronize(st));
    for (int i = 0; i < nloc; ++i) {
      hv[(size_t)lo + i] = 0.5 * (hsq[i] - hsq[(size_t)nloc + i] - hsq[2 * (size_t)nloc + i]);
      hv[(size_t)m + lo + i] = hsb[(size_t)i * 4 + 3] + hsg[(size_t)i * 4 + 3];
    }
  }
  if ((rc = allreduce_dev(ctx, b_gt.as<double>(), ngt))) return rc;
  std::vector<double> hgt(ngt);
  CU(copy_out(ctx, hgt.data(), b_gt.p, ngt * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  if ((rc = allreduce_host(ctx, hv))) return rc;

  // d/dy (training): T' γ
  if (grad_train_y) {
    const size_t ny = (size_t)p * N;
    DevBuf b_gy;
    CU(b_gy.alloc(ctx, 2 * ny * sizeof(double)));
    CU(cudaMemsetAsync(b_gy.p, 0, 2 * ny * sizeof(double), st));
    if (nloc > 0) {
      std::vector<double> Hneg((size_t)p * m);  // backproject with "H" = -T' applied to -γ
      for (int i = 0; i < m; ++i)
        for (int j = 0; j < p; ++j) Hneg[(size_t)i * p + j] = -pr.T[(size_t)j * m + i];
      DevBuf b_Hn;
      CU(b_Hn.alloc(ctx, Hneg.size() * sizeof(double)));
      CU(copy_in(ctx, b_Hn.as<double>(), Hneg.data(), Hneg.size()));
      CU(launch_backproject(st, b_Hn.as<double>(), p, m, lo, nloc, b_g.as<double>(), b_g.as<double>(), npad, N, 0.0, 0.0, 0,
                            b_gy.as<double>(), b_gy.as<double>() + ny));
      ++ctx->launches;
      CU(cudaStreamSynchronize(st));  // Hneg goes out of scope
    }
    if ((rc = allreduce_dev(ctx, b_gy.as<double>(), ny))) return rc;
    CU(copy_out(ctx, grad_train_y, b_gy.p, ny * sizeof(double)));
    CU(cudaStreamSynchronize(st));
  }

  // U and S: bar_T[i, :] = γ_i Y' - β_i Y*' through T = S^{-1/2} U' (both sides), plus the test-side regulariser R* Z*'/σ*²
  const size_t npm = (size_t)p * m;
  std::vector<double> hGU;
  if (orth && (grad_U || grad_S)) {
    DevBuf b_GU, b_R, b_Z, b_P, b_Q, b_tys, b_zero, b_pt;
    CU(b_GU.alloc(ctx, 2 * npm * sizeof(double)));
    CU(cudaMemsetAsync(b_GU.p, 0, 2 * npm * sizeof(double), st));
    if (nloc > 0) {
      CU(launch_abt(st, d_ytr, (size_t)N, p, b_g.as<double>(), npad, nloc, N, -1.0, b_GU.as<double>() + (size_t)lo * p));
      CU(launch_abt(st, d_ys, (size_t)Ns, p, keep.beta.as<double>(), nspad, nloc, Ns, -1.0, b_GU.as<double>() + (size_t)lo * p));
      ctx->launches += 2;
    }
    if (ctx->rank == 0) {  // the regulariser is counted once
      CU(b_P.alloc(ctx, pr.P.size() * sizeof(double)));
      CU(copy_in(ctx, b_P.as<double>(), pr.P.data(), pr.P.size()));
      CU(b_Q.alloc(ctx, pr.Q.size() * sizeof(double)));
      CU(copy_in(ctx, b_Q.as<double>(), pr.Q.data(), pr.Q.size()));
      CU(b_R.alloc(ctx, (size_t)p * Ns * sizeof(double)));
      CU(b_Z.alloc(ctx, (size_t)m * Ns * sizeof(double)));
      CU(b_tys.alloc(ctx, (size_t)nl * nspad * sizeof(double)));
      CU(cudaMemsetAsync(b_tys.p, 0, (size_t)nl * nspad * sizeof(double), st));
      CU(b_zero.alloc(ctx, (size_t)nl * sizeof(double)));
      CU(cudaMemsetAsync(b_zero.p, 0, (size_t)nl * sizeof(double), st));
      const int nblk = project_max_partials(Ns);
      CU(b_pt.alloc(ctx, (size_t)nblk * sizeof(double)));
      CU(cudaMemsetAsync(b_pt.p, 0, (size_t)nblk * sizeof(double), st));
      CU(launch_project(st, d_ys, Ns, p, b_T.as<double>(), m, lo, nloc, b_zero.as<double>(), b_tys.as<double>(), nspad, b_P.as<double>(),
                        b_Q.as<double>(), b_pt.as<double>(), nullptr, b_R.as<double>(), b_Z.as<double>()));
      CU(launch_abt(st, b_R.as<double>(), (size_t)Ns, p, b_Z.as<double>(), (size_t)Ns, m, Ns, 1.0, b_GU.as<double>() + npm));
      ctx->launches += 2;
    }
    if ((rc = allreduce_dev(ctx, b_GU.as<double>(), 2 * npm))) return rc;
    hGU.resize(2 * npm);
    CU(copy_out(ctx, hGU.data(), b_GU.p, 2 * npm * sizeof(double)));
    CU(cudaStreamSynchronize(st));
  }

  // ---- host assembly
  std::vector<double> terms((size_t)m * TERM_SLOTS);
  for (size_t k = 0; k < terms.size(); ++k) terms[k] = (hgt[k] + hgt[(size_t)m * TERM_SLOTS + k]) + hgt[2 * (size_t)m * TERM_SLOTS + k];
  if (grad_terms) std::copy(terms.begin(), terms.end(), grad_terms);
  for (int i = 0; i < m; ++i) {
    const double* t0 = terms.data() + (size_t)i * TERM_SLOTS;
    if (grad_latents) {
      grad_latents[(size_t)i * 3 + 0] = t0[0];
      grad_latents[(size_t)i * 3 + 1] = t0[1];
      grad_latents[(size_t)i * 3 + 2] = hv[(size_t)m + i];
    }
    if (grad_ard)
      for (int k = 0; k < D; ++k) grad_ard[(size_t)i * D + k] = (post->descs[i].ard && k < MAX_ARD) ? t0[3 + k] : 0.0;
  }
  if (grad_train_sigma2) {
    double s = 0.0;
    for (int i = 0; i < m; ++i) s += hv[i] * (orth ? 1.0 / post->S[i] : 1.0);  // ν_i = σ²/S_i (OILMM) or σ²
    *grad_train_sigma2 = s;
  }
  if (orth && grad_S)
    for (int i = 0; i < m; ++i) {
      const double Si = post->S[i];
      double bt_u = 0.0;  // Σ_j bar_T[i, j] U[j, i]
      for (int j = 0; j < p; ++j) bt_u += hGU[(size_t)i * p + j] * post->U[(size_t)i * p + j];
      const double tr_ss = 0.5 * (keep.hg[i] - keep.hg[(size_t)m + i]);
      grad_S[i] = -bt_u / (2.0 * Si * std::sqrt(Si)) - hv[i] * s2t / (Si * Si) - tr_ss * sigma2 / (Si * Si) - (double)Ns / (2.0 * Si);
    }
  if (orth && grad_U)
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < p; ++j)
        grad_U[(size_t)i * p + j] = hGU[(size_t)i * p + j] / std::sqrt(post->S[i]) + hGU[npm + (size_t)i * p + j] / sigma2;
  return LMM_OK;
}
