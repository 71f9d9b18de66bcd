// rrule of logpdf (OILMM, IndependentMOGP, general ILMM), sequential conditioning of per-latent posteriors, prior
// cross-covariance of an IndependentMOGP.
#include <algorithm>

#include "host_internal.h"

// ------------------------------------------------------------------------------------------------
// Sequential conditioning: posterior(post(x2, σ²), y2) on an OILMM / IndependentMOGP posterior
// (src/oilmm.jl:116-134 / src/independent_mogp.jl:119-126 applied to PosteriorGP latents).  Each latent's prior is
// conditioned on the union [x; x2] with per-point noise [Σ1_i .. ; Σ2_i ..] -- the exact-GP identity "posterior of a
// posterior = prior conditioned on the union" -- and, as AbstractGPs does, the existing factor is EXTENDED by a block
// Cholesky update (O(N² N₂)) instead of re-factorising the union (O((N + N₂)³); option "condition_update" = 0).
// ------------------------------------------------------------------------------------------------

extern "C" int lmm_post_condition(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, lmm_post** out_post,
                                  int* info_latent) {
  if (!post || !xs || Ns <= 0 || !ys || !out_post) return LMM_E_ARG;
  *out_post = nullptr;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (post->kind == POST_VFE) return ctx->fail(LMM_E_UNSUPPORTED, VFE_POST_ONLY);
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  if (post->kind == POST_MASKED) return ctx->fail(LMM_E_UNSUPPORTED, "a missing-data posterior offers mean_and_var only");
  if (post->joint()) return ilmm_post_condition(post, xs, Ns, sigma2, ys, out_post, info_latent);
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p, D = post->D, N1 = post->N, N2 = N1 + Ns, lo = post->lo, nloc = post->nloc();
  const int nt2 = ntiles(N2);
  const size_t npad1 = post->npad(), npad2 = (size_t)nt2 * TILE;
  Projection pr;
  std::vector<double> H;
  int rc;
  if (post->kind == POST_OILMM) {
    if ((rc = oilmm_projection(ctx, post->U.data(), post->S.data(), p, m, sigma2, Ns, pr, H))) return rc;
  } else {
    if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
    pr.T.assign((size_t)m * m, 0.0);
    for (int i = 0; i < m; ++i) pr.T[(size_t)i * m + i] = 1.0;
    pr.noise.assign(m, sigma2);
  }
  const int nl = nloc > 0 ? nloc : 1;
  DevBuf b_x, b_y, b_T, b_means, b_delta, b_part, b_noise_new, b_nv, b_L, b_W, b_alpha, b_r, b_z, b_logdet, b_info, b_params, b_H;
  // x' = [x; xs]
  CU(b_x.alloc(ctx, npad2 * D * sizeof(double)));
  CU(cudaMemsetAsync(b_x.p, 0, npad2 * D * sizeof(double), st));
  CU(cudaMemcpyAsync(b_x.p, post->d_xpad, (size_t)N1 * D * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(copy_in(ctx, b_x.as<double>() + (size_t)N1 * D, xs, (size_t)Ns * D));
  // δ' = [δ; T y2 - mean]
  const double* d_y = ys;
  if (!is_device_ptr(ys)) {
    CU(b_y.alloc(ctx, (size_t)p * Ns * sizeof(double)));
    CU(copy_in(ctx, b_y.as<double>(), ys, (size_t)p * Ns));
    d_y = b_y.as<double>();
  }
  CU(b_T.alloc(ctx, pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, b_T.as<double>(), pr.T.data(), pr.T.size()));
  std::vector<double> hmeans(nl, 0.0), hnoise(nl, 0.0);
  for (int i = lo; i < post->hi; ++i) {
    hmeans[i - lo] = post->descs[i].mean_const;
    hnoise[i - lo] = pr.noise[i];
  }
  CU(b_means.alloc(ctx, (size_t)nl * sizeof(double)));
  CU(copy_in(ctx, b_means.as<double>(), hmeans.data(), (size_t)nl));
  CU(b_noise_new.alloc(ctx, (size_t)nl * sizeof(double)));
  CU(copy_in(ctx, b_noise_new.as<double>(), hnoise.data(), (size_t)nl));
  CU(b_delta.alloc(ctx, (size_t)nl * npad2 * sizeof(double)));
  CU(cudaMemsetAsync(b_delta.p, 0, (size_t)nl * npad2 * sizeof(double), st));
  CU(b_part.alloc(ctx, (size_t)project_max_partials(Ns) * sizeof(double)));
  if (nloc > 0) {
    CU(cudaMemcpy2DAsync(b_delta.p, npad2 * sizeof(double), post->d_delta, npad1 * sizeof(double), (size_t)N1 * sizeof(double),
                         (size_t)nloc, cudaMemcpyDeviceToDevice, st));
    CU(launch_project(st, d_y, Ns, p, b_T.as<double>(), m, lo, nloc, b_means.as<double>(), b_delta.as<double>() + N1, npad2, nullptr,
                      nullptr, b_part.as<double>(), nullptr));
    ++ctx->launches;
  }
  // per-point noise
  CU(b_nv.alloc(ctx, (size_t)nl * npad2 * sizeof(double)));
  CU(cudaMemsetAsync(b_nv.p, 0, (size_t)nl * npad2 * sizeof(double), st));
  if (nloc > 0) {
    CU(launch_fill_noise(st, nloc, b_nv.as<double>(), npad2, N1, Ns, post->d_noise_vec, npad1, post->d_params, b_noise_new.as<double>()));
    ++ctx->launches;
  }
  std::vector<int> hinfo(nl, 0);
  CU(b_params.alloc(ctx, (size_t)(nl + 1) * sizeof(LatentParams)));
  if (nloc > 0) {
    CU(cudaMemcpyAsync(b_params.p, post->d_params, (size_t)nloc * sizeof(LatentParams), cudaMemcpyDeviceToDevice, st));
    CU(b_L.alloc(ctx, (size_t)nloc * sym_tiles(nt2) * TT * sizeof(double)));
    CU(b_W.alloc(ctx, (size_t)nloc * nt2 * TT * sizeof(double)));
    CU(b_alpha.alloc(ctx, (size_t)nloc * npad2 * sizeof(double)));
    CU(b_r.alloc(ctx, (size_t)nloc * npad2 * sizeof(double)));
    CU(b_z.alloc(ctx, (size_t)nloc * npad2 * sizeof(double)));
    CU(b_logdet.alloc(ctx, (size_t)nloc * sizeof(double)));
    CU(b_info.alloc(ctx, (size_t)nloc * sizeof(int)));
    CU(cudaMemsetAsync(b_logdet.p, 0, (size_t)nloc * sizeof(double), st));
    CU(cudaMemsetAsync(b_info.p, 0, (size_t)nloc * sizeof(int), st));
    TiledSym L{b_L.as<double>(), nt2, sym_tiles(nt2) * TT};
    const size_t wstride = (size_t)nt2 * TT;
    // Block-Cholesky update (what AbstractGPs does when a FiniteGP{<:PosteriorGP} is conditioned again, SURVEY App. A.2;
    // exercised at test/oilmm.jl:20-26): the tile rows of the old factor that lie entirely above the new points are final
    // -- L = [L11 0; L21 L22], L21 = K21 L11^{-T}, L22 = chol(K22 + Σ2 - L21 L21') -- so they are copied, and only the tile
    // rows from jstart = floor(N1 / 128) on are built and factored (the last, partly filled old tile row is recomputed
    // together with the new rows: its old rows come out bit-identical, a row of a TRSM / update depends on that row only).
    const int jstart = ctx->condition_update ? N1 / TILE : 0;
    if (jstart > 0) {
      const size_t pre_l = sym_tiles(jstart) * TT, pre_w = (size_t)jstart * TT;
      const size_t ls1 = sym_tiles(post->nt) * TT, ws1 = (size_t)post->nt * TT, ls2 = sym_tiles(nt2) * TT;
      for (int i = 0; i < nloc; ++i) {
        CU(cudaMemcpyAsync(b_L.as<double>() + (size_t)i * ls2, post->d_L + (size_t)i * ls1, pre_l * sizeof(double), cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(b_W.as<double>() + (size_t)i * wstride, post->d_W + (size_t)i * ws1, pre_w * sizeof(double), cudaMemcpyDeviceToDevice, st));
      }
    }
    CU(launch_kmat_sym(st, L, nloc, b_x.as<double>(), N2, D, b_params.as<LatentParams>(), ctx->distance_form, b_nv.as<double>(), npad2, jstart));
    ++ctx->launches;
    CU(chol_factor(ctx, L, b_W.as<double>(), wstride, nloc, b_logdet.as<double>(), b_info.as<int>(), jstart));
    CU(cudaMemcpyAsync(b_r.p, b_delta.p, (size_t)nloc * npad2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CU(launch_fwd_solve(st, L, b_W.as<double>(), wstride, b_r.as<double>(), b_z.as<double>(), npad2, nloc, &ctx->launches));
    CU(cudaMemcpyAsync(b_r.p, b_z.p, (size_t)nloc * npad2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CU(launch_bwd_solve(st, L, b_W.as<double>(), wstride, b_r.as<double>(), b_alpha.as<double>(), npad2, nloc, &ctx->launches));
    CU(copy_out(ctx, hinfo.data(), b_info.p, (size_t)nloc * sizeof(int)));
  }
  CU(b_H.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(cudaMemcpyAsync(b_H.p, post->d_H, (size_t)p * m * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(cudaStreamSynchronize(st));
  {
    std::vector<int> hi(hinfo.begin(), hinfo.begin() + nloc);
    if ((rc = report_info(ctx, hi, lo, N2, info_latent))) return rc;  // collective: also the ranks without latents
  }
  lmm_post* P = new lmm_post();
  P->ctx = ctx; P->kind = post->kind; P->m = m; P->p = p; P->N = N2; P->D = D; P->nt = nt2; P->lo = lo; P->hi = post->hi;
  P->adopt_descs(post->descs.data(), m, D); P->noise = post->noise; P->H = post->H; P->U = post->U; P->S = post->S; P->sigma2 = sigma2;
  P->bytes = (size_t)nloc * (factor_bytes_per_latent(nt2) + 3 * npad2 * sizeof(double)) + npad2 * D * sizeof(double);
  P->d_xpad = (double*)b_x.detach();
  P->d_L = (double*)b_L.detach();
  P->d_W = (double*)b_W.detach();
  P->d_alpha = (double*)b_alpha.detach();
  P->d_delta = (double*)b_delta.detach();
  P->d_params = (LatentParams*)b_params.detach();
  P->d_H = (double*)b_H.detach();
  P->d_noise_vec = (double*)b_nv.detach();
  *out_post = P;
  return LMM_OK;
}
// ------------------------------------------------------------------------------------------------
// rrule of logpdf (SURVEY.md §8f-1): value + gradients w.r.t. the per-latent hyper-parameters
// (variance, inv_lengthscale, mean_const), the observation noise σ² and the observations y.
//   G_i = d lml_i / dC_i = (α_i α_i' - C_i^{-1}) / 2,   C_i^{-1} = L^{-T} L^{-1}  (batched potri)
// potri on the tensor pipe: X = L^{-T} by the triangular-aware TRSM sweep on an identity
// (N³/3 flop), then -C^{-1} = -X X' by a triangular-aware SYRK into the factor's own tiles
// (N³/3 flop): the gradient costs about 3x the logpdf.
// ------------------------------------------------------------------------------------------------
namespace lmm_host {

// Launch bounds of the per-term contraction for latents [lo, hi): the most terms, and whether any term has an ARDTransform.
void terms_shape(const lmm_gp_desc* latents, int lo, int hi, int& max_terms, bool& any_ard) {
  max_terms = 1;
  any_ard = false;
  for (int i = lo; i < hi; ++i) {
    max_terms = std::max(max_terms, 1 + latents[i].n_extra);
    any_ard |= latents[i].ard != nullptr;
    for (int t = 0; t < latents[i].n_extra; ++t) any_ard |= latents[i].extra[t].ard != nullptr;
  }
}

// grad_terms -> outputs: the whole per-term block, and term 0's values in place of the single-kernel contraction's
// grad_latents[:, 0:2] / grad_ard rows for composite latents (single-kernel latents keep kgrad / kgrad_ard's values).
void scatter_terms(const lmm_gp_desc* latents, int m, int D, const std::vector<double>& ht, double* grad_terms, double* grad_latents,
                   double* grad_ard) {
  std::copy(ht.begin(), ht.end(), grad_terms);
  for (int i = 0; i < m; ++i) {
    if (!desc_is_composite(latents[i])) continue;
    const double* g = ht.data() + (size_t)i * TERM_SLOTS;
    if (grad_latents) {
      grad_latents[(size_t)i * 3 + 0] = g[0];
      grad_latents[(size_t)i * 3 + 1] = g[1];
    }
    if (grad_ard)
      for (int k = 0; k < D && k < MAX_ARD; ++k) grad_ard[(size_t)i * D + k] = latents[i].ard ? g[3 + k] : 0.0;
  }
}

int grad_run_setup(lmm_ctx* ctx, bool orth, const lmm_gp_desc* latents, int m, const double* x, int N, int D, int p, const double* y,
                   const Projection& pr, const GradOut& out, GradRun& s) {
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  shard_range(ctx, m, s.lo, s.hi);
  const int lo = s.lo, hi = s.hi;
  s.mloc = hi - lo;
  s.nt = ntiles(N);
  s.npad = (size_t)s.nt * TILE;
  s.multi = ctx->comm && ctx->nranks > 1;
  const int mloc = s.mloc;
  const size_t npad = s.npad;
  CU(cudaEventRecord(ctx->ev[0], st));
  int rc = stage_xpad(ctx, s.b_x, x, N, D);
  if (rc) return rc;
  s.d_y = y;
  if (!is_device_ptr(y)) {
    CU(s.b_y.alloc(ctx, (size_t)p * N * sizeof(double)));
    CU(copy_in(ctx, s.b_y.as<double>(), y, (size_t)p * N));
    s.d_y = s.b_y.as<double>();
  }
  CU(s.b_T.alloc(ctx, pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, s.b_T.as<double>(), pr.T.data(), pr.T.size()));
  if (pr.has_reg) {
    CU(s.b_P.alloc(ctx, pr.P.size() * sizeof(double)));
    CU(copy_in(ctx, s.b_P.as<double>(), pr.P.data(), pr.P.size()));
    CU(s.b_Q.alloc(ctx, pr.Q.size() * sizeof(double)));
    CU(copy_in(ctx, s.b_Q.as<double>(), pr.Q.data(), pr.Q.size()));
  }
  s.nl = mloc > 0 ? mloc : 1;
  const int nl = s.nl;
  std::vector<double> hmeans(nl, 0.0);
  for (int i = lo; i < hi; ++i) hmeans[i - lo] = latents[i].mean_const;
  CU(s.b_means.alloc(ctx, (size_t)nl * sizeof(double)));
  CU(copy_in(ctx, s.b_means.as<double>(), hmeans.data(), (size_t)nl));
  if ((rc = upload_params(ctx, s.b_params, latents, pr.noise.data(), lo, hi, D))) return rc;
  CU(s.b_ty.alloc(ctx, (size_t)nl * npad * sizeof(double)));
  CU(cudaMemsetAsync(s.b_ty.p, 0, (size_t)nl * npad * sizeof(double), st));
  const int nblk = project_max_partials(N);
  CU(s.b_part.alloc(ctx, (size_t)nblk * sizeof(double)));
  CU(cudaMemsetAsync(s.b_part.p, 0, (size_t)nblk * sizeof(double), st));
  CU(s.b_resid.alloc(ctx, sizeof(double)));
  CU(cudaMemsetAsync(s.b_resid.p, 0, sizeof(double), st));
  s.do_reg = pr.has_reg && ctx->rank == 0;
  s.want_U = orth && out.grad_U;
  s.want_R = s.do_reg && (out.grad_y || s.want_U);
  s.want_Z = s.do_reg && s.want_U;
  if (s.want_R) CU(s.b_R.alloc(ctx, (size_t)p * N * sizeof(double)));
  if (s.want_Z) CU(s.b_Z.alloc(ctx, (size_t)m * N * sizeof(double)));
  CU(launch_project(st, s.d_y, N, p, s.b_T.as<double>(), m, lo, mloc, s.b_means.as<double>(), s.b_ty.as<double>(), npad,
                    s.do_reg ? s.b_P.as<double>() : nullptr, s.do_reg ? s.b_Q.as<double>() : nullptr, s.b_part.as<double>(), nullptr,
                    s.want_R ? s.b_R.as<double>() : nullptr, s.want_Z ? s.b_Z.as<double>() : nullptr));
  ++ctx->launches;
  if (s.do_reg) {
    CU(launch_sum_partials(st, s.b_part.as<double>(), nblk, s.b_resid.as<double>()));
    ++ctx->launches;
  }
  // reduction vector: [lml (m) | gv (m) | gs (m) | gmean (m) | gnoise (m) | resid (1) | quad (m)]
  s.nvec = (size_t)6 * m + 1;
  CU(s.b_vec.alloc(ctx, s.nvec * sizeof(double)));
  CU(cudaMemsetAsync(s.b_vec.p, 0, s.nvec * sizeof(double), st));
  double* d_vec = s.b_vec.as<double>();
  if (s.do_reg) CU(cudaMemcpyAsync(d_vec + 5 * m, s.b_resid.p, sizeof(double), cudaMemcpyDeviceToDevice, st));
  s.want_ard = false;
  if (out.grad_ard) {
    for (int i = 0; i < m; ++i) s.want_ard |= latents[i].ard != nullptr;
    for (size_t i = 0; i < (size_t)m * D; ++i) out.grad_ard[i] = 0.0;
  }
  if (s.want_ard) {
    CU(s.b_gard.alloc(ctx, (size_t)m * MAX_ARD * sizeof(double)));
    CU(cudaMemsetAsync(s.b_gard.p, 0, (size_t)m * MAX_ARD * sizeof(double), st));
  }
  s.max_terms = 1;
  s.terms_ard = false;
  if (out.grad_terms) {
    terms_shape(latents, lo, hi, s.max_terms, s.terms_ard);
    CU(s.b_gterms.alloc(ctx, (size_t)m * TERM_SLOTS * sizeof(double)));
    CU(cudaMemsetAsync(s.b_gterms.p, 0, (size_t)m * TERM_SLOTS * sizeof(double), st));
  }
  return LMM_OK;
}

int grad_run_finish(lmm_ctx* ctx, bool orth, const lmm_gp_desc* latents, int m, int N, int D, int p, double sigma2, const Projection& pr,
                    const double* Shost, GradOut out, GradRun& s, const double* d_a, const std::vector<int>& hinfo,
                    const std::vector<double>& hg4, const std::vector<double>& hquad) {
  cudaStream_t st = ctx->stream;
  const int lo = s.lo, mloc = s.mloc;
  const size_t npad = s.npad, nvec = s.nvec;
  const bool multi = s.multi, want_ard = s.want_ard, want_U = s.want_U, want_R = s.want_R, want_Z = s.want_Z;
  double* d_vec = s.b_vec.as<double>();
  int rc;
  DevBuf b_gy;
  if (mloc > 0) {
    // scatter the local gradients into the reduction vector
    std::vector<double> hv(nvec, 0.0);
    for (int i = 0; i < mloc; ++i) hv[(size_t)5 * m + 1 + lo + i] = hquad[i];
    for (int i = 0; i < mloc; ++i) {
      hv[(size_t)m + lo + i] = hg4[(size_t)i * 4 + 0];
      hv[(size_t)2 * m + lo + i] = hg4[(size_t)i * 4 + 1];
      hv[(size_t)3 * m + lo + i] = hg4[(size_t)i * 4 + 3];
      hv[(size_t)4 * m + lo + i] = hg4[(size_t)i * 4 + 2];
    }
    DevBuf b_hv;
    CU(b_hv.alloc(ctx, nvec * sizeof(double)));
    CU(copy_in(ctx, b_hv.as<double>(), hv.data(), nvec));
    CU(launch_axpy(st, d_vec, b_hv.as<double>(), nvec, 1.0));
    CU(cudaStreamSynchronize(st));
  }
  std::vector<double> hgard;
  if (want_ard) {
    if (multi) {
      int r = nccl_api().AllReduce(s.b_gard.p, s.b_gard.p, (size_t)m * MAX_ARD, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
      if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
    }
    hgard.resize((size_t)m * MAX_ARD);
    CU(copy_out(ctx, hgard.data(), s.b_gard.p, hgard.size() * sizeof(double)));
    CU(cudaStreamSynchronize(st));
    for (int i = 0; i < m; ++i)
      for (int k = 0; k < D && k < MAX_ARD; ++k) out.grad_ard[(size_t)i * D + k] = latents[i].ard ? hgard[(size_t)i * MAX_ARD + k] : 0.0;
  }
  std::vector<double> hterms;
  if (out.grad_terms) {
    if (multi) {
      int r = nccl_api().AllReduce(s.b_gterms.p, s.b_gterms.p, (size_t)m * TERM_SLOTS, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
      if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
    }
    hterms.resize((size_t)m * TERM_SLOTS);
    CU(copy_out(ctx, hterms.data(), s.b_gterms.p, hterms.size() * sizeof(double)));
    CU(cudaStreamSynchronize(st));
  }
  // d/dy: -sum_i T[i,:]' a_i  (- R/σ² from the regulariser on rank 0)
  if (out.grad_y) {
    const size_t ny = (size_t)p * N;
    CU(b_gy.alloc(ctx, 2 * ny * sizeof(double)));
    CU(cudaMemsetAsync(b_gy.p, 0, 2 * ny * sizeof(double), st));
    if (mloc > 0) {
      // backproject with "H" = -T' (p x m column-major): Hneg[j + i*p] = -T[i + j*m]
      std::vector<double> Hneg((size_t)p * m);
      for (int i = 0; i < m; ++i)
        for (int j = 0; j < p; ++j) Hneg[(size_t)i * p + j] = -pr.T[(size_t)j * m + i];
      DevBuf b_Hn;
      CU(b_Hn.alloc(ctx, Hneg.size() * sizeof(double)));
      CU(copy_in(ctx, b_Hn.as<double>(), Hneg.data(), Hneg.size()));
      CU(launch_backproject(st, b_Hn.as<double>(), p, m, lo, mloc, d_a, d_a, npad, N, 0.0, 0.0, 0,
                            b_gy.as<double>(), b_gy.as<double>() + ny));
      ++ctx->launches;
      CU(cudaStreamSynchronize(st));
    }
    if (want_R) {
      CU(launch_axpy(st, b_gy.as<double>(), s.b_R.as<double>(), ny, -1.0 / sigma2));
      ++ctx->launches;
    }
    if (multi) {
      int r = nccl_api().AllReduce(b_gy.p, b_gy.p, ny, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
      if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
    }
    CU(copy_out(ctx, out.grad_y, b_gy.p, ny * sizeof(double)));
  }
  // d/dU: -(Y a_i)/sqrt(S_i) per column (latent) + R Z'/σ² from the regulariser (rank 0)
  std::vector<double> hGU;
  if (want_U) {
    DevBuf b_GU;
    const size_t npm = (size_t)p * m;
    CU(b_GU.alloc(ctx, 2 * npm * sizeof(double)));
    CU(cudaMemsetAsync(b_GU.p, 0, 2 * npm * sizeof(double), st));
    if (mloc > 0) {
      CU(launch_abt(st, s.d_y, (size_t)N, p, d_a, npad, mloc, N, 1.0, b_GU.as<double>() + (size_t)lo * p));
      ++ctx->launches;
    }
    if (want_Z) {
      CU(launch_abt(st, s.b_R.as<double>(), (size_t)N, p, s.b_Z.as<double>(), (size_t)N, m, N, 1.0, b_GU.as<double>() + npm));
      ++ctx->launches;
    }
    if (multi) {
      int r = nccl_api().AllReduce(b_GU.p, b_GU.p, 2 * npm, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
      if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
    }
    hGU.resize(2 * npm);
    CU(copy_out(ctx, hGU.data(), b_GU.p, 2 * npm * sizeof(double)));
    CU(cudaStreamSynchronize(st));
  }
  if (multi) {
    int r = nccl_api().AllReduce(d_vec, d_vec, nvec, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
    if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
  }
  std::vector<double> hv(nvec, 0.0);
  CU(copy_out(ctx, hv.data(), d_vec, nvec * sizeof(double)));
  CU(cudaEventRecord(ctx->ev[1], st));
  CU(cudaStreamSynchronize(st));
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
  ctx->timings[0] = ms;
  {
    std::vector<int> hi2(hinfo.begin(), hinfo.begin() + mloc);
    if ((rc = report_info(ctx, hi2, lo, N, out.info_latent))) return rc;  // collective: also the ranks without latents
  }
  const double resid = hv[(size_t)5 * m];
  double reg = 0.0, dreg = 0.0;
  if (pr.has_reg) {
    reg = -(pr.reg_c0 + resid / sigma2) / 2.0;
    // d/dσ² of -(n (p-m) log(2πσ²) + R/σ²)/2
    dreg = -((double)N * (double)(p - m) / sigma2 - resid / (sigma2 * sigma2)) / 2.0;
  }
  if (out.logpdf) {
    double sum = 0.0;
    for (int i = 0; i < m; ++i) sum += hv[i];
    *out.logpdf = sum + reg;
  }
  if (out.grad_latents)
    for (int i = 0; i < m; ++i) {
      out.grad_latents[(size_t)i * 3 + 0] = hv[(size_t)m + i];
      out.grad_latents[(size_t)i * 3 + 1] = hv[(size_t)2 * m + i];
      out.grad_latents[(size_t)i * 3 + 2] = hv[(size_t)3 * m + i];
    }
  if (out.grad_terms) scatter_terms(latents, m, D, hterms, out.grad_terms, out.grad_latents, out.grad_ard);
  if (out.grad_sigma2) {
    double sum = dreg;
    for (int i = 0; i < m; ++i) sum += hv[(size_t)4 * m + i] * (orth ? 1.0 / Shost[i] : 1.0);  // ν_i = σ²/S_i (OILMM) or σ²
    *out.grad_sigma2 = sum;
  }
  if (orth && out.grad_S)
    for (int i = 0; i < m; ++i) {
      // δ_i = U_i'Y/sqrt(S_i) - m_i, ν_i = σ²/S_i, reg ∋ -n log(S_i)/2
      const double a_dot_ty = hv[(size_t)5 * m + 1 + i] + latents[i].mean_const * hv[(size_t)3 * m + i];
      out.grad_S[i] = a_dot_ty / (2.0 * Shost[i]) - hv[(size_t)4 * m + i] * sigma2 / (Shost[i] * Shost[i]) - (double)N / (2.0 * Shost[i]);
    }
  if (want_U) {
    const size_t npm = (size_t)p * m;
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < p; ++j)
        out.grad_U[(size_t)i * p + j] = -hGU[(size_t)i * p + j] / std::sqrt(Shost[i]) + hGU[npm + (size_t)i * p + j] / sigma2;
  }
  return LMM_OK;
}

int latents_grad_run(lmm_ctx* ctx, bool orth, const lmm_gp_desc* latents, int m, const double* x, int N, int D, int p, double sigma2,
                     const double* y, const Projection& pr, const double* Shost, GradOut out) {
  GradRun s;
  int rc = grad_run_setup(ctx, orth, latents, m, x, N, D, p, y, pr, out, s);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  const int lo = s.lo, mloc = s.mloc, nt = s.nt, nl = s.nl, max_terms = s.max_terms;
  const bool want_ard = s.want_ard, terms_ard = s.terms_ard;
  const size_t npad = s.npad;
  double* d_vec = s.b_vec.as<double>();
  DevBuf b_L, b_W, b_X, b_alpha, b_r, b_z, b_logdet, b_quad, b_info, b_gpart, b_g4, b_apart, b_tpart;
  std::vector<int> hinfo(nl, 0);
  std::vector<double> hg4((size_t)nl * 4, 0.0), hquad(nl, 0.0);
  if (mloc > 0) {
    const size_t per_lat = factor_bytes_per_latent(nt) + (size_t)nt * nt * TT * sizeof(double) + 6 * npad * sizeof(double);
    int chunk = 0;
    CU(mem_fit(ctx, per_lat, mloc, &chunk));
    const int ntl = (int)sym_tiles(nt);
    CU(b_L.alloc(ctx, (size_t)chunk * sym_tiles(nt) * TT * sizeof(double)));
    CU(b_W.alloc(ctx, (size_t)chunk * nt * TT * sizeof(double)));
    CU(b_X.alloc(ctx, (size_t)chunk * nt * nt * TT * sizeof(double)));
    CU(b_alpha.alloc(ctx, (size_t)mloc * npad * sizeof(double)));
    CU(b_r.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    CU(b_z.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    CU(b_logdet.alloc(ctx, (size_t)mloc * sizeof(double)));
    CU(b_quad.alloc(ctx, (size_t)mloc * sizeof(double)));
    CU(b_info.alloc(ctx, (size_t)mloc * sizeof(int)));
    CU(b_gpart.alloc(ctx, (size_t)chunk * ntl * 3 * sizeof(double)));
    CU(b_g4.alloc(ctx, (size_t)mloc * 4 * sizeof(double)));
    if (want_ard) CU(b_apart.alloc(ctx, (size_t)chunk * ntl * MAX_ARD * sizeof(double)));
    if (out.grad_terms) CU(b_tpart.alloc(ctx, (size_t)chunk * ntl * TERM_SLOTS * sizeof(double)));
    CU(cudaMemsetAsync(b_logdet.p, 0, (size_t)mloc * sizeof(double), st));
    CU(cudaMemsetAsync(b_info.p, 0, (size_t)mloc * sizeof(int), st));
    for (int c0 = 0; c0 < mloc; c0 += chunk) {
      const int nb = (c0 + chunk <= mloc) ? chunk : mloc - c0;
      TiledSym L{b_L.as<double>(), nt, sym_tiles(nt) * TT};
      TiledRect X{b_X.as<double>(), nt, nt, (size_t)nt * nt * TT};
      double* W = b_W.as<double>();
      const size_t wstride = (size_t)nt * TT;
      const LatentParams* dp = s.b_params.as<LatentParams>() + c0;
      double* delta = s.b_ty.as<double>() + (size_t)c0 * npad;
      double* alpha = b_alpha.as<double>() + (size_t)c0 * npad;
      CU(launch_kmat_sym(st, L, nb, s.b_x.as<double>(), N, D, dp, ctx->distance_form));
      CU(chol_factor(ctx, L, W, wstride, nb, b_logdet.as<double>() + c0, b_info.as<int>() + c0));
      CU(cudaMemcpyAsync(b_r.p, delta, (size_t)nb * npad * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_fwd_solve(st, L, W, wstride, b_r.as<double>(), b_z.as<double>(), npad, nb, &ctx->launches));
      CU(launch_sumsq(st, b_z.as<double>(), npad, (int)npad, nb, b_quad.as<double>() + c0));
      CU(cudaMemcpyAsync(b_r.p, b_z.p, (size_t)nb * npad * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_bwd_solve(st, L, W, wstride, b_r.as<double>(), alpha, npad, nb, &ctx->launches));
      CU(launch_lml_terms(st, d_vec, lo + c0, nb, b_logdet.as<double>() + c0, b_quad.as<double>() + c0, N, LOG2PI));
      // potri: X = L^{-T}, then -C^{-1} = -X X' into the (no longer needed) factor tiles
      CU(launch_rect_identity(st, X, nb));
      CU(trsm_right_lt_upper(ctx, st, X, L, W, wstride, nb));
      CU(cudaMemsetAsync(b_L.p, 0, (size_t)nb * sym_tiles(nt) * TT * sizeof(double), st));
      GemmArgs g{};
      g.A = operand(X); g.B = operand(X); g.C = operand(L);
      g.i0 = 0; g.j0 = 0; g.k0 = 0; g.k1 = nt; g.sym = 1; g.k_from_row = 1;
      CU(launch_gemm(st, GEMM_UPDATE, g, nt, nt, nb));
      CU(launch_kgrad(st, L, nb, s.b_x.as<double>(), N, D, dp, alpha, npad, ctx->distance_form, b_gpart.as<double>()));
      CU(launch_kgrad_finish(st, b_gpart.as<double>(), ntl, nb, alpha, npad, N, b_g4.as<double>() + (size_t)c0 * 4));
      ctx->launches += 8;
      if (want_ard) {
        CU(launch_kgrad_ard(st, L.base, L.batch_stride, 0, s.b_x.as<double>(), N, D, dp, nb, alpha, npad, ctx->distance_form,
                            b_apart.as<double>(), s.b_gard.as<double>() + (size_t)(lo + c0) * MAX_ARD));
        ctx->launches += 2;
      }
      if (out.grad_terms) {
        CU(launch_kgrad_terms(st, L.base, L.batch_stride, 0, s.b_x.as<double>(), N, D, dp, nb, max_terms, terms_ard, alpha, npad,
                              ctx->distance_form, b_tpart.as<double>(), s.b_gterms.as<double>() + (size_t)(lo + c0) * TERM_SLOTS));
        ctx->launches += 2;
      }
    }
    CU(copy_out(ctx, hinfo.data(), b_info.p, (size_t)mloc * sizeof(int)));
    CU(copy_out(ctx, hg4.data(), b_g4.p, (size_t)mloc * 4 * sizeof(double)));
    CU(copy_out(ctx, hquad.data(), b_quad.p, (size_t)mloc * sizeof(double)));
    CU(cudaStreamSynchronize(st));
  }
  return grad_run_finish(ctx, orth, latents, m, N, D, p, sigma2, pr, Shost, out, s, b_alpha.as<double>(), hinfo, hg4, hquad);
}

}  // namespace lmm_host

namespace lmm_host {
// The single-kernel entry points (grad_terms == NULL) reject composite / periodic latents: their grad_latents has no
// place for the further terms' hyper-parameters.  The _terms entry points accept every latent the value path accepts.
int reject_composite(lmm_ctx* ctx, const lmm_gp_desc* latents, int m) {
  for (int i = 0; i < m; ++i)
    if (desc_is_composite(latents[i]))
      return ctx->fail(LMM_E_UNSUPPORTED, "the logpdf gradient is built for single (Sq)Euclidean base kernels; composite / periodic latents: value only");
  return LMM_OK;
}

int oilmm_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U, const double* S, int p,
                      double sigma2, const double* y, int out_dim, double* out_logpdf, double* grad_latents, double* grad_ard,
                      double* grad_sigma2, double* grad_y, double* grad_U, double* grad_S, double* grad_terms, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!grad_terms && (rc = reject_composite(ctx, latents, m))) return rc;
  if (!U || !S || !y) return ctx->fail(LMM_E_ARG, "null pointer");
  if (m > p) return ctx->fail(LMM_E_ARG, "more latents than outputs");
  Projection pr;
  std::vector<double> H;
  if ((rc = oilmm_projection(ctx, U, S, p, m, sigma2, N, pr, H))) return rc;
  GradOut out{out_logpdf, grad_latents, grad_sigma2, grad_y, info_latent};
  out.grad_U = grad_U;
  out.grad_S = grad_S;
  out.grad_ard = grad_ard;
  out.grad_terms = grad_terms;
  return latents_grad_run(ctx, true, latents, m, x, N, D, p, sigma2, y, pr, S, out);
}

int imogp_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, double sigma2, const double* y, int out_dim,
                      double* out_logpdf, double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_terms,
                      int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, fs, m, x, N, D, m, out_dim);
  if (rc) return rc;
  if (!grad_terms && (rc = reject_composite(ctx, fs, m))) return rc;
  if (!y) return ctx->fail(LMM_E_ARG, "null pointer");
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  Projection pr;
  pr.T.assign((size_t)m * m, 0.0);
  for (int i = 0; i < m; ++i) pr.T[(size_t)i * m + i] = 1.0;
  pr.noise.assign(m, sigma2);
  pr.has_reg = false;
  GradOut out{out_logpdf, grad_latents, grad_sigma2, grad_y, info_latent};
  out.grad_ard = grad_ard;
  out.grad_terms = grad_terms;
  return latents_grad_run(ctx, false, fs, m, x, N, D, m, sigma2, y, pr, nullptr, out);
}
}  // namespace lmm_host

extern "C" int lmm_oilmm_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U,
                                     const double* S, int p, double sigma2, const double* y, int out_dim, double* out_logpdf,
                                     double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_U,
                                     double* grad_S, int* info_latent) {
  return oilmm_logpdf_grad(ctx, latents, m, x, N, D, U, S, p, sigma2, y, out_dim, out_logpdf, grad_latents, grad_ard, grad_sigma2, grad_y,
                           grad_U, grad_S, nullptr, info_latent);
}
extern "C" int lmm_oilmm_logpdf_grad_terms(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U,
                                           const double* S, int p, double sigma2, const double* y, int out_dim, double* out_logpdf,
                                           double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_U,
                                           double* grad_S, double* grad_terms, int* info_latent) {
  if (ctx && !grad_terms) return ctx->fail(LMM_E_ARG, "null grad_terms");
  return oilmm_logpdf_grad(ctx, latents, m, x, N, D, U, S, p, sigma2, y, out_dim, out_logpdf, grad_latents, grad_ard, grad_sigma2, grad_y,
                           grad_U, grad_S, grad_terms, info_latent);
}

extern "C" int lmm_imogp_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, double sigma2,
                                     const double* y, int out_dim, double* out_logpdf, double* grad_latents, double* grad_ard,
                                     double* grad_sigma2, double* grad_y, int* info_latent) {
  return imogp_logpdf_grad(ctx, fs, m, x, N, D, sigma2, y, out_dim, out_logpdf, grad_latents, grad_ard, grad_sigma2, grad_y, nullptr,
                           info_latent);
}
extern "C" int lmm_imogp_logpdf_grad_terms(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, double sigma2,
                                           const double* y, int out_dim, double* out_logpdf, double* grad_latents, double* grad_ard,
                                           double* grad_sigma2, double* grad_y, double* grad_terms, int* info_latent) {
  if (ctx && !grad_terms) return ctx->fail(LMM_E_ARG, "null grad_terms");
  return imogp_logpdf_grad(ctx, fs, m, x, N, D, sigma2, y, out_dim, out_logpdf, grad_latents, grad_ard, grad_sigma2, grad_y, grad_terms,
                           info_latent);
}
// ------------------------------------------------------------------------------------------------
// cov(f::IndependentMOGP, x, y): dense block-diagonal cross-covariance of the PRIOR process between
// two isotopic inputs, by outputs  (src/independent_mogp.jl:66-71; the by-features variants
// :188-215 permute this result on the host side).
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_imogp_cross_cov(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* xa, int Na, const double* xb, int Nb, int D,
                                   double* out) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!fs || !xa || !xb || !out || m <= 0 || Na <= 0 || Nb <= 0 || D <= 0 || D > 64) return ctx->fail(LMM_E_ARG, "bad argument");
  int rc = check_descs(ctx, fs, m, D);
  if (rc) return rc;
  if ((int64_t)m * Na > 46000 || (int64_t)m * Nb > 46000) return ctx->fail(LMM_E_UNSUPPORTED, "dense covariance output too large");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  DevBuf b_xa, b_xb, b_params, b_V, b_out;
  if ((rc = stage_xpad(ctx, b_xa, xa, Na, D))) return rc;
  if ((rc = stage_xpad(ctx, b_xb, xb, Nb, D))) return rc;
  std::vector<double> noise(m, 0.0);
  if ((rc = upload_params(ctx, b_params, fs, noise.data(), 0, m, D))) return rc;
  const int nta = ntiles(Na), ntb = ntiles(Nb);
  CU(b_V.alloc(ctx, (size_t)m * nta * ntb * TT * sizeof(double)));
  TiledRect V{b_V.as<double>(), nta, ntb, (size_t)nta * ntb * TT};
  CU(launch_kmat_cross(st, V, m, b_xa.as<double>(), Na, b_xb.as<double>(), Nb, D, b_params.as<LatentParams>(), ctx->distance_form));
  const size_t rows = (size_t)m * Na, cols = (size_t)m * Nb;
  CU(b_out.alloc(ctx, rows * cols * sizeof(double)));
  CU(cudaMemsetAsync(b_out.p, 0, rows * cols * sizeof(double), st));
  CU(launch_untile_rect_blockdiag(st, V, m, Na, Nb, b_out.as<double>(), rows));
  ctx->launches += 2;
  CU(copy_out(ctx, out, b_out.p, rows * cols * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  return LMM_OK;
}
// ------------------------------------------------------------------------------------------------
// rrule of the general-ILMM logpdf (projected form, src/ilmm.jl:150-163 incl. `project` :61-68 and
// `regulariser` :171-181; `gradient(logpdf, ilmmx, y_train)` at test/ilmm.jl:31).
//   δ = vec((TY)') - μ, α = C^{-1}δ, G = (αα' - C^{-1})/2 over the joint (mN) matrix
//   C = blockdiag(K_a) + ΣT ⊗ I:  d/dθ_a = <G_aa, dK_a/dθ>,  d/dΣT = block traces of G,
//   d/d(TY) = -A (A = α as m x N).  The big contractions run on the device (joint potri on the
//   tensor pipe + fused kernel-gradient pass); the chain through T = M^{-1}H'/σ², M = H'H/σ² + 1e-9 I
//   and ΣT = σ² T T' is m x m / m x p host arithmetic.
// ------------------------------------------------------------------------------------------------

namespace lmm_host {
// Joint potri of one factor (batch 1): X = L^{-T} by the triangular-aware TRSM sweep on an identity, then -C^{-1} = -X X'
// by a triangular-aware SYRK into L's own tiles.  X: L.nt x L.nt tiles of scratch.
cudaError_t joint_neg_inverse(lmm_ctx* ctx, cudaStream_t st, TiledSym L, const double* W, size_t wstride, TiledRect X) {
  cudaError_t e;
  if ((e = launch_rect_identity(st, X, 1)) != cudaSuccess) return e;
  if ((e = trsm_right_lt_upper(ctx, st, X, L, W, wstride, 1)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(L.base, 0, sym_tiles(L.nt) * TT * sizeof(double), st)) != cudaSuccess) return e;
  GemmArgs g{};
  g.A = operand(X); g.B = operand(X); g.C = operand(L);
  g.i0 = 0; g.j0 = 0; g.k0 = 0; g.k1 = L.nt; g.sym = 1; g.k_from_row = 1;
  return launch_gemm(st, GEMM_UPDATE, g, L.nt, L.nt, 1);
}

int ilmm_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H, int p, double sigma2,
                     const double* y, int out_dim, double* out_logpdf, double* grad_latents, double* grad_ard, double* grad_sigma2,
                     double* grad_y, double* grad_H, double* grad_terms, int* info) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!grad_terms && (rc = reject_composite(ctx, latents, m))) return rc;
  if (!H || !y) return ctx->fail(LMM_E_ARG, "null pointer");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  GeneralProjection gp;
  if ((rc = general_projection(ctx, H, p, m, sigma2, N, gp))) return rc;
  const int64_t big64 = (int64_t)m * N;
  if (big64 > (1 << 20)) return ctx->fail(LMM_E_UNSUPPORTED, "joint dimension too large");
  const int big = (int)big64, bnt = ntiles(big);
  const size_t bpad = (size_t)bnt * TILE, wstride = (size_t)bnt * TT;
  CU(cudaEventRecord(ctx->ev[0], st));
  DevBuf b_x, b_y, b_T, b_Q, b_means, b_zero, b_delta, b_part, b_resid, b_params, b_E, b_H, b_Ht, b_Tt, b_L, b_W, b_X, b_logdet, b_info,
      b_r, b_z, b_quad, b_alpha, b_R, b_Z, b_HtR, b_V, b_gpart, b_g3, b_B, b_bT, b_bH, b_gy;
  CU(b_x.alloc(ctx, (size_t)N * D * sizeof(double)));
  CU(copy_in(ctx, b_x.as<double>(), x, (size_t)N * D));
  const double* d_y = y;
  if (!is_device_ptr(y)) {
    CU(b_y.alloc(ctx, (size_t)p * N * sizeof(double)));
    CU(copy_in(ctx, b_y.as<double>(), y, (size_t)p * N));
    d_y = b_y.as<double>();
  }
  std::vector<double> noise0(m, 0.0);
  if ((rc = upload_params(ctx, b_params, latents, noise0.data(), 0, m, D))) return rc;
  std::vector<double> Hh(H, H + (size_t)p * m), Ht((size_t)m * p), Tt((size_t)p * m);
  for (int a = 0; a < m; ++a)
    for (int j = 0; j < p; ++j) {
      Ht[(size_t)j * m + a] = Hh[(size_t)a * p + j];        // H' as m x p col-major
      Tt[(size_t)a * p + j] = gp.pr.T[(size_t)j * m + a];   // T' as p x m col-major
    }
  CU(b_H.alloc(ctx, Hh.size() * sizeof(double)));
  CU(copy_in(ctx, b_H.as<double>(), Hh.data(), Hh.size()));
  CU(b_Ht.alloc(ctx, Ht.size() * sizeof(double)));
  CU(copy_in(ctx, b_Ht.as<double>(), Ht.data(), Ht.size()));
  CU(b_Tt.alloc(ctx, Tt.size() * sizeof(double)));
  CU(copy_in(ctx, b_Tt.as<double>(), Tt.data(), Tt.size()));
  CU(b_T.alloc(ctx, gp.pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, b_T.as<double>(), gp.pr.T.data(), gp.pr.T.size()));
  std::vector<double> hmeans(m);
  for (int i = 0; i < m; ++i) hmeans[i] = latents[i].mean_const;
  CU(b_means.alloc(ctx, (size_t)m * sizeof(double)));
  CU(copy_in(ctx, b_means.as<double>(), hmeans.data(), (size_t)m));
  CU(b_zero.alloc(ctx, (size_t)m * sizeof(double)));
  CU(cudaMemsetAsync(b_zero.p, 0, (size_t)m * sizeof(double), st));
  CU(b_delta.alloc(ctx, bpad * sizeof(double)));
  CU(cudaMemsetAsync(b_delta.p, 0, bpad * sizeof(double), st));
  const int nblk = project_max_partials(N);
  CU(b_part.alloc(ctx, (size_t)nblk * sizeof(double)));
  CU(cudaMemsetAsync(b_part.p, 0, (size_t)nblk * sizeof(double), st));
  CU(b_resid.alloc(ctx, sizeof(double)));
  CU(b_R.alloc(ctx, (size_t)p * N * sizeof(double)));
  CU(b_Z.alloc(ctx, (size_t)m * N * sizeof(double)));
  // δ = vec((TY)') - μ (latent-major, stride N), Z = T Y, R = Y - H Z, |R|²
  CU(launch_project(st, d_y, N, p, b_T.as<double>(), m, 0, m, b_means.as<double>(), b_delta.as<double>(), (size_t)N, b_T.as<double>(),
                    b_H.as<double>(), b_part.as<double>(), nullptr, b_R.as<double>(), b_Z.as<double>()));
  CU(launch_sum_partials(st, b_part.as<double>(), nblk, b_resid.as<double>()));
  ctx->launches += 2;
  CU(b_E.alloc(ctx, gp.ST.size() * sizeof(double)));
  CU(copy_in(ctx, b_E.as<double>(), gp.ST.data(), gp.ST.size()));
  CU(b_L.alloc(ctx, sym_tiles(bnt) * TT * sizeof(double)));
  CU(b_W.alloc(ctx, (size_t)bnt * TT * sizeof(double)));
  CU(b_logdet.alloc(ctx, sizeof(double)));
  CU(b_info.alloc(ctx, sizeof(int)));
  CU(b_quad.alloc(ctx, sizeof(double)));
  CU(cudaMemsetAsync(b_logdet.p, 0, sizeof(double), st));
  CU(cudaMemsetAsync(b_info.p, 0, sizeof(int), st));
  TiledSym L{b_L.as<double>(), bnt, sym_tiles(bnt) * TT};
  CU(launch_assemble_ilmm(st, L, b_x.as<double>(), N, D, b_params.as<LatentParams>(), m, m, b_E.as<double>(), b_H.as<double>(), 0,
                          ctx->distance_form));
  ++ctx->launches;
  {
    PartitionScope scope(ctx);
    CU(chol_factor(ctx, L, b_W.as<double>(), wstride, 1, b_logdet.as<double>(), b_info.as<int>()));
  }
  CU(b_r.alloc(ctx, bpad * sizeof(double)));
  CU(b_z.alloc(ctx, bpad * sizeof(double)));
  CU(b_alpha.alloc(ctx, bpad * sizeof(double)));
  CU(cudaMemcpyAsync(b_r.p, b_delta.p, bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(launch_fwd_solve(st, L, b_W.as<double>(), wstride, b_r.as<double>(), b_z.as<double>(), bpad, 1, &ctx->launches));
  CU(launch_sumsq(st, b_z.as<double>(), bpad, (int)bpad, 1, b_quad.as<double>()));
  CU(cudaMemcpyAsync(b_r.p, b_z.p, bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(launch_bwd_solve(st, L, b_W.as<double>(), wstride, b_r.as<double>(), b_alpha.as<double>(), bpad, 1, &ctx->launches));
  ++ctx->launches;
  CU(b_X.alloc(ctx, (size_t)bnt * bnt * TT * sizeof(double)));
  TiledRect X{b_X.as<double>(), bnt, bnt, (size_t)bnt * bnt * TT};
  CU(joint_neg_inverse(ctx, st, L, b_W.as<double>(), wstride, X));
  const int nchunks = (int)sym_tiles(ntiles(N));
  CU(b_gpart.alloc(ctx, (size_t)m * nchunks * 2 * sizeof(double)));
  CU(b_g3.alloc(ctx, (size_t)m * 3 * sizeof(double)));
  CU(b_B.alloc(ctx, (size_t)m * m * sizeof(double)));
  CU(launch_kgrad_joint(st, L, b_x.as<double>(), N, D, b_params.as<LatentParams>(), m, b_alpha.as<double>(), ctx->distance_form,
                        b_gpart.as<double>(), b_g3.as<double>(), b_B.as<double>()));
  ctx->launches += 6;
  bool want_ard = false;
  DevBuf b_apart, b_gard;
  std::vector<double> hgard;
  if (grad_ard) {
    for (int a = 0; a < m; ++a) want_ard |= latents[a].ard != nullptr;
    for (size_t i = 0; i < (size_t)m * D; ++i) grad_ard[i] = 0.0;
  }
  if (want_ard) {
    CU(b_apart.alloc(ctx, (size_t)m * nchunks * MAX_ARD * sizeof(double)));
    CU(b_gard.alloc(ctx, (size_t)m * MAX_ARD * sizeof(double)));
    CU(launch_kgrad_ard(st, L.base, 0, N, b_x.as<double>(), N, D, b_params.as<LatentParams>(), m, b_alpha.as<double>(), (size_t)N,
                        ctx->distance_form, b_apart.as<double>(), b_gard.as<double>()));
    ctx->launches += 2;
    hgard.resize((size_t)m * MAX_ARD);
    CU(copy_out(ctx, hgard.data(), b_gard.p, hgard.size() * sizeof(double)));
  }
  DevBuf b_tpart, b_gterms;
  std::vector<double> hterms;
  if (grad_terms) {
    int max_terms;
    bool terms_ard;
    terms_shape(latents, 0, m, max_terms, terms_ard);
    CU(b_tpart.alloc(ctx, (size_t)m * nchunks * TERM_SLOTS * sizeof(double)));
    CU(b_gterms.alloc(ctx, (size_t)m * TERM_SLOTS * sizeof(double)));
    CU(launch_kgrad_terms(st, L.base, 0, N, b_x.as<double>(), N, D, b_params.as<LatentParams>(), m, max_terms, terms_ard, b_alpha.as<double>(),
                          (size_t)N, ctx->distance_form, b_tpart.as<double>(), b_gterms.as<double>()));
    ctx->launches += 2;
    hterms.resize((size_t)m * TERM_SLOTS);
    CU(copy_out(ctx, hterms.data(), b_gterms.p, hterms.size() * sizeof(double)));
  }
  // V = H'R/σ² - A ;  dT(direct) = V Y' ;  dH(direct) = R Z'/σ² ;  dy = T'V - R/σ²
  CU(b_HtR.alloc(ctx, (size_t)m * N * sizeof(double)));
  CU(launch_project(st, b_R.as<double>(), N, p, b_Ht.as<double>(), m, 0, m, b_zero.as<double>(), b_HtR.as<double>(), (size_t)N, nullptr,
                    nullptr, b_part.as<double>(), nullptr));
  CU(b_V.alloc(ctx, (size_t)m * N * sizeof(double)));
  CU(launch_scale_sub(st, b_V.as<double>(), b_HtR.as<double>(), 1.0 / sigma2, b_alpha.as<double>(), (size_t)m * N));
  const size_t npm = (size_t)p * m;
  CU(b_bT.alloc(ctx, npm * sizeof(double)));
  CU(b_bH.alloc(ctx, npm * sizeof(double)));
  CU(cudaMemsetAsync(b_bT.p, 0, npm * sizeof(double), st));
  CU(cudaMemsetAsync(b_bH.p, 0, npm * sizeof(double), st));
  CU(launch_abt(st, b_V.as<double>(), (size_t)N, m, d_y, (size_t)N, p, N, 1.0, b_bT.as<double>()));            // m x p
  CU(launch_abt(st, b_R.as<double>(), (size_t)N, p, b_Z.as<double>(), (size_t)N, m, N, 1.0 / sigma2, b_bH.as<double>()));  // p x m
  ctx->launches += 4;
  if (grad_y) {
    const size_t ny = (size_t)p * N;
    CU(b_gy.alloc(ctx, 2 * ny * sizeof(double)));
    CU(launch_backproject(st, b_Tt.as<double>(), p, m, 0, m, b_V.as<double>(), b_V.as<double>(), (size_t)N, N, 0.0, 0.0, 0,
                          b_gy.as<double>(), b_gy.as<double>() + ny));
    CU(launch_axpy(st, b_gy.as<double>(), b_R.as<double>(), ny, -1.0 / sigma2));
    ctx->launches += 2;
    CU(copy_out(ctx, grad_y, b_gy.p, ny * sizeof(double)));
  }
  double hlogdet = 0.0, hquad = 0.0, hres = 0.0;
  int hinfo = 0;
  std::vector<double> g3((size_t)m * 3), B((size_t)m * m), bT(npm), bH(npm);
  CU(copy_out(ctx, &hlogdet, b_logdet.p, sizeof(double)));
  CU(copy_out(ctx, &hquad, b_quad.p, sizeof(double)));
  CU(copy_out(ctx, &hres, b_resid.p, sizeof(double)));
  CU(copy_out(ctx, &hinfo, b_info.p, sizeof(int)));
  CU(copy_out(ctx, g3.data(), b_g3.p, g3.size() * sizeof(double)));
  CU(copy_out(ctx, B.data(), b_B.p, B.size() * sizeof(double)));
  CU(copy_out(ctx, bT.data(), b_bT.p, npm * sizeof(double)));
  CU(copy_out(ctx, bH.data(), b_bH.p, npm * sizeof(double)));
  CU(cudaEventRecord(ctx->ev[1], st));
  CU(cudaStreamSynchronize(st));
  {
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    ctx->timings[0] = ms;
  }
  if (hinfo > 0) {
    if (info) *info = hinfo > big ? big : hinfo;
    ctx->err = "PosDefException: the joint ILMM covariance is not positive definite";
    return hinfo > big ? big : hinfo;
  }
  if (info) *info = 0;
  if (out_logpdf) *out_logpdf = -((double)big * LOG2PI + hlogdet + hquad) / 2.0 - (gp.pr.reg_c0 + hres / sigma2) / 2.0;
  if (want_ard)
    for (int a = 0; a < m; ++a)
      for (int k = 0; k < D && k < MAX_ARD; ++k) grad_ard[(size_t)a * D + k] = latents[a].ard ? hgard[(size_t)a * MAX_ARD + k] : 0.0;
  if (grad_latents)
    for (int a = 0; a < m; ++a) {
      grad_latents[(size_t)a * 3 + 0] = g3[(size_t)a * 3 + 0];
      grad_latents[(size_t)a * 3 + 1] = g3[(size_t)a * 3 + 1];
      grad_latents[(size_t)a * 3 + 2] = g3[(size_t)a * 3 + 2];
    }
  if (grad_terms) scatter_terms(latents, m, D, hterms, grad_terms, grad_latents, grad_ard);
  if (grad_sigma2 || grad_H) {
    rc = ilmm_grad_chain(ctx, gp, Hh, p, m, N, sigma2, hres, B, bT, bH, grad_sigma2, grad_H);
    if (rc != LMM_OK) return rc;
  }
  return LMM_OK;
}
}  // namespace lmm_host

extern "C" int lmm_ilmm_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H,
                                    int p, double sigma2, const double* y, int out_dim, double* out_logpdf, double* grad_latents,
                                    double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_H, int* info) {
  return ilmm_logpdf_grad(ctx, latents, m, x, N, D, H, p, sigma2, y, out_dim, out_logpdf, grad_latents, grad_ard, grad_sigma2, grad_y, grad_H,
                          nullptr, info);
}
extern "C" int lmm_ilmm_logpdf_grad_terms(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H,
                                          int p, double sigma2, const double* y, int out_dim, double* out_logpdf, double* grad_latents,
                                          double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_H, double* grad_terms, int* info) {
  if (ctx && !grad_terms) return ctx->fail(LMM_E_ARG, "null grad_terms");
  return ilmm_logpdf_grad(ctx, latents, m, x, N, D, H, p, sigma2, y, out_dim, out_logpdf, grad_latents, grad_ard, grad_sigma2, grad_y, grad_H,
                          grad_terms, info);
}
// ------------------------------------------------------------------------------------------------
// rrule of the missing-data logpdf of the dense model (the value of lmm_ilmm_masked_posterior).  Over the observed entries
// a = (j_a, i_a):  C_ab = Σ_l H[j_a,l] H[j_b,l] k_l(x_{i_a}, x_{i_b}) + σ² [a = b],  δ_a = y_a - Σ_l H[j_a,l] m_l,
// α = C^{-1}δ,  G = (αα' - C^{-1})/2:
//   d/dθ_{l,t} = Σ_ab G_ab H[j_a,l] H[j_b,l] ∂k_l/∂θ_t            (kgrad_masked_kernel, with the potri's -C^{-1})
//   d/dH[j,l]  = 2 Σ_{a: j_a = j} Σ_b G_ab H[j_b,l] k_l(a,b) + m_l Σ_{a: j_a = j} α_a
//   d/dm_l     = Σ_a α_a H[j_a,l],   d/dσ² = tr G = (α'α - tr C^{-1})/2,   d/dy_a = -α_a (0 at NaN entries)
// Workspace: the packed factor and the potri's square X (≈ 12 nobs² bytes); X is freed before the contraction's partials.
// ------------------------------------------------------------------------------------------------
namespace lmm_host {
int ilmm_masked_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H, int p,
                            double sigma2, const double* y, int out_dim, double* out_logpdf, double* grad_latents, double* grad_ard,
                            double* grad_sigma2, double* grad_y, double* grad_H, double* grad_terms, int* n_observed, int* info) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!grad_terms && (rc = reject_composite(ctx, latents, m))) return rc;
  if (!H || !y) return ctx->fail(LMM_E_ARG, "null pointer");
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  if (is_device_ptr(y) || is_device_ptr(H)) return ctx->fail(LMM_E_UNSUPPORTED, "the missing-data path takes host y and H (the mask is read on the host)");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  std::vector<int> obs;
  std::vector<double> delta;
  masked_observations(latents, m, H, p, N, y, obs, delta);
  const int nobs = (int)obs.size();
  if (n_observed) *n_observed = nobs;
  if (nobs == 0) return ctx->fail(LMM_E_ARG, "every observation is missing");
  if (nobs > (1 << 20)) return ctx->fail(LMM_E_UNSUPPORTED, "joint dimension too large");
  const int bnt = ntiles(nobs), ntl = (int)sym_tiles(bnt);
  const size_t bpad = (size_t)bnt * TILE, wstride = (size_t)bnt * TT;
  std::vector<int> seg(p + 1, 0);  // the entries of output j are [seg[j], seg[j+1]) (obs is sorted by outputs)
  for (int o : obs) ++seg[o / N + 1];
  for (int j = 0; j < p; ++j) seg[j + 1] += seg[j];
  CU(cudaEventRecord(ctx->ev[0], st));
  DevBuf b_x, b_params, b_H, b_obs, b_seg, b_delta, b_L, b_W, b_X, b_logdet, b_info, b_quad, b_r, b_z, b_alpha, b_tpart, b_rpart, b_cpart,
      b_v, b_gterms, b_gH, b_diag;
  CU(b_x.alloc(ctx, (size_t)N * D * sizeof(double)));
  CU(copy_in(ctx, b_x.as<double>(), x, (size_t)N * D));
  std::vector<double> noise0(m, 0.0);
  if ((rc = upload_params(ctx, b_params, latents, noise0.data(), 0, m, D))) return rc;
  CU(b_H.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(copy_in(ctx, b_H.as<double>(), H, (size_t)p * m));
  CU(b_obs.alloc(ctx, (size_t)nobs * sizeof(int)));
  CU(b_seg.alloc(ctx, (size_t)(p + 1) * sizeof(int)));
  ctx->h2d += (int64_t)((size_t)(nobs + p + 1) * sizeof(int));
  CU(cudaMemcpyAsync(b_obs.p, obs.data(), (size_t)nobs * sizeof(int), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(b_seg.p, seg.data(), (size_t)(p + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
  CU(b_delta.alloc(ctx, bpad * sizeof(double)));
  CU(cudaMemsetAsync(b_delta.p, 0, bpad * sizeof(double), st));
  CU(copy_in(ctx, b_delta.as<double>(), delta.data(), (size_t)nobs));
  // factor, logdet, α (as lmm_ilmm_masked_posterior)
  CU(b_L.alloc(ctx, sym_tiles(bnt) * TT * sizeof(double)));
  CU(b_W.alloc(ctx, (size_t)bnt * TT * sizeof(double)));
  CU(b_logdet.alloc(ctx, sizeof(double)));
  CU(b_info.alloc(ctx, sizeof(int)));
  CU(b_quad.alloc(ctx, sizeof(double)));
  CU(cudaMemsetAsync(b_logdet.p, 0, sizeof(double), st));
  CU(cudaMemsetAsync(b_info.p, 0, sizeof(int), st));
  TiledSym L{b_L.as<double>(), bnt, sym_tiles(bnt) * TT};
  CU(launch_assemble_masked(st, L, b_obs.as<int>(), nobs, b_x.as<double>(), N, D, b_params.as<LatentParams>(), m, p, b_H.as<double>(), sigma2,
                            ctx->distance_form));
  ++ctx->launches;
  {
    PartitionScope scope(ctx);
    CU(chol_factor(ctx, L, b_W.as<double>(), wstride, 1, b_logdet.as<double>(), b_info.as<int>()));
  }
  CU(b_r.alloc(ctx, bpad * sizeof(double)));
  CU(b_z.alloc(ctx, bpad * sizeof(double)));
  CU(b_alpha.alloc(ctx, bpad * sizeof(double)));
  CU(cudaMemcpyAsync(b_r.p, b_delta.p, bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(launch_fwd_solve(st, L, b_W.as<double>(), wstride, b_r.as<double>(), b_z.as<double>(), bpad, 1, &ctx->launches));
  CU(launch_sumsq(st, b_z.as<double>(), bpad, (int)bpad, 1, b_quad.as<double>()));
  CU(cudaMemcpyAsync(b_r.p, b_z.p, bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(launch_bwd_solve(st, L, b_W.as<double>(), wstride, b_r.as<double>(), b_alpha.as<double>(), bpad, 1, &ctx->launches));
  ++ctx->launches;
  // potri into the factor's tiles, then the contraction (X is released first: the partials reuse its memory)
  CU(b_X.alloc(ctx, (size_t)bnt * bnt * TT * sizeof(double)));
  TiledRect X{b_X.as<double>(), bnt, bnt, (size_t)bnt * bnt * TT};
  CU(joint_neg_inverse(ctx, st, L, b_W.as<double>(), wstride, X));
  b_X.release();
  b_W.release();
  int max_terms;
  bool terms_ard;
  terms_shape(latents, 0, m, max_terms, terms_ard);
  CU(b_tpart.alloc(ctx, (size_t)m * ntl * TERM_SLOTS * sizeof(double)));
  CU(b_rpart.alloc(ctx, (size_t)m * ntl * TILE * sizeof(double)));
  CU(b_cpart.alloc(ctx, (size_t)m * ntl * TILE * sizeof(double)));
  CU(b_v.alloc(ctx, (size_t)m * nobs * sizeof(double)));
  CU(b_gterms.alloc(ctx, (size_t)m * TERM_SLOTS * sizeof(double)));
  CU(b_gH.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(b_diag.alloc(ctx, sizeof(double)));
  CU(launch_kgrad_masked(st, L, b_obs.as<int>(), nobs, b_x.as<double>(), N, D, b_params.as<LatentParams>(), m, p, b_H.as<double>(),
                         b_alpha.as<double>(), max_terms, terms_ard, ctx->distance_form, b_seg.as<int>(), b_tpart.as<double>(),
                         b_rpart.as<double>(), b_cpart.as<double>(), b_v.as<double>(), b_gterms.as<double>(), b_gH.as<double>(),
                         b_diag.as<double>()));
  ctx->launches += 5;
  double hlogdet = 0.0, hquad = 0.0, hdiag = 0.0;
  int hinfo = 0;
  std::vector<double> ha(nobs), hterms((size_t)m * TERM_SLOTS), hgH((size_t)p * m);
  CU(copy_out(ctx, &hlogdet, b_logdet.p, sizeof(double)));
  CU(copy_out(ctx, &hquad, b_quad.p, sizeof(double)));
  CU(copy_out(ctx, &hinfo, b_info.p, sizeof(int)));
  CU(copy_out(ctx, &hdiag, b_diag.p, sizeof(double)));
  CU(copy_out(ctx, ha.data(), b_alpha.p, (size_t)nobs * sizeof(double)));
  CU(copy_out(ctx, hterms.data(), b_gterms.p, hterms.size() * sizeof(double)));
  CU(copy_out(ctx, hgH.data(), b_gH.p, hgH.size() * sizeof(double)));
  CU(cudaEventRecord(ctx->ev[1], st));
  CU(cudaStreamSynchronize(st));
  {
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    ctx->timings[0] = ms;
  }
  if (hinfo > 0) {
    if (info) *info = hinfo > nobs ? nobs : hinfo;
    ctx->err = "PosDefException: the covariance of the observed entries is not positive definite";
    return hinfo > nobs ? nobs : hinfo;
  }
  if (info) *info = 0;
  if (out_logpdf) *out_logpdf = -((double)nobs * LOG2PI + hlogdet + hquad) / 2.0;
  std::vector<double> asum(p, 0.0);  // Σ_{a: j_a = j} α_a
  double aa = 0.0;
  for (int j = 0; j < p; ++j)
    for (int a = seg[j]; a < seg[j + 1]; ++a) asum[j] += ha[a];
  for (int a = 0; a < nobs; ++a) aa += ha[a] * ha[a];
  if (grad_latents)
    for (int l = 0; l < m; ++l) {
      double gm = 0.0;
      for (int j = 0; j < p; ++j) gm += H[(size_t)l * p + j] * asum[j];
      grad_latents[(size_t)l * 3 + 0] = hterms[(size_t)l * TERM_SLOTS + 0];
      grad_latents[(size_t)l * 3 + 1] = hterms[(size_t)l * TERM_SLOTS + 1];
      grad_latents[(size_t)l * 3 + 2] = gm;
    }
  if (grad_ard)
    for (int l = 0; l < m; ++l)
      for (int k = 0; k < D; ++k)
        grad_ard[(size_t)l * D + k] = (latents[l].ard && k < MAX_ARD) ? hterms[(size_t)l * TERM_SLOTS + 3 + k] : 0.0;
  if (grad_terms) std::copy(hterms.begin(), hterms.end(), grad_terms);
  if (grad_sigma2) *grad_sigma2 = 0.5 * (aa + hdiag);
  if (grad_y) {
    std::fill(grad_y, grad_y + (size_t)p * N, 0.0);
    for (int a = 0; a < nobs; ++a) grad_y[obs[a]] = -ha[a];
  }
  if (grad_H)
    for (int l = 0; l < m; ++l)
      for (int j = 0; j < p; ++j) grad_H[(size_t)l * p + j] = hgH[(size_t)l * p + j] + latents[l].mean_const * asum[j];
  return LMM_OK;
}
}  // namespace lmm_host

extern "C" int lmm_ilmm_masked_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H,
                                           int p, double sigma2, const double* y, int out_dim, double* out_logpdf, double* grad_latents,
                                           double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_H, double* grad_terms,
                                           int* n_observed, int* info) {
  return ilmm_masked_logpdf_grad(ctx, latents, m, x, N, D, H, p, sigma2, y, out_dim, out_logpdf, grad_latents, grad_ard, grad_sigma2, grad_y,
                                 grad_H, grad_terms, n_observed, info);
}

// Per-input mask: the OILMM gradient on the observed inputs (gather, call, scatter); grad_y is 0 at the missing inputs.
extern "C" int lmm_oilmm_masked_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U,
                                            const double* S, int p, double sigma2, const double* y, int out_dim, double* out_logpdf,
                                            double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_U,
                                            double* grad_S, double* grad_terms, int* n_observed_inputs, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  {
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
    if (rc) return rc;
    if (!U || !S || !y) return ctx->fail(LMM_E_ARG, "null pointer");
    if (is_device_ptr(y) || is_device_ptr(x)) return ctx->fail(LMM_E_UNSUPPORTED, "the missing-data path takes host x and y (the mask is read on the host)");
  }
  std::vector<int> keep;
  if (!per_input_mask(y, p, N, keep)) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->fail(LMM_E_UNSUPPORTED, "the mask is not per-input (some outputs observed, some missing at one input): use lmm_ilmm_masked_logpdf_grad");
  }
  const int No = (int)keep.size();
  if (n_observed_inputs) *n_observed_inputs = No;
  if (No == 0) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->fail(LMM_E_ARG, "every observation is missing");
  }
  std::vector<double> xo((size_t)No * D), yo((size_t)p * No), gyo(grad_y ? (size_t)p * No : 0);
  for (int k = 0; k < No; ++k) {
    for (int d = 0; d < D; ++d) xo[(size_t)k * D + d] = x[(size_t)keep[k] * D + d];
    for (int j = 0; j < p; ++j) yo[(size_t)j * No + k] = y[(size_t)j * N + keep[k]];
  }
  const int rc = oilmm_logpdf_grad(ctx, latents, m, xo.data(), No, D, U, S, p, sigma2, yo.data(), out_dim, out_logpdf, grad_latents, grad_ard,
                                   grad_sigma2, grad_y ? gyo.data() : nullptr, grad_U, grad_S, grad_terms, info_latent);
  if (rc == LMM_OK && grad_y) {
    std::fill(grad_y, grad_y + (size_t)p * N, 0.0);
    for (int k = 0; k < No; ++k)
      for (int j = 0; j < p; ++j) grad_y[(size_t)j * N + keep[k]] = gyo[(size_t)j * No + k];
  }
  return rc;
}
