// The per-latent exact-GP driver shared by OILMM (src/oilmm.jl:79-93, 116-134) and IndependentMOGP
// (src/independent_mogp.jl:74-80, 119-126): logpdf, posterior handles, marginals.
#include "host_internal.h"

// ------------------------------------------------------------------------------------------------
// Core: per-latent exact GP logpdf / posterior over a set of independent latents
// ------------------------------------------------------------------------------------------------
namespace lmm_host {



// The shared driver for OILMM (src/oilmm.jl:79-93, 116-134) and IndependentMOGP
// (src/independent_mogp.jl:74-80, 119-126).
int latents_run(lmm_ctx* ctx, int kind, const lmm_gp_desc* latents, int m, const double* x, int N, int D, int p, double sigma2,
                const double* y, const Projection& pr, const double* Hhost, const double* Uhost, const double* Shost, RunOut out,
                const double* noise_vec /* per-point noise, m*N by outputs (IndependentMOGP with Σy = Diagonal(v)) */) {
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  int lo, hi;
  shard_range(ctx, m, lo, hi);
  const int mloc = hi - lo;
  const int nt = ntiles(N);
  const size_t npad = (size_t)nt * TILE;
  const bool keep = out.post != nullptr;

  CU(cudaEventRecord(ctx->ev[0], st));
  // ---- stage inputs
  DevBuf b_x, b_y, b_T, b_P, b_Q, b_means, b_ty, b_resid_part, b_resid, b_terms;
  CU(b_x.alloc(ctx, npad * D * sizeof(double)));
  CU(cudaMemsetAsync(b_x.p, 0, npad * D * sizeof(double), st));
  CU(copy_in(ctx, b_x.as<double>(), x, (size_t)N * D));
  const double* d_y = y;
  if (!is_device_ptr(y)) {
    CU(b_y.alloc(ctx, (size_t)p * N * sizeof(double)));
    CU(copy_in(ctx, b_y.as<double>(), y, (size_t)p * N));
    d_y = b_y.as<double>();
  }
  CU(b_T.alloc(ctx, pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, b_T.as<double>(), pr.T.data(), pr.T.size()));
  if (pr.has_reg) {
    CU(b_P.alloc(ctx, pr.P.size() * sizeof(double)));
    CU(copy_in(ctx, b_P.as<double>(), pr.P.data(), pr.P.size()));
    CU(b_Q.alloc(ctx, pr.Q.size() * sizeof(double)));
    CU(copy_in(ctx, b_Q.as<double>(), pr.Q.data(), pr.Q.size()));
  }
  std::vector<double> hmeans(mloc > 0 ? mloc : 1, 0.0);
  for (int i = lo; i < hi; ++i) hmeans[i - lo] = latents[i].mean_const;
  CU(b_means.alloc(ctx, hmeans.size() * sizeof(double)));
  CU(copy_in(ctx, b_means.as<double>(), hmeans.data(), hmeans.size()));
  std::vector<LatentParams> hparams;
  fill_params(hparams, latents, pr.noise.data(), lo, hi, D);
  DevBuf b_params;
  CU(b_params.alloc(ctx, (hparams.size() + 1) * sizeof(LatentParams)));
  if (mloc > 0) {
    ctx->h2d += (int64_t)(hparams.size() * sizeof(LatentParams));
    CU(cudaMemcpyAsync(b_params.p, hparams.data(), hparams.size() * sizeof(LatentParams), cudaMemcpyHostToDevice, st));
  }

  // ---- projection + residual (K2/K3)
  CU(b_ty.alloc(ctx, (size_t)(mloc > 0 ? mloc : 1) * npad * sizeof(double)));
  CU(cudaMemsetAsync(b_ty.p, 0, (size_t)(mloc > 0 ? mloc : 1) * npad * sizeof(double), st));
  const int nblk = project_max_partials(N);
  CU(b_resid_part.alloc(ctx, (size_t)nblk * sizeof(double)));
  CU(cudaMemsetAsync(b_resid_part.p, 0, (size_t)nblk * sizeof(double), st));
  CU(b_resid.alloc(ctx, sizeof(double)));
  CU(b_terms.alloc(ctx, (size_t)(m + 1) * sizeof(double)));
  CU(cudaMemsetAsync(b_terms.p, 0, (size_t)(m + 1) * sizeof(double), st));
  const bool do_reg = pr.has_reg && ctx->rank == 0;
  {
    int nb_out = 0;
    CU(launch_project(st, d_y, N, p, b_T.as<double>(), m, lo, mloc, b_means.as<double>(), b_ty.as<double>(), npad,
                      do_reg ? b_P.as<double>() : nullptr, do_reg ? b_Q.as<double>() : nullptr, b_resid_part.as<double>(), &nb_out));
    ++ctx->launches;
    if (do_reg) {
      CU(launch_sum_partials(st, b_resid_part.as<double>(), nblk, b_resid.as<double>()));
      CU(launch_regulariser(st, b_terms.as<double>() + m, pr.reg_c0, b_resid.as<double>(), sigma2));
      ctx->launches += 2;
    }
  }
  CU(cudaEventRecord(ctx->ev[1], st));

  // ---- factor storage: all local latents when a posterior is kept, else a streamed arena
  const size_t per_lat = factor_bytes_per_latent(nt);
  int chunk = mloc;
  if (!keep && mloc > 0) CU(mem_fit(ctx, per_lat + 6 * npad * sizeof(double), mloc, &chunk));
  DevBuf b_L, b_W, b_alpha, b_r, b_z, b_logdet, b_quad, b_info, b_nv, b_env, b_fb, b_rowoff;
  if (noise_vec) {
    const int nl = mloc > 0 ? mloc : 1;
    CU(b_nv.alloc(ctx, (size_t)nl * npad * sizeof(double)));
    CU(cudaMemsetAsync(b_nv.p, 0, (size_t)nl * npad * sizeof(double), st));
    if (mloc > 0) {
      const bool dev = is_device_ptr(noise_vec);
      if (!dev) ctx->h2d += (int64_t)((size_t)mloc * N * sizeof(double));
      CU(cudaMemcpy2DAsync(b_nv.p, npad * sizeof(double), noise_vec + (size_t)lo * N, (size_t)N * sizeof(double), (size_t)N * sizeof(double),
                           (size_t)mloc, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    }
  }
  std::vector<int> hinfo(mloc > 0 ? mloc : 1, 0);
  // tile envelope of each chunk's kernel matrices: far-apart points give exact zeros that the factorisation and the solves skip
  std::vector<int> henv;
  // the kernel-matrix build skips the tiles that are provably exact zeros (launch_kmat_bound) where the factorisation takes the envelope
  std::vector<int> hrowoff;
  bool skipped = false;
  float ms_kmat = 0, ms_chol = 0, ms_solve = 0;
  if (mloc > 0) {
    henv.resize((size_t)chunk * nt);
    hrowoff.resize(henv.size() + 1);
    CU(b_env.alloc(ctx, henv.size() * sizeof(int)));
    CU(b_fb.alloc(ctx, henv.size() * sizeof(int)));
    CU(b_rowoff.alloc(ctx, hrowoff.size() * sizeof(int)));
    CU(b_L.alloc(ctx, (size_t)chunk * sym_tiles(nt) * TT * sizeof(double)));
    CU(b_W.alloc(ctx, (size_t)chunk * nt * TT * sizeof(double)));
    CU(b_r.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    CU(b_z.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    if (keep) CU(b_alpha.alloc(ctx, (size_t)mloc * npad * sizeof(double)));
    CU(b_logdet.alloc(ctx, (size_t)mloc * sizeof(double)));
    CU(b_quad.alloc(ctx, (size_t)mloc * sizeof(double)));
    CU(b_info.alloc(ctx, (size_t)mloc * sizeof(int)));
    CU(cudaMemsetAsync(b_logdet.p, 0, (size_t)mloc * sizeof(double), st));
    CU(cudaMemsetAsync(b_info.p, 0, (size_t)mloc * sizeof(int), st));
    for (int c0 = 0; c0 < mloc; c0 += chunk) {
      const int nb = (c0 + chunk <= mloc) ? chunk : mloc - c0;
      TiledSym L{b_L.as<double>(), nt, sym_tiles(nt) * TT};
      double* W = b_W.as<double>();
      const size_t wstride = (size_t)nt * TT;
      const LatentParams* dp = b_params.as<LatentParams>() + c0;
      double* delta = b_ty.as<double>() + (size_t)c0 * npad;
      CU(cudaEventRecord(ctx->ev[2], st));
      const int* env = b_env.as<int>();
      const bool skip = ctx->kmat_skip && chol_takes_envelope(ctx, nt, nb);
      if (skip) {
        // fb (one small launch) -> host: the build's grid is the tiles (I, fb[b][I] .. I) of all nb latents
        CU(launch_kmat_bound(st, nb, b_x.as<double>(), N, D, nt, dp, b_fb.as<int>()));
        ++ctx->launches;
        CU(copy_out(ctx, henv.data(), b_fb.p, (size_t)nb * nt * sizeof(int)));
        CU(cudaStreamSynchronize(st));
        hrowoff[0] = 0;
        for (int r = 0; r < nb * nt; ++r) hrowoff[r + 1] = hrowoff[r] + (r % nt) + 1 - henv[r];
        ctx->h2d += (int64_t)((size_t)(nb * nt + 1) * sizeof(int));
        CU(cudaMemcpyAsync(b_rowoff.p, hrowoff.data(), (size_t)(nb * nt + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
        skipped = true;
      }
      CU(launch_kmat_sym(st, L, nb, b_x.as<double>(), N, D, dp, ctx->distance_form,
                         noise_vec ? b_nv.as<double>() + (size_t)c0 * npad : nullptr, npad, 0, b_env.as<int>(),
                         skip ? b_rowoff.as<int>() : nullptr, hrowoff[nb * nt]));
      ++ctx->launches;
      CU(cudaEventRecord(ctx->ev[3], st));
      CU(copy_out(ctx, henv.data(), env, (size_t)nb * nt * sizeof(int)));  // sizes the factorisation's grids
      CU(cudaStreamSynchronize(st));
      CU(chol_factor(ctx, L, W, wstride, nb, b_logdet.as<double>() + c0, b_info.as<int>() + c0, 0, env, henv.data()));
      CU(cudaEventRecord(ctx->ev[4], st));
      CU(cudaMemcpyAsync(b_r.p, delta, (size_t)nb * npad * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_fwd_solve(st, L, W, wstride, b_r.as<double>(), b_z.as<double>(), npad, nb, &ctx->launches, env));
      CU(launch_sumsq(st, b_z.as<double>(), npad, (int)npad, nb, b_quad.as<double>() + c0));
      ++ctx->launches;
      if (keep) {
        CU(cudaMemcpyAsync(b_r.p, b_z.p, (size_t)nb * npad * sizeof(double), cudaMemcpyDeviceToDevice, st));
        CU(launch_bwd_solve(st, L, W, wstride, b_r.as<double>(), b_alpha.as<double>() + (size_t)c0 * npad, npad, nb, &ctx->launches, env));
      }
      CU(launch_lml_terms(st, b_terms.as<double>(), lo + c0, nb, b_logdet.as<double>() + c0, b_quad.as<double>() + c0, N, LOG2PI));
      ++ctx->launches;
      CU(cudaEventRecord(ctx->ev[5], st));
      {
        // accumulate stage timings per chunk: the stage events are reused by the next chunk, so they
        // are read here (one host sync per chunk; negligible next to a chunk's factorisation)
        CU(cudaEventSynchronize(ctx->ev[5]));
        float a = 0, bq = 0, c = 0;
        cudaEventElapsedTime(&a, ctx->ev[2], ctx->ev[3]);
        cudaEventElapsedTime(&bq, ctx->ev[3], ctx->ev[4]);
        cudaEventElapsedTime(&c, ctx->ev[4], ctx->ev[5]);
        ms_kmat += a; ms_chol += bq; ms_solve += c;
      }
    }
  }
  // ---- reduce the per-latent terms across ranks (one NCCL all-reduce over NVLink) and read back
  if (ctx->comm && ctx->nranks > 1) {
    int r = nccl_api().AllReduce(b_terms.p, b_terms.p, (size_t)(m + 1), NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
    if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
  }
  std::vector<double> hterms(m + 1, 0.0);
  CU(copy_out(ctx, hterms.data(), b_terms.p, (size_t)(m + 1) * sizeof(double)));
  if (mloc > 0) CU(copy_out(ctx, hinfo.data(), b_info.p, (size_t)mloc * sizeof(int)));
  CU(cudaEventRecord(ctx->ev[6], st));
  CU(cudaStreamSynchronize(st));
  {
    float tot = 0, prj = 0;
    cudaEventElapsedTime(&tot, ctx->ev[0], ctx->ev[6]);
    cudaEventElapsedTime(&prj, ctx->ev[0], ctx->ev[1]);
    ctx->timings[0] = tot; ctx->timings[1] = ms_kmat; ctx->timings[2] = ms_chol; ctx->timings[3] = ms_solve; ctx->timings[4] = prj;
  }
  {
    // collective verdict: every rank returns the same PosDef code / latent, none emits a value (ADVICE r01)
    const int rc_info = report_info(ctx, std::vector<int>(hinfo.begin(), hinfo.begin() + mloc), lo, N, out.info_latent);
    if (rc_info) return rc_info;
  }
  if (out.lml_terms) memcpy(out.lml_terms, hterms.data(), (size_t)(m + 1) * sizeof(double));
  if (out.logpdf) {
    double s = 0.0;
    for (int i = 0; i < m; ++i) s += hterms[i];
    *out.logpdf = s + hterms[m];
  }
  if (keep) {
    DevBuf b_H;
    CU(b_H.alloc(ctx, (size_t)p * m * sizeof(double)));
    CU(copy_in(ctx, b_H.as<double>(), Hhost, (size_t)p * m));
    CU(cudaStreamSynchronize(st));
    lmm_post* P = new lmm_post();  // nothing below can fail: ownership of the device buffers moves to P
    P->ctx = ctx; P->kind = kind; P->m = m; P->p = p; P->N = N; P->D = D; P->nt = nt; P->lo = lo; P->hi = hi;
    P->adopt_descs(latents, m, D);
    P->noise = pr.noise;
    P->H.assign(Hhost, Hhost + (size_t)p * m);
    if (Uhost) P->U.assign(Uhost, Uhost + (size_t)p * m);
    if (Shost) P->S.assign(Shost, Shost + m);
    P->sigma2 = sigma2;
    P->bytes = (size_t)mloc * (per_lat + 2 * npad * sizeof(double)) + npad * D * sizeof(double);
    P->d_xpad = (double*)b_x.detach();
    P->d_L = (double*)b_L.detach();
    P->d_W = (double*)b_W.detach();
    P->d_alpha = (double*)b_alpha.detach();
    P->d_delta = (double*)b_ty.detach();
    P->d_params = (LatentParams*)b_params.detach();
    P->d_H = (double*)b_H.detach();
    if (noise_vec) P->d_noise_vec = (double*)b_nv.detach();
    if (skipped) {  // a kept posterior holds every latent in one chunk: b_env is the envelope of all of them
      P->d_env = (int*)b_env.detach();
      P->zeros_pending = true;
    }
    *out.post = P;
  }
  return LMM_OK;
}

int oilmm_projection(lmm_ctx* ctx, const double* U, const double* S, int p, int m, double sigma2, int N, Projection& pr,
                     std::vector<double>& H) {
  for (int i = 0; i < m; ++i)
    if (!(S[i] > 0.0)) return ctx->fail(LMM_E_ARG, "S must have positive entries");
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  pr.T.resize((size_t)m * p);
  pr.P.resize((size_t)m * p);
  pr.Q.assign(U, U + (size_t)p * m);
  pr.noise.resize(m);
  H.resize((size_t)p * m);
  double logdetS = 0.0;
  for (int i = 0; i < m; ++i) {
    const double rs = std::sqrt(S[i]);
    for (int j = 0; j < p; ++j) {
      const double u = U[(size_t)i * p + j];
      pr.T[(size_t)j * m + i] = u / rs;  // T = sqrt(S) \ U'        src/oilmm.jl:24
      pr.P[(size_t)j * m + i] = u;       // U'
      H[(size_t)i * p + j] = u * rs;     // U * sqrt(S)             src/oilmm.jl:69
    }
    pr.noise[i] = sigma2 * (1.0 / S[i]);  // diag(σ² * inv(S))      src/oilmm.jl:27
    logdetS += std::log(S[i]);
  }
  // -(n (logdet(S) + (p-m) log(2πσ²)) + |(I-UU')Y|²/σ²)/2          src/oilmm.jl:111-112
  pr.reg_c0 = (double)N * (logdetS + (double)(p - m) * std::log(2.0 * M_PI * sigma2));
  pr.has_reg = true;
  return LMM_OK;
}

int check_common(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const void* x, int N, int D, int p, int out_dim) {
  if (!latents || !x || m <= 0 || N <= 0 || D <= 0 || p <= 0) return ctx->fail(LMM_E_ARG, "null pointer or non-positive size");
  if (D > 64) return ctx->fail(LMM_E_UNSUPPORTED, "input dimension D > 64 is not supported");
  if (out_dim != p) return ctx->fail(LMM_E_OUT_DIM, "out dim of x != out dim of f.");
  return check_descs(ctx, latents, m, D);
}

}  // namespace lmm_host

// ------------------------------------------------------------------------------------------------
// OILMM
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_oilmm_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                                   const double* U, const double* S, int p, double sigma2, const double* y, int out_dim,
                                   lmm_post** out_post, double* out_logpdf, double* lml_terms, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (out_post) *out_post = nullptr;
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!U || !S || !y) return ctx->fail(LMM_E_ARG, "null pointer");
  if (m > p) return ctx->fail(LMM_E_ARG, "more latents than outputs");
  Projection pr;
  std::vector<double> H;
  if ((rc = oilmm_projection(ctx, U, S, p, m, sigma2, N, pr, H))) return rc;
  RunOut out{out_post, out_logpdf, lml_terms, info_latent};
  return latents_run(ctx, POST_OILMM, latents, m, x, N, D, p, sigma2, y, pr, H.data(), U, S, out);
}

extern "C" int lmm_oilmm_logpdf(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U,
                                const double* S, int p, double sigma2, const double* y, int out_dim, double* out_logpdf,
                                double* lml_terms, int* info_latent) {
  if (!out_logpdf && !lml_terms) return LMM_E_ARG;
  return lmm_oilmm_posterior(ctx, latents, m, x, N, D, U, S, p, sigma2, y, out_dim, nullptr, out_logpdf, lml_terms, info_latent);
}

// ------------------------------------------------------------------------------------------------
// IndependentMOGP
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_imogp_posterior(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, double sigma2,
                                   const double* y, int out_dim, lmm_post** out_post, double* out_logpdf, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (out_post) *out_post = nullptr;
  int rc = check_common(ctx, fs, m, x, N, D, m, out_dim);
  if (rc) return rc;
  if (!y) return ctx->fail(LMM_E_ARG, "null pointer");
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  Projection pr;
  pr.T.assign((size_t)m * m, 0.0);
  for (int i = 0; i < m; ++i) pr.T[(size_t)i * m + i] = 1.0;
  pr.noise.assign(m, sigma2);
  pr.has_reg = false;
  std::vector<double> H = pr.T;
  RunOut out{out_post, out_logpdf, nullptr, info_latent};
  return latents_run(ctx, POST_IMOGP, fs, m, x, N, D, m, sigma2, y, pr, H.data(), nullptr, nullptr, out);
}

extern "C" int lmm_imogp_logpdf(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, double sigma2,
                                const double* y, int out_dim, double* out_logpdf, double* lml_terms, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, fs, m, x, N, D, m, out_dim);
  if (rc) return rc;
  if (!y || (!out_logpdf && !lml_terms)) return ctx->fail(LMM_E_ARG, "null pointer");
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  Projection pr;
  pr.T.assign((size_t)m * m, 0.0);
  for (int i = 0; i < m; ++i) pr.T[(size_t)i * m + i] = 1.0;
  pr.noise.assign(m, sigma2);
  pr.has_reg = false;
  std::vector<double> H = pr.T;
  RunOut out{nullptr, out_logpdf, lml_terms, info_latent};
  return latents_run(ctx, POST_IMOGP, fs, m, x, N, D, m, sigma2, y, pr, H.data(), nullptr, nullptr, out);
}

// ------------------------------------------------------------------------------------------------
// Posterior handle
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_post_free(lmm_post* post) {
  if (!post) return LMM_E_ARG;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  cudaSetDevice(ctx->device);
  void* ptrs[] = {post->d_xpad, post->d_L, post->d_W, post->d_alpha, post->d_delta, post->d_params, post->d_H, post->d_noise_vec,
                  post->d_Ept, post->d_obs, post->d_env};
  for (void* q : ptrs)
    if (q) cudaFreeAsync(q, ctx->stream);
  cudaStreamSynchronize(ctx->stream);
  delete post;
  return LMM_OK;
}

extern "C" int lmm_post_info(lmm_post* post, int* kind, int* m, int* p, int* N, int* D, int64_t* device_bytes) {
  if (!post) return LMM_E_ARG;
  if (kind) *kind = post->kind;
  if (m) *m = post->m;
  if (p) *p = post->p;
  if (N) *N = post->N;
  if (D) *D = post->D;
  if (device_bytes) *device_bytes = (int64_t)post->bytes;
  return LMM_OK;
}

extern "C" int lmm_post_export(lmm_post* post, int i, double* Lout, double* alpha, double* delta) {
  if (!post) return LMM_E_ARG;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  int b, n;
  if (post->joint()) {
    if (i != 0) return ctx->fail(LMM_E_ARG, "a joint posterior has one factor (i = 0)");
    b = 0;
    n = post->big_n;
  } else {
    if (i < post->lo || i >= post->hi) return ctx->fail(LMM_E_ARG, "latent not resident on this rank");
    b = i - post->lo;
    n = post->N;
  }
  const size_t vstride = post->joint() ? (size_t)post->big_nt * TILE : post->npad();
  if (Lout) {
    DevBuf dense;
    CU(dense.alloc(ctx, (size_t)n * n * sizeof(double)));
    CU(cudaMemsetAsync(dense.p, 0, (size_t)n * n * sizeof(double), ctx->stream));
    CU(launch_untile_lower(ctx->stream, post->Lsym(), b, dense.as<double>(), n));
    ++ctx->launches;
    CU(copy_out(ctx, Lout, dense.p, (size_t)n * n * sizeof(double)));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  if (alpha) CU(copy_out(ctx, alpha, post->d_alpha + (size_t)b * vstride, (size_t)n * sizeof(double)));
  if (delta) CU(copy_out(ctx, delta, post->d_delta + (size_t)b * vstride, (size_t)n * sizeof(double)));
  CU(cudaStreamSynchronize(ctx->stream));
  return LMM_OK;
}

namespace lmm_host {

int post_fill_zeros(lmm_post* post) {
  if (!post->zeros_pending) return LMM_OK;
  lmm_ctx* ctx = post->ctx;
  CU(launch_kmat_zero(ctx->stream, post->Lsym(), post->nloc(), post->d_env));
  ++ctx->launches;
  post->zeros_pending = false;
  return LMM_OK;
}

// Latent posterior marginals at xs for the resident latents: ML/VL [nloc][nspad] on the device.
// mean*_i = m_i + K(x*,x) α_i ; var*_i = k(x*,x*) - colsumsq(L_i^{-1} K(x,x*))   (AbstractGPs)
// `first` / `count` select a sub-range of the resident latents (default: all of them); d_ML / d_VL rows are relative to it.
int post_latent_marginals(lmm_post* post, const double* d_xspad, int Ns, int nts, double* d_ML, double* d_VL, int first, int count) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  const int nloc = count < 0 ? post->nloc() - first : count, nt = post->nt;
  const size_t nspad = (size_t)nts * TILE;
  if (nloc <= 0) return LMM_OK;
  const size_t per_lat = (size_t)nts * nt * TT * sizeof(double);
  int chunk = 0;
  CU(mem_fit(ctx, per_lat, nloc, &chunk));
  DevBuf b_V;
  CU(b_V.alloc(ctx, (size_t)chunk * per_lat));
  const TiledSym L = post->Lsym();
  for (int c0 = 0; c0 < nloc; c0 += chunk) {
    const int nb = (c0 + chunk <= nloc) ? chunk : nloc - c0;
    TiledRect V{b_V.as<double>(), nts, nt, (size_t)nts * nt * TT};
    const int g0 = first + c0;  // index among the resident latents
    TiledSym Lc{L.base + (size_t)g0 * L.batch_stride, nt, L.batch_stride};
    const double* Wc = post->d_W + (size_t)g0 * post->wstride();
    const LatentParams* dp = post->d_params + g0;
    CU(launch_kmat_cross(st, V, nb, d_xspad, Ns, post->d_xpad, post->N, post->D, dp, ctx->distance_form));
    CU(launch_rect_gemv(st, V, post->d_alpha + (size_t)g0 * post->npad(), post->npad(), d_ML + (size_t)c0 * nspad, nspad, dp, 1, nb));
    ctx->launches += 2;
    CU(trsm_right_lt(ctx, V, Lc, Wc, post->wstride(), nb, dp));  // dp: k(x*,x*) bounds the row norms (int8 path, if the option is on)
    CU(launch_rect_rowsumsq(st, V, d_VL + (size_t)c0 * nspad, nspad, dp, nb));
    ++ctx->launches;
  }
  return LMM_OK;
}

}  // namespace lmm_host


extern "C" int lmm_post_mean_and_var(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean, double* var) {
  if (!post || !xs || Ns <= 0 || !mean || !var) return LMM_E_ARG;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  if (post->kind == POST_MASKED) return masked_post_mean_and_var(post, xs, Ns, sigma2, mean, var);
  if (post->joint()) return ilmm_post_mean_and_var(post, xs, Ns, sigma2, mean, var);
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  const int nts = ntiles(Ns), nloc = post->nloc(), p = post->p, m = post->m;
  const size_t nspad = (size_t)nts * TILE;
  CU(cudaEventRecord(ctx->ev[0], st));
  DevBuf b_xs, b_ML, b_VL, b_mean, b_var;
  CU(b_xs.alloc(ctx, nspad * post->D * sizeof(double)));
  CU(cudaMemsetAsync(b_xs.p, 0, nspad * post->D * sizeof(double), st));
  CU(copy_in(ctx, b_xs.as<double>(), xs, (size_t)Ns * post->D));
  CU(b_ML.alloc(ctx, (size_t)(nloc > 0 ? nloc : 1) * nspad * sizeof(double)));
  CU(b_VL.alloc(ctx, (size_t)(nloc > 0 ? nloc : 1) * nspad * sizeof(double)));
  int rc = post_latent_marginals(post, b_xs.as<double>(), Ns, nts, b_ML.as<double>(), b_VL.as<double>());
  if (rc) return rc;
  // one buffer [mean | var] so that a single all-reduce covers both
  const size_t nout = (size_t)p * Ns;
  CU(b_mean.alloc(ctx, 2 * nout * sizeof(double)));
  double* d_mean = b_mean.as<double>();
  double* d_var = d_mean + nout;
  const bool multi = ctx->comm && ctx->nranks > 1;
  if (post->kind == POST_OILMM) {
    // M = H M_lat ; V = (H∘H)(V_lat + 1e-18) + σ²     src/oilmm.jl:61-75 (1e-18: default FiniteGP noise)
    CU(cudaMemsetAsync(d_mean, 0, 2 * nout * sizeof(double), st));
    CU(launch_backproject(st, post->d_H, p, m, post->lo, nloc, b_ML.as<double>(), b_VL.as<double>(), nspad, Ns, 1e-18, sigma2,
                          multi ? 0 : 1, d_mean, d_var));
    ++ctx->launches;
  } else {
    // IndependentMOGP: mean/var concatenated by outputs, var + σ²   src/independent_mogp.jl:50-57
    CU(cudaMemsetAsync(d_mean, 0, 2 * nout * sizeof(double), st));
    if (nloc > 0) {
      CU(launch_copy_add(st, nloc, d_mean + (size_t)post->lo * Ns, Ns, b_ML.as<double>(), nspad, Ns, 0.0));
      CU(launch_copy_add(st, nloc, d_var + (size_t)post->lo * Ns, Ns, b_VL.as<double>(), nspad, Ns, multi ? 0.0 : sigma2));
      ctx->launches += 2;
    }
  }
  if (multi) {
    int r = nccl_api().AllReduce(d_mean, d_mean, 2 * nout, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
    if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
    CU(launch_add_scalar(st, d_var, nout, sigma2));
    ++ctx->launches;
  }
  CU(copy_out(ctx, mean, d_mean, nout * sizeof(double)));
  CU(copy_out(ctx, var, d_var, nout * sizeof(double)));
  CU(cudaEventRecord(ctx->ev[1], st));
  CU(cudaStreamSynchronize(st));
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
  ctx->timings[0] = ms;
  ctx->timings[5] = ms;
  return LMM_OK;
}

// mean_and_var(post.f.fs[i](x*, σ²)): one PosteriorGP latent evaluated on its own (AbstractGPs FiniteGP{<:PosteriorGP}
// mean_and_var = (m_i + K*x α_i, k** - colsumsq(L_i^{-1} K x*) + σ²)); src/oilmm.jl:61 calls exactly this per latent.
extern "C" int lmm_post_latent_mean_and_var(lmm_post* post, int i, const double* xs, int Ns, double sigma2, double* mean, double* var) {
  if (!post || !xs || Ns <= 0 || !mean || !var) return LMM_E_ARG;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  if (post->joint()) return ctx->fail(LMM_E_UNSUPPORTED, "a joint posterior has no independent latent posteriors");
  if (i < post->lo || i >= post->hi) return ctx->fail(LMM_E_ARG, "latent not resident on this rank");
  cudaStream_t st = ctx->stream;
  const int nts = ntiles(Ns);
  const size_t nspad = (size_t)nts * TILE;
  DevBuf b_xs, b_ML, b_VL;
  CU(b_xs.alloc(ctx, nspad * post->D * sizeof(double)));
  CU(cudaMemsetAsync(b_xs.p, 0, nspad * post->D * sizeof(double), st));
  CU(copy_in(ctx, b_xs.as<double>(), xs, (size_t)Ns * post->D));
  CU(b_ML.alloc(ctx, nspad * sizeof(double)));
  CU(b_VL.alloc(ctx, nspad * sizeof(double)));
  int rc = post_latent_marginals(post, b_xs.as<double>(), Ns, nts, b_ML.as<double>(), b_VL.as<double>(), i - post->lo, 1);
  if (rc) return rc;
  CU(launch_add_scalar(st, b_VL.as<double>(), (size_t)Ns, sigma2));
  ++ctx->launches;
  CU(copy_out(ctx, mean, b_ML.p, (size_t)Ns * sizeof(double)));
  CU(copy_out(ctx, var, b_VL.p, (size_t)Ns * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  return LMM_OK;
}

// ------------------------------------------------------------------------------------------------
// OILMM prior marginals: src/oilmm.jl:57-76 with GP latents (mean const, var = variance + 1e-18)
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_oilmm_prior_mean_and_var(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* xs, int Ns, int D,
                                            const double* U, const double* S, int p, double sigma2, int out_dim, double* mean,
                                            double* var) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, xs, Ns, D, p, out_dim);
  if (rc) return rc;
  if (!U || !S || !mean || !var) return ctx->fail(LMM_E_ARG, "null pointer");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  Projection pr;
  std::vector<double> H;
  if ((rc = oilmm_projection(ctx, U, S, p, m, sigma2, Ns, pr, H))) return rc;
  // latent marginals are constants along n: build ML/VL on the host side of the (tiny) m x Ns arrays
  std::vector<double> ML((size_t)m * Ns), VL((size_t)m * Ns);
  for (int i = 0; i < m; ++i)
    for (int n = 0; n < Ns; ++n) {
      ML[(size_t)i * Ns + n] = latents[i].mean_const;
      VL[(size_t)i * Ns + n] = desc_kdiag(latents[i]);
    }
  DevBuf b_H, b_ML, b_VL, b_out;
  CU(b_H.alloc(ctx, H.size() * sizeof(double)));
  CU(copy_in(ctx, b_H.as<double>(), H.data(), H.size()));
  CU(b_ML.alloc(ctx, ML.size() * sizeof(double)));
  CU(copy_in(ctx, b_ML.as<double>(), ML.data(), ML.size()));
  CU(b_VL.alloc(ctx, VL.size() * sizeof(double)));
  CU(copy_in(ctx, b_VL.as<double>(), VL.data(), VL.size()));
  const size_t nout = (size_t)p * Ns;
  CU(b_out.alloc(ctx, 2 * nout * sizeof(double)));
  CU(launch_backproject(st, b_H.as<double>(), p, m, 0, m, b_ML.as<double>(), b_VL.as<double>(), Ns, Ns, 1e-18, sigma2, 1,
                        b_out.as<double>(), b_out.as<double>() + nout));
  ++ctx->launches;
  CU(copy_out(ctx, mean, b_out.p, nout * sizeof(double)));
  CU(copy_out(ctx, var, b_out.as<double>() + nout, nout * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  return LMM_OK;
}
