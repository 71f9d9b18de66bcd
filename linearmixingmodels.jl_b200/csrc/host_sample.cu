// Sampling (src/oilmm.jl:40-54, src/ilmm.jl:78-87, src/independent_mogp.jl:83-86), posterior-predictive logpdf and
// its gradient, hyper-parameter sweep (BASELINE config 5).
#include "host_internal.h"

namespace lmm_host {

// Upload LatentParams for latents [lo, hi) of `descs` with per-latent noise values.
int upload_params(lmm_ctx* ctx, DevBuf& buf, const lmm_gp_desc* descs, const double* noise_all, int lo, int hi, int D) {
  std::vector<LatentParams> hp;
  fill_params(hp, descs, noise_all, lo, hi, D);
  CU(buf.alloc(ctx, (hp.size() + 1) * sizeof(LatentParams)));
  if (!hp.empty()) {
    ctx->h2d += (int64_t)(hp.size() * sizeof(LatentParams));
    CU(cudaMemcpyAsync(buf.p, hp.data(), hp.size() * sizeof(LatentParams), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));  // hp goes out of scope
  }
  return LMM_OK;
}

// Copy z (m*N, latent-major, host or device) rows [lo,hi) into a zero-padded [nloc][npad] buffer.
int stage_latent_vectors(lmm_ctx* ctx, DevBuf& buf, const double* z, int N, size_t npad, int lo, int hi) {
  const int nloc = hi - lo;
  CU(buf.alloc(ctx, (size_t)(nloc > 0 ? nloc : 1) * npad * sizeof(double)));
  CU(cudaMemsetAsync(buf.p, 0, (size_t)(nloc > 0 ? nloc : 1) * npad * sizeof(double), ctx->stream));
  const bool dev = is_device_ptr(z);
  if (nloc > 0) {
    if (!dev) ctx->h2d += (int64_t)((size_t)nloc * N * sizeof(double));
    CU(cudaMemcpy2DAsync(buf.p, npad * sizeof(double), z + (size_t)lo * N, (size_t)N * sizeof(double), (size_t)N * sizeof(double),
                         (size_t)nloc, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
  }
  return LMM_OK;
}

// PosDef report for a set of sharded factorizations.  hinfo holds this rank's LAPACK-style info words for the units
// lo, lo + 1, ...  With a communicator the verdict is made COLLECTIVE: one MIN all-reduce of a single double that encodes
// (first failing unit, pivot), so that every rank returns the same code and the same info_latent and no rank goes on with a
// value summed from a failed factorisation's garbage (ADVICE r01: rank-local PosDef status desynchronised the ranks, and a
// return between the factorisation and a later collective left the other ranks hanging in NCCL).  EVERY rank of the
// communicator must therefore reach this call, also one that owns no unit (hinfo empty), and callers must not return a
// rank-local PosDef code before it.
int report_info(lmm_ctx* ctx, const std::vector<int>& hinfo, int lo, int nmax, int* info_latent) {
  constexpr double NONE = 1e300;
  double key = NONE;  // unit * 2^31 + pivot of the first failing local unit
  for (size_t i = 0; i < hinfo.size(); ++i)
    if (hinfo[i] > 0) {
      const int pivot = hinfo[i] > nmax ? nmax : hinfo[i];
      key = (double)(lo + (int)i) * 2147483648.0 + (double)pivot;
      break;
    }
  if (ctx->comm && ctx->nranks > 1) {
    DevBuf b_key;
    CU(b_key.alloc(ctx, sizeof(double)));
    CU(cudaMemcpyAsync(b_key.p, &key, sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    int r = nccl_api().AllReduce(b_key.p, b_key.p, 1, NCCL_DOUBLE, NCCL_MIN, ctx->comm, ctx->stream);
    if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
    CU(cudaMemcpyAsync(&key, b_key.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  if (key < NONE) {
    const int unit = (int)std::floor(key / 2147483648.0);
    const int pivot = (int)(key - (double)unit * 2147483648.0);
    if (info_latent) *info_latent = unit;
    char buf[128];
    snprintf(buf, sizeof buf, "PosDefException: latent %d is not positive definite (pivot %d)", unit, pivot);
    ctx->err = buf;
    return pivot;
  }
  if (info_latent) *info_latent = -1;
  return LMM_OK;
}

// Prior samples of the resident latents: X_i = mean_i + chol(K_i + noise_i I) z_i  -> d_X [nloc][npad]
// (AbstractGPs `rand(rng, f(x, σ²)) = m + C.U' z`; reference call sites src/oilmm.jl:47,
// src/independent_mogp.jl:85, src/ilmm.jl:84)
int prior_latent_samples(lmm_ctx* ctx, const lmm_gp_desc* descs, const double* noise_all, int lo, int hi, const double* d_xpad, int N,
                         int D, const double* d_z, double* d_X, int* info_latent) {
  cudaStream_t st = ctx->stream;
  const int nloc = hi - lo, nt = ntiles(N);
  const size_t npad = (size_t)nt * TILE;
  if (nloc == 0) return report_info(ctx, std::vector<int>(), lo, N, info_latent);  // collective: every rank takes part
  DevBuf b_params, b_L, b_W, b_logdet, b_info;
  int rc = upload_params(ctx, b_params, descs, noise_all, lo, hi, D);
  if (rc) return rc;
  int chunk = 0;
  CU(mem_fit(ctx, factor_bytes_per_latent(nt), nloc, &chunk));
  CU(b_L.alloc(ctx, (size_t)chunk * sym_tiles(nt) * TT * sizeof(double)));
  CU(b_W.alloc(ctx, (size_t)chunk * nt * TT * sizeof(double)));
  CU(b_logdet.alloc(ctx, (size_t)nloc * sizeof(double)));
  CU(b_info.alloc(ctx, (size_t)nloc * sizeof(int)));
  CU(cudaMemsetAsync(b_logdet.p, 0, (size_t)nloc * sizeof(double), st));
  CU(cudaMemsetAsync(b_info.p, 0, (size_t)nloc * sizeof(int), st));
  for (int c0 = 0; c0 < nloc; c0 += chunk) {
    const int nb = (c0 + chunk <= nloc) ? chunk : nloc - c0;
    TiledSym L{b_L.as<double>(), nt, sym_tiles(nt) * TT};
    CU(launch_kmat_sym(st, L, nb, d_xpad, N, D, b_params.as<LatentParams>() + c0, ctx->distance_form));
    ++ctx->launches;
    CU(chol_factor(ctx, L, b_W.as<double>(), (size_t)nt * TT, nb, b_logdet.as<double>() + c0, b_info.as<int>() + c0));
    CU(launch_lower_gemv(st, L, d_z + (size_t)c0 * npad, npad, d_X + (size_t)c0 * npad, npad, nb));
    CU(launch_add_mean(st, nb, d_X + (size_t)c0 * npad, npad, N, b_params.as<LatentParams>() + c0));
    ctx->launches += 2;
  }
  std::vector<int> hinfo(nloc, 0);
  CU(copy_out(ctx, hinfo.data(), b_info.p, (size_t)nloc * sizeof(int)));
  CU(cudaStreamSynchronize(st));
  return report_info(ctx, hinfo, lo, N, info_latent);
}

// out[j*N+n] = sum_i H[j,i] X[i][n] (+ all-reduce over ranks) + sqrt(sigma2) * z_noise
int mix_and_add_noise(lmm_ctx* ctx, const double* Hhost, int p, int m, int lo, int hi, const double* d_X, size_t npad, int N,
                      double sigma2, const double* z_noise, double* out) {
  cudaStream_t st = ctx->stream;
  const size_t nout = (size_t)p * N;
  DevBuf b_H, b_out, b_zn;
  CU(b_H.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(copy_in(ctx, b_H.as<double>(), Hhost, (size_t)p * m));
  CU(b_out.alloc(ctx, 2 * nout * sizeof(double)));
  CU(cudaMemsetAsync(b_out.p, 0, 2 * nout * sizeof(double), st));
  CU(launch_backproject(st, b_H.as<double>(), p, m, lo, hi - lo, d_X, d_X, npad, N, 0.0, 0.0, 0, b_out.as<double>(),
                        b_out.as<double>() + nout));
  ++ctx->launches;
  if (ctx->comm && ctx->nranks > 1) {
    int r = nccl_api().AllReduce(b_out.p, b_out.p, nout, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
    if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
  }
  if (z_noise) {
    const double* dzn = z_noise;
    if (!is_device_ptr(z_noise)) {
      CU(b_zn.alloc(ctx, nout * sizeof(double)));
      CU(copy_in(ctx, b_zn.as<double>(), z_noise, nout));
      dzn = b_zn.as<double>();
    }
    CU(launch_axpy(st, b_out.as<double>(), dzn, nout, std::sqrt(sigma2)));
    ++ctx->launches;
  }
  CU(copy_out(ctx, out, b_out.p, nout * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  return LMM_OK;
}

int stage_xpad(lmm_ctx* ctx, DevBuf& buf, const double* x, int N, int D) {
  const size_t npad = (size_t)ntiles(N) * TILE;
  CU(buf.alloc(ctx, npad * D * sizeof(double)));
  CU(cudaMemsetAsync(buf.p, 0, npad * D * sizeof(double), ctx->stream));
  CU(copy_in(ctx, buf.as<double>(), x, (size_t)N * D));
  return LMM_OK;
}

}  // namespace lmm_host

// ------------------------------------------------------------------------------------------------
// rand on prior latents
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_oilmm_rand(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U,
                              const double* S, int p, double sigma2, int out_dim, const double* z_latent, const double* z_noise,
                              double* out, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!U || !S || !z_latent || !z_noise || !out) return ctx->fail(LMM_E_ARG, "null pointer");
  CU(cudaSetDevice(ctx->device));
  Projection pr;
  std::vector<double> H;
  if ((rc = oilmm_projection(ctx, U, S, p, m, sigma2, N, pr, H))) return rc;
  int lo, hi;
  shard_range(ctx, m, lo, hi);
  const size_t npad = (size_t)ntiles(N) * TILE;
  DevBuf b_x, b_z, b_X;
  if ((rc = stage_xpad(ctx, b_x, x, N, D))) return rc;
  if ((rc = stage_latent_vectors(ctx, b_z, z_latent, N, npad, lo, hi))) return rc;
  CU(b_X.alloc(ctx, (size_t)(hi - lo > 0 ? hi - lo : 1) * npad * sizeof(double)));
  std::vector<double> noise(m, 1e-18);  // `f(x)` default FiniteGP noise, src/oilmm.jl:47
  if ((rc = prior_latent_samples(ctx, latents, noise.data(), lo, hi, b_x.as<double>(), N, D, b_z.as<double>(), b_X.as<double>(), info_latent)))
    return rc;
  return mix_and_add_noise(ctx, H.data(), p, m, lo, hi, b_X.as<double>(), npad, N, sigma2, z_noise, out);
}

extern "C" int lmm_ilmm_rand(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H, int p,
                             double sigma2, int out_dim, const double* z_latent, const double* z_noise, double* out, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!H || !z_latent || !z_noise || !out) return ctx->fail(LMM_E_ARG, "null pointer");
  CU(cudaSetDevice(ctx->device));
  int lo, hi;
  shard_range(ctx, m, lo, hi);
  const size_t npad = (size_t)ntiles(N) * TILE;
  DevBuf b_x, b_z, b_X;
  if ((rc = stage_xpad(ctx, b_x, x, N, D))) return rc;
  if ((rc = stage_latent_vectors(ctx, b_z, z_latent, N, npad, lo, hi))) return rc;
  CU(b_X.alloc(ctx, (size_t)(hi - lo > 0 ? hi - lo : 1) * npad * sizeof(double)));
  std::vector<double> noise(m, 1e-12);  // src/ilmm.jl:84
  if ((rc = prior_latent_samples(ctx, latents, noise.data(), lo, hi, b_x.as<double>(), N, D, b_z.as<double>(), b_X.as<double>(), info_latent)))
    return rc;
  return mix_and_add_noise(ctx, H, p, m, lo, hi, b_X.as<double>(), npad, N, sigma2, z_noise, out);
}

extern "C" int lmm_imogp_rand(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, double sigma2, int out_dim,
                              const double* z, double* out, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, fs, m, x, N, D, m, out_dim);
  if (rc) return rc;
  if (!z || !out) return ctx->fail(LMM_E_ARG, "null pointer");
  CU(cudaSetDevice(ctx->device));
  int lo, hi;
  shard_range(ctx, m, lo, hi);
  const size_t npad = (size_t)ntiles(N) * TILE;
  DevBuf b_x, b_z, b_X;
  if ((rc = stage_xpad(ctx, b_x, x, N, D))) return rc;
  if ((rc = stage_latent_vectors(ctx, b_z, z, N, npad, lo, hi))) return rc;
  CU(b_X.alloc(ctx, (size_t)(hi - lo > 0 ? hi - lo : 1) * npad * sizeof(double)));
  std::vector<double> noise(m, sigma2);  // finite_gps(ft, σ²), src/independent_mogp.jl:84
  if ((rc = prior_latent_samples(ctx, fs, noise.data(), lo, hi, b_x.as<double>(), N, D, b_z.as<double>(), b_X.as<double>(), info_latent)))
    return rc;
  std::vector<double> I((size_t)m * m, 0.0);
  for (int i = 0; i < m; ++i) I[(size_t)i * m + i] = 1.0;
  return mix_and_add_noise(ctx, I.data(), m, m, lo, hi, b_X.as<double>(), npad, N, 0.0, nullptr, out);
}

// ------------------------------------------------------------------------------------------------
// Posterior predictive over the resident latents: factor of K** - V V' + noise I, mean*.
// ------------------------------------------------------------------------------------------------
namespace lmm_host {


// Builds, for ALL resident latents, the predictive mean (ML [nloc][nspad]) and the Cholesky factor
// of the predictive covariance K(x*,x*) - K(x*,x)(K+Σ)^{-1}K(x,x*) + noise_i I (C tiles, W inverse
// diagonal tiles).  AbstractGPs: cov(post, x*) = K** - (C.U'\K_{x*})'(C.U'\K_{x*}).
int build_predictive(lmm_post* post, const double* xs, int Ns, const std::vector<double>& noise_all, Predictive& P, int* info_latent,
                     bool factor) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  const int nloc = post->nloc(), nt = post->nt;
  P.nts = ntiles(Ns);
  P.nspad = (size_t)P.nts * TILE;
  int rc = stage_xpad(ctx, P.xs, xs, Ns, post->D);
  if (rc) return rc;
  if ((rc = upload_params(ctx, P.params, post->descs.data(), noise_all.data(), post->lo, post->hi, post->D))) return rc;
  const int nl = nloc > 0 ? nloc : 1;
  CU(P.ML.alloc(ctx, (size_t)nl * P.nspad * sizeof(double)));
  CU(P.C.alloc(ctx, (size_t)nl * sym_tiles(P.nts) * TT * sizeof(double)));
  CU(P.W.alloc(ctx, (size_t)nl * P.nts * TT * sizeof(double)));
  CU(P.logdet.alloc(ctx, (size_t)nl * sizeof(double)));
  CU(P.info.alloc(ctx, (size_t)nl * sizeof(int)));
  CU(cudaMemsetAsync(P.logdet.p, 0, (size_t)nl * sizeof(double), st));
  CU(cudaMemsetAsync(P.info.p, 0, (size_t)nl * sizeof(int), st));
  if (nloc == 0) return factor ? report_info(ctx, std::vector<int>(), post->lo, Ns, info_latent) : LMM_OK;  // collective
  const size_t per_lat = (size_t)P.nts * nt * TT * sizeof(double);
  int chunk = 0;
  CU(mem_fit(ctx, per_lat, nloc, &chunk));
  CU(P.V.alloc(ctx, (size_t)chunk * per_lat));
  const TiledSym L = post->Lsym();
  TiledSym Call{P.C.as<double>(), P.nts, sym_tiles(P.nts) * TT};
  CU(launch_kmat_sym(st, Call, nloc, P.xs.as<double>(), Ns, post->D, P.params.as<LatentParams>(), ctx->distance_form));
  ++ctx->launches;
  for (int c0 = 0; c0 < nloc; c0 += chunk) {
    const int nb = (c0 + chunk <= nloc) ? chunk : nloc - c0;
    TiledRect V{P.V.as<double>(), P.nts, nt, (size_t)P.nts * nt * TT};
    TiledSym Lc{L.base + (size_t)c0 * L.batch_stride, nt, L.batch_stride};
    TiledSym Cc{Call.base + (size_t)c0 * Call.batch_stride, P.nts, Call.batch_stride};
    const LatentParams* dp = P.params.as<LatentParams>() + c0;
    CU(launch_kmat_cross(st, V, nb, P.xs.as<double>(), Ns, post->d_xpad, post->N, post->D, dp, ctx->distance_form));
    CU(launch_rect_gemv(st, V, post->d_alpha + (size_t)c0 * post->npad(), post->npad(), P.ML.as<double>() + (size_t)c0 * P.nspad,
                        P.nspad, dp, 1, nb));
    ctx->launches += 2;
    CU(trsm_right_lt(ctx, V, Lc, post->d_W + (size_t)c0 * post->wstride(), post->wstride(), nb));
    GemmArgs g{};
    g.A = operand(V); g.B = operand(V); g.C = operand(Cc);
    g.i0 = 0; g.j0 = 0; g.k0 = 0; g.k1 = nt; g.sym = 1;
    CU(launch_gemm(st, GEMM_UPDATE, g, P.nts, P.nts, nb));
    ++ctx->launches;
  }
  if (!factor) return LMM_OK;
  CU(chol_factor(ctx, Call, P.W.as<double>(), (size_t)P.nts * TT, nloc, P.logdet.as<double>(), P.info.as<int>()));
  std::vector<int> hinfo(nloc, 0);
  CU(copy_out(ctx, hinfo.data(), P.info.p, (size_t)nloc * sizeof(int)));
  CU(cudaStreamSynchronize(st));
  return report_info(ctx, hinfo, post->lo, Ns, info_latent);
}

}  // namespace lmm_host


extern "C" int lmm_post_rand(lmm_post* post, const double* xs, int Ns, double sigma2, const double* z_latent, const double* z_noise,
                             double* out, int* info_latent) {
  if (!post || !xs || Ns <= 0 || !z_latent || !out) return LMM_E_ARG;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  if (post->kind != POST_IMOGP && post->kind != POST_JOINT && post->kind != POST_MASKED && !z_noise) return ctx->fail(LMM_E_ARG, "null pointer");
  if (post->kind == POST_MASKED) return masked_post_rand(post, xs, Ns, sigma2, z_latent, out, info_latent);  // z_latent: p*Ns normals
  if (post->joint()) return ilmm_post_rand(post, xs, Ns, sigma2, z_latent, z_noise, out, info_latent);
  cudaStream_t st = ctx->stream;
  // OILMM: latents sampled at the default FiniteGP noise 1e-18 (src/oilmm.jl:47); IndependentMOGP: σ²
  std::vector<double> noise(post->m, post->kind == POST_OILMM ? 1e-18 : sigma2);
  Predictive P;
  int rc = build_predictive(post, xs, Ns, noise, P, info_latent);
  if (rc) return rc;
  const int nloc = post->nloc();
  DevBuf b_z, b_X;
  if ((rc = stage_latent_vectors(ctx, b_z, z_latent, Ns, P.nspad, post->lo, post->hi))) return rc;
  CU(b_X.alloc(ctx, (size_t)(nloc > 0 ? nloc : 1) * P.nspad * sizeof(double)));
  if (nloc > 0) {
    TiledSym Call{P.C.as<double>(), P.nts, sym_tiles(P.nts) * TT};
    CU(launch_lower_gemv(st, Call, b_z.as<double>(), P.nspad, b_X.as<double>(), P.nspad, nloc));
    CU(launch_axpy(st, b_X.as<double>(), P.ML.as<double>(), (size_t)nloc * P.nspad, 1.0));
    ctx->launches += 2;
  }
  if (post->kind == POST_OILMM)
    return mix_and_add_noise(ctx, post->H.data(), post->p, post->m, post->lo, post->hi, b_X.as<double>(), P.nspad, Ns, sigma2, z_noise, out);
  std::vector<double> I((size_t)post->m * post->m, 0.0);
  for (int i = 0; i < post->m; ++i) I[(size_t)i * post->m + i] = 1.0;
  return mix_and_add_noise(ctx, I.data(), post->m, post->m, post->lo, post->hi, b_X.as<double>(), P.nspad, Ns, 0.0, nullptr, out);
}

namespace lmm_host {
// logpdf(post(x*, σ²), y*) and, optionally, its gradient w.r.t. σ² and y* (the posterior's own data
// α, C, x and the kernel hyper-parameters are held fixed):
//   d/dy* = -T' α* - R/σ²,   d/dν_i = (α*_i'α*_i - tr(C*_i^{-1}))/2 with ν_i = σ²/S_i (OILMM) or σ².
// keep (nullable): hands the predictive factors, β and the gradient pieces to the caller (requires grad_sigma2).
int post_logpdf_impl(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, double* out_logpdf, double* grad_sigma2,
                     double* grad_y, int* info_latent, PredictiveKeep* keep) {
  lmm_ctx* ctx = post->ctx;
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  if (post->kind == POST_MASKED) return ctx->fail(LMM_E_UNSUPPORTED, "a missing-data posterior offers mean_and_var only");
  if (post->joint()) return ilmm_post_logpdf(post, xs, Ns, sigma2, ys, out_logpdf, grad_sigma2, grad_y, info_latent);
  const bool want_grad = grad_sigma2 || grad_y;
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p, nloc = post->nloc(), lo = post->lo;
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
    pr.has_reg = false;
  }
  Predictive P_own;
  Predictive& P = keep ? keep->P : P_own;
  if ((rc = build_predictive(post, xs, Ns, pr.noise, P, info_latent))) return rc;
  // project y*: δ*_i = (T Y*)_i  (means handled below: predictive mean ML already includes m_i)
  DevBuf b_y, b_T, b_Pm, b_Q, b_zero, b_ty, b_part, b_resid, b_terms, b_r, b_z, b_quad;
  const double* d_y = ys;
  if (!is_device_ptr(ys)) {
    CU(b_y.alloc(ctx, (size_t)p * Ns * sizeof(double)));
    CU(copy_in(ctx, b_y.as<double>(), ys, (size_t)p * Ns));
    d_y = b_y.as<double>();
  }
  CU(b_T.alloc(ctx, pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, b_T.as<double>(), pr.T.data(), pr.T.size()));
  const bool do_reg = pr.has_reg && ctx->rank == 0;
  if (pr.has_reg) {
    CU(b_Pm.alloc(ctx, pr.P.size() * sizeof(double)));
    CU(copy_in(ctx, b_Pm.as<double>(), pr.P.data(), pr.P.size()));
    CU(b_Q.alloc(ctx, pr.Q.size() * sizeof(double)));
    CU(copy_in(ctx, b_Q.as<double>(), pr.Q.data(), pr.Q.size()));
  }
  const int nl = nloc > 0 ? nloc : 1;
  CU(b_zero.alloc(ctx, (size_t)nl * sizeof(double)));
  CU(cudaMemsetAsync(b_zero.p, 0, (size_t)nl * sizeof(double), st));
  CU(b_ty.alloc(ctx, (size_t)nl * P.nspad * sizeof(double)));
  CU(cudaMemsetAsync(b_ty.p, 0, (size_t)nl * P.nspad * sizeof(double), st));
  const int nblk = project_max_partials(Ns);
  CU(b_part.alloc(ctx, (size_t)nblk * sizeof(double)));
  CU(cudaMemsetAsync(b_part.p, 0, (size_t)nblk * sizeof(double), st));
  CU(b_resid.alloc(ctx, sizeof(double)));
  CU(b_terms.alloc(ctx, (size_t)(m + 1) * sizeof(double)));
  CU(cudaMemsetAsync(b_terms.p, 0, (size_t)(m + 1) * sizeof(double), st));
  DevBuf b_R, b_alpha_own, b_X, b_tr, b_gy, b_gvec;
  DevBuf& b_alpha = keep ? keep->beta : b_alpha_own;
  const bool want_R = do_reg && want_grad;
  if (want_R) CU(b_R.alloc(ctx, (size_t)p * Ns * sizeof(double)));
  CU(cudaMemsetAsync(b_resid.p, 0, sizeof(double), st));
  CU(launch_project(st, d_y, Ns, p, b_T.as<double>(), m, lo, nloc, b_zero.as<double>(), b_ty.as<double>(), P.nspad,
                    do_reg ? b_Pm.as<double>() : nullptr, do_reg ? b_Q.as<double>() : nullptr, b_part.as<double>(), nullptr,
                    want_R ? b_R.as<double>() : nullptr, nullptr));
  ++ctx->launches;
  if (do_reg) {
    CU(launch_sum_partials(st, b_part.as<double>(), nblk, b_resid.as<double>()));
    CU(launch_regulariser(st, b_terms.as<double>() + m, pr.reg_c0, b_resid.as<double>(), sigma2));
    ctx->launches += 2;
  }
  if (nloc > 0) {
    // δ = Ty* - mean*   (padding rows: ML padding holds mean_i + 0, ty padding 0 -> force to 0 below)
    const size_t tot = (size_t)nloc * P.nspad;
    CU(launch_axpy(st, b_ty.as<double>(), P.ML.as<double>(), tot, -1.0));
    if (P.nspad > (size_t)Ns)
      CU(cudaMemset2DAsync(b_ty.as<double>() + Ns, P.nspad * sizeof(double), 0, (P.nspad - Ns) * sizeof(double), (size_t)nloc, st));
    CU(b_r.alloc(ctx, tot * sizeof(double)));
    CU(b_z.alloc(ctx, tot * sizeof(double)));
    CU(b_quad.alloc(ctx, (size_t)nloc * sizeof(double)));
    CU(cudaMemcpyAsync(b_r.p, b_ty.p, tot * sizeof(double), cudaMemcpyDeviceToDevice, st));
    TiledSym Call{P.C.as<double>(), P.nts, sym_tiles(P.nts) * TT};
    CU(launch_fwd_solve(st, Call, P.W.as<double>(), (size_t)P.nts * TT, b_r.as<double>(), b_z.as<double>(), P.nspad, nloc, &ctx->launches));
    CU(launch_sumsq(st, b_z.as<double>(), P.nspad, (int)P.nspad, nloc, b_quad.as<double>()));
    CU(launch_lml_terms(st, b_terms.as<double>(), lo, nloc, P.logdet.as<double>(), b_quad.as<double>(), Ns, LOG2PI));
    ctx->launches += 3;
  }
  const bool multi = ctx->comm && ctx->nranks > 1;
  // gradient pieces: [α*'α* (m) | tr(C*^{-1}) (m) | |R|² (1)] reduced over ranks
  const size_t ngv = (size_t)2 * m + 1;
  if (want_grad) {
    CU(b_gvec.alloc(ctx, ngv * sizeof(double)));
    CU(cudaMemsetAsync(b_gvec.p, 0, ngv * sizeof(double), st));
    if (do_reg) CU(cudaMemcpyAsync(b_gvec.as<double>() + 2 * m, b_resid.p, sizeof(double), cudaMemcpyDeviceToDevice, st));
    const size_t ny = (size_t)p * Ns;
    if (grad_y) {
      CU(b_gy.alloc(ctx, 2 * ny * sizeof(double)));
      CU(cudaMemsetAsync(b_gy.p, 0, 2 * ny * sizeof(double), st));
    }
    if (nloc > 0) {
      const size_t tot = (size_t)nloc * P.nspad;
      TiledSym Call{P.C.as<double>(), P.nts, sym_tiles(P.nts) * TT};
      const size_t wst = (size_t)P.nts * TT;
      CU(b_alpha.alloc(ctx, tot * sizeof(double)));
      CU(cudaMemcpyAsync(b_r.p, b_z.p, tot * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CU(launch_bwd_solve(st, Call, P.W.as<double>(), wst, b_r.as<double>(), b_alpha.as<double>(), P.nspad, nloc, &ctx->launches));
      CU(launch_sumsq(st, b_alpha.as<double>(), P.nspad, (int)P.nspad, nloc, b_gvec.as<double>() + lo));
      ++ctx->launches;
      if (grad_sigma2) {
        // tr(C^{-1}) = |L^{-T}|_F²: triangular TRSM sweep on an identity, chunked by free memory
        const size_t per_lat = (size_t)P.nts * P.nts * TT * sizeof(double);
        int chunk = 0;
        CU(mem_fit(ctx, per_lat, nloc, &chunk));
        CU(b_X.alloc(ctx, (size_t)chunk * per_lat));
        for (int c0 = 0; c0 < nloc; c0 += chunk) {
          const int nb = (c0 + chunk <= nloc) ? chunk : nloc - c0;
          TiledRect X{b_X.as<double>(), P.nts, P.nts, (size_t)P.nts * P.nts * TT};
          TiledSym Lc{Call.base + (size_t)c0 * Call.batch_stride, P.nts, Call.batch_stride};
          CU(launch_rect_identity(st, X, nb));
          CU(trsm_right_lt_upper(ctx, st, X, Lc, P.W.as<double>() + (size_t)c0 * wst, wst, nb));
          CU(launch_sumsq(st, b_X.as<double>(), (size_t)P.nts * P.nts * TT, P.nts * P.nts * TT, nb, b_gvec.as<double>() + m + lo + c0));
          ctx->launches += 2;
        }
        // the identity padding of the factor contributes (nspad - Ns) ones to each trace
        CU(launch_add_scalar(st, b_gvec.as<double>() + m + lo, (size_t)nloc, -(double)(P.nspad - (size_t)Ns)));
        ++ctx->launches;
      }
      if (grad_y) {
        std::vector<double> Hneg((size_t)p * m);
        for (int i = 0; i < m; ++i)
          for (int j = 0; j < p; ++j) Hneg[(size_t)i * p + j] = -pr.T[(size_t)j * m + i];
        DevBuf b_Hn;
        CU(b_Hn.alloc(ctx, Hneg.size() * sizeof(double)));
        CU(copy_in(ctx, b_Hn.as<double>(), Hneg.data(), Hneg.size()));
        CU(launch_backproject(st, b_Hn.as<double>(), p, m, lo, nloc, b_alpha.as<double>(), b_alpha.as<double>(), P.nspad, Ns, 0.0, 0.0, 0,
                              b_gy.as<double>(), b_gy.as<double>() + ny));
        ++ctx->launches;
        CU(cudaStreamSynchronize(st));  // Hneg / b_Hn go out of scope
      }
    }
    if (grad_y) {
      if (want_R) {
        CU(launch_axpy(st, b_gy.as<double>(), b_R.as<double>(), ny, -1.0 / sigma2));
        ++ctx->launches;
      }
      if (multi) {
        int r = nccl_api().AllReduce(b_gy.p, b_gy.p, ny, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
        if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
      }
      CU(copy_out(ctx, grad_y, b_gy.p, ny * sizeof(double)));
    }
    if (multi) {
      int r = nccl_api().AllReduce(b_gvec.p, b_gvec.p, ngv, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
      if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
    }
  }
  if (multi) {
    int r = nccl_api().AllReduce(b_terms.p, b_terms.p, (size_t)(m + 1), NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
    if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
  }
  std::vector<double> ht(m + 1, 0.0), hg(ngv, 0.0);
  CU(copy_out(ctx, ht.data(), b_terms.p, (size_t)(m + 1) * sizeof(double)));
  if (want_grad) CU(copy_out(ctx, hg.data(), b_gvec.p, ngv * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  if (keep) keep->hg = hg;
  double s = 0.0;
  for (int i = 0; i < m; ++i) s += ht[i];
  if (out_logpdf) *out_logpdf = s + ht[m];
  if (grad_sigma2) {
    double g = 0.0;
    for (int i = 0; i < m; ++i) g += 0.5 * (hg[i] - hg[(size_t)m + i]) * (post->kind == POST_OILMM ? 1.0 / post->S[i] : 1.0);
    if (pr.has_reg) g += -0.5 * ((double)Ns * (double)(p - m) / sigma2 - hg[(size_t)2 * m] / (sigma2 * sigma2));
    *grad_sigma2 = g;
  }
  return LMM_OK;
}
}  // namespace lmm_host

extern "C" int lmm_post_logpdf(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, double* out_logpdf,
                               int* info_latent) {
  if (!post || !xs || Ns <= 0 || !ys || !out_logpdf) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(post->ctx->mu);
  return post_logpdf_impl(post, xs, Ns, sigma2, ys, out_logpdf, nullptr, nullptr, info_latent);
}

extern "C" int lmm_post_logpdf_grad(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, double* out_logpdf,
                                    double* grad_sigma2, double* grad_y, int* info_latent) {
  if (!post || !xs || Ns <= 0 || !ys) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(post->ctx->mu);
  return post_logpdf_impl(post, xs, Ns, sigma2, ys, out_logpdf, grad_sigma2, grad_y, info_latent);
}

// ------------------------------------------------------------------------------------------------
// Hyper-parameter sweep (BASELINE config 5): (sweep x latent) grid of independent factorisations
// streamed through one arena; the grid is block-sharded over ranks.
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_oilmm_logpdf_sweep(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U,
                                      const double* S, int p, double sigma2, const double* y, int out_dim,
                                      const double* inv_lengthscale_scales, int n_sweep, double* out_logpdfs, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!U || !S || !y || !inv_lengthscale_scales || n_sweep <= 0 || !out_logpdfs) return ctx->fail(LMM_E_ARG, "null pointer");
  for (int s = 0; s < n_sweep; ++s)
    if (!(inv_lengthscale_scales[s] > 0.0)) return ctx->fail(LMM_E_ARG, "lengthscale scales must be positive");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  Projection pr;
  std::vector<double> H;
  if ((rc = oilmm_projection(ctx, U, S, p, m, sigma2, N, pr, H))) return rc;
  const int nt = ntiles(N);
  const size_t npad = (size_t)nt * TILE;
  const int units = n_sweep * m;
  const int ulo = (int)(((int64_t)units * ctx->rank) / ctx->nranks), uhi = (int)(((int64_t)units * (ctx->rank + 1)) / ctx->nranks);
  const int nu = uhi - ulo;
  CU(cudaEventRecord(ctx->ev[0], st));
  DevBuf b_x, b_y, b_T, b_Pm, b_Q, b_means, b_ty, b_part, b_resid, b_terms;
  if ((rc = stage_xpad(ctx, b_x, x, N, D))) return rc;
  const double* d_y = y;
  if (!is_device_ptr(y)) {
    CU(b_y.alloc(ctx, (size_t)p * N * sizeof(double)));
    CU(copy_in(ctx, b_y.as<double>(), y, (size_t)p * N));
    d_y = b_y.as<double>();
  }
  CU(b_T.alloc(ctx, pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, b_T.as<double>(), pr.T.data(), pr.T.size()));
  CU(b_Pm.alloc(ctx, pr.P.size() * sizeof(double)));
  CU(copy_in(ctx, b_Pm.as<double>(), pr.P.data(), pr.P.size()));
  CU(b_Q.alloc(ctx, pr.Q.size() * sizeof(double)));
  CU(copy_in(ctx, b_Q.as<double>(), pr.Q.data(), pr.Q.size()));
  std::vector<double> hmeans(m);
  for (int i = 0; i < m; ++i) hmeans[i] = latents[i].mean_const;
  CU(b_means.alloc(ctx, (size_t)m * sizeof(double)));
  CU(copy_in(ctx, b_means.as<double>(), hmeans.data(), (size_t)m));
  CU(b_ty.alloc(ctx, (size_t)m * npad * sizeof(double)));
  CU(cudaMemsetAsync(b_ty.p, 0, (size_t)m * npad * sizeof(double), st));
  const int nblk = project_max_partials(N);
  CU(b_part.alloc(ctx, (size_t)nblk * sizeof(double)));
  CU(cudaMemsetAsync(b_part.p, 0, (size_t)nblk * sizeof(double), st));
  CU(b_resid.alloc(ctx, sizeof(double)));
  CU(b_terms.alloc(ctx, (size_t)(units + 1) * sizeof(double)));
  CU(cudaMemsetAsync(b_terms.p, 0, (size_t)(units + 1) * sizeof(double), st));
  const bool do_reg = ctx->rank == 0;
  CU(launch_project(st, d_y, N, p, b_T.as<double>(), m, 0, m, b_means.as<double>(), b_ty.as<double>(), npad,
                    do_reg ? b_Pm.as<double>() : nullptr, do_reg ? b_Q.as<double>() : nullptr, b_part.as<double>(), nullptr));
  ++ctx->launches;
  if (do_reg) {
    CU(launch_sum_partials(st, b_part.as<double>(), nblk, b_resid.as<double>()));
    CU(launch_regulariser(st, b_terms.as<double>() + units, pr.reg_c0, b_resid.as<double>(), sigma2));
    ctx->launches += 2;
  }
  std::vector<int> hinfo(nu > 0 ? nu : 1, 0);
  if (nu > 0) {
    int chunk = 0;
    CU(mem_fit(ctx, (factor_bytes_per_latent(nt) + 4 * npad * sizeof(double)), nu, &chunk));
    DevBuf b_L, b_W, b_r, b_z, b_logdet, b_quad, b_info, b_params, b_idx;
    CU(b_L.alloc(ctx, (size_t)chunk * sym_tiles(nt) * TT * sizeof(double)));
    CU(b_W.alloc(ctx, (size_t)chunk * nt * TT * sizeof(double)));
    CU(b_r.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    CU(b_z.alloc(ctx, (size_t)chunk * npad * sizeof(double)));
    CU(b_logdet.alloc(ctx, (size_t)nu * sizeof(double)));
    CU(b_quad.alloc(ctx, (size_t)nu * sizeof(double)));
    CU(b_info.alloc(ctx, (size_t)nu * sizeof(int)));
    CU(cudaMemsetAsync(b_logdet.p, 0, (size_t)nu * sizeof(double), st));
    CU(cudaMemsetAsync(b_info.p, 0, (size_t)nu * sizeof(int), st));
    std::vector<LatentParams> hp(nu);
    std::vector<int> hidx(nu);
    for (int u = ulo; u < uhi; ++u) {
      const int s = u / m, i = u % m;
      LatentParams& q = hp[u - ulo];
      set_params(q, latents[i], pr.noise[i], inv_lengthscale_scales[s], D);
      hidx[u - ulo] = i;
    }
    CU(b_params.alloc(ctx, (size_t)nu * sizeof(LatentParams)));
    CU(cudaMemcpyAsync(b_params.p, hp.data(), (size_t)nu * sizeof(LatentParams), cudaMemcpyHostToDevice, st));
    CU(b_idx.alloc(ctx, (size_t)nu * sizeof(int)));
    CU(cudaMemcpyAsync(b_idx.p, hidx.data(), (size_t)nu * sizeof(int), cudaMemcpyHostToDevice, st));
    for (int c0 = 0; c0 < nu; c0 += chunk) {
      const int nb = (c0 + chunk <= nu) ? chunk : nu - c0;
      TiledSym L{b_L.as<double>(), nt, sym_tiles(nt) * TT};
      CU(launch_kmat_sym(st, L, nb, b_x.as<double>(), N, D, b_params.as<LatentParams>() + c0, ctx->distance_form));
      CU(chol_factor(ctx, L, b_W.as<double>(), (size_t)nt * TT, nb, b_logdet.as<double>() + c0, b_info.as<int>() + c0));
      CU(launch_gather_rows(st, b_r.as<double>(), b_ty.as<double>(), b_idx.as<int>() + c0, npad, nb));
      CU(launch_fwd_solve(st, L, b_W.as<double>(), (size_t)nt * TT, b_r.as<double>(), b_z.as<double>(), npad, nb, &ctx->launches));
      CU(launch_sumsq(st, b_z.as<double>(), npad, (int)npad, nb, b_quad.as<double>() + c0));
      CU(launch_lml_terms(st, b_terms.as<double>(), ulo + c0, nb, b_logdet.as<double>() + c0, b_quad.as<double>() + c0, N, LOG2PI));
      ctx->launches += 4;
    }
    CU(copy_out(ctx, hinfo.data(), b_info.p, (size_t)nu * sizeof(int)));
    CU(cudaStreamSynchronize(st));
  }
  if (ctx->comm && ctx->nranks > 1) {
    int r = nccl_api().AllReduce(b_terms.p, b_terms.p, (size_t)(units + 1), NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
    if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
  }
  std::vector<double> ht(units + 1, 0.0);
  CU(copy_out(ctx, ht.data(), b_terms.p, (size_t)(units + 1) * sizeof(double)));
  CU(cudaEventRecord(ctx->ev[1], st));
  CU(cudaStreamSynchronize(st));
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
  ctx->timings[0] = ms;
  {
    int unit = -1;
    const int rc_info = report_info(ctx, std::vector<int>(hinfo.begin(), hinfo.begin() + nu), ulo, N, &unit);  // collective
    if (rc_info) {
      if (info_latent) *info_latent = unit >= 0 ? unit % m : -1;
      if (rc_info > 0) {
        char buf[160];
        snprintf(buf, sizeof buf, "PosDefException in hyper-parameter sweep: latent %d at sweep point %d (pivot %d)", unit % m, unit / m, rc_info);
        ctx->err = buf;
      }
      return rc_info;
    }
  }
  if (info_latent) *info_latent = -1;
  for (int s = 0; s < n_sweep; ++s) {
    double acc = 0.0;
    for (int i = 0; i < m; ++i) acc += ht[(size_t)s * m + i];
    out_logpdfs[s] = acc + ht[units];
  }
  return LMM_OK;
}
