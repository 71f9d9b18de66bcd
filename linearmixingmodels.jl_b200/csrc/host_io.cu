// Serialisable posterior handles and the generic MVN logpdf / rand on an explicit (mean, covariance).
#include "host_internal.h"

// ------------------------------------------------------------------------------------------------
// Serialisable posterior (SURVEY.md §8f-3: the on-disk / wire format of the path's output).  The file is
// the handle's host metadata followed by its device arrays verbatim (tiled factor, inverse diagonal
// tiles, α, δ, inputs, per-point noise), little-endian Float64: loading needs no recomputation and the
// restored handle answers every lmm_post_* call bit-identically.  Multi-GPU: each rank saves / loads
// its own shard (the file records [lo, hi)).
// ------------------------------------------------------------------------------------------------
namespace lmm_host {
struct PostFileHeader {
  char magic[8];  // "LMMPOST3"
  int32_t kind, m, p, N, D, nt, lo, hi, big_n, big_nt, has_U, has_noise_vec, has_Ept, n_obs;  // n_obs: POST_MASKED observed entries (ints after the arrays)
  double sigma2;
  uint64_t n_x, n_L, n_W, n_alpha, n_delta, n_params, n_H, n_noise_vec, n_Ept;  // element counts (doubles; params: structs)
};

void post_array_sizes(const lmm_post* P, PostFileHeader& h) {
  const bool joint = P->joint();
  const int nloc = joint ? 1 : P->nloc();
  const int nt = joint ? P->big_nt : P->nt;
  const size_t vstride = (size_t)nt * TILE;
  h.n_x = joint ? (uint64_t)P->N * P->D : (uint64_t)P->npad() * P->D;
  h.n_L = (uint64_t)nloc * sym_tiles(nt) * TT;
  h.n_W = (uint64_t)nloc * nt * TT;
  h.n_alpha = (uint64_t)nloc * vstride;
  // the per-latent kinds allocate δ for max(nloc, 1) latents; the joint kinds one padded joint vector
  h.n_delta = (uint64_t)(joint ? 1 : (nloc > 0 ? nloc : 1)) * vstride;
  h.n_params = (uint64_t)(joint ? P->m : nloc);
  h.n_H = (uint64_t)P->p * P->m;
  h.n_noise_vec = P->d_noise_vec ? (uint64_t)(nloc > 0 ? nloc : 1) * vstride : 0;
  h.n_Ept = P->d_Ept ? (uint64_t)P->N * P->m * P->m : 0;
}

int stream_out(lmm_ctx* ctx, FILE* f, const void* dptr, size_t bytes) {
  const size_t CH = (size_t)64 << 20;
  std::vector<char> buf(bytes < CH ? bytes : CH);
  for (size_t off = 0; off < bytes; off += CH) {
    const size_t n = bytes - off < CH ? bytes - off : CH;
    CU(cudaMemcpyAsync(buf.data(), (const char*)dptr + off, n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->d2h += (int64_t)n;
    if (fwrite(buf.data(), 1, n, f) != n) return ctx->fail(LMM_E_ARG, "short write while saving a posterior");
  }
  return LMM_OK;
}
int stream_in(lmm_ctx* ctx, FILE* f, void* dptr, size_t bytes) {
  const size_t CH = (size_t)64 << 20;
  std::vector<char> buf(bytes < CH ? bytes : CH);
  for (size_t off = 0; off < bytes; off += CH) {
    const size_t n = bytes - off < CH ? bytes - off : CH;
    if (fread(buf.data(), 1, n, f) != n) return ctx->fail(LMM_E_ARG, "truncated posterior file");
    CU(cudaMemcpyAsync((char*)dptr + off, buf.data(), n, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->h2d += (int64_t)n;
  }
  return LMM_OK;
}
}  // namespace lmm_host

extern "C" int lmm_post_save(lmm_post* post, const char* path) {
  if (!post || !path) return LMM_E_ARG;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (post->kind == POST_VFE) return ctx->fail(LMM_E_UNSUPPORTED, VFE_POST_ONLY);
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  FILE* f = fopen(path, "wb");
  if (!f) return ctx->fail(LMM_E_ARG, std::string("cannot open ") + path + " for writing");
  PostFileHeader h{};
  memcpy(h.magic, "LMMPOST3", 8);
  h.kind = post->kind; h.m = post->m; h.p = post->p; h.N = post->N; h.D = post->D; h.nt = post->nt; h.lo = post->lo; h.hi = post->hi;
  h.big_n = post->big_n; h.big_nt = post->big_nt; h.has_U = post->U.empty() ? 0 : 1;
  h.has_noise_vec = post->d_noise_vec ? 1 : 0; h.has_Ept = post->d_Ept ? 1 : 0;
  h.n_obs = post->kind == POST_MASKED ? post->big_n : 0;
  h.sigma2 = post->sigma2;
  post_array_sizes(post, h);
  int rc = LMM_OK;
  bool ok = fwrite(&h, sizeof h, 1, f) == 1 && fwrite(post->descs.data(), sizeof(lmm_gp_desc), post->m, f) == (size_t)post->m &&
            fwrite(post->noise.data(), sizeof(double), post->m, f) == (size_t)post->m &&
            fwrite(post->H.data(), sizeof(double), post->H.size(), f) == post->H.size();
  // the descriptions hold host pointers (ARD vectors): the file carries the vectors and re-points on load (a non-null
  // pointer in the raw desc only marks "this latent has one")
  if (ok) ok = fwrite(post->ard_store.data(), sizeof(double), post->ard_store.size(), f) == post->ard_store.size();
  // composite kernels: the extra terms and their ARD vectors, fixed-size blocks (m x 3 terms, m x 3 x D multipliers)
  if (ok) ok = fwrite(post->term_store.data(), sizeof(lmm_kernel_term), post->term_store.size(), f) == post->term_store.size() &&
               fwrite(post->term_ard_store.data(), sizeof(double), post->term_ard_store.size(), f) == post->term_ard_store.size();
  if (ok && h.has_U)
    ok = fwrite(post->U.data(), sizeof(double), post->U.size(), f) == post->U.size() &&
         fwrite(post->S.data(), sizeof(double), post->S.size(), f) == post->S.size();
  if (!ok) rc = ctx->fail(LMM_E_ARG, "short write while saving a posterior");
  const void* arrs[] = {post->d_xpad, post->d_L, post->d_W, post->d_alpha, post->d_delta, post->d_params, post->d_H, post->d_noise_vec, post->d_Ept};
  const uint64_t cnt[] = {h.n_x, h.n_L, h.n_W, h.n_alpha, h.n_delta, h.n_params, h.n_H, h.n_noise_vec, h.n_Ept};
  for (int k = 0; k < 9 && rc == LMM_OK; ++k) {
    const size_t bytes = (size_t)cnt[k] * (k == 5 ? sizeof(LatentParams) : sizeof(double));
    if (bytes && arrs[k]) rc = stream_out(ctx, f, arrs[k], bytes);
  }
  if (rc == LMM_OK && h.n_obs > 0) rc = stream_out(ctx, f, post->d_obs, (size_t)h.n_obs * sizeof(int));
  if (fclose(f) != 0 && rc == LMM_OK) rc = ctx->fail(LMM_E_ARG, "close failed while saving a posterior");
  return rc;
}

extern "C" int lmm_post_load(lmm_ctx* ctx, const char* path, lmm_post** out_post) {
  if (!ctx || !path || !out_post) return LMM_E_ARG;
  *out_post = nullptr;
  std::lock_guard<std::mutex> lk(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  FILE* f = fopen(path, "rb");
  if (!f) return ctx->fail(LMM_E_ARG, std::string("cannot open ") + path);
  PostFileHeader h{};
  auto bail = [&](const char* msg) {
    fclose(f);
    return ctx->fail(LMM_E_ARG, msg);
  };
  if (fread(&h, sizeof h, 1, f) != 1 || memcmp(h.magic, "LMMPOST3", 8) != 0) return bail("not a liblmm posterior file");
  if (h.kind < POST_OILMM || h.kind > POST_MASKED || (h.kind == POST_MASKED) != (h.n_obs > 0) || (h.kind == POST_MASKED && h.n_obs != h.big_n) || h.m <= 0 || h.p <= 0 || h.N <= 0 || h.D <= 0 || h.lo < 0 || h.hi < h.lo || h.hi > h.m)
    return bail("corrupt posterior header");
  lmm_post* P = new lmm_post();
  P->ctx = ctx; P->kind = h.kind; P->m = h.m; P->p = h.p; P->N = h.N; P->D = h.D; P->nt = h.nt; P->lo = h.lo; P->hi = h.hi;
  P->big_n = h.big_n; P->big_nt = h.big_nt; P->sigma2 = h.sigma2;
  P->descs.resize(h.m); P->noise.resize(h.m); P->H.resize((size_t)h.p * h.m);
  bool ok = fread(P->descs.data(), sizeof(lmm_gp_desc), h.m, f) == (size_t)h.m && fread(P->noise.data(), sizeof(double), h.m, f) == (size_t)h.m &&
            fread(P->H.data(), sizeof(double), P->H.size(), f) == P->H.size();
  if (ok) {
    P->ard_store.resize((size_t)h.m * h.D);
    ok = fread(P->ard_store.data(), sizeof(double), P->ard_store.size(), f) == P->ard_store.size();
    if (ok) {
      constexpr int XT = LMM_MAX_TERMS - 1;
      P->term_store.resize((size_t)h.m * XT);
      P->term_ard_store.resize((size_t)h.m * XT * h.D);
      ok = fread(P->term_store.data(), sizeof(lmm_kernel_term), P->term_store.size(), f) == P->term_store.size() &&
           fread(P->term_ard_store.data(), sizeof(double), P->term_ard_store.size(), f) == P->term_ard_store.size();
      for (int i = 0; ok && i < h.m; ++i)
        if (P->descs[i].n_extra < 0 || P->descs[i].n_extra > XT) ok = false;
    }
    if (ok) P->repoint_descs(h.D);
  }
  if (ok && h.has_U) {
    P->U.resize((size_t)h.p * h.m); P->S.resize(h.m);
    ok = fread(P->U.data(), sizeof(double), P->U.size(), f) == P->U.size() && fread(P->S.data(), sizeof(double), P->S.size(), f) == P->S.size();
  }
  PostFileHeader chk = h;
  if (ok) {
    // the array sizes follow from the metadata: a file whose counts disagree is rejected before any allocation
    P->d_noise_vec = h.has_noise_vec ? (double*)1 : nullptr;
    P->d_Ept = h.has_Ept ? (double*)1 : nullptr;
    post_array_sizes(P, chk);
    P->d_noise_vec = nullptr;
    P->d_Ept = nullptr;
    ok = chk.n_x == h.n_x && chk.n_L == h.n_L && chk.n_W == h.n_W && chk.n_alpha == h.n_alpha && chk.n_delta == h.n_delta &&
         chk.n_params == h.n_params && chk.n_H == h.n_H && chk.n_noise_vec == h.n_noise_vec && chk.n_Ept == h.n_Ept &&
         h.nt == ntiles(h.N) && (!P->joint() || (h.big_nt == ntiles(h.big_n) && h.big_n > 0));
  }
  if (!ok) {
    delete P;
    return bail("corrupt or truncated posterior file");
  }
  void** slots[] = {(void**)&P->d_xpad, (void**)&P->d_L, (void**)&P->d_W, (void**)&P->d_alpha, (void**)&P->d_delta, (void**)&P->d_params,
                    (void**)&P->d_H, (void**)&P->d_noise_vec, (void**)&P->d_Ept};
  const uint64_t cnt[] = {h.n_x, h.n_L, h.n_W, h.n_alpha, h.n_delta, h.n_params, h.n_H, h.n_noise_vec, h.n_Ept};
  int rc = LMM_OK;
  size_t total = 0;
  for (int k = 0; k < 9 && rc == LMM_OK; ++k) {
    size_t bytes = (size_t)cnt[k] * (k == 5 ? sizeof(LatentParams) : sizeof(double));
    if (k == 7 && !h.has_noise_vec) continue;
    if (k == 8 && !h.has_Ept) continue;
    total += bytes;
    void* d = nullptr;
    cudaError_t e = cudaMallocAsync(&d, bytes ? bytes + (k == 5 ? sizeof(LatentParams) : 0) : 8, ctx->stream);
    if (e != cudaSuccess) {
      rc = ctx->fail_cuda(e, "cudaMallocAsync (posterior load)", __LINE__);
      break;
    }
    *slots[k] = d;
    if (bytes) rc = stream_in(ctx, f, d, bytes);
  }
  if (rc == LMM_OK && h.n_obs > 0) {  // missing-data posterior: the list of observed entries
    void* d = nullptr;
    cudaError_t e = cudaMallocAsync(&d, (size_t)h.n_obs * sizeof(int), ctx->stream);
    if (e != cudaSuccess) rc = ctx->fail_cuda(e, "cudaMallocAsync (posterior load)", __LINE__);
    else {
      P->d_obs = (int*)d;
      total += (size_t)h.n_obs * sizeof(int);
      rc = stream_in(ctx, f, d, (size_t)h.n_obs * sizeof(int));
    }
  }
  fclose(f);
  if (rc != LMM_OK) {
    if (P->d_obs) cudaFreeAsync(P->d_obs, ctx->stream);
    for (void** sl : slots)
      if (*sl) cudaFreeAsync(*sl, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    delete P;
    return rc;
  }
  P->bytes = total;
  *out_post = P;
  return LMM_OK;
}
// ------------------------------------------------------------------------------------------------
// AbstractGPs generic FiniteGP verbs on an explicit (mean, covariance): `logpdf(fx, y)` =
// -(n log 2π + logdet C + |C.U'^{-1}(y - m)|²)/2 and `rand(rng, fx)` = m + C.U' z with
// C = cholesky(Symmetric(cov)).  Used for FiniteGPs the fast paths do not cover (a posterior evaluated
// under a vector / dense Σy, test/independent_mogp.jl:120-133): mean_and_cov comes from the library,
// the dense factorisation and solve stay on the device too.
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_mvn_logpdf_rand(lmm_ctx* ctx, const double* mean, const double* cov, int n, const double* y, double* out_logpdf,
                                   const double* z, double* out_sample, int* info) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!mean || !cov || n <= 0 || (!(y && out_logpdf) && !(z && out_sample))) return ctx->fail(LMM_E_ARG, "null pointer or non-positive size");
  if (n > 46000) return ctx->fail(LMM_E_UNSUPPORTED, "dense covariance too large");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int nt = ntiles(n);
  const size_t npad = (size_t)nt * TILE, wstride = (size_t)nt * TT;
  DevBuf b_A, b_L, b_W, b_logdet, b_info, b_m, b_r, b_z, b_quad, b_s;
  const double* dA = cov;
  if (!is_device_ptr(cov)) {
    CU(b_A.alloc(ctx, (size_t)n * n * sizeof(double)));
    CU(copy_in(ctx, b_A.as<double>(), cov, (size_t)n * n));
    dA = b_A.as<double>();
  }
  CU(b_L.alloc(ctx, sym_tiles(nt) * TT * sizeof(double)));
  CU(b_W.alloc(ctx, (size_t)nt * TT * sizeof(double)));
  CU(b_logdet.alloc(ctx, sizeof(double)));
  CU(b_info.alloc(ctx, sizeof(int)));
  CU(cudaMemsetAsync(b_logdet.p, 0, sizeof(double), st));
  CU(cudaMemsetAsync(b_info.p, 0, sizeof(int), st));
  TiledSym L{b_L.as<double>(), nt, sym_tiles(nt) * TT};
  CU(launch_tile_from_dense(st, L, 1, dA, n));
  ++ctx->launches;
  CU(chol_factor(ctx, L, b_W.as<double>(), wstride, 1, b_logdet.as<double>(), b_info.as<int>()));
  CU(b_m.alloc(ctx, npad * sizeof(double)));
  CU(cudaMemsetAsync(b_m.p, 0, npad * sizeof(double), st));
  CU(copy_in(ctx, b_m.as<double>(), mean, (size_t)n));
  double hlogdet = 0.0, hquad = 0.0;
  int hinfo = 0;
  if (y && out_logpdf) {
    CU(b_r.alloc(ctx, npad * sizeof(double)));
    CU(b_z.alloc(ctx, npad * sizeof(double)));
    CU(b_quad.alloc(ctx, sizeof(double)));
    CU(cudaMemsetAsync(b_r.p, 0, npad * sizeof(double), st));
    CU(copy_in(ctx, b_r.as<double>(), y, (size_t)n));
    CU(launch_axpy(st, b_r.as<double>(), b_m.as<double>(), npad, -1.0));
    CU(launch_fwd_solve(st, L, b_W.as<double>(), wstride, b_r.as<double>(), b_z.as<double>(), npad, 1, &ctx->launches));
    CU(launch_sumsq(st, b_z.as<double>(), npad, (int)npad, 1, b_quad.as<double>()));
    ctx->launches += 2;
    CU(copy_out(ctx, &hquad, b_quad.p, sizeof(double)));
  }
  if (z && out_sample) {
    DevBuf b_zz;
    CU(b_zz.alloc(ctx, npad * sizeof(double)));
    CU(cudaMemsetAsync(b_zz.p, 0, npad * sizeof(double), st));
    CU(copy_in(ctx, b_zz.as<double>(), z, (size_t)n));
    CU(b_s.alloc(ctx, npad * sizeof(double)));
    CU(launch_lower_gemv(st, L, b_zz.as<double>(), npad, b_s.as<double>(), npad, 1));
    CU(launch_axpy(st, b_s.as<double>(), b_m.as<double>(), npad, 1.0));
    ctx->launches += 2;
    CU(copy_out(ctx, out_sample, b_s.p, (size_t)n * sizeof(double)));
    CU(cudaStreamSynchronize(st));  // b_zz goes out of scope
  }
  CU(copy_out(ctx, &hlogdet, b_logdet.p, sizeof(double)));
  CU(copy_out(ctx, &hinfo, b_info.p, sizeof(int)));
  CU(cudaStreamSynchronize(st));
  if (hinfo > 0) {
    if (info) *info = hinfo > n ? n : hinfo;
    ctx->err = "PosDefException: the covariance is not positive definite";
    return hinfo > n ? n : hinfo;
  }
  if (info) *info = 0;
  if (y && out_logpdf) *out_logpdf = -((double)n * LOG2PI + hlogdet + hquad) / 2.0;
  return LMM_OK;
}
