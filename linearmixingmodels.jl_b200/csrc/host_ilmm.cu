// General-H ILMM (src/ilmm.jl): projection, the joint (mN) factor, posterior, marginals, dense covariances, joint
// predictive rand / logpdf, sequential conditioning; IndependentMOGP under a vector / dense Σy.
#include "host_internal.h"

// ------------------------------------------------------------------------------------------------
// General-H ILMM (src/ilmm.jl)
// ------------------------------------------------------------------------------------------------
namespace lmm_host {

// Small dense host helpers (m x m, column-major) for `project` src/ilmm.jl:61-68.
bool host_chol(std::vector<double>& A, int n) {  // in place, lower
  for (int j = 0; j < n; ++j) {
    double d = A[(size_t)j * n + j];
    for (int k = 0; k < j; ++k) d -= A[(size_t)k * n + j] * A[(size_t)k * n + j];
    if (!(d > 0.0)) return false;
    d = std::sqrt(d);
    A[(size_t)j * n + j] = d;
    for (int i = j + 1; i < n; ++i) {
      double s = A[(size_t)j * n + i];
      for (int k = 0; k < j; ++k) s -= A[(size_t)k * n + i] * A[(size_t)k * n + j];
      A[(size_t)j * n + i] = s / d;
    }
  }
  return true;
}
void host_chol_solve(const std::vector<double>& L, int n, double* b) {  // solves (L L') x = b
  for (int i = 0; i < n; ++i) {
    double s = b[i];
    for (int k = 0; k < i; ++k) s -= L[(size_t)k * n + i] * b[k];
    b[i] = s / L[(size_t)i * n + i];
  }
  for (int i = n - 1; i >= 0; --i) {
    double s = b[i];
    for (int k = i + 1; k < n; ++k) s -= L[(size_t)i * n + k] * b[k];
    b[i] = s / L[(size_t)i * n + i];
  }
}


// T = chol(H'H/σ² + 1e-9 I) \ H' * (1/σ²) ;  ΣT = T (σ² I) T'      src/ilmm.jl:62-65
int general_projection(lmm_ctx* ctx, const double* H, int p, int m, double sigma2, int N, GeneralProjection& gp) {
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  const double inv = 1.0 / sigma2;
  std::vector<double> A((size_t)m * m);
  for (int a = 0; a < m; ++a)
    for (int b = 0; b < m; ++b) {
      double s = 0.0;
      for (int j = 0; j < p; ++j) s += (H[(size_t)a * p + j] * inv) * H[(size_t)b * p + j];
      A[(size_t)b * m + a] = s + (a == b ? 1e-9 : 0.0);
    }
  if (!host_chol(A, m)) return ctx->fail(LMM_E_ARG, "H'H/σ² + 1e-9 I is not positive definite");
  gp.pr.T.assign((size_t)m * p, 0.0);
  std::vector<double> col(m);
  gp.Winv.assign((size_t)m * m, 0.0);
  for (int b = 0; b < m; ++b) {
    gp.Winv[(size_t)b * m + b] = 1.0;
    host_chol_solve(A, m, gp.Winv.data() + (size_t)b * m);
  }
  for (int j = 0; j < p; ++j) {
    for (int a = 0; a < m; ++a) col[a] = H[(size_t)a * p + j];
    host_chol_solve(A, m, col.data());
    for (int a = 0; a < m; ++a) gp.pr.T[(size_t)j * m + a] = col[a] * inv;
  }
  gp.ST.assign((size_t)m * m, 0.0);
  for (int a = 0; a < m; ++a)
    for (int b = 0; b < m; ++b) {
      double s = 0.0;
      for (int j = 0; j < p; ++j) s += (gp.pr.T[(size_t)j * m + a] * sigma2) * gp.pr.T[(size_t)j * m + b];
      gp.ST[(size_t)b * m + a] = s;
    }
  std::vector<double> C = gp.ST;
  if (!host_chol(C, m)) return ctx->fail(LMM_E_ARG, "projected noise ΣT is not positive definite");
  gp.logdet_ST = 0.0;
  for (int a = 0; a < m; ++a) gp.logdet_ST += 2.0 * std::log(C[(size_t)a * m + a]);
  gp.pr.P = gp.pr.T;
  gp.pr.Q.assign(H, H + (size_t)p * m);
  gp.pr.noise.assign(m, 0.0);
  gp.pr.has_reg = true;
  // -(n((p-m) log 2π + (p log σ² - logdet ΣT)) + Σ|Y - HTY|²/σ²)/2      src/ilmm.jl:179-180
  gp.pr.reg_c0 = (double)N * ((double)(p - m) * LOG2PI + ((double)p * std::log(sigma2) - gp.logdet_ST));
  return LMM_OK;
}

// POST_JOINT (IndependentMOGP under the AbstractGPs generic path): no projection -- T = I, ΣT = σ² I, regulariser 0.
void identity_projection(int m, double sigma2, GeneralProjection& gp) {
  gp.pr.T.assign((size_t)m * m, 0.0);
  gp.ST.assign((size_t)m * m, 0.0);
  for (int a = 0; a < m; ++a) {
    gp.pr.T[(size_t)a * m + a] = 1.0;
    gp.ST[(size_t)a * m + a] = sigma2;
  }
  gp.Winv = gp.pr.T;
  gp.pr.P = gp.pr.T;
  gp.pr.Q = gp.pr.T;
  gp.pr.noise.assign(m, 0.0);
  gp.pr.has_reg = true;
  gp.pr.reg_c0 = 0.0;
  gp.logdet_ST = (double)m * std::log(sigma2);
}

// C (ra x cb, col-major) = op(A) * op(B) for tiny host matrices: A is ar x ac, B is br x bc.
std::vector<double> hmm(const std::vector<double>& A, int ar, int ac, bool ta, const std::vector<double>& B, int br, int bc, bool tb) {
  const int r = ta ? ac : ar, k = ta ? ar : ac, c = tb ? br : bc;
  std::vector<double> C((size_t)r * c, 0.0);
  for (int j = 0; j < c; ++j)
    for (int l = 0; l < k; ++l) {
      const double b = tb ? B[(size_t)l * br + j] : B[(size_t)j * br + l];
      if (b == 0.0) continue;
      for (int i = 0; i < r; ++i) C[(size_t)j * r + i] += (ta ? A[(size_t)i * ar + l] : A[(size_t)l * ar + i]) * b;
    }
  return C;
}
double hdot(const std::vector<double>& A, const std::vector<double>& B) {
  double s = 0.0;
  for (size_t i = 0; i < A.size(); ++i) s += A[i] * B[i];
  return s;
}

// Host chain of the general-ILMM gradient (all m x m / m x p, column-major): from the device-side
// cotangents B = d lml/dΣT (block traces of G), bT = direct d/dT, bH = direct d/dH and |R|² to
// d/dσ² and d/dH through ΣT = σ² T T', T = W H'/σ², W = (H'H/σ² + 1e-9 I)^{-1}  (src/ilmm.jl:61-68).
int ilmm_grad_chain(lmm_ctx* ctx, const GeneralProjection& gp, const std::vector<double>& Hh, int p, int m, int N, double sigma2,
                    double hres, const std::vector<double>& B, std::vector<double> bT, const std::vector<double>& bH,
                    double* grad_sigma2, double* grad_H) {
  const size_t npm = (size_t)p * m;
  const std::vector<double>& T = gp.pr.T;    // m x p
  const std::vector<double>& Wi = gp.Winv;   // m x m
  std::vector<double> STinv = gp.ST;
  if (!host_chol(STinv, m)) return ctx->fail(LMM_E_ARG, "projected noise ΣT is not positive definite");
  std::vector<double> bST = B;  // dΣT = B + (N/2) ΣT^{-1}
  {
    std::vector<double> col(m);
    for (int b = 0; b < m; ++b) {
      for (int a = 0; a < m; ++a) col[a] = (a == b) ? 1.0 : 0.0;
      host_chol_solve(STinv, m, col.data());
      for (int a = 0; a < m; ++a) bST[(size_t)b * m + a] += 0.5 * (double)N * col[a];
    }
  }
  double gs2 = -0.5 * ((double)N * (double)p / sigma2 - hres / (sigma2 * sigma2));
  const std::vector<double> TTt = hmm(T, m, p, false, T, m, p, true);  // m x m
  gs2 += hdot(bST, TTt);
  std::vector<double> bSTs(bST.size());
  for (int a = 0; a < m; ++a)
    for (int b = 0; b < m; ++b) bSTs[(size_t)b * m + a] = sigma2 * (bST[(size_t)b * m + a] + bST[(size_t)a * m + b]);
  const std::vector<double> add = hmm(bSTs, m, m, false, T, m, p, false);  // m x p
  for (size_t i = 0; i < npm; ++i) bT[i] += add[i];
  gs2 -= hdot(bT, T) / sigma2;
  const std::vector<double> Zm0 = hmm(bT, m, p, false, Hh, p, m, false);  // bT H : m x m
  std::vector<double> bM = hmm(hmm(Wi, m, m, false, Zm0, m, m, false), m, m, false, Wi, m, m, false);
  for (double& v : bM) v = -v / sigma2;  // bM = -W (bT H / σ²) W
  const std::vector<double> HtH = hmm(Hh, p, m, true, Hh, p, m, false);
  gs2 -= hdot(bM, HtH) / (sigma2 * sigma2);
  if (grad_sigma2) *grad_sigma2 = gs2;
  if (grad_H) {
    const std::vector<double> t1 = hmm(bT, m, p, true, Wi, m, m, false);  // bT' W : p x m
    std::vector<double> bMs(bM.size());
    for (int a = 0; a < m; ++a)
      for (int b = 0; b < m; ++b) bMs[(size_t)b * m + a] = bM[(size_t)b * m + a] + bM[(size_t)a * m + b];
    const std::vector<double> t2 = hmm(Hh, p, m, false, bMs, m, m, false);  // H (bM + bM') : p x m
    for (size_t i = 0; i < npm; ++i) grad_H[i] = bH[i] + (t1[i] + t2[i]) / sigma2;
  }
  return LMM_OK;
}


// Returns LMM_OK, a positive pivot (PosDefException) or a negative error.  Stage timings [1] assemble,
// [2] Cholesky, [3] solves are written to ctx->timings.
// logpdf-only evaluation with the joint matrix DISTRIBUTED over the ranks (option "partition_ilmm" = 2): this rank assembles
// and stores only the tile rows it owns (1/G of the matrix), the right-hand side rides along as one extra tile row, and
// chol_factor_rowcyclic_dist leaves logdet (every rank) and z = L^{-1} δ (every rank) -- no full copy of the matrix
// exists anywhere, so a joint dimension that does not fit one GPU runs.  Same outputs and stage timings as joint_factor.
static int joint_factor_distributed(lmm_ctx* ctx, JointBuild& J, int* info) {
  cudaStream_t st = ctx->stream;
  const int G = ctx->nranks, me = ctx->rank, nc = J.bnt, nrows = nc + 1;
  const size_t own_tiles = cyc_tiles(nrows, G, me);
  const size_t ws_tiles = rowcyclic_dist_workspace_tiles(nrows, G, rowcyclic_dist_block(ctx, nc));
  DevBuf b_z;
  CU(J.L.alloc(ctx, (own_tiles > 0 ? own_tiles : 1) * TT * sizeof(double)));
  CU(J.W.alloc(ctx, (size_t)nc * TT * sizeof(double)));
  CU(J.logdet.alloc(ctx, sizeof(double)));
  CU(J.info.alloc(ctx, sizeof(int)));
  CU(J.quad.alloc(ctx, sizeof(double)));
  CU(b_z.alloc(ctx, J.bpad * sizeof(double)));
  CU(cudaMemsetAsync(J.logdet.p, 0, sizeof(double), st));
  CU(cudaMemsetAsync(J.info.p, 0, sizeof(int), st));
  TiledSym Lown{J.L.as<double>(), nc, 0};
  Lown.cyc_G = G; Lown.cyc_r = me;
  CU(cudaEventRecord(ctx->ev[1], st));
  CU(launch_assemble_ilmm(st, Lown, J.x.as<double>(), J.N, J.D, J.params.as<LatentParams>(), J.m, J.q, J.E.as<double>(), J.H.as<double>(),
                          J.mode, ctx->distance_form));
  ++ctx->launches;
  if (nc % G == me) {  // the owner of the extra tile row writes the right-hand side
    CU(launch_rhs_row(st, Lown, nc, J.delta.as<double>()));
    ++ctx->launches;
  }
  CU(cudaEventRecord(ctx->ev[2], st));
  Lown.nt = nrows;
  CU(chol_factor_rowcyclic_dist(ctx, Lown, nrows, nc, J.W.as<double>(), (size_t)nc * TT, J.logdet.as<double>(), J.info.as<int>(), b_z.as<double>()));
  CU(cudaEventRecord(ctx->ev[3], st));
  CU(launch_sumsq(st, b_z.as<double>(), J.bpad, (int)J.bpad, 1, J.quad.as<double>()));
  ++ctx->launches;
  int hinfo = 0;
  CU(copy_out(ctx, &J.hlogdet, J.logdet.p, sizeof(double)));
  CU(copy_out(ctx, &J.hquad, J.quad.p, sizeof(double)));
  CU(copy_out(ctx, &hinfo, J.info.p, sizeof(int)));
  CU(cudaEventRecord(ctx->ev[4], st));
  CU(cudaStreamSynchronize(st));
  {
    float a = 0, b = 0, c = 0, d = 0;
    cudaEventElapsedTime(&a, ctx->ev[0], ctx->ev[4]);
    cudaEventElapsedTime(&b, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&c, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&d, ctx->ev[3], ctx->ev[4]);
    ctx->timings[0] = a; ctx->timings[1] = b; ctx->timings[2] = c; ctx->timings[3] = d;
    // memory of this evaluation, in bytes: the matrix rows this rank holds, its exchange / window workspace, the whole matrix
    const double tb = (double)TT * sizeof(double);
    ctx->timings[4] = (double)own_tiles * tb; ctx->timings[5] = (double)ws_tiles * tb; ctx->timings[7] = (double)sym_tiles(nc) * tb;
  }
  if (hinfo > 0) {
    if (info) *info = hinfo > J.big ? J.big : hinfo;
    ctx->err = "PosDefException: the joint covariance is not positive definite";
    return hinfo > J.big ? J.big : hinfo;
  }
  if (info) *info = 0;
  return LMM_OK;
}

int joint_factor(lmm_ctx* ctx, JointBuild& J, bool want_alpha, int* info) {
  cudaStream_t st = ctx->stream;
  if (!want_alpha && ctx->partition_ilmm == 2 && ctx->comm && ctx->nranks > 1 && J.bnt >= 2 * ctx->nranks && nccl_api().AllGather)
    return joint_factor_distributed(ctx, J, info);
  CU(J.L.alloc(ctx, sym_tiles(J.bnt) * TT * sizeof(double)));
  CU(J.W.alloc(ctx, (size_t)J.bnt * TT * sizeof(double)));
  CU(J.logdet.alloc(ctx, sizeof(double)));
  CU(J.info.alloc(ctx, sizeof(int)));
  CU(J.quad.alloc(ctx, sizeof(double)));
  CU(cudaMemsetAsync(J.logdet.p, 0, sizeof(double), st));
  CU(cudaMemsetAsync(J.info.p, 0, sizeof(int), st));
  TiledSym L{J.L.as<double>(), J.bnt, sym_tiles(J.bnt) * TT};
  const size_t wstride = (size_t)J.bnt * TT;
  CU(cudaEventRecord(ctx->ev[1], st));
  CU(launch_assemble_ilmm(st, L, J.x.as<double>(), J.N, J.D, J.params.as<LatentParams>(), J.m, J.q, J.E.as<double>(), J.H.as<double>(),
                          J.mode, ctx->distance_form));
  ++ctx->launches;
  CU(cudaEventRecord(ctx->ev[2], st));
  {
    PartitionScope scope(ctx);  // ILMM calls are replicated on every rank: the joint factor may be partitioned
    CU(chol_factor(ctx, L, J.W.as<double>(), wstride, 1, J.logdet.as<double>(), J.info.as<int>()));
  }
  CU(cudaEventRecord(ctx->ev[3], st));
  DevBuf b_r, b_z;
  CU(b_r.alloc(ctx, J.bpad * sizeof(double)));
  CU(b_z.alloc(ctx, J.bpad * sizeof(double)));
  CU(cudaMemcpyAsync(b_r.p, J.delta.p, J.bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(launch_fwd_solve(st, L, J.W.as<double>(), wstride, b_r.as<double>(), b_z.as<double>(), J.bpad, 1, &ctx->launches));
  CU(launch_sumsq(st, b_z.as<double>(), J.bpad, (int)J.bpad, 1, J.quad.as<double>()));
  ++ctx->launches;
  if (want_alpha) {
    CU(J.alpha.alloc(ctx, J.bpad * sizeof(double)));
    CU(cudaMemcpyAsync(b_r.p, b_z.p, J.bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CU(launch_bwd_solve(st, L, J.W.as<double>(), wstride, b_r.as<double>(), J.alpha.as<double>(), J.bpad, 1, &ctx->launches));
  }
  int hinfo = 0;
  CU(copy_out(ctx, &J.hlogdet, J.logdet.p, sizeof(double)));
  CU(copy_out(ctx, &J.hquad, J.quad.p, sizeof(double)));
  CU(copy_out(ctx, &hinfo, J.info.p, sizeof(int)));
  CU(cudaEventRecord(ctx->ev[4], st));
  CU(cudaStreamSynchronize(st));
  {
    float a = 0, b = 0, c = 0, d = 0;
    cudaEventElapsedTime(&a, ctx->ev[0], ctx->ev[4]);
    cudaEventElapsedTime(&b, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&c, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&d, ctx->ev[3], ctx->ev[4]);
    ctx->timings[0] = a; ctx->timings[1] = b; ctx->timings[2] = c; ctx->timings[3] = d;
  }
  if (hinfo > 0) {
    if (info) *info = hinfo > J.big ? J.big : hinfo;
    ctx->err = "PosDefException: the joint covariance is not positive definite";
    return hinfo > J.big ? J.big : hinfo;
  }
  if (info) *info = 0;
  return LMM_OK;
}

// Ownership of the device buffers moves to the new handle (nothing here can fail).
lmm_post* joint_make_post(lmm_ctx* ctx, JointBuild& J, int kind, const lmm_gp_desc* latents, const double* Hhost, int p, double sigma2,
                          DevBuf& Ept) {
  lmm_post* P = new lmm_post();
  P->ctx = ctx; P->kind = kind; P->m = J.m; P->p = p; P->N = J.N; P->D = J.D; P->nt = ntiles(J.N); P->lo = 0; P->hi = J.m;
  P->adopt_descs(latents, J.m, J.D);
  P->noise.assign(J.m, 0.0);
  P->H.assign(Hhost, Hhost + (size_t)p * J.m);
  P->sigma2 = sigma2;
  P->big_n = J.big; P->big_nt = J.bnt;
  P->bytes = (sym_tiles(J.bnt) + J.bnt) * TT * sizeof(double) + 2 * J.bpad * sizeof(double);
  P->d_xpad = (double*)J.x.detach();  // unpadded [N][D] for the joint kinds
  P->d_L = (double*)J.L.detach();
  P->d_W = (double*)J.W.detach();
  P->d_alpha = (double*)J.alpha.detach();
  P->d_delta = (double*)J.delta.detach();
  P->d_params = (LatentParams*)J.params.detach();
  P->d_H = (double*)J.H.detach();
  P->d_Ept = (double*)Ept.detach();
  return P;
}



int ilmm_run(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H, int p, double sigma2,
             const double* y, int form, lmm_post** out_post, double* out_logpdf, int* info, const double* dense_noise) {
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  if (form != LMM_ILMM_FORM_PROJECTED && form != LMM_ILMM_FORM_DENSE && form != FORM_IMOGP_DENSE) return ctx->fail(LMM_E_ARG, "unknown ILMM form");
  if (out_post && form == LMM_ILMM_FORM_DENSE) return ctx->fail(LMM_E_UNSUPPORTED, "posterior uses the projected form");
  GeneralProjection gp;
  int rc;
  if (form != FORM_IMOGP_DENSE && (rc = general_projection(ctx, H, p, m, sigma2, N, gp))) return rc;
  JointBuild J;
  J.m = m; J.N = N; J.D = D;
  J.q = (form == LMM_ILMM_FORM_DENSE) ? p : m;
  const int64_t big64 = (int64_t)J.q * N;
  if (big64 > (1 << 20)) return ctx->fail(LMM_E_UNSUPPORTED, "joint dimension too large");
  J.big = (int)big64; J.bnt = ntiles(J.big); J.bpad = (size_t)J.bnt * TILE;
  CU(cudaEventRecord(ctx->ev[0], st));
  DevBuf b_y, b_T, b_Q, b_means, b_part, b_resid, b_Ept;
  CU(J.x.alloc(ctx, (size_t)N * D * sizeof(double)));
  CU(copy_in(ctx, J.x.as<double>(), x, (size_t)N * D));
  const double* d_y = y;
  if (!is_device_ptr(y)) {
    CU(b_y.alloc(ctx, (size_t)p * N * sizeof(double)));
    CU(copy_in(ctx, b_y.as<double>(), y, (size_t)p * N));
    d_y = b_y.as<double>();
  }
  std::vector<double> noise0(m, 0.0);
  if ((rc = upload_params(ctx, J.params, latents, noise0.data(), 0, m, D))) return rc;
  CU(J.H.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(copy_in(ctx, J.H.as<double>(), H, (size_t)p * m));
  CU(J.delta.alloc(ctx, J.bpad * sizeof(double)));
  CU(cudaMemsetAsync(J.delta.p, 0, J.bpad * sizeof(double), st));
  double reg = 0.0;
  if (form == LMM_ILMM_FORM_PROJECTED) {
    CU(b_T.alloc(ctx, gp.pr.T.size() * sizeof(double)));
    CU(copy_in(ctx, b_T.as<double>(), gp.pr.T.data(), gp.pr.T.size()));
    CU(b_Q.alloc(ctx, gp.pr.Q.size() * sizeof(double)));
    CU(copy_in(ctx, b_Q.as<double>(), gp.pr.Q.data(), gp.pr.Q.size()));
    std::vector<double> hmeans(m);
    for (int i = 0; i < m; ++i) hmeans[i] = latents[i].mean_const;
    CU(b_means.alloc(ctx, (size_t)m * sizeof(double)));
    CU(copy_in(ctx, b_means.as<double>(), hmeans.data(), (size_t)m));
    const int nblk = project_max_partials(N);
    CU(b_part.alloc(ctx, (size_t)nblk * sizeof(double)));
    CU(cudaMemsetAsync(b_part.p, 0, (size_t)nblk * sizeof(double), st));
    CU(b_resid.alloc(ctx, sizeof(double)));
    // δ = vec((TY)') - mean: latent-major with stride N (the joint vector is padded only at its end)
    CU(launch_project(st, d_y, N, p, b_T.as<double>(), m, 0, m, b_means.as<double>(), J.delta.as<double>(), (size_t)N,
                      b_T.as<double>(), b_Q.as<double>(), b_part.as<double>(), nullptr));
    CU(launch_sum_partials(st, b_part.as<double>(), nblk, b_resid.as<double>()));
    ctx->launches += 2;
    double hres = 0.0;
    CU(copy_out(ctx, &hres, b_resid.p, sizeof(double)));
    CU(cudaStreamSynchronize(st));
    reg = -(gp.pr.reg_c0 + hres / sigma2) / 2.0;
    CU(J.E.alloc(ctx, gp.ST.size() * sizeof(double)));
    CU(copy_in(ctx, J.E.as<double>(), gp.ST.data(), gp.ST.size()));
    J.mode = 0;
  } else {
    // dense forms: δ = y - (H ⊗ I) mean
    std::vector<double> hm(p, 0.0);
    for (int j = 0; j < p; ++j)
      for (int a = 0; a < m; ++a) hm[j] += H[(size_t)a * p + j] * latents[a].mean_const;
    CU(cudaMemcpyAsync(J.delta.p, d_y, (size_t)p * N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    for (int j = 0; j < p; ++j)
      if (hm[j] != 0.0) {
        CU(launch_add_scalar(st, J.delta.as<double>() + (size_t)j * N, (size_t)N, -hm[j]));
        ++ctx->launches;
      }
    if (form == LMM_ILMM_FORM_DENSE) {
      CU(J.E.alloc(ctx, sizeof(double)));
      CU(copy_in(ctx, J.E.as<double>(), &sigma2, 1));
      J.mode = 1;
    } else {
      CU(J.E.alloc(ctx, (size_t)J.big * J.big * sizeof(double)));
      CU(copy_in(ctx, J.E.as<double>(), dense_noise, (size_t)J.big * J.big));
      J.mode = 2;
    }
  }
  if ((rc = joint_factor(ctx, J, out_post != nullptr, info))) return rc;
  if (out_logpdf) *out_logpdf = -((double)J.big * LOG2PI + J.hlogdet + J.hquad) / 2.0 + reg;
  if (out_post) {
    if (form == LMM_ILMM_FORM_PROJECTED) {
      // per-point projected noise blocks (all equal to ΣT here): what sequential conditioning extends
      const size_t tot = (size_t)N * m * m;
      CU(b_Ept.alloc(ctx, tot * sizeof(double)));
      CU(launch_repeat_block(st, b_Ept.as<double>(), J.E.as<double>(), m * m, tot));
      ++ctx->launches;
      CU(cudaStreamSynchronize(st));
    }
    *out_post = joint_make_post(ctx, J, form == FORM_IMOGP_DENSE ? POST_JOINT : POST_ILMM, latents, H, p, sigma2, b_Ept);
  }
  return LMM_OK;
}

// mean_and_var of ILMM(PosteriorGP{IndependentMOGP}, H) at x*: src/ilmm.jl:108-129 (computed
// directly from the joint factor; never forms kron(H, I) nor factorises the latent covariance).
int ilmm_post_mean_and_var(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean, double* var) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p, N = post->N, D = post->D;
  const int ntr = ntiles(m * Ns), bnt = post->big_nt;
  DevBuf b_xs, b_V, b_ml, b_out;
  CU(b_xs.alloc(ctx, (size_t)Ns * D * sizeof(double)));
  CU(copy_in(ctx, b_xs.as<double>(), xs, (size_t)Ns * D));
  CU(b_V.alloc(ctx, (size_t)ntr * bnt * TT * sizeof(double)));
  TiledRect V{b_V.as<double>(), ntr, bnt, (size_t)ntr * bnt * TT};
  CU(launch_assemble_cross_blockdiag(st, V, b_xs.as<double>(), Ns, post->d_xpad, N, D, post->d_params, m, ctx->distance_form));
  CU(b_ml.alloc(ctx, (size_t)ntr * TILE * sizeof(double)));
  CU(launch_rect_gemv(st, V, post->d_alpha, (size_t)bnt * TILE, b_ml.as<double>(), (size_t)ntr * TILE, post->d_params, 0, 1));
  ctx->launches += 2;
  CU(trsm_right_lt(ctx, V, post->Lsym(), post->d_W, post->wstride(), 1));
  const size_t nout = (size_t)p * Ns;
  CU(b_out.alloc(ctx, 2 * nout * sizeof(double)));
  CU(launch_ilmm_predict(st, V, Ns, m, p, post->d_H, post->d_params, b_ml.as<double>(), sigma2, b_out.as<double>(),
                         b_out.as<double>() + nout));
  ++ctx->launches;
  CU(copy_out(ctx, mean, b_out.p, nout * sizeof(double)));
  CU(copy_out(ctx, var, b_out.as<double>() + nout, nout * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  return LMM_OK;
}

}  // namespace lmm_host

extern "C" int lmm_ilmm_logpdf(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H, int p,
                               double sigma2, const double* y, int out_dim, int form, double* out_logpdf, int* info) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!H || !y || !out_logpdf) return ctx->fail(LMM_E_ARG, "null pointer");
  return ilmm_run(ctx, latents, m, x, N, D, H, p, sigma2, y, form, nullptr, out_logpdf, info);
}

extern "C" int lmm_ilmm_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H,
                                  int p, double sigma2, const double* y, int out_dim, lmm_post** out_post, double* out_logpdf,
                                  int* info) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (out_post) *out_post = nullptr;
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!H || !y || !out_post) return ctx->fail(LMM_E_ARG, "null pointer");
  return ilmm_run(ctx, latents, m, x, N, D, H, p, sigma2, y, LMM_ILMM_FORM_PROJECTED, out_post, out_logpdf, info);
}

extern "C" int lmm_ilmm_prior_mean_and_var(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* xs, int Ns, int D,
                                           const double* H, int p, double sigma2, int out_dim, double* mean, double* var) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, xs, Ns, D, p, out_dim);
  if (rc) return rc;
  if (!H || !mean || !var) return ctx->fail(LMM_E_ARG, "null pointer");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // prior latent covariance is block diagonal: diag((H⊗I)(C_lat + 1e-18 I)(H⊗I)') = Σ_a H[j,a]² (k_a(x,x) + 1e-18)
  std::vector<double> ML((size_t)m * Ns), VL((size_t)m * Ns);
  for (int i = 0; i < m; ++i)
    for (int n = 0; n < Ns; ++n) {
      ML[(size_t)i * Ns + n] = latents[i].mean_const;
      VL[(size_t)i * Ns + n] = desc_kdiag(latents[i]);
    }
  DevBuf b_H, b_ML, b_VL, b_out;
  CU(b_H.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(copy_in(ctx, b_H.as<double>(), H, (size_t)p * m));
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

// ------------------------------------------------------------------------------------------------
// mean_and_cov / cov: dense (p Ns)^2 outputs (AbstractGPs API surface; src/ilmm.jl:132-139,147,
// src/independent_mogp.jl:60-63).  Meant for small Ns (the reference builds kron(H, I) here).
// ------------------------------------------------------------------------------------------------
namespace lmm_host {

int finish_cov(lmm_ctx* ctx, double* d_cov, double* d_mean, int dim, double sigma2, double* mean, double* cov) {
  cudaStream_t st = ctx->stream;
  if (ctx->comm && ctx->nranks > 1) {
    int r = nccl_api().AllReduce(d_cov, d_cov, (size_t)dim * dim, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
    if (r == 0 && d_mean) r = nccl_api().AllReduce(d_mean, d_mean, (size_t)dim, NCCL_DOUBLE, NCCL_SUM, ctx->comm, st);
    if (r != 0) return ctx->fail(LMM_E_NCCL, "ncclAllReduce failed");
  }
  CU(launch_add_diag(st, d_cov, dim, sigma2));
  ++ctx->launches;
  if (mean && d_mean) CU(copy_out(ctx, mean, d_mean, (size_t)dim * sizeof(double)));
  CU(copy_out(ctx, cov, d_cov, (size_t)dim * dim * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  return LMM_OK;
}

}  // namespace lmm_host

extern "C" int lmm_prior_mean_and_cov(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* xs, int Ns, int D, const double* H,
                                      int p, double sigma2, double latent_jitter, int out_dim, double* mean, double* cov) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  int rc = check_common(ctx, latents, m, xs, Ns, D, p, out_dim);
  if (rc) return rc;
  if (!H || !cov) return ctx->fail(LMM_E_ARG, "null pointer");
  if ((int64_t)p * Ns > 46000) return ctx->fail(LMM_E_UNSUPPORTED, "dense covariance output too large");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  int lo, hi;
  shard_range(ctx, m, lo, hi);
  const int nloc = hi - lo, nts = ntiles(Ns), dim = p * Ns;
  DevBuf b_xs, b_params, b_C, b_H, b_cov, b_mean;
  if ((rc = stage_xpad(ctx, b_xs, xs, Ns, D))) return rc;
  std::vector<double> noise(m, latent_jitter);
  if ((rc = upload_params(ctx, b_params, latents, noise.data(), lo, hi, D))) return rc;
  CU(b_C.alloc(ctx, (size_t)(nloc > 0 ? nloc : 1) * sym_tiles(nts) * TT * sizeof(double)));
  TiledSym C{b_C.as<double>(), nts, sym_tiles(nts) * TT};
  if (nloc > 0) {
    CU(launch_kmat_sym(st, C, nloc, b_xs.as<double>(), Ns, D, b_params.as<LatentParams>(), ctx->distance_form));
    ++ctx->launches;
  }
  CU(b_H.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(copy_in(ctx, b_H.as<double>(), H, (size_t)p * m));
  CU(b_cov.alloc(ctx, (size_t)dim * dim * sizeof(double)));
  CU(launch_mix_cov(st, C, nloc, lo, b_H.as<double>(), p, Ns, b_cov.as<double>()));
  ++ctx->launches;
  std::vector<double> hm((size_t)dim, 0.0);
  if (ctx->rank == 0 || !(ctx->comm && ctx->nranks > 1))
    for (int j = 0; j < p; ++j) {
      double s = 0.0;
      for (int a = 0; a < m; ++a) s += H[(size_t)a * p + j] * latents[a].mean_const;
      for (int n = 0; n < Ns; ++n) hm[(size_t)j * Ns + n] = s;
    }
  CU(b_mean.alloc(ctx, (size_t)dim * sizeof(double)));
  CU(copy_in(ctx, b_mean.as<double>(), hm.data(), (size_t)dim));
  return finish_cov(ctx, b_cov.as<double>(), b_mean.as<double>(), dim, sigma2, mean, cov);
}

extern "C" int lmm_post_mean_and_cov(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean, double* cov) {
  if (!post || !xs || Ns <= 0 || !cov) return LMM_E_ARG;
  lmm_ctx* ctx = post->ctx;
  std::lock_guard<std::mutex> lk(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  if (int rcz = post_fill_zeros(post)) return rcz;  // the factor is read below
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p, dim = p * Ns;
  if ((int64_t)p * Ns > 46000) return ctx->fail(LMM_E_UNSUPPORTED, "dense covariance output too large");
  DevBuf b_cov, b_mean;
  CU(b_cov.alloc(ctx, (size_t)dim * dim * sizeof(double)));
  CU(b_mean.alloc(ctx, 2 * (size_t)dim * sizeof(double)));
  CU(cudaMemsetAsync(b_mean.p, 0, 2 * (size_t)dim * sizeof(double), st));
  if (post->kind == POST_MASKED) return masked_post_mean_and_cov(post, xs, Ns, sigma2, mean, cov);
  if (post->joint()) {
    // joint latent posterior: C_lat = blockdiag(K**) + 1e-18 I - V V',  V = Kc L^{-T}
    const int N = post->N, D = post->D, bnt = post->big_nt, ntr = ntiles(m * Ns);
    DevBuf b_xs, b_V, b_Cl, b_E, b_ml;
    CU(b_xs.alloc(ctx, (size_t)Ns * D * sizeof(double)));
    CU(copy_in(ctx, b_xs.as<double>(), xs, (size_t)Ns * D));
    CU(b_V.alloc(ctx, (size_t)ntr * bnt * TT * sizeof(double)));
    TiledRect V{b_V.as<double>(), ntr, bnt, (size_t)ntr * bnt * TT};
    CU(launch_assemble_cross_blockdiag(st, V, b_xs.as<double>(), Ns, post->d_xpad, N, D, post->d_params, m, ctx->distance_form));
    CU(b_ml.alloc(ctx, (size_t)ntr * TILE * sizeof(double)));
    CU(launch_rect_gemv(st, V, post->d_alpha, (size_t)bnt * TILE, b_ml.as<double>(), (size_t)ntr * TILE, post->d_params, 0, 1));
    CU(trsm_right_lt(ctx, V, post->Lsym(), post->d_W, post->wstride(), 1));
    std::vector<double> E((size_t)m * m, 0.0);
    for (int a = 0; a < m; ++a) E[(size_t)a * m + a] = post->kind == POST_JOINT ? 0.0 : 1e-18;  // default FiniteGP noise, src/ilmm.jl:115
    CU(b_E.alloc(ctx, E.size() * sizeof(double)));
    CU(copy_in(ctx, b_E.as<double>(), E.data(), E.size()));
    CU(b_Cl.alloc(ctx, sym_tiles(ntr) * TT * sizeof(double)));
    TiledSym Cl{b_Cl.as<double>(), ntr, sym_tiles(ntr) * TT};
    CU(launch_assemble_ilmm(st, Cl, b_xs.as<double>(), Ns, D, post->d_params, m, m, b_E.as<double>(), post->d_H, 0, ctx->distance_form));
    GemmArgs g{};
    g.A = operand(V); g.B = operand(V); g.C = operand(Cl);
    g.i0 = 0; g.j0 = 0; g.k0 = 0; g.k1 = bnt; g.sym = 1;
    CU(launch_gemm(st, GEMM_UPDATE, g, ntr, ntr, 1));
    CU(launch_mix_cov_joint(st, Cl, m, post->d_H, p, Ns, b_cov.as<double>()));
    // mean: reuse the predictive kernel's formula on the host-visible pieces
    CU(launch_ilmm_predict(st, V, Ns, m, p, post->d_H, post->d_params, b_ml.as<double>(), sigma2, b_mean.as<double>(),
                           b_mean.as<double>() + dim));
    ctx->launches += 7;
    CU(launch_add_diag(st, b_cov.as<double>(), dim, sigma2));
    if (mean) CU(copy_out(ctx, mean, b_mean.p, (size_t)dim * sizeof(double)));
    CU(copy_out(ctx, cov, b_cov.p, (size_t)dim * dim * sizeof(double)));
    CU(cudaStreamSynchronize(st));
    return LMM_OK;
  }
  // independent posterior latents: C_a = K** - V V' + jitter I
  const bool oilmm = post->kind == POST_OILMM;
  std::vector<double> noise(m, oilmm ? 1e-18 : 0.0);
  Predictive P;
  int rc = build_predictive(post, xs, Ns, noise, P, nullptr, false);
  if (rc) return rc;
  const int nloc = post->nloc();
  TiledSym Call{P.C.as<double>(), P.nts, sym_tiles(P.nts) * TT};
  CU(launch_mix_cov(st, Call, nloc, post->lo, post->d_H, p, Ns, b_cov.as<double>()));
  ++ctx->launches;
  // mean = H M_lat (partial over resident latents)
  if (nloc > 0) {
    CU(launch_backproject(st, post->d_H, p, m, post->lo, nloc, P.ML.as<double>(), P.ML.as<double>(), P.nspad, Ns, 0.0, 0.0, 0,
                          b_mean.as<double>(), b_mean.as<double>() + dim));
    ++ctx->launches;
  }
  return finish_cov(ctx, b_cov.as<double>(), b_mean.as<double>(), dim, sigma2, mean, cov);
}

// ------------------------------------------------------------------------------------------------
// rand / logpdf on a general-ILMM posterior: ILMM(PosteriorGP{IndependentMOGP}, H)
//   rand   src/ilmm.jl:78-87 : latent = m* + chol(C* + 1e-12 I) z ; out = (H⊗I) latent + sqrt(σ²) ε
//   logpdf src/ilmm.jl:150-163: N(vec((TY*)') | m*, C* + ΣT ⊗ I) + regulariser
// with the joint latent posterior m* = m + Kc α, C* = blockdiag(K**) - V V', V = Kc L^{-T}.
// ------------------------------------------------------------------------------------------------
namespace lmm_host {

struct JointPredictive {
  DevBuf xs, V, ml, Cl, W, logdet, info, E;
  int ntr = 0;
};

// Builds m* (ml, length ntr*128, WITHOUT the prior means) and the Cholesky factor of C* + E ⊗ I.
int build_joint_predictive(lmm_post* post, const double* xs, int Ns, const std::vector<double>& E, JointPredictive& P, int* info) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  const int m = post->m, N = post->N, D = post->D, bnt = post->big_nt;
  P.ntr = ntiles(m * Ns);
  CU(P.xs.alloc(ctx, (size_t)Ns * D * sizeof(double)));
  CU(copy_in(ctx, P.xs.as<double>(), xs, (size_t)Ns * D));
  CU(P.V.alloc(ctx, (size_t)P.ntr * bnt * TT * sizeof(double)));
  TiledRect V{P.V.as<double>(), P.ntr, bnt, (size_t)P.ntr * bnt * TT};
  CU(launch_assemble_cross_blockdiag(st, V, P.xs.as<double>(), Ns, post->d_xpad, N, D, post->d_params, m, ctx->distance_form));
  CU(P.ml.alloc(ctx, (size_t)P.ntr * TILE * sizeof(double)));
  CU(launch_rect_gemv(st, V, post->d_alpha, (size_t)bnt * TILE, P.ml.as<double>(), (size_t)P.ntr * TILE, post->d_params, 0, 1));
  CU(trsm_right_lt(ctx, V, post->Lsym(), post->d_W, post->wstride(), 1));
  CU(P.E.alloc(ctx, E.size() * sizeof(double)));
  CU(copy_in(ctx, P.E.as<double>(), E.data(), E.size()));
  CU(P.Cl.alloc(ctx, sym_tiles(P.ntr) * TT * sizeof(double)));
  TiledSym Cl{P.Cl.as<double>(), P.ntr, sym_tiles(P.ntr) * TT};
  CU(launch_assemble_ilmm(st, Cl, P.xs.as<double>(), Ns, D, post->d_params, m, m, P.E.as<double>(), post->d_H, 0, ctx->distance_form));
  GemmArgs g{};
  g.A = operand(V); g.B = operand(V); g.C = operand(Cl);
  g.i0 = 0; g.j0 = 0; g.k0 = 0; g.k1 = bnt; g.sym = 1;
  CU(launch_gemm(st, GEMM_UPDATE, g, P.ntr, P.ntr, 1));
  ctx->launches += 4;
  CU(P.W.alloc(ctx, (size_t)P.ntr * TT * sizeof(double)));
  CU(P.logdet.alloc(ctx, sizeof(double)));
  CU(P.info.alloc(ctx, sizeof(int)));
  CU(cudaMemsetAsync(P.logdet.p, 0, sizeof(double), st));
  CU(cudaMemsetAsync(P.info.p, 0, sizeof(int), st));
  CU(chol_factor(ctx, Cl, P.W.as<double>(), (size_t)P.ntr * TT, 1, P.logdet.as<double>(), P.info.as<int>()));
  int hinfo = 0;
  CU(copy_out(ctx, &hinfo, P.info.p, sizeof(int)));
  CU(cudaStreamSynchronize(st));
  if (hinfo > 0) {
    const int big = m * Ns;
    if (info) *info = hinfo > big ? big : hinfo;
    ctx->err = "PosDefException: the joint ILMM posterior covariance is not positive definite";
    return hinfo > big ? big : hinfo;
  }
  if (info) *info = 0;
  return LMM_OK;
}

int ilmm_post_rand(lmm_post* post, const double* xs, int Ns, double sigma2, const double* z_latent, const double* z_noise, double* out,
                   int* info) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p;
  const bool generic = post->kind == POST_JOINT;  // AbstractGPs generic rand: m* + chol(C* + σ² I) z, no separate noise draw
  std::vector<double> E((size_t)m * m, 0.0);
  for (int a = 0; a < m; ++a) E[(size_t)a * m + a] = generic ? sigma2 : 1e-12;  // src/ilmm.jl:84
  JointPredictive P;
  int rc = build_joint_predictive(post, xs, Ns, E, P, info);
  if (rc) return rc;
  const size_t bpad = (size_t)P.ntr * TILE;
  DevBuf b_z, b_X, b_means;
  CU(b_z.alloc(ctx, bpad * sizeof(double)));
  CU(cudaMemsetAsync(b_z.p, 0, bpad * sizeof(double), st));
  CU(copy_in(ctx, b_z.as<double>(), z_latent, (size_t)m * Ns));
  CU(b_X.alloc(ctx, bpad * sizeof(double)));
  TiledSym Cl{P.Cl.as<double>(), P.ntr, sym_tiles(P.ntr) * TT};
  CU(launch_lower_gemv(st, Cl, b_z.as<double>(), bpad, b_X.as<double>(), bpad, 1));
  CU(launch_axpy(st, b_X.as<double>(), P.ml.as<double>(), bpad, 1.0));
  // add the prior means m_a to each latent's segment (stride Ns)
  CU(launch_add_mean(st, m, b_X.as<double>(), (size_t)Ns, Ns, post->d_params));
  ctx->launches += 3;
  return mix_and_add_noise(ctx, post->H.data(), p, m, 0, m, b_X.as<double>(), (size_t)Ns, Ns, sigma2, generic ? nullptr : z_noise, out);
}

int ilmm_post_logpdf(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, double* out_logpdf, double* grad_sigma2,
                     double* grad_y, int* info) {
  lmm_ctx* ctx = post->ctx;
  const bool want_grad = grad_sigma2 || grad_y;
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p;
  GeneralProjection gp;
  int rc = LMM_OK;
  if (post->kind == POST_JOINT) {
    if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
    identity_projection(m, sigma2, gp);
  } else if ((rc = general_projection(ctx, post->H.data(), p, m, sigma2, Ns, gp))) {
    return rc;
  }
  JointPredictive P;
  if ((rc = build_joint_predictive(post, xs, Ns, gp.ST, P, info))) return rc;
  const size_t bpad = (size_t)P.ntr * TILE;
  DevBuf b_y, b_T, b_Q, b_means, b_delta, b_part, b_resid, b_r, b_z, b_quad;
  const double* d_y = ys;
  if (!is_device_ptr(ys)) {
    CU(b_y.alloc(ctx, (size_t)p * Ns * sizeof(double)));
    CU(copy_in(ctx, b_y.as<double>(), ys, (size_t)p * Ns));
    d_y = b_y.as<double>();
  }
  CU(b_T.alloc(ctx, gp.pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, b_T.as<double>(), gp.pr.T.data(), gp.pr.T.size()));
  CU(b_Q.alloc(ctx, gp.pr.Q.size() * sizeof(double)));
  CU(copy_in(ctx, b_Q.as<double>(), gp.pr.Q.data(), gp.pr.Q.size()));
  std::vector<double> hmeans(m);
  for (int i = 0; i < m; ++i) hmeans[i] = post->descs[i].mean_const;
  CU(b_means.alloc(ctx, (size_t)m * sizeof(double)));
  CU(copy_in(ctx, b_means.as<double>(), hmeans.data(), (size_t)m));
  CU(b_delta.alloc(ctx, bpad * sizeof(double)));
  CU(cudaMemsetAsync(b_delta.p, 0, bpad * sizeof(double), st));
  const int nblk = project_max_partials(Ns);
  CU(b_part.alloc(ctx, (size_t)nblk * sizeof(double)));
  CU(cudaMemsetAsync(b_part.p, 0, (size_t)nblk * sizeof(double), st));
  CU(b_resid.alloc(ctx, sizeof(double)));
  DevBuf b_R, b_Ht, b_Tt, b_HtR, b_V, b_alpha, b_X, b_B, b_bT, b_gy, b_zero;
  if (want_grad) CU(b_R.alloc(ctx, (size_t)p * Ns * sizeof(double)));
  CU(launch_project(st, d_y, Ns, p, b_T.as<double>(), m, 0, m, b_means.as<double>(), b_delta.as<double>(), (size_t)Ns, b_T.as<double>(),
                    b_Q.as<double>(), b_part.as<double>(), nullptr, want_grad ? b_R.as<double>() : nullptr, nullptr));
  CU(launch_sum_partials(st, b_part.as<double>(), nblk, b_resid.as<double>()));
  // δ = vec((TY*)') - m_prior - Kc α   (ml padding is zero beyond m*Ns because Kc rows are zero there)
  CU(launch_axpy(st, b_delta.as<double>(), P.ml.as<double>(), bpad, -1.0));
  CU(b_r.alloc(ctx, bpad * sizeof(double)));
  CU(b_z.alloc(ctx, bpad * sizeof(double)));
  CU(b_quad.alloc(ctx, sizeof(double)));
  CU(cudaMemcpyAsync(b_r.p, b_delta.p, bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
  TiledSym Cl{P.Cl.as<double>(), P.ntr, sym_tiles(P.ntr) * TT};
  CU(launch_fwd_solve(st, Cl, P.W.as<double>(), (size_t)P.ntr * TT, b_r.as<double>(), b_z.as<double>(), bpad, 1, &ctx->launches));
  CU(launch_sumsq(st, b_z.as<double>(), bpad, (int)bpad, 1, b_quad.as<double>()));
  ctx->launches += 4;
  const size_t npm = (size_t)p * m;
  std::vector<double> B((size_t)m * m, 0.0), bT(npm, 0.0), Hh(post->H);
  if (want_grad) {
    // α* = C*^{-1} δ*, V = H'R/σ² - A, d/dy* = T'V - R/σ²; d/dσ² through ΣT, T (host chain, d/dH discarded)
    const size_t wst = (size_t)P.ntr * TT;
    std::vector<double> Ht((size_t)m * p), Tt((size_t)p * m);
    for (int a = 0; a < m; ++a)
      for (int j = 0; j < p; ++j) {
        Ht[(size_t)j * m + a] = Hh[(size_t)a * p + j];
        Tt[(size_t)a * p + j] = gp.pr.T[(size_t)j * m + a];
      }
    CU(b_Ht.alloc(ctx, Ht.size() * sizeof(double)));
    CU(copy_in(ctx, b_Ht.as<double>(), Ht.data(), Ht.size()));
    CU(b_Tt.alloc(ctx, Tt.size() * sizeof(double)));
    CU(copy_in(ctx, b_Tt.as<double>(), Tt.data(), Tt.size()));
    CU(b_zero.alloc(ctx, (size_t)m * sizeof(double)));
    CU(cudaMemsetAsync(b_zero.p, 0, (size_t)m * sizeof(double), st));
    CU(b_alpha.alloc(ctx, bpad * sizeof(double)));
    CU(cudaMemcpyAsync(b_r.p, b_z.p, bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CU(launch_bwd_solve(st, Cl, P.W.as<double>(), wst, b_r.as<double>(), b_alpha.as<double>(), bpad, 1, &ctx->launches));
    CU(b_HtR.alloc(ctx, (size_t)m * Ns * sizeof(double)));
    CU(launch_project(st, b_R.as<double>(), Ns, p, b_Ht.as<double>(), m, 0, m, b_zero.as<double>(), b_HtR.as<double>(), (size_t)Ns, nullptr,
                      nullptr, b_part.as<double>(), nullptr));
    CU(b_V.alloc(ctx, (size_t)m * Ns * sizeof(double)));
    CU(launch_scale_sub(st, b_V.as<double>(), b_HtR.as<double>(), 1.0 / sigma2, b_alpha.as<double>(), (size_t)m * Ns));
    ctx->launches += 2;
    if (grad_y) {
      const size_t ny = (size_t)p * Ns;
      CU(b_gy.alloc(ctx, 2 * ny * sizeof(double)));
      CU(launch_backproject(st, b_Tt.as<double>(), p, m, 0, m, b_V.as<double>(), b_V.as<double>(), (size_t)Ns, Ns, 0.0, 0.0, 0,
                            b_gy.as<double>(), b_gy.as<double>() + ny));
      CU(launch_axpy(st, b_gy.as<double>(), b_R.as<double>(), ny, -1.0 / sigma2));
      ctx->launches += 2;
      CU(copy_out(ctx, grad_y, b_gy.p, ny * sizeof(double)));
    }
    if (grad_sigma2) {
      // joint potri of the predictive covariance: X = L^{-T}, -C^{-1} = -X X' into Cl's tiles; B = block traces of G
      CU(b_X.alloc(ctx, (size_t)P.ntr * P.ntr * TT * sizeof(double)));
      TiledRect X{b_X.as<double>(), P.ntr, P.ntr, (size_t)P.ntr * P.ntr * TT};
      CU(launch_rect_identity(st, X, 1));
      CU(trsm_right_lt_upper(ctx, st, X, Cl, P.W.as<double>(), wst, 1));
      CU(cudaMemsetAsync(P.Cl.p, 0, sym_tiles(P.ntr) * TT * sizeof(double), st));
      GemmArgs g{};
      g.A = operand(X); g.B = operand(X); g.C = operand(Cl);
      g.i0 = 0; g.j0 = 0; g.k0 = 0; g.k1 = P.ntr; g.sym = 1; g.k_from_row = 1;
      CU(launch_gemm(st, GEMM_UPDATE, g, P.ntr, P.ntr, 1));
      CU(b_B.alloc(ctx, B.size() * sizeof(double)));
      CU(launch_block_trace(st, Cl, b_alpha.as<double>(), Ns, m, b_B.as<double>()));
      CU(b_bT.alloc(ctx, npm * sizeof(double)));
      CU(cudaMemsetAsync(b_bT.p, 0, npm * sizeof(double), st));
      CU(launch_abt(st, b_V.as<double>(), (size_t)Ns, m, d_y, (size_t)Ns, p, Ns, 1.0, b_bT.as<double>()));
      ctx->launches += 4;
      CU(copy_out(ctx, B.data(), b_B.p, B.size() * sizeof(double)));
      CU(copy_out(ctx, bT.data(), b_bT.p, npm * sizeof(double)));
    }
  }
  double hres = 0.0, hlogdet = 0.0, hquad = 0.0;
  CU(copy_out(ctx, &hres, b_resid.p, sizeof(double)));
  CU(copy_out(ctx, &hlogdet, P.logdet.p, sizeof(double)));
  CU(copy_out(ctx, &hquad, b_quad.p, sizeof(double)));
  CU(cudaStreamSynchronize(st));
  const double reg = -(gp.pr.reg_c0 + hres / sigma2) / 2.0;
  if (out_logpdf) *out_logpdf = -((double)m * Ns * LOG2PI + hlogdet + hquad) / 2.0 + reg;
  if (grad_sigma2) {
    if (post->kind == POST_JOINT) {  // ΣT = σ² I, T constant: d/dσ² = tr(B)
      double g = 0.0;
      for (int a = 0; a < m; ++a) g += B[(size_t)a * m + a];
      *grad_sigma2 = g;
    } else {
      std::vector<double> bH(npm, 0.0);
      rc = ilmm_grad_chain(ctx, gp, Hh, p, m, Ns, sigma2, hres, B, bT, bH, grad_sigma2, nullptr);
      if (rc != LMM_OK) return rc;
    }
  }
  return LMM_OK;
}

}  // namespace lmm_host
// ------------------------------------------------------------------------------------------------
// Sequential conditioning of a general-ILMM posterior: posterior(post(x2, σ²), y2)  (src/ilmm.jl:184-198
// applied to ILMM(PosteriorGP{IndependentMOGP}, H)).  The exact-GP identity "posterior of a posterior =
// prior conditioned on the union" in latent-major order: inputs [x; x2], projected observations
// [δ_a; (T2 Y2)_a - m_a] per latent and per-point projected noise blocks [ΣT1 ... ; ΣT2 ...].
// ------------------------------------------------------------------------------------------------
namespace lmm_host {
int ilmm_post_condition(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, lmm_post** out_post, int* info) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  if (post->kind != POST_ILMM || !post->d_Ept)
    return ctx->fail(LMM_E_UNSUPPORTED, "sequential conditioning is built for OILMM, IndependentMOGP (scalar noise) and general-ILMM posteriors");
  const int m = post->m, p = post->p, D = post->D, N1 = post->N, N2 = N1 + Ns;
  GeneralProjection gp;
  int rc = general_projection(ctx, post->H.data(), p, m, sigma2, Ns, gp);
  if (rc) return rc;
  JointBuild J;
  J.m = m; J.q = m; J.N = N2; J.D = D; J.mode = 3;
  const int64_t big64 = (int64_t)m * N2;
  if (big64 > (1 << 20)) return ctx->fail(LMM_E_UNSUPPORTED, "joint dimension too large");
  J.big = (int)big64; J.bnt = ntiles(J.big); J.bpad = (size_t)J.bnt * TILE;
  CU(cudaEventRecord(ctx->ev[0], st));
  DevBuf b_y, b_T, b_means, b_part, b_E2, b_Ept;
  CU(J.x.alloc(ctx, (size_t)N2 * D * sizeof(double)));
  CU(cudaMemcpyAsync(J.x.p, post->d_xpad, (size_t)N1 * D * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(copy_in(ctx, J.x.as<double>() + (size_t)N1 * D, xs, (size_t)Ns * D));
  const double* d_y = ys;
  if (!is_device_ptr(ys)) {
    CU(b_y.alloc(ctx, (size_t)p * Ns * sizeof(double)));
    CU(copy_in(ctx, b_y.as<double>(), ys, (size_t)p * Ns));
    d_y = b_y.as<double>();
  }
  CU(J.params.alloc(ctx, (size_t)(m + 1) * sizeof(LatentParams)));
  CU(cudaMemcpyAsync(J.params.p, post->d_params, (size_t)m * sizeof(LatentParams), cudaMemcpyDeviceToDevice, st));
  CU(J.H.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(cudaMemcpyAsync(J.H.p, post->d_H, (size_t)p * m * sizeof(double), cudaMemcpyDeviceToDevice, st));
  // δ' (latent-major, stride N2) = [δ_a ; (T2 Y2)_a - mean_a]
  CU(J.delta.alloc(ctx, J.bpad * sizeof(double)));
  CU(cudaMemsetAsync(J.delta.p, 0, J.bpad * sizeof(double), st));
  CU(cudaMemcpy2DAsync(J.delta.p, (size_t)N2 * sizeof(double), post->d_delta, (size_t)N1 * sizeof(double), (size_t)N1 * sizeof(double),
                       (size_t)m, cudaMemcpyDeviceToDevice, st));
  CU(b_T.alloc(ctx, gp.pr.T.size() * sizeof(double)));
  CU(copy_in(ctx, b_T.as<double>(), gp.pr.T.data(), gp.pr.T.size()));
  std::vector<double> hmeans(m);
  for (int i = 0; i < m; ++i) hmeans[i] = post->descs[i].mean_const;
  CU(b_means.alloc(ctx, (size_t)m * sizeof(double)));
  CU(copy_in(ctx, b_means.as<double>(), hmeans.data(), (size_t)m));
  CU(b_part.alloc(ctx, (size_t)project_max_partials(Ns) * sizeof(double)));
  CU(launch_project(st, d_y, Ns, p, b_T.as<double>(), m, 0, m, b_means.as<double>(), J.delta.as<double>() + N1, (size_t)N2, nullptr, nullptr,
                    b_part.as<double>(), nullptr));
  ++ctx->launches;
  // per-point noise blocks: the old points keep theirs, the new points get ΣT(σ²)
  const size_t mm = (size_t)m * m;
  CU(b_Ept.alloc(ctx, (size_t)N2 * mm * sizeof(double)));
  CU(cudaMemcpyAsync(b_Ept.p, post->d_Ept, (size_t)N1 * mm * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(b_E2.alloc(ctx, mm * sizeof(double)));
  CU(copy_in(ctx, b_E2.as<double>(), gp.ST.data(), mm));
  CU(launch_repeat_block(st, b_Ept.as<double>() + (size_t)N1 * mm, b_E2.as<double>(), (int)mm, (size_t)Ns * mm));
  ++ctx->launches;
  // the assemble kernel reads E from J.E: alias the per-point blocks (ownership stays with b_Ept)
  CU(J.E.alloc(ctx, (size_t)N2 * mm * sizeof(double)));
  CU(cudaMemcpyAsync(J.E.p, b_Ept.p, (size_t)N2 * mm * sizeof(double), cudaMemcpyDeviceToDevice, st));
  if ((rc = joint_factor(ctx, J, true, info))) return rc;
  *out_post = joint_make_post(ctx, J, POST_ILMM, post->descs.data(), post->H.data(), p, sigma2, b_Ept);
  return LMM_OK;
}
}  // namespace lmm_host
// ------------------------------------------------------------------------------------------------
// IndependentMOGP with non-isotropic observation noise: the reference dispatches its fast methods on
// Σy::Diagonal{<:Real,<:Fill} only (src/independent_mogp.jl:44-46); f(x, v::Vector) and
// f(x, Σ::Matrix) fall to the AbstractGPs generic FiniteGP path (test/independent_mogp.jl:72-75 runs the
// public-interface checks on `f(x_train_mo, Σy)` with a dense Σy).  Diagonal noise keeps the latents
// independent (batched per-latent factorisations with per-point noise); a dense Σy couples them: one
// joint (mN x mN) factor of blockdiag(K_a) + Σy.
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_imogp_posterior_noise(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, const double* Sigma_y,
                                         int noise_kind, const double* y, int out_dim, lmm_post** out_post, double* out_logpdf,
                                         int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (out_post) *out_post = nullptr;
  int rc = check_common(ctx, fs, m, x, N, D, m, out_dim);
  if (rc) return rc;
  if (!y || !Sigma_y || (!out_post && !out_logpdf)) return ctx->fail(LMM_E_ARG, "null pointer");
  if (noise_kind == LMM_NOISE_DIAG) {
    Projection pr;
    pr.T.assign((size_t)m * m, 0.0);
    for (int i = 0; i < m; ++i) pr.T[(size_t)i * m + i] = 1.0;
    pr.noise.assign(m, 0.0);
    pr.has_reg = false;
    std::vector<double> H = pr.T;
    RunOut out{out_post, out_logpdf, nullptr, info_latent};
    return latents_run(ctx, POST_IMOGP, fs, m, x, N, D, m, 0.0, y, pr, H.data(), nullptr, nullptr, out, Sigma_y);
  }
  if (noise_kind != LMM_NOISE_DENSE) return ctx->fail(LMM_E_ARG, "noise_kind must be LMM_NOISE_DIAG or LMM_NOISE_DENSE");
  std::vector<double> I((size_t)m * m, 0.0);
  for (int i = 0; i < m; ++i) I[(size_t)i * m + i] = 1.0;
  rc = ilmm_run(ctx, fs, m, x, N, D, I.data(), m, 0.0, y, FORM_IMOGP_DENSE, out_post, out_logpdf, info_latent, Sigma_y);
  if (info_latent && rc <= 0) *info_latent = -1;
  return rc;
}

// ------------------------------------------------------------------------------------------------
// Heterotopic / missing-data ILMM (SURVEY.md §8f-4; the reference leaves it unsupported,
// examples/oilmm_and_ilmm.ipynb:112).  Entries of y that are NaN are unobserved.  Exact inference on the observed entries
// of the dense multi-output model  y ~ N((H ⊗ I) m, Σ_l (h_l h_l') ⊗ K_l + σ² I)  (the model the reference's tests use as
// the ground truth of the ILMM, test/ilmm.jl:5): one factor of the (n_obs x n_obs) covariance, assembled straight into the
// factor tiles from the index list of observed entries.  With nothing missing it equals the ILMM's dense form.
// ------------------------------------------------------------------------------------------------
namespace lmm_host {
// Observed entries of a by-outputs y (host, NaN = missing): obs[a] = j*N + i ascending, δ_a = y_a - (H m)_j.
void masked_observations(const lmm_gp_desc* latents, int m, const double* H, int p, int N, const double* y, std::vector<int>& obs,
                         std::vector<double>& delta) {
  std::vector<double> hm(p, 0.0);
  for (int j = 0; j < p; ++j)
    for (int a = 0; a < m; ++a) hm[j] += H[(size_t)a * p + j] * latents[a].mean_const;
  for (int j = 0; j < p; ++j)
    for (int i = 0; i < N; ++i) {
      const double v = y[(size_t)j * N + i];
      if (v == v) {  // not NaN
        obs.push_back(j * N + i);
        delta.push_back(v - hm[j]);
      }
    }
}
// Inputs at which every output is observed, for a PER-INPUT mask (at each input all p outputs observed or all NaN).
// Returns false if the mask is not per-input.
bool per_input_mask(const double* y, int p, int N, std::vector<int>& keep) {
  for (int i = 0; i < N; ++i) {
    int nan = 0;
    for (int j = 0; j < p; ++j) nan += (y[(size_t)j * N + i] != y[(size_t)j * N + i]) ? 1 : 0;
    if (nan == 0) keep.push_back(i);
    else if (nan != p) return false;
  }
  return true;
}
}  // namespace lmm_host

extern "C" int lmm_ilmm_masked_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H,
                                         int p, double sigma2, const double* y, int out_dim, lmm_post** out_post, double* out_logpdf,
                                         int* n_observed, int* info) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (out_post) *out_post = nullptr;
  int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
  if (rc) return rc;
  if (!H || !y || (!out_post && !out_logpdf)) return ctx->fail(LMM_E_ARG, "null pointer");
  if (!(sigma2 > 0.0)) return ctx->fail(LMM_E_ARG, "noise variance must be positive");
  if (is_device_ptr(y) || is_device_ptr(H)) return ctx->fail(LMM_E_UNSUPPORTED, "the missing-data path takes host y and H (the mask is read on the host)");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  // observed entries and centred observations (host: a scan of p*N doubles)
  std::vector<int> obs;
  std::vector<double> delta;
  masked_observations(latents, m, H, p, N, y, obs, delta);
  const int nobs = (int)obs.size();
  if (n_observed) *n_observed = nobs;
  if (nobs == 0) return ctx->fail(LMM_E_ARG, "every observation is missing");
  if (nobs > (1 << 20)) return ctx->fail(LMM_E_UNSUPPORTED, "joint dimension too large");
  JointBuild J;
  J.m = m; J.q = p; J.N = N; J.D = D;
  J.big = nobs; J.bnt = ntiles(nobs); J.bpad = (size_t)J.bnt * TILE;
  CU(cudaEventRecord(ctx->ev[0], st));
  DevBuf b_obs;
  CU(J.x.alloc(ctx, (size_t)N * D * sizeof(double)));
  CU(copy_in(ctx, J.x.as<double>(), x, (size_t)N * D));
  std::vector<double> noise0(m, 0.0);
  if ((rc = upload_params(ctx, J.params, latents, noise0.data(), 0, m, D))) return rc;
  CU(J.H.alloc(ctx, (size_t)p * m * sizeof(double)));
  CU(copy_in(ctx, J.H.as<double>(), H, (size_t)p * m));
  CU(b_obs.alloc(ctx, (size_t)nobs * sizeof(int)));
  ctx->h2d += (int64_t)((size_t)nobs * sizeof(int));
  CU(cudaMemcpyAsync(b_obs.p, obs.data(), (size_t)nobs * sizeof(int), cudaMemcpyHostToDevice, st));
  CU(J.delta.alloc(ctx, J.bpad * sizeof(double)));
  CU(cudaMemsetAsync(J.delta.p, 0, J.bpad * sizeof(double), st));
  CU(copy_in(ctx, J.delta.as<double>(), delta.data(), (size_t)nobs));
  // factor storage + assembly + factor + solves (joint_factor assembles through launch_assemble_ilmm: do it here instead)
  CU(J.L.alloc(ctx, sym_tiles(J.bnt) * TT * sizeof(double)));
  CU(J.W.alloc(ctx, (size_t)J.bnt * TT * sizeof(double)));
  CU(J.logdet.alloc(ctx, sizeof(double)));
  CU(J.info.alloc(ctx, sizeof(int)));
  CU(J.quad.alloc(ctx, sizeof(double)));
  CU(cudaMemsetAsync(J.logdet.p, 0, sizeof(double), st));
  CU(cudaMemsetAsync(J.info.p, 0, sizeof(int), st));
  TiledSym L{J.L.as<double>(), J.bnt, sym_tiles(J.bnt) * TT};
  const size_t wstride = (size_t)J.bnt * TT;
  CU(cudaEventRecord(ctx->ev[1], st));
  CU(launch_assemble_masked(st, L, b_obs.as<int>(), nobs, J.x.as<double>(), N, D, J.params.as<LatentParams>(), m, p, J.H.as<double>(), sigma2,
                            ctx->distance_form));
  ++ctx->launches;
  CU(cudaEventRecord(ctx->ev[2], st));
  {
    PartitionScope scope(ctx);
    CU(chol_factor(ctx, L, J.W.as<double>(), wstride, 1, J.logdet.as<double>(), J.info.as<int>()));
  }
  CU(cudaEventRecord(ctx->ev[3], st));
  DevBuf b_r, b_z;
  CU(b_r.alloc(ctx, J.bpad * sizeof(double)));
  CU(b_z.alloc(ctx, J.bpad * sizeof(double)));
  CU(cudaMemcpyAsync(b_r.p, J.delta.p, J.bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CU(launch_fwd_solve(st, L, J.W.as<double>(), wstride, b_r.as<double>(), b_z.as<double>(), J.bpad, 1, &ctx->launches));
  CU(launch_sumsq(st, b_z.as<double>(), J.bpad, (int)J.bpad, 1, J.quad.as<double>()));
  ++ctx->launches;
  if (out_post) {
    CU(J.alpha.alloc(ctx, J.bpad * sizeof(double)));
    CU(cudaMemcpyAsync(b_r.p, b_z.p, J.bpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CU(launch_bwd_solve(st, L, J.W.as<double>(), wstride, b_r.as<double>(), J.alpha.as<double>(), J.bpad, 1, &ctx->launches));
  }
  int hinfo = 0;
  CU(copy_out(ctx, &J.hlogdet, J.logdet.p, sizeof(double)));
  CU(copy_out(ctx, &J.hquad, J.quad.p, sizeof(double)));
  CU(copy_out(ctx, &hinfo, J.info.p, sizeof(int)));
  CU(cudaEventRecord(ctx->ev[4], st));
  CU(cudaStreamSynchronize(st));
  {
    float a = 0, b = 0, c = 0, d = 0;
    cudaEventElapsedTime(&a, ctx->ev[0], ctx->ev[4]);
    cudaEventElapsedTime(&b, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&c, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&d, ctx->ev[3], ctx->ev[4]);
    ctx->timings[0] = a; ctx->timings[1] = b; ctx->timings[2] = c; ctx->timings[3] = d;
  }
  if (hinfo > 0) {
    if (info) *info = hinfo > nobs ? nobs : hinfo;
    ctx->err = "PosDefException: the covariance of the observed entries is not positive definite";
    return hinfo > nobs ? nobs : hinfo;
  }
  if (info) *info = 0;
  if (out_logpdf) *out_logpdf = -((double)nobs * LOG2PI + J.hlogdet + J.hquad) / 2.0;
  if (out_post) {
    DevBuf none;
    lmm_post* P = joint_make_post(ctx, J, POST_MASKED, latents, H, p, sigma2, none);
    P->d_obs = (int*)b_obs.detach();
    P->bytes += (size_t)nobs * sizeof(int);
    *out_post = P;
  }
  return LMM_OK;
}

namespace lmm_host {
// mean_and_var(post(x*, σ²)) of the missing-data posterior: all p outputs at x*.
//   mean = (H m)_j + K_{*,obs} α ;  var = Σ_l H[j,l]² k_l(x*,x*) - rowsumsq(K_{*,obs} L^{-T}) + σ²
int masked_post_mean_and_var(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean, double* var) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p, N = post->N, D = post->D, bnt = post->big_nt, nobs = post->big_n;
  const int64_t rows64 = (int64_t)p * Ns;
  if (rows64 > (1 << 22)) return ctx->fail(LMM_E_UNSUPPORTED, "too many prediction points");
  const int rows = (int)rows64, ntr = ntiles(rows);
  DevBuf b_xs, b_V, b_m, b_v, b_zero;
  CU(b_xs.alloc(ctx, (size_t)Ns * D * sizeof(double)));
  CU(copy_in(ctx, b_xs.as<double>(), xs, (size_t)Ns * D));
  CU(b_V.alloc(ctx, (size_t)ntr * bnt * TT * sizeof(double)));
  TiledRect V{b_V.as<double>(), ntr, bnt, (size_t)ntr * bnt * TT};
  CU(launch_assemble_masked_cross(st, V, b_xs.as<double>(), Ns, post->d_obs, nobs, post->d_xpad, N, D, post->d_params, m, p, post->d_H,
                                  ctx->distance_form));
  // a zeroed LatentParams turns rect_gemv / rect_rowsumsq into plain K α and -rowsumsq
  CU(b_zero.alloc(ctx, sizeof(LatentParams)));
  CU(cudaMemsetAsync(b_zero.p, 0, sizeof(LatentParams), st));
  CU(b_m.alloc(ctx, (size_t)ntr * TILE * sizeof(double)));
  CU(b_v.alloc(ctx, (size_t)ntr * TILE * sizeof(double)));
  CU(launch_rect_gemv(st, V, post->d_alpha, (size_t)bnt * TILE, b_m.as<double>(), (size_t)ntr * TILE, b_zero.as<LatentParams>(), 0, 1));
  CU(trsm_right_lt(ctx, V, post->Lsym(), post->d_W, post->wstride(), 1));
  CU(launch_rect_rowsumsq(st, V, b_v.as<double>(), (size_t)ntr * TILE, b_zero.as<LatentParams>(), 1));
  ctx->launches += 3;
  CU(copy_out(ctx, mean, b_m.p, (size_t)rows * sizeof(double)));
  CU(copy_out(ctx, var, b_v.p, (size_t)rows * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  // prior mean and variance of output j (constants along n): Σ_l H[j,l] m_l and Σ_l H[j,l]² variance_l
  for (int j = 0; j < p; ++j) {
    double pm = 0.0, pv = 0.0;
    for (int l = 0; l < m; ++l) {
      const double h = post->H[(size_t)l * p + j];
      pm += h * post->descs[l].mean_const;
      pv += h * h * desc_kdiag(post->descs[l]);
    }
    for (int n = 0; n < Ns; ++n) {
      mean[(size_t)j * Ns + n] += pm;
      var[(size_t)j * Ns + n] += pv + sigma2;
    }
  }
  return LMM_OK;
}
}  // namespace lmm_host

namespace lmm_host {
// Predictive pieces of the missing-data (dense-model) posterior at x*: mean (p Ns, by outputs) and the tiled
// covariance  C = Σ_l (h_l h_l') ⊗ K_l(x*, x*) + e0 I - V V',  V = K_{*,obs} L^{-T}  (dimension p Ns).
struct MaskedPredictive {
  DevBuf xs, V, mean, C;
  int ntr = 0, rows = 0;
};
int masked_predictive(lmm_post* post, const double* xs, int Ns, double e0, MaskedPredictive& P) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  const int m = post->m, p = post->p, N = post->N, D = post->D, bnt = post->big_nt, nobs = post->big_n;
  if ((int64_t)p * Ns > 46000) return ctx->fail(LMM_E_UNSUPPORTED, "dense covariance output too large");
  P.rows = p * Ns;
  P.ntr = ntiles(P.rows);
  DevBuf b_zero, b_e0, b_pm;
  CU(P.xs.alloc(ctx, (size_t)Ns * D * sizeof(double)));
  CU(copy_in(ctx, P.xs.as<double>(), xs, (size_t)Ns * D));
  CU(P.V.alloc(ctx, (size_t)P.ntr * bnt * TT * sizeof(double)));
  TiledRect V{P.V.as<double>(), P.ntr, bnt, (size_t)P.ntr * bnt * TT};
  CU(launch_assemble_masked_cross(st, V, P.xs.as<double>(), Ns, post->d_obs, nobs, post->d_xpad, N, D, post->d_params, m, p, post->d_H,
                                  ctx->distance_form));
  CU(b_zero.alloc(ctx, sizeof(LatentParams)));
  CU(cudaMemsetAsync(b_zero.p, 0, sizeof(LatentParams), st));
  CU(P.mean.alloc(ctx, (size_t)P.ntr * TILE * sizeof(double)));
  CU(launch_rect_gemv(st, V, post->d_alpha, (size_t)bnt * TILE, P.mean.as<double>(), (size_t)P.ntr * TILE, b_zero.as<LatentParams>(), 0, 1));
  CU(trsm_right_lt(ctx, V, post->Lsym(), post->d_W, post->wstride(), 1));
  // prior means of the outputs (constants along n) added on the device
  std::vector<double> pm((size_t)P.rows, 0.0);
  for (int j = 0; j < p; ++j) {
    double v = 0.0;
    for (int l = 0; l < m; ++l) v += post->H[(size_t)l * p + j] * post->descs[l].mean_const;
    for (int n = 0; n < Ns; ++n) pm[(size_t)j * Ns + n] = v;
  }
  CU(b_pm.alloc(ctx, (size_t)P.rows * sizeof(double)));
  CU(copy_in(ctx, b_pm.as<double>(), pm.data(), (size_t)P.rows));
  CU(launch_axpy(st, P.mean.as<double>(), b_pm.as<double>(), (size_t)P.rows, 1.0));
  CU(b_e0.alloc(ctx, sizeof(double)));
  CU(copy_in(ctx, b_e0.as<double>(), &e0, 1));
  CU(P.C.alloc(ctx, sym_tiles(P.ntr) * TT * sizeof(double)));
  TiledSym C{P.C.as<double>(), P.ntr, sym_tiles(P.ntr) * TT};
  CU(launch_assemble_ilmm(st, C, P.xs.as<double>(), Ns, D, post->d_params, m, p, b_e0.as<double>(), post->d_H, 1, ctx->distance_form));
  GemmArgs g{};
  g.A = operand(V); g.B = operand(V); g.C = operand(C);
  g.i0 = 0; g.j0 = 0; g.k0 = 0; g.k1 = bnt; g.sym = 1;
  CU(launch_gemm(st, GEMM_UPDATE, g, P.ntr, P.ntr, 1));
  ctx->launches += 5;
  CU(cudaStreamSynchronize(st));  // the host-side staging vectors go out of scope
  return LMM_OK;
}

// mean_and_cov(post(x*, σ²)) of the missing-data posterior: dense (p Ns)², by outputs.
int masked_post_mean_and_cov(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean, double* cov) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  MaskedPredictive P;
  int rc = masked_predictive(post, xs, Ns, sigma2, P);
  if (rc) return rc;
  DevBuf dense;
  CU(dense.alloc(ctx, (size_t)P.rows * P.rows * sizeof(double)));
  CU(cudaMemsetAsync(dense.p, 0, (size_t)P.rows * P.rows * sizeof(double), st));
  TiledSym C{P.C.as<double>(), P.ntr, sym_tiles(P.ntr) * TT};
  CU(launch_untile_lower(st, C, 0, dense.as<double>(), P.rows));
  ++ctx->launches;
  std::vector<double> h((size_t)P.rows * P.rows);
  CU(copy_out(ctx, h.data(), dense.p, h.size() * sizeof(double)));
  if (mean) CU(copy_out(ctx, mean, P.mean.p, (size_t)P.rows * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  for (int c = 0; c < P.rows; ++c)  // mirror the lower triangle
    for (int r = c; r < P.rows; ++r) {
      cov[(size_t)c * P.rows + r] = h[(size_t)c * P.rows + r];
      cov[(size_t)r * P.rows + c] = h[(size_t)c * P.rows + r];
    }
  return LMM_OK;
}

// rand(rng, post(x*, σ²)) of the missing-data posterior -- AbstractGPs' generic FiniteGP rand on the dense model:
// mean + chol(C + σ² I) z with ONE vector z of p Ns standard normals (by outputs).
int masked_post_rand(lmm_post* post, const double* xs, int Ns, double sigma2, const double* z, double* out, int* info) {
  lmm_ctx* ctx = post->ctx;
  cudaStream_t st = ctx->stream;
  MaskedPredictive P;
  int rc = masked_predictive(post, xs, Ns, sigma2, P);
  if (rc) return rc;
  const size_t bpad = (size_t)P.ntr * TILE;
  DevBuf b_W, b_logdet, b_info, b_z, b_X;
  CU(b_W.alloc(ctx, (size_t)P.ntr * TT * sizeof(double)));
  CU(b_logdet.alloc(ctx, sizeof(double)));
  CU(b_info.alloc(ctx, sizeof(int)));
  CU(cudaMemsetAsync(b_logdet.p, 0, sizeof(double), st));
  CU(cudaMemsetAsync(b_info.p, 0, sizeof(int), st));
  TiledSym C{P.C.as<double>(), P.ntr, sym_tiles(P.ntr) * TT};
  CU(chol_factor(ctx, C, b_W.as<double>(), (size_t)P.ntr * TT, 1, b_logdet.as<double>(), b_info.as<int>()));
  CU(b_z.alloc(ctx, bpad * sizeof(double)));
  CU(cudaMemsetAsync(b_z.p, 0, bpad * sizeof(double), st));
  CU(copy_in(ctx, b_z.as<double>(), z, (size_t)P.rows));
  CU(b_X.alloc(ctx, bpad * sizeof(double)));
  CU(launch_lower_gemv(st, C, b_z.as<double>(), bpad, b_X.as<double>(), bpad, 1));
  CU(launch_axpy(st, b_X.as<double>(), P.mean.as<double>(), (size_t)P.rows, 1.0));
  ctx->launches += 2;
  int hinfo = 0;
  CU(copy_out(ctx, &hinfo, b_info.p, sizeof(int)));
  CU(copy_out(ctx, out, b_X.p, (size_t)P.rows * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  if (hinfo > 0) {
    if (info) *info = hinfo > P.rows ? P.rows : hinfo;
    ctx->err = "PosDefException: the missing-data predictive covariance is not positive definite";
    return hinfo > P.rows ? P.rows : hinfo;
  }
  if (info) *info = -1;
  return LMM_OK;
}
}  // namespace lmm_host

// Heterotopic OILMM whose mask is PER INPUT (at every input either all p outputs are observed or none is: sensors that drop
// whole time steps).  Conditioning on the observed entries is then the ordinary OILMM on the observed inputs -- the
// projection T*Y stays exact, the latents stay independent, cost O(m N_obs³) instead of the dense model's O((p N)³) -- and the
// returned handle is a full OILMM posterior (marginals, cov, rand, logpdf, conditioning, gradients, save / load).
// A mask that is not per-input returns LMM_E_UNSUPPORTED: use lmm_ilmm_masked_posterior (dense model) with H = U sqrt(S).
extern "C" int lmm_oilmm_masked_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* U,
                                          const double* S, int p, double sigma2, const double* y, int out_dim, lmm_post** out_post,
                                          double* out_logpdf, int* n_observed_inputs, int* info_latent) {
  if (!ctx) return LMM_E_ARG;
  {
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (out_post) *out_post = nullptr;
    int rc = check_common(ctx, latents, m, x, N, D, p, out_dim);
    if (rc) return rc;
    if (!U || !S || !y || (!out_post && !out_logpdf)) return ctx->fail(LMM_E_ARG, "null pointer");
    if (is_device_ptr(y) || is_device_ptr(x)) return ctx->fail(LMM_E_UNSUPPORTED, "the missing-data path takes host x and y (the mask is read on the host)");
  }
  std::vector<int> keep;
  if (!per_input_mask(y, p, N, keep)) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->fail(LMM_E_UNSUPPORTED, "the mask is not per-input (some outputs observed, some missing at one input): use lmm_ilmm_masked_posterior");
  }
  const int No = (int)keep.size();
  if (n_observed_inputs) *n_observed_inputs = No;
  if (No == 0) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->fail(LMM_E_ARG, "every observation is missing");
  }
  std::vector<double> xo((size_t)No * D), yo((size_t)p * No);
  for (int k = 0; k < No; ++k) {
    for (int d = 0; d < D; ++d) xo[(size_t)k * D + d] = x[(size_t)keep[k] * D + d];
    for (int j = 0; j < p; ++j) yo[(size_t)j * No + k] = y[(size_t)j * N + keep[k]];
  }
  return lmm_oilmm_posterior(ctx, latents, m, xo.data(), No, D, U, S, p, sigma2, yo.data(), out_dim, out_post, out_logpdf, nullptr, info_latent);
}
