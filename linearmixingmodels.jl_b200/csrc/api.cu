// liblmm C ABI (include/lmm.h): contexts, communicators, options and the host-only entry points; the shared host
// helpers (pointer classification, staged copies, shard ranges).  See host_internal.h for the file map.
#include <algorithm>

#include "host_internal.h"

// NCCL through dlopen: no link-time dependency; picks up the libnccl.so.2 already loaded by the host process (torch
// bundles one) or the system one.
NcclApi& nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (api.handle) break;
    }
    if (!api.handle) return;
    api.GetUniqueId = (int (*)(NcclId*))dlsym(api.handle, "ncclGetUniqueId");
    api.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(api.handle, "ncclCommInitRank");
    api.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(api.handle, "ncclAllReduce");
    api.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(api.handle, "ncclAllGather");
    api.CommSplit = (int (*)(void*, int, int, void**, void*))dlsym(api.handle, "ncclCommSplit");
    api.CommDestroy = (int (*)(void*))dlsym(api.handle, "ncclCommDestroy");
    api.GetErrorString = (const char* (*)(int))dlsym(api.handle, "ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.AllReduce && api.CommDestroy;
  });
  return api;
}

namespace lmm_host {

bool is_device_ptr(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Copy n doubles from a caller pointer (host or device) into device memory at dst.
cudaError_t copy_in(lmm_ctx* ctx, double* dst, const double* src, size_t n) {
  if (is_device_ptr(src)) return cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream);
  ctx->h2d += (int64_t)(n * sizeof(double));
  return cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
}
cudaError_t copy_out(lmm_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes) {
  ctx->d2h += (int64_t)bytes;
  return cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, ctx->stream);
}

void shard_range(const lmm_ctx* ctx, int m, int& lo, int& hi) {
  lo = (int)(((int64_t)m * ctx->rank) / ctx->nranks);
  hi = (int)(((int64_t)m * (ctx->rank + 1)) / ctx->nranks);
}

static int check_term(lmm_ctx* ctx, int kind, double variance, double inv_ls, double param, const double* ard, int D) {
  if (kind < 0 || kind > LMM_KERNEL_PERIODIC)
    return ctx->fail(LMM_E_UNSUPPORTED, "unsupported kernel kind (SE, Matern32, Matern52, Exponential, RationalQuadratic, Periodic)");
  if (kind == LMM_KERNEL_RATIONAL_QUADRATIC && !(param > 0.0)) return ctx->fail(LMM_E_ARG, "RationalQuadraticKernel needs α > 0 in `param`");
  if (kind == LMM_KERNEL_PERIODIC && !(param > 0.0)) return ctx->fail(LMM_E_ARG, "PeriodicKernel needs r > 0 in `param`");
  if (!(variance > 0.0) || !(inv_ls > 0.0)) return ctx->fail(LMM_E_ARG, "kernel variance and inv_lengthscale must be positive");
  if (ard) {
    if (D > LMM_MAX_ARD) return ctx->fail(LMM_E_UNSUPPORTED, "ARDTransform is supported for input dimension D <= 8");
    for (int k = 0; k < D; ++k)
      if (!(ard[k] > 0.0)) return ctx->fail(LMM_E_ARG, "ARD multipliers must be positive");
  }
  return LMM_OK;
}

int check_descs(lmm_ctx* ctx, const lmm_gp_desc* d, int m, int D) {
  for (int i = 0; i < m; ++i) {
    int rc = check_term(ctx, d[i].kind, d[i].variance, d[i].inv_lengthscale, d[i].param, d[i].ard, D);
    if (rc) return rc;
    if (d[i].compose < LMM_COMPOSE_NONE || d[i].compose > LMM_COMPOSE_PRODUCT) return ctx->fail(LMM_E_ARG, "lmm_gp_desc.compose must be 0 (none), 1 (sum) or 2 (product)");
    if (d[i].n_extra < 0 || d[i].n_extra > LMM_MAX_TERMS - 1) return ctx->fail(LMM_E_UNSUPPORTED, "a composite kernel has at most LMM_MAX_TERMS = 4 terms");
    if (d[i].compose == LMM_COMPOSE_NONE && d[i].n_extra != 0) return ctx->fail(LMM_E_ARG, "n_extra must be 0 for a single kernel (compose = 0)");
    if (d[i].n_extra > 0 && !d[i].extra) return ctx->fail(LMM_E_ARG, "n_extra > 0 with a null `extra` pointer");
    for (int t = 0; t < d[i].n_extra; ++t) {
      const lmm_kernel_term& q = d[i].extra[t];
      if ((rc = check_term(ctx, q.kind, q.variance, q.inv_lengthscale, q.param, q.ard, D))) return rc;
    }
  }
  return LMM_OK;
}

// k(x, x) of a latent's whole kernel (κ(0) = 1 for every supported base kernel): Σ or Π of the term variances.
double desc_kdiag(const lmm_gp_desc& d) {
  double v = d.variance;
  for (int t = 0; t < d.n_extra; ++t) v = (d.compose == LMM_COMPOSE_PRODUCT) ? v * d.extra[t].variance : v + d.extra[t].variance;
  return v;
}
bool desc_is_composite(const lmm_gp_desc& d) { return d.n_extra > 0 || d.kind == LMM_KERNEL_PERIODIC; }

size_t factor_bytes_per_latent(int nt) { return (sym_tiles(nt) + (size_t)nt) * TT * sizeof(double); }

// Device-side description of one latent (noise = what is added on the diagonal of its kernel matrix).
void set_params(LatentParams& q, const lmm_gp_desc& d, double noise, double ls_scale, int D) {
  q.kind = d.kind;
  q.ard_dim = d.ard ? D : 0;
  q.variance = d.variance;
  q.inv_ls = d.inv_lengthscale * ls_scale;
  q.noise = noise;
  q.mean = d.mean_const;
  q.param = d.param;
  static_assert(MAX_ARD == LMM_MAX_ARD, "device and ABI limits must agree");
  static_assert(MAX_TERMS == LMM_MAX_TERMS, "device and ABI limits must agree");
  for (int k = 0; k < MAX_ARD; ++k) q.ard[k] = (d.ard && k < D) ? d.ard[k] : 1.0;
  q.nterms = 1 + d.n_extra;
  q.compose = d.compose;
  q.kdiag = desc_kdiag(d);
  for (int t = 0; t < MAX_TERMS - 1; ++t) {
    TermParams& e = q.extra[t];
    if (t < d.n_extra) {
      const lmm_kernel_term& src = d.extra[t];
      e.kind = src.kind;
      e.ard_dim = src.ard ? D : 0;
      e.variance = src.variance;
      e.inv_ls = src.inv_lengthscale * ls_scale;  // a lengthscale sweep stretches every term
      e.param = src.param;
      for (int k = 0; k < MAX_ARD; ++k) e.ard[k] = (src.ard && k < D) ? src.ard[k] : 1.0;
    } else {
      e.kind = 0; e.ard_dim = 0; e.variance = 0.0; e.inv_ls = 1.0; e.param = 1.0;
      for (int k = 0; k < MAX_ARD; ++k) e.ard[k] = 1.0;
    }
  }
}

void fill_params(std::vector<LatentParams>& hp, const lmm_gp_desc* d, const double* noise, int lo, int hi, int D, double ls_scale) {
  hp.resize(hi - lo);
  for (int i = lo; i < hi; ++i) set_params(hp[i - lo], d[i], noise[i], ls_scale, D);
}

}  // namespace lmm_host

// ------------------------------------------------------------------------------------------------
// C ABI: context
// ------------------------------------------------------------------------------------------------
extern "C" const char* lmm_version(void) { return "liblmm 0.1.0 (sm_100a)"; }

extern "C" int lmm_ctx_create(int device, lmm_ctx** out) {
  if (!out) return LMM_E_ARG;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return LMM_E_CUDA;  // no CPU fallback
  }
  if (device < 0 || device >= ndev) return LMM_E_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return LMM_E_CUDA;
  lmm_ctx* ctx = new lmm_ctx();
  ctx->device = device;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return LMM_E_CUDA;
  }
  for (auto& e : ctx->ev) cudaEventCreate(&e);
  for (auto& g : ctx->gstream) cudaStreamCreateWithFlags(&g, cudaStreamNonBlocking);
  {
    int lo_pri = 0, hi_pri = 0;
    cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri);
    cudaStreamCreateWithPriority(&ctx->panel_stream, cudaStreamNonBlocking, hi_pri);
    cudaStreamCreateWithPriority(&ctx->update_stream, cudaStreamNonBlocking, lo_pri);
  }
  cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
  for (auto& e : ctx->ev_join) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  // LMM_OZAKI=6|7|8: start with the integer-slice trailing update switched on (runs a whole test suite / application on it unchanged)
  if (const char* oz = getenv("LMM_OZAKI")) {
    const int v = atoi(oz);
    if (v == 6 || v == 7 || v == 8) ctx->ozaki = v;
  }
  if (const char* ob = getenv("LMM_OZAKI_BITS")) {
    const int v = atoi(ob);
    if (v == 7 || v == 8) ctx->ozaki_bits = v;
  }
  *out = ctx;
  return LMM_OK;
}

extern "C" int lmm_ctx_destroy(lmm_ctx* ctx) {
  if (!ctx) return LMM_E_ARG;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->comm_small && nccl_api().ok) nccl_api().CommDestroy(ctx->comm_small);
  if (ctx->comm && nccl_api().ok) nccl_api().CommDestroy(ctx->comm);
  if (ctx->chain_cnt) cudaFree(ctx->chain_cnt);
  for (auto& e : ctx->ev) cudaEventDestroy(e);
  for (auto& g : ctx->gstream) cudaStreamDestroy(g);
  if (ctx->xbuf) cudaFree(ctx->xbuf);
  if (ctx->oz_slices) cudaFree(ctx->oz_slices);
  if (ctx->oz_scale) cudaFree(ctx->oz_scale);
  if (ctx->oz_fp) cudaFree(ctx->oz_fp);
  if (ctx->oz_x) cudaFree(ctx->oz_x);
  for (auto& e : ctx->oz_events) cudaEventDestroy(e);  // "ozaki_time" events nobody read back
  cudaStreamDestroy(ctx->panel_stream);
  cudaStreamDestroy(ctx->update_stream);
  for (auto& e : ctx->blk_ev) cudaEventDestroy(e);
  cudaEventDestroy(ctx->ev_fork);
  for (auto& e : ctx->ev_join) cudaEventDestroy(e);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
  return LMM_OK;
}

extern "C" const char* lmm_last_error(lmm_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int lmm_ctx_set_option(lmm_ctx* ctx, const char* key, double value) {
  if (!ctx || !key) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  std::string k(key);
  if (k == "distance_form") {
    if (value != 0.0 && value != 1.0) return ctx->fail(LMM_E_ARG, "distance_form must be 0 or 1");
    ctx->distance_form = (int)value;
  } else if (k == "outer_block") {
    if (value == 0.0) {  // back to the built-in choice
      ctx->outer_block = 8;
      ctx->outer_block_user = false;
      return LMM_OK;
    }
    if (value < 1 || value > 64) return ctx->fail(LMM_E_ARG, "outer_block must be in [1, 64] (0 = automatic)");
    ctx->outer_block = (int)value;
    ctx->outer_block_user = true;
  } else if (k == "streams") {
    if (value < 1 || value > lmm_ctx::MAX_GROUPS) return ctx->fail(LMM_E_ARG, "streams must be in [1, 8]");
    ctx->ngroups = (int)value;
  } else if (k == "lookahead") {
    if (value != 0.0 && value != 1.0) return ctx->fail(LMM_E_ARG, "lookahead must be 0 (plain) or 1 (right-looking block schedule on two streams)");
    ctx->lookahead = (int)value;
  } else if (k == "kmat_skip") {
    if (value != 0.0 && value != 1.0) return ctx->fail(LMM_E_ARG, "kmat_skip must be 0 (build every kernel-matrix tile) or 1");
    ctx->kmat_skip = (int)value;
  } else if (k == "vfe_chunk") {
    if (value < 0 || value > 1e6 || value != (double)(int)value) return ctx->fail(LMM_E_ARG, "vfe_chunk must be a whole number of tile rows >= 0 (0 = by memory)");
    ctx->vfe_chunk = (int)value;
  } else if (k == "chain_fused") {
    if (value != 0.0 && value != 1.0 && value != 2.0) return ctx->fail(LMM_E_ARG, "chain_fused must be 0, 1 (where it pays off) or 2 (everywhere)");
    ctx->chain_fused = (int)value;
  } else if (k == "pdl") {
    set_pdl(value != 0.0);
  } else if (k == "nccl_small_ctas") {  // takes effect at lmm_comm_init
    if (value < 0 || value > 32) return ctx->fail(LMM_E_ARG, "nccl_small_ctas must be in [0, 32]");
    ctx->nccl_small_ctas = (int)value;
  } else if (k == "partition_ilmm") {
    if (value != 0.0 && value != 1.0 && value != 2.0) return ctx->fail(LMM_E_ARG, "partition_ilmm must be 0, 1 or 2");
    ctx->partition_ilmm = (int)value;
  } else if (k == "ozaki") {
    if (value != 0.0 && value != 6.0 && value != 7.0 && value != 8.0) return ctx->fail(LMM_E_ARG, "ozaki must be 0 (DMMA) or 6, 7, 8 (int8 digit planes)");
    ctx->ozaki = (int)value;
  } else if (k == "ozaki_bits") {
    if (value != 7.0 && value != 8.0) return ctx->fail(LMM_E_ARG, "ozaki_bits must be 7 (radix 128) or 8 (radix 256)");
    ctx->ozaki_bits = (int)value;
  } else if (k == "ozaki_time") {
    if (value != 0.0 && value != 1.0) return ctx->fail(LMM_E_ARG, "ozaki_time must be 0 or 1");
    ctx->ozaki_time = (int)value;
  } else if (k == "ozaki_single_nt") {
    if (value < 0 || value > 65536) return ctx->fail(LMM_E_ARG, "ozaki_single_nt must be in [0, 65536]");
    ctx->ozaki_single_nt = (int)value;
  } else if (k == "ozaki_min_k") {
    if (value < 1 || value > 4096) return ctx->fail(LMM_E_ARG, "ozaki_min_k must be in [1, 4096]");
    ctx->ozaki_min_k = (int)value;
  } else if (k == "trsm_slice") {
    if (value != 0.0 && value != 1.0) return ctx->fail(LMM_E_ARG, "trsm_slice must be 0 or 1");
    ctx->trsm_slice = (int)value;
  } else if (k == "gemm_small") {
    if (value < 0 || value > 4096) return ctx->fail(LMM_E_ARG, "gemm_small must be in [0, 4096]");
    set_gemm_small_threshold((int)value);
  } else if (k == "project_impl") {
    if (value != 0.0 && value != 1.0) return ctx->fail(LMM_E_UNSUPPORTED, "project_impl must be 0 or 1");
    set_project_impl((int)value);
  } else if (k == "condition_update") {
    if (value != 0.0 && value != 1.0) return ctx->fail(LMM_E_UNSUPPORTED, "condition_update must be 0 or 1");
    ctx->condition_update = (int)value;
  } else if (k == "solve_impl") {
    if (value != 0.0 && value != 1.0) return ctx->fail(LMM_E_UNSUPPORTED, "solve_impl must be 0 or 1");
    set_solve_impl((int)value);
  } else {
    return ctx->fail(LMM_E_UNSUPPORTED, "unknown option " + k);
  }
  return LMM_OK;
}

extern "C" int lmm_ctx_counters(lmm_ctx* ctx, int64_t* kernel_launches, int64_t* h2d_bytes, int64_t* d2h_bytes) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (kernel_launches) *kernel_launches = ctx->launches;
  if (h2d_bytes) *h2d_bytes = ctx->h2d;
  if (d2h_bytes) *d2h_bytes = ctx->d2h;
  return LMM_OK;
}

extern "C" int lmm_ctx_last_timings(lmm_ctx* ctx, double out_ms[8]) {
  if (!ctx || !out_ms) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  for (int i = 0; i < 8; ++i) out_ms[i] = ctx->timings[i];
  if (!ctx->oz_events.empty()) {  // "ozaki_time": the int8 update launches of the last call(s), summed; events are consumed here
    double sum = 0.0;
    for (size_t i = 0; i + 1 < ctx->oz_events.size(); i += 2) {
      float ms = 0.f;
      if (cudaEventSynchronize(ctx->oz_events[i + 1]) == cudaSuccess && cudaEventElapsedTime(&ms, ctx->oz_events[i], ctx->oz_events[i + 1]) == cudaSuccess)
        sum += ms;
      cudaEventDestroy(ctx->oz_events[i]);
      cudaEventDestroy(ctx->oz_events[i + 1]);
    }
    ctx->oz_events.clear();
    out_ms[7] = sum;
    out_ms[5] = ctx->oz_tile_products;
    ctx->oz_tile_products = 0.0;
  }
  return LMM_OK;
}

extern "C" int lmm_comm_unique_id(void* out_128_bytes) {
  if (!out_128_bytes) return LMM_E_ARG;
  NcclApi& api = nccl_api();
  if (!api.ok) return LMM_E_NCCL;
  NcclId id;
  if (api.GetUniqueId(&id) != 0) return LMM_E_NCCL;
  memcpy(out_128_bytes, &id, 128);
  return LMM_OK;
}

extern "C" int lmm_comm_set_shard(lmm_ctx* ctx, int nranks, int rank) {
  if (!ctx || nranks < 1 || rank < 0 || rank >= nranks) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  ctx->nranks = nranks;
  ctx->rank = rank;
  return LMM_OK;
}

extern "C" int lmm_comm_init(lmm_ctx* ctx, const void* unique_id_128_bytes, int nranks, int rank) {
  if (!ctx || !unique_id_128_bytes || nranks < 1 || rank < 0 || rank >= nranks) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  NcclApi& api = nccl_api();
  if (!api.ok) return ctx->fail(LMM_E_NCCL, "libnccl.so.2 not found (dlopen)");
  if (cudaSetDevice(ctx->device) != cudaSuccess) return LMM_E_CUDA;
  NcclId id;
  memcpy(&id, unique_id_128_bytes, 128);
  int r = api.CommInitRank(&ctx->comm, nranks, id, rank);
  if (r != 0) return ctx->fail(LMM_E_NCCL, std::string("ncclCommInitRank: ") + (api.GetErrorString ? api.GetErrorString(r) : "?"));
  ctx->nranks = nranks;
  ctx->rank = rank;
  // Communicators of the partitioned factorisation (optional: without them it uses the main one).  Their exchanges sit on
  // the panel chain while the trailing GEMMs hold every SM (one 192 KB CTA each), so an NCCL kernel waits for as many
  // SMs to drain as it has CTAs: cap them (ncclConfig_t minCTAs / maxCTAs; the prefix of the struct as of NCCL 2.18).
  if (api.CommSplit && nranks > 1) {
    struct { size_t size; unsigned magic; unsigned version; int blocking, cgaClusterSize, minCTAs, maxCTAs; const char* netName; int splitShare; } cfg;
    const int UNDEF = -2147483647 - 1;
    auto split = [&](void** out, int max_ctas) {
      cfg = {sizeof(cfg), 0xcafebeefu, 21800u, UNDEF, UNDEF, 1, max_ctas, nullptr, UNDEF};
      if (api.CommSplit(ctx->comm, 0, rank, out, &cfg) != 0) {
        *out = nullptr;
        if (api.CommSplit(ctx->comm, 0, rank, out, nullptr) != 0) *out = nullptr;
      }
    };
    if (ctx->nccl_small_ctas > 0) split(&ctx->comm_small, ctx->nccl_small_ctas);
  }
  return LMM_OK;
}

// ------------------------------------------------------------------------------------------------
// Orthogonal validation (host): src/orthogonal_matrix.jl:21-23  isapprox(U'U, I)
// ------------------------------------------------------------------------------------------------
// Largest |eigenvalue| of a symmetric n x n matrix (= its operator 2-norm): cyclic Jacobi rotations on the host.
// n = m (number of latents), so O(n³) per sweep is negligible; converges quadratically, 6-10 sweeps.
static double sym_opnorm(std::vector<double> A, int n) {
  for (int sweep = 0; sweep < 60; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int a = 0; a < n; ++a)
      for (int b = 0; b < n; ++b) (a == b ? diag : off) += A[(size_t)a * n + b] * A[(size_t)a * n + b];
    if (off <= 1e-32 * (diag + off) || off == 0.0) break;
    for (int pI = 0; pI < n - 1; ++pI)
      for (int q = pI + 1; q < n; ++q) {
        const double apq = A[(size_t)pI * n + q];
        if (apq == 0.0) continue;
        const double theta = (A[(size_t)q * n + q] - A[(size_t)pI * n + pI]) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), sn = t * c;
        for (int k = 0; k < n; ++k) {  // columns p, q
          const double akp = A[(size_t)k * n + pI], akq = A[(size_t)k * n + q];
          A[(size_t)k * n + pI] = c * akp - sn * akq;
          A[(size_t)k * n + q] = sn * akp + c * akq;
        }
        for (int k = 0; k < n; ++k) {  // rows p, q
          const double apk = A[(size_t)pI * n + k], aqk = A[(size_t)q * n + k];
          A[(size_t)pI * n + k] = c * apk - sn * aqk;
          A[(size_t)q * n + k] = sn * apk + c * aqk;
        }
      }
  }
  double mx = 0.0;
  for (int a = 0; a < n; ++a) mx = std::max(mx, std::fabs(A[(size_t)a * n + a]));
  return mx;
}

// Julia: `isapprox(U'U, I)` against a UniformScaling uses the OPERATOR 2-norm with |I| = 1
// (LinearAlgebra: norm(A - J) <= max(atol, rtol * max(norm(A), |λ|)), norm = opnorm, rtol = sqrt(eps)).
extern "C" int lmm_orthogonal_validate(const double* U, int p, int m) {
  if (!U || p <= 0 || m <= 0) return LMM_E_ARG;
  std::vector<double> G((size_t)m * m), Dm((size_t)m * m);
  for (int a = 0; a < m; ++a)
    for (int b = 0; b <= a; ++b) {
      double s = 0.0;
      for (int j = 0; j < p; ++j) s += U[(size_t)a * p + j] * U[(size_t)b * p + j];
      if (!std::isfinite(s)) return LMM_E_NOT_ORTHOGONAL;
      G[(size_t)a * m + b] = G[(size_t)b * m + a] = s;
      Dm[(size_t)a * m + b] = Dm[(size_t)b * m + a] = s - (a == b ? 1.0 : 0.0);
    }
  const double rtol = 1.4901161193847656e-08;  // sqrt(eps(Float64))
  const double nrm = std::max(sym_opnorm(G, m), 1.0);
  if (!(sym_opnorm(Dm, m) <= rtol * nrm)) return LMM_E_NOT_ORTHOGONAL;
  return LMM_OK;
}

extern "C" int lmm_reorder_indices(int N, int p, int direction, int64_t* out) {
  if (N <= 0 || p <= 0 || !out || (direction != 0 && direction != 1)) return LMM_E_ARG;
  // direction 0: vec(reshape(1:pN, N, p)')  (src/independent_mogp.jl:138)
  // direction 1: vec(reshape(1:pN, p, N)')  (src/independent_mogp.jl:144)
  if (direction == 0) {
    for (int i = 0; i < N; ++i)
      for (int j = 0; j < p; ++j) out[(size_t)i * p + j] = (int64_t)j * N + i;
  } else {
    for (int j = 0; j < p; ++j)
      for (int i = 0; i < N; ++i) out[(size_t)j * N + i] = (int64_t)i * p + j;
  }
  return LMM_OK;
}
