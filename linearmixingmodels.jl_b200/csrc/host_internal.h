// Internal header of the liblmm host side (not installed): the context / posterior-handle structs, the device-buffer
// RAII helper and the prototypes shared by the host translation units
//   api.cu           contexts, communicators, options, host-only entry points
//   host_chol.cu     batched blocked Cholesky schedules (stream groups, look-ahead, row-cyclic multi-GPU), TRSM sweeps
//   host_latents.cu  the per-latent exact-GP driver: OILMM / IndependentMOGP logpdf, posterior, marginals
//   host_sample.cu   rand, posterior-predictive logpdf (+ gradient), hyper-parameter sweep
//   host_ilmm.cu     general-ILMM joint factor: logpdf, posterior, marginals, covariances, conditioning, dense-noise IMOGP
//   host_grad.cu     rrule of logpdf (OILMM, IndependentMOGP, general ILMM), sequential conditioning, cross-covariance
//   host_io.cu       serialisable posteriors, generic MVN logpdf / rand
// There is no CPU fallback anywhere on the host side: every compute entry point needs a CUDA device.
#pragma once
#include <cmath>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/lmm.h"
#include "kernels.h"

using namespace lmm;

constexpr double LOG2PI = 1.8378770664093453;  // log(2π)

// ------------------------------------------------------------------------------------------------
// NCCL through dlopen: no link-time dependency; picks up the libnccl.so.2 already loaded by the
// host process (torch bundles one) or the system one.
// ------------------------------------------------------------------------------------------------
struct NcclId { char internal[128]; };
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*CommSplit)(void*, int, int, void**, void*) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
};
NcclApi& nccl_api();
constexpr int NCCL_DOUBLE = 8, NCCL_SUM = 0, NCCL_MIN = 3;  // ncclFloat64, ncclSum, ncclMin

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct lmm_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::mutex mu;
  std::string err;
  int distance_form = 0;
  int outer_block = 8;
  bool outer_block_user = false;
  int nranks = 1, rank = 0;
  void* comm = nullptr;
  void* comm_small = nullptr;  // few-CTA communicator for the small, latency-critical exchanges on the panel chain
  int nccl_small_ctas = 0;  // 0: NCCL's own choice
  int64_t launches = 0, h2d = 0, d2h = 0;
  size_t total_mem = 0;  // device memory size, queried once (mem_fit)
  double timings[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  cudaEvent_t ev[8];
  // latent groups run their (latency-bound) panel steps on separate streams so that one group's
  // diagonal-tile factorisation overlaps the other groups' trailing updates
  static constexpr int MAX_GROUPS = 8;
  int ngroups = 4;
  cudaStream_t gstream[MAX_GROUPS];
  cudaEvent_t ev_fork, ev_join[MAX_GROUPS];
  // block-level look-ahead for small batches (ILMM: batch 1): panel stream (high priority) +
  // trailing-update stream, chained by per-block events
  cudaStream_t panel_stream = nullptr, update_stream = nullptr;
  std::vector<cudaEvent_t> blk_ev;
  int lookahead = 1;  // small batches (<= 2): 1 = right-looking block schedule on two streams (default), 0 = plain
  int chain_fused = 1;  // panel chain of a column (TRSM + next-column update + next diagonal tile) as ONE launch where the grids are small
  void* chain_cnt = nullptr;  // ready counters of the fused chain kernel
  size_t chain_cnt_bytes = 0;
  // one large factor (general ILMM, batch 1) partitioned row-cyclically over the ranks of the communicator
  int partition_ilmm = 0;
  int kmat_skip = 1;  // OILMM / IndependentMOGP evals: build only the kernel-matrix tiles that are not provably exact zeros (kmat.cu)
  int condition_update = 1;  // sequential conditioning of per-latent posteriors: 1 = block-Cholesky update of the factor, 0 = re-factorise the union
  int partition_now = 0;  // set by the callers whose factorisation is replicated on every rank (ILMM joint factor)
  int dist_error = 0;  // NCCL failure inside the partitioned schedule (reported by the caller)
  // integer-slice (Ozaki) trailing update on the int8 tensor cores: 0 = off (DMMA, default), 6 / 7 / 8 = digit planes
  int ozaki = 0;
  int ozaki_bits = 7;         // bits per digit plane: 7 = radix 128 (digits |q| <= 64), 8 = radix 256 (digits in [-128, 127])
  int ozaki_time = 0;         // 1: CUDA events around every int8 update launch; their sum (ms) and the tile products they cover are
                              // reported by lmm_ctx_last_timings in slots [7] and [5] (meaningful with "streams" = 1: serial launches)
  std::vector<cudaEvent_t> oz_events;
  double oz_tile_products = 0.0;
  int ozaki_single_nt = 96;   // batch <= 2: use the batched schedule (and with it the int8 update) from this many tile rows on (0 = never)
  int ozaki_min_k = 4;        // wide updates over fewer k-tiles stay on DMMA (the int8 epilogue is per output tile, not per k)
  int trsm_slice = 1;         // 1: the panel TRSMs of the int8 Cholesky write the digit planes of the tiles they finish; 0: a
                              // separate slice launch per block column (the same bytes)
  void* oz_slices = nullptr;  // [latents in flight][sym_tiles][S * 16 KB], grown on demand
  size_t oz_slices_bytes = 0;
  void* oz_x = nullptr;       // prediction sweep: digit planes + row scales of X
  size_t oz_x_bytes = 0;
  double* oz_scale = nullptr;
  size_t oz_scale_bytes = 0;
  uint8_t* oz_fp = nullptr;   // [latents in flight][sym_tiles]: first digit plane of each sliced factor tile with a nonzero digit (S: none)
  size_t oz_fp_bytes = 0;
  void* xbuf = nullptr;  // exchange buffers of the row-cyclic schedule (send | all-gathered), grown on demand
  size_t xbuf_bytes = 0;

  int fail(int code, const std::string& msg) {
    err = msg;
    return code;
  }
  int fail_cuda(cudaError_t e, const char* what, int line, const char* file = "liblmm") {
    char buf[512];
    snprintf(buf, sizeof buf, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e), file, line, what);
    err = buf;
    cudaGetLastError();  // clear non-sticky error state
    return e == cudaErrorMemoryAllocation ? LMM_E_OOM : LMM_E_CUDA;
  }
};

#define CU(expr)                                                        \
  do {                                                                  \
    cudaError_t e__ = (expr);                                           \
    if (e__ != cudaSuccess) return ctx->fail_cuda(e__, #expr, __LINE__, __FILE__); \
  } while (0)


namespace lmm_host {

struct DevBuf {
  lmm_ctx* c = nullptr;
  void* p = nullptr;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFreeAsync(p, c->stream);
    p = nullptr;
  }
  cudaError_t alloc(lmm_ctx* ctx, size_t bytes) {
    release();
    c = ctx;
    if (bytes == 0) bytes = 8;
    return cudaMallocAsync(&p, bytes, ctx->stream);
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
  void* detach() {
    void* q = p;
    p = nullptr;
    return q;
  }
};

inline int ntiles(int n) { return (n + TILE - 1) / TILE; }

// How many of `units` work items of `per_unit` bytes fit into 80 % of the free device memory (>= 1).  cudaMemGetInfo
// synchronises with the device and costs ~0.5 ms -- as much as a whole small-N eval -- so requests below 2 % of the
// device's memory skip it (an allocation that does not fit after all still fails cleanly with LMM_E_OOM).
inline cudaError_t mem_fit(lmm_ctx* ctx, size_t per_unit, int units, int* chunk) {
  size_t fr = 0, tot = 0;
  cudaError_t e;
  if (ctx->total_mem == 0) {
    if ((e = cudaMemGetInfo(&fr, &tot)) != cudaSuccess) return e;
    ctx->total_mem = tot;
  }
  if ((double)per_unit * (double)units <= 0.02 * (double)ctx->total_mem) {
    *chunk = units;
    return cudaSuccess;
  }
  if ((e = cudaMemGetInfo(&fr, &tot)) != cudaSuccess) return e;
  size_t fit = (size_t)((double)fr * 0.8) / (per_unit ? per_unit : 1);
  if (fit < 1) fit = 1;
  *chunk = (size_t)units < fit ? units : (int)fit;
  return cudaSuccess;
}

// Marks a factorisation that every rank of the communicator performs on identical inputs (the joint ILMM factor,
// the batch-1 potrf primitive): with the "partition_ilmm" option such a call runs the row-cyclic multi-GPU schedule.
struct PartitionScope {
  lmm_ctx* c;
  explicit PartitionScope(lmm_ctx* ctx) : c(ctx) { c->partition_now = 1; }
  ~PartitionScope() { c->partition_now = 0; }
};

}  // namespace lmm_host

// POST_JOINT: IndependentMOGP conditioned under a dense Σy (AbstractGPs generic path): one joint (mN) factor like
// POST_ILMM, identity mixing, no projection.
// POST_MASKED: heterotopic / missing-data dense model -- one factor over the observed entries (d_obs), any mixing matrix.
enum { POST_OILMM = 0, POST_IMOGP = 1, POST_ILMM = 2, POST_JOINT = 3, POST_MASKED = 4 };

struct lmm_post {
  lmm_ctx* ctx = nullptr;
  int kind = POST_OILMM;
  int m = 0, p = 0, N = 0, D = 1, nt = 0;
  int lo = 0, hi = 0;  // resident latents [lo, hi)
  std::vector<lmm_gp_desc> descs;  // descs[i].ard points into ard_store (or is NULL)
  std::vector<double> ard_store;   // m x D copies of the callers' ARD vectors
  std::vector<double> noise;  // per latent (all m)
  std::vector<double> H;      // p x m column-major (U sqrt(S) for OILMM)
  std::vector<double> U, S;
  double sigma2 = 0.0;
  // device
  double* d_xpad = nullptr;  // [Npad][D]
  double* d_L = nullptr;     // TiledSym, batch = hi - lo (ILMM: batch 1 over mN)
  double* d_W = nullptr;     // [batch][nt] tiles
  double* d_alpha = nullptr; // [batch][Npad]
  double* d_delta = nullptr; // [batch][Npad]
  LatentParams* d_params = nullptr;
  double* d_H = nullptr;
  double* d_noise_vec = nullptr;  // [nloc][Npad] per-point training noise (sequentially conditioned posteriors), else null
  int* d_obs = nullptr;           // POST_MASKED: observed entries j*N + i (big_n of them)
  double* d_Ept = nullptr;        // POST_ILMM: [N][m*m] per-point projected noise blocks ΣT (extended by sequential conditioning)
  int* d_env = nullptr;           // [nloc][nt] tile envelope of the factors (OILMM / IndependentMOGP built inside it), else null
  bool zeros_pending = false;     // the tiles (I, k < env) of d_L were never written: post_fill_zeros writes them before a read
  size_t bytes = 0;
  int big_n = 0, big_nt = 0;  // ILMM joint dimension mN and its tile count

  std::vector<lmm_kernel_term> term_store;  // m x (LMM_MAX_TERMS-1) copies of the callers' extra terms (composite kernels)
  std::vector<double> term_ard_store;       // m x (LMM_MAX_TERMS-1) x D copies of their ARD vectors
  // deep copy of the latent descriptions (the caller's ARD / extra-term arrays are only valid during its call)
  void adopt_descs(const lmm_gp_desc* d, int m_, int D_) {
    constexpr int XT = LMM_MAX_TERMS - 1;
    descs.assign(d, d + m_);
    ard_store.assign((size_t)m_ * D_, 0.0);
    term_store.assign((size_t)m_ * XT, lmm_kernel_term{});
    term_ard_store.assign((size_t)m_ * XT * D_, 0.0);
    for (int i = 0; i < m_; ++i) {
      if (d[i].ard) {
        for (int k = 0; k < D_; ++k) ard_store[(size_t)i * D_ + k] = d[i].ard[k];
      }
      for (int t = 0; t < d[i].n_extra && t < XT; ++t) {
        lmm_kernel_term q = d[i].extra[t];
        if (q.ard)
          for (int k = 0; k < D_; ++k) term_ard_store[((size_t)i * XT + t) * D_ + k] = q.ard[k];
        term_store[(size_t)i * XT + t] = q;
      }
    }
    repoint_descs(D_);
  }
  // make every pointer inside descs / term_store refer to this handle's own copies (after adopt_descs or a load)
  void repoint_descs(int D_) {
    constexpr int XT = LMM_MAX_TERMS - 1;
    for (size_t i = 0; i < descs.size(); ++i) {
      if (descs[i].ard) descs[i].ard = ard_store.data() + i * D_;
      for (int t = 0; t < XT; ++t) {
        lmm_kernel_term& q = term_store[i * XT + t];
        if (q.ard) q.ard = term_ard_store.data() + (i * XT + t) * D_;
      }
      descs[i].extra = descs[i].n_extra > 0 ? term_store.data() + i * XT : nullptr;
    }
  }
  int nloc() const { return hi - lo; }
  size_t npad() const { return (size_t)nt * TILE; }
  bool joint() const { return kind == POST_ILMM || kind == POST_JOINT || kind == POST_MASKED; }
  TiledSym Lsym() const { return TiledSym{d_L, joint() ? big_nt : nt, sym_tiles(joint() ? big_nt : nt) * TT}; }
  size_t wstride() const { return (size_t)(joint() ? big_nt : nt) * TT; }
};

namespace lmm_host {

// Projection description (host): Ty = T Y  (m x p), residual |Y - Q (P Y)|², regulariser constant.
struct Projection {
  std::vector<double> T;      // m x p col-major
  std::vector<double> P, Q;   // m x p, p x m (empty: no regulariser)
  std::vector<double> noise;  // per latent diagonal noise
  double reg_c0 = 0.0;        // n * (...) part of the regulariser
  bool has_reg = false;
};

struct RunOut {
  lmm_post** post = nullptr;
  double* logpdf = nullptr;
  double* lml_terms = nullptr;
  int* info_latent = nullptr;
};

struct Predictive {
  DevBuf params, xs, V, C, W, logdet, info, ML;
  int nts = 0;
  size_t nspad = 0;
};

struct GeneralProjection {
  Projection pr;            // T, P (= T), Q (= H), has_reg
  std::vector<double> ST;   // ΣT m x m col-major
  std::vector<double> Winv; // (H'H/σ² + 1e-9 I)^{-1}, m x m col-major (gradient chain)
  double logdet_ST = 0.0;
};

// One joint (q*N x q*N) exact-GP solve shared by the general ILMM (projected / dense form), the
// IndependentMOGP with a dense Σy and sequential conditioning of a joint posterior: assemble the
// covariance straight into the factor tiles, factor, z = L^{-1}δ, quad = |z|², optionally α = L^{-T}z.
struct JointBuild {
  int m = 0, q = 0, N = 0, D = 1, mode = 0;  // assemble mode (assemble.cu)
  int big = 0, bnt = 0;
  size_t bpad = 0;
  DevBuf x, params, H, E, delta, L, W, alpha, logdet, info, quad;
  double hlogdet = 0.0, hquad = 0.0;
};

constexpr int FORM_IMOGP_DENSE = 2;  // internal: IndependentMOGP with a dense Σy (AbstractGPs generic path)

// ---- prototypes (definitions in the host_*.cu files)
bool is_device_ptr(const void* p);
cudaError_t copy_in(lmm_ctx* ctx, double* dst, const double* src, size_t n);
cudaError_t copy_out(lmm_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes);
void shard_range(const lmm_ctx* ctx, int m, int& lo, int& hi);
int check_descs(lmm_ctx* ctx, const lmm_gp_desc* d, int m, int D);
double desc_kdiag(const lmm_gp_desc& d);         // k(x, x) of the whole (possibly composite) kernel
bool desc_is_composite(const lmm_gp_desc& d);   // more than one term, or a non-(Sq)Euclidean metric (PeriodicKernel)
void set_params(LatentParams& q, const lmm_gp_desc& d, double noise, double ls_scale, int D);
size_t factor_bytes_per_latent(int nt);
void fill_params(std::vector<LatentParams>& hp, const lmm_gp_desc* d, const double* noise, int lo, int hi, int D, double ls_scale = 1.0);
int latents_run(lmm_ctx* ctx, int kind, const lmm_gp_desc* latents, int m, const double* x, int N, int D, int p, double sigma2, const double* y, const Projection& pr, const double* Hhost, const double* Uhost, const double* Shost, RunOut out, const double* noise_vec = nullptr);
int oilmm_projection(lmm_ctx* ctx, const double* U, const double* S, int p, int m, double sigma2, int N, Projection& pr, std::vector<double>& H);
int check_common(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const void* x, int N, int D, int p, int out_dim);
// Every entry point that reads a posterior's factor calls this first: it writes the exact zeros the kernel-matrix build left out.
int post_fill_zeros(lmm_post* post);
int post_latent_marginals(lmm_post* post, const double* d_xspad, int Ns, int nts, double* d_ML, double* d_VL, int first = 0, int count = -1);
int upload_params(lmm_ctx* ctx, DevBuf& buf, const lmm_gp_desc* descs, const double* noise_all, int lo, int hi, int D);
int stage_latent_vectors(lmm_ctx* ctx, DevBuf& buf, const double* z, int N, size_t npad, int lo, int hi);
int report_info(lmm_ctx* ctx, const std::vector<int>& hinfo, int lo, int nmax, int* info_latent);
int prior_latent_samples(lmm_ctx* ctx, const lmm_gp_desc* descs, const double* noise_all, int lo, int hi, const double* d_xpad, int N, int D, const double* d_z, double* d_X, int* info_latent);
int mix_and_add_noise(lmm_ctx* ctx, const double* Hhost, int p, int m, int lo, int hi, const double* d_X, size_t npad, int N, double sigma2, const double* z_noise, double* out);
int stage_xpad(lmm_ctx* ctx, DevBuf& buf, const double* x, int N, int D);
int build_predictive(lmm_post* post, const double* xs, int Ns, const std::vector<double>& noise_all, Predictive& P, int* info_latent, bool factor = true);
bool host_chol(std::vector<double>& A, int n);
void host_chol_solve(const std::vector<double>& L, int n, double* b);
int general_projection(lmm_ctx* ctx, const double* H, int p, int m, double sigma2, int N, GeneralProjection& gp);
void identity_projection(int m, double sigma2, GeneralProjection& gp);
std::vector<double> hmm(const std::vector<double>& A, int ar, int ac, bool ta, const std::vector<double>& B, int br, int bc, bool tb);
double hdot(const std::vector<double>& A, const std::vector<double>& B);
int ilmm_grad_chain(lmm_ctx* ctx, const GeneralProjection& gp, const std::vector<double>& Hh, int p, int m, int N, double sigma2, double hres, const std::vector<double>& B, std::vector<double> bT, const std::vector<double>& bH, double* grad_sigma2, double* grad_H);
int joint_factor(lmm_ctx* ctx, JointBuild& J, bool want_alpha, int* info);
lmm_post* joint_make_post(lmm_ctx* ctx, JointBuild& J, int kind, const lmm_gp_desc* latents, const double* Hhost, int p, double sigma2, DevBuf& Ept);
int ilmm_run(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D, const double* H, int p, double sigma2, const double* y, int form, lmm_post** out_post, double* out_logpdf, int* info, const double* dense_noise = nullptr);
int ilmm_post_mean_and_var(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean, double* var);
int ilmm_post_rand(lmm_post* post, const double* xs, int Ns, double sigma2, const double* z_latent, const double* z_noise, double* out, int* info);
int ilmm_post_logpdf(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, double* out_logpdf, double* grad_sigma2, double* grad_y, int* info);
int ilmm_post_condition(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, lmm_post** out_post, int* info);
// env_d / env_h (both or neither; jstart = 0): the tile envelope of the batch (launch_kmat_sym) on the device and a host copy of it.
// The batched left-looking schedule then skips every tile product, TRSM and slice that has an all-zero operand -- the factor is
// bit-identical to the dense schedule's -- and sizes its grids from the host copy.  The other schedules ignore it.
// Whether chol_factor (jstart = 0) factors `batch` matrices of nt tile rows on the batched left-looking schedule, the one that
// takes the envelope.  The others read every tile: chol_factor writes the zeros outside the envelope before it runs them.
bool chol_takes_envelope(const lmm_ctx* ctx, int nt, int batch);
cudaError_t chol_factor(lmm_ctx* ctx, TiledSym L, double* W, size_t wstride, int batch, double* logdet, int* info, int jstart = 0,
                        const int* env_d = nullptr, const int* env_h = nullptr);
cudaError_t chol_factor_rowcyclic_dist(lmm_ctx* ctx, TiledSym Lown, int nrows, int nc, double* W, size_t wstride, double* logdet, int* info,
                                       double* zvec);
size_t rowcyclic_dist_workspace_tiles(int nrows, int G, int ob);
int rowcyclic_dist_block(const lmm_ctx* ctx, int nc);
cudaError_t trsm_right_lt(lmm_ctx* ctx, TiledRect X, TiledSym L, const double* W, size_t wstride, int batch, const LatentParams* xbound = nullptr);
cudaError_t trsm_right_lt_upper(lmm_ctx* ctx, cudaStream_t st, TiledRect X, TiledSym L, const double* W, size_t wstride, int batch);
void masked_observations(const lmm_gp_desc* latents, int m, const double* H, int p, int N, const double* y, std::vector<int>& obs,
                         std::vector<double>& delta);
bool per_input_mask(const double* y, int p, int N, std::vector<int>& keep);

constexpr int TERM_SLOTS = LMM_MAX_TERMS * LMM_GRAD_TERM_STRIDE;  // grad_terms doubles per latent
void terms_shape(const lmm_gp_desc* latents, int lo, int hi, int& max_terms, bool& any_ard);

struct GradOut {
  double* logpdf;
  double* grad_latents;  // m x 3: d/d variance, d/d inv_lengthscale, d/d mean_const
  double* grad_sigma2;
  double* grad_y;        // p*N by outputs (nullable)
  int* info_latent;
  double* grad_U = nullptr;  // p x m column-major (OILMM only, nullable)
  double* grad_S = nullptr;  // m (OILMM only, nullable)
  const double* Yhost_or_dev = nullptr;
  double* grad_ard = nullptr;  // m x D row-major: d/d ARD multiplier (zeros for latents without an ARDTransform; nullable)
  double* grad_terms = nullptr;  // m x LMM_MAX_TERMS x LMM_GRAD_TERM_STRIDE: per-term gradients (nullable)
};

// The OILMM / IndependentMOGP logpdf gradient (host_grad.cu) and the LOO driver (host_loo.cu) share everything but the
// per-latent loop.  grad_run_setup stages the inputs, projects the data (δ = T y - m in b_ty, regulariser pieces) and
// allocates the reduction buffers; the loop leaves per latent a [mloc][npad] vector a (α for the logpdf, w for LOO) with
// dvalue/dδ = -a, hg4[i*4 + {0,1,2,3}] = {d/d variance, d/d inv_lengthscale, d/d noise, Σ a}, hdot[i] = a·δ, the value
// terms in b_vec[lo + i] and (when asked) b_gard / b_gterms; grad_run_finish runs the chain to U, S, σ², y and the means.
struct GradRun {
  int lo = 0, hi = 0, mloc = 0, nt = 0, nl = 1;
  size_t npad = 0, nvec = 0;
  bool multi = false, do_reg = false, want_U = false, want_R = false, want_Z = false, want_ard = false;
  int max_terms = 1;
  bool terms_ard = false;
  const double* d_y = nullptr;
  DevBuf b_x, b_y, b_T, b_P, b_Q, b_means, b_ty, b_part, b_resid, b_R, b_Z, b_params, b_vec, b_gard, b_gterms;
};
int grad_run_setup(lmm_ctx* ctx, bool orth, const lmm_gp_desc* latents, int m, const double* x, int N, int D, int p, const double* y,
                   const Projection& pr, const GradOut& out, GradRun& s);
int grad_run_finish(lmm_ctx* ctx, bool orth, const lmm_gp_desc* latents, int m, int N, int D, int p, double sigma2, const Projection& pr,
                    const double* Shost, GradOut out, GradRun& s, const double* d_a, const std::vector<int>& hinfo,
                    const std::vector<double>& hg4, const std::vector<double>& hdot);
// What post_logpdf_impl leaves behind for the gradient through the conditioning (host_post_grad.cu): the predictive factors
// and inputs (P), β_i = Σ*_i⁻¹(ỹ*_i - μ_i) of the resident latents [nloc][P.nspad], and the rank-summed gradient pieces
// hg = [β_i'β_i (m) | tr(Σ*_i⁻¹) (m) | |R*|² (1)].
struct PredictiveKeep {
  Predictive P;
  DevBuf beta;
  std::vector<double> hg;
};
int post_logpdf_impl(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys, double* out_logpdf, double* grad_sigma2,
                     double* grad_y, int* info_latent, PredictiveKeep* keep = nullptr);

}  // namespace lmm_host
namespace lmm_host {
int masked_post_mean_and_var(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean, double* var);
int masked_post_mean_and_cov(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean, double* cov);
int masked_post_rand(lmm_post* post, const double* xs, int Ns, double sigma2, const double* z, double* out, int* info);
}
using namespace lmm_host;
