/*
 * lmm.h -- C ABI of liblmm.so: the B200 (sm_100a) implementation of the LinearMixingModels.jl
 * inference hot path.  This is the drop-in boundary: the Julia shim
 * (linearmixingmodels.jl_b200/julia/LinearMixingModelsB200.jl) binds these symbols with `ccall`
 * and keeps the reference's exported types/method signatures; the Python host mirror
 * (linearmixingmodels.jl_b200/api.py) binds the same symbols with ctypes.
 *
 * The reference has no FFI of its own (pure Julia multiple dispatch).  Each entry point below
 * names the reference method body (file:line under /root/reference) it replaces.
 *
 * Conventions
 *  - Every function returns int: 0 = ok; > 0 = LAPACK-style `info` (1-based index of the first
 *    non-positive pivot; the failing latent is reported through lmm_last_error and *info_latent)
 *    -> Julia PosDefException(info); < 0 = LMM_E_* below.
 *  - All matrices are column-major Float64 (Julia Matrix / NumPy order='F').  Multi-output vectors
 *    are "by outputs": y[(j-1)N + i] = output j at input i == the N x p column-major matrix
 *    (src/ilmm.jl:43 reshape_y).  x is D x N column-major (ColVecs; a Vector{Float64} has D = 1).
 *  - Pointer arguments are HOST memory owned by the caller unless documented otherwise; x / y
 *    / U / S / H inputs may alternatively be DEVICE pointers on the context's GPU (detected with
 *    cudaPointerGetAttributes) -- bench.py's HBM-resident timing uses that.  The library never
 *    retains a caller pointer after return.
 *  - Calls are synchronous and thread-safe per context (one mutex per lmm_ctx; cudaSetDevice on
 *    entry).  A posterior handle belongs to the context that created it: free every lmm_post
 *    before destroying its lmm_ctx.  There is no CPU fallback: without a CUDA device every compute entry returns
 *    LMM_E_CUDA.
 */
#ifndef LMM_H_
#define LMM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LMM_OK 0
#define LMM_E_ARG (-1)            /* bad argument / null pointer / non-positive size          */
#define LMM_E_OUT_DIM (-2)        /* "out dim of x != out dim of f."  src/ilmm.jl:52          */
#define LMM_E_UNSUPPORTED (-3)    /* kernel / mean / option outside the supported set         */
#define LMM_E_CUDA (-4)           /* CUDA runtime error or no device                          */
#define LMM_E_NCCL (-5)           /* NCCL unavailable or failed                               */
#define LMM_E_NOT_ORTHOGONAL (-6) /* "`U` is not an orthogonal matrix" src/orthogonal_matrix.jl:22 */
#define LMM_E_OOM (-7)            /* device memory exhausted                                  */

/* Base kernels (KernelFunctions.jl): SEKernel, Matern32Kernel, Matern52Kernel, ExponentialKernel (= Matern12Kernel,
 * κ(d) = exp(-d)), RationalQuadraticKernel(α) (κ(d²) = (1 + d²/(2α))^(-α), α in `param`) and PeriodicKernel(r)
 * (metric Sinus(r): κ = exp(-0.5 Σ_k (sinpi(x_k - x'_k) / r)²), one r for all dimensions, in `param`). */
#define LMM_KERNEL_SE 0
#define LMM_KERNEL_MATERN32 1
#define LMM_KERNEL_MATERN52 2
#define LMM_KERNEL_EXPONENTIAL 3
#define LMM_KERNEL_RATIONAL_QUADRATIC 4
#define LMM_KERNEL_PERIODIC 5

/* Composite kernels (KernelFunctions `k1 + k2` = KernelSum, `k1 * k2` = KernelProduct; the reference accepts any
 * AbstractGP latent, src/independent_mogp.jl:10-12): a flat sum or product of up to LMM_MAX_TERMS scaled, stretched base
 * kernels.  Term 0 is the descriptor's own (kind, variance, inv_lengthscale, ard, param); terms 1.. are `extra[0..n_extra)`.
 *   LMM_COMPOSE_SUM:      k(x,x') = Σ_t variance_t κ_t(s_t x, s_t x')     (seasonal + trend latents)
 *   LMM_COMPOSE_PRODUCT:  k(x,x') = Π_t variance_t κ_t(s_t x, s_t x')     (locally periodic latents)
 * Each term is evaluated exactly like a single kernel (own input scaling, own pairwise distances), then combined left
 * to right, as KernelFunctions' kernelmatrix(::KernelSum / ::KernelProduct) does. */
#define LMM_COMPOSE_NONE 0
#define LMM_COMPOSE_SUM 1
#define LMM_COMPOSE_PRODUCT 2
#define LMM_MAX_TERMS 4
typedef struct lmm_kernel_term {
  int32_t kind;           /* LMM_KERNEL_*                                   */
  int32_t reserved;       /* must be 0                                      */
  double variance;        /* ScaledKernel σ² of this term                   */
  double inv_lengthscale; /* ScaleTransform s of this term                  */
  double param;           /* shape parameter (α / r) of this term's kernel  */
  const double* ard;      /* ARDTransform multipliers of this term (D values) or NULL */
} lmm_kernel_term;

/* One latent `GP(mean_const, variance * (base_kernel ∘ ScaleTransform(inv_lengthscale) [∘ ARDTransform(ard)]))`, optionally
 * summed / multiplied with further terms (above).  Inputs are multiplied by inv_lengthscale (and, per dimension, by ard[k])
 * BEFORE distances are taken (KernelFunctions semantics, SURVEY.md App. A.3). */
#define LMM_MAX_ARD 8
typedef struct lmm_gp_desc {
  int32_t kind;           /* LMM_KERNEL_*                                   */
  int32_t compose;        /* LMM_COMPOSE_NONE (single kernel), _SUM or _PRODUCT over term 0 and `extra` */
  double variance;        /* ScaledKernel σ² (1.0 for a plain kernel)       */
  double inv_lengthscale; /* ScaleTransform s (1.0 for a plain kernel)      */
  double mean_const;      /* ZeroMean -> 0.0; ConstMean(c) -> c             */
  const double* ard;      /* ARDTransform v: D positive per-dimension multipliers (D <= LMM_MAX_ARD), or NULL;
                             read during the call only (posterior handles keep their own copy)           */
  double param;           /* shape parameter of the base kernel: α of RationalQuadraticKernel, r of PeriodicKernel; else ignored */
  int32_t n_extra;        /* number of further terms, 0 .. LMM_MAX_TERMS - 1 (must be 0 when compose == LMM_COMPOSE_NONE) */
  int32_t reserved2;      /* must be 0                                      */
  const lmm_kernel_term* extra; /* n_extra terms, read during the call only (or NULL)                        */
} lmm_gp_desc;

typedef struct lmm_ctx lmm_ctx;   /* owns device, stream, memory pool, optional NCCL communicator */
typedef struct lmm_post lmm_post; /* device-resident posterior: per-latent factor L_i, α_i, δ_i, x */

/* ---- context ------------------------------------------------------------------------------ */
int lmm_ctx_create(int device, lmm_ctx** out);
int lmm_ctx_destroy(lmm_ctx* ctx);
const char* lmm_last_error(lmm_ctx* ctx);
const char* lmm_version(void);
/* Tunables (key, value):
 *   "distance_form"   0 = Distances.jl form |a|²+|b|²-2a·b clamped at 0 [default], 1 = direct differences
 *   "outer_block"     tile columns per outer Cholesky step (default 8 for batched work, 1-4 by size for the
 *                     look-ahead schedules); 0 = back to automatic
 *   "streams"         latent groups factored concurrently on separate CUDA streams (default 4, 1..8)
 *   "lookahead"       schedule for batches <= 2: 1 = right-looking block schedule, the next block column on a high-priority
 *                     panel stream, the rest of the trailing update as one large GEMM on a second stream [default]; 0 = plain
 *   "kmat_skip"       OILMM / IndependentMOGP logpdf and posterior: 1 = build only the kernel-matrix tiles that are not provably
 *                     exact zeros (far-apart point tiles of the SE / Matern kernels) [default]; a kept posterior writes those
 *                     zeros on its first read.  0 = build every tile.  The results are the same bits either way.
 *   "chain_fused"     1 = where the grids are small (batches <= 2, or few latents x few tile rows) the panel chain of a tile
 *                     column -- TRSM of the column, update of the next column(s), factorisation of the next diagonal tile --
 *                     is ONE launch whose CTAs hand tiles to each other through ready counters in global memory, the
 *                     critical tiles first [default: single factors up to N = 4096, the last 31 tile columns of larger ones
 *                     and small batched grids -- where the chain is the run time]; 2 = everywhere (measured slower from
 *                     N = 8192 on: the trailing GEMMs set the time there); 0 = one launch per operation, chained by "pdl"
 *   "pdl"             programmatic dependent launch along the panel chain: the diagonal-tile kernel, the small direct GEMMs
 *                     and the fused chain kernel are launched with programmatic stream serialisation, wait on
 *                     `griddepcontrol.wait` before their first read and release their successor before their final
 *                     stores.  Default 1; 0 = plain launches.            [process-wide]
 *   "partition_ilmm"  1 = the joint factor of a general ILMM (one large matrix, factored by every rank of the communicator
 *                     on identical inputs) is partitioned row-cyclically over the ranks: one ncclAllGather of the current
 *                     block column per step, panels redundant.  Every rank must make the same calls.  Default 0 (replicas).
 *                     2 = as 1, and lmm_ilmm_logpdf additionally DISTRIBUTES THE STORAGE: every rank assembles and keeps only
 *                     the tile rows it owns (1/G of the joint matrix) plus two block-column windows; both operands of every
 *                     trailing update come from the all-gathered window, the right-hand side rides along as an extra tile
 *                     row (z = L^{-1} δ falls out of the panel TRSMs), so a joint dimension that does not fit one GPU runs.
 *                     Calls that need the whole factor afterwards (posterior, gradient) behave as with 1.
 *   "nccl_small_ctas" CTA cap of the panel-chain communicator (takes effect at lmm_comm_init; 0 = NCCL's choice)
 *   "gemm_small"      grids of at most this many tiles use the latency-optimised direct kernel (8 row slices per tile, no
 *                     shared memory, zero blocks of the triangular inverse skipped) instead of the TMA-pipelined one
 *                     (default 74, 0 = never)                            [process-wide]
 *   "project_impl"    projection + regulariser residual (T*Y, (I - UU')Y): 1 = FP64 tensor-core (DMMA) kernel with the column
 *                     block / row split sized to the SM count (default); 0 = register-tiled scalar-FMA kernel  [process-wide]
 *   "condition_update" lmm_post_condition on an OILMM / IndependentMOGP posterior: 1 = block-Cholesky update of each latent's
 *                     factor, L21 = K21 L11^{-T}, L22 = chol(K22 + Σ2 - L21 L21'), O(N² N₂) (default, what AbstractGPs does);
 *                     0 = re-factorise the union of the inputs, O((N + N₂)³)
 *   "ozaki"           6 | 7 | 8: the WIDE trailing update of the batched blocked Cholesky runs as an integer-slice (Ozaki-scheme) product on
 *                     the int8 tensor cores (tcgen05.mma kind::i8, exact int32 accumulation in TMEM) with that many 7-bit digit
 *                     planes per FP64 operand, instead of FP64 DMMA -- and so do the wide updates of the prediction sweep K(x*,x) L^{-T} of
 *                     per-latent posteriors (mean_and_var / marginals); everything else (panels, in-block updates, TRSMs, solves, kernel
 *                     matrices) stays FP64.  8 planes truncate at 2^-56 of the row scale (measured normwise factor error 2e-14, DMMA 6e-16 .. 2e-14);
 *                     each plane less costs 2^7 in accuracy and saves ~12 % of the update time.  Default 0 = DMMA (the north
 *                     star's prescription); LMM_OZAKI in the environment sets the initial value.
 *   "ozaki_bits"      bits per digit plane: 7 = radix 128, digits |q| <= 64 (default; P planes carry 6 + 7 (P - 1) bits, exact int32 sums for
 *                     K * P < 524288 columns) or 8 = radix 256, balanced digits in [-128, 127] (6 + 8 (P - 1) bits: 7 planes = 54 bits with 28
 *                     instead of 36 MMAs per tile product; exact int32 sums for K * P < 131072 columns, i.e. N <= 18724 at 7 planes --
 *                     beyond that the update of a block column falls back to DMMA).  LMM_OZAKI_BITS sets the initial value.
 *   "ozaki_min_k"     wide updates over fewer k-tiles than this stay on DMMA (default 4: the int8 epilogue costs per output tile); with
 *                     "ozaki" on, "outer_block" defaults to 2 tile columns (the in-block updates stay on DMMA), and to 1 for the
 *                     banded factors of the OILMM / IndependentMOGP eval from 64 tile rows (N >= 8192) on (every update of a column by
 *                     earlier ones takes the int8 path)
 *   "trsm_slice"      with "ozaki" on: 1 (default) = the panel TRSMs write the int8 digit planes of the tiles they finish; 0 = a separate
 *                     slice pass per block column (the same bytes: results are bit-identical)
 *   "ozaki_single_nt" with "ozaki" on, batches <= 2 keep the right-looking DMMA schedule unless the factor has at least this many tile
 *                     rows (two thirds of it for a batch of 2), from which on it takes the batched schedule and with it the int8 update
 *                     (default 96, i.e. N >= 12288: N = 16384: 45.9 -> 33 ms, two factors 88.9 -> 44 ms, while a single N = 8192
 *                     factor is faster on the right-looking DMMA schedule: 7.1 vs 8.6 ms; 0 = never)
 *   "ozaki_time"      1 = time every int8 update launch with CUDA events: see lmm_ctx_last_timings (default 0)
 *   "solve_impl"      triangular vector solves (z = L^{-1} r, a = L^{-T} z): 1 = ONE persistent launch per direction, tile rows /
 *                     columns chained through ready flags in global memory (default); 0 = one launch per tile column
 *                                                                 [process-wide] */
int lmm_ctx_set_option(lmm_ctx* ctx, const char* key, double value);
/* Counters since context creation: kernels launched by this library, bytes copied H2D / D2H. */
int lmm_ctx_counters(lmm_ctx* ctx, int64_t* kernel_launches, int64_t* h2d_bytes, int64_t* d2h_bytes);
/* CUDA-event time (ms) of the device work of the most recent compute call, and of its dominant
 * stages: [0] total, [1] kernel-matrix build, [2] Cholesky, [3] solves, [4] projection,
 * [5] prediction (cross-cov + TRSM + back-projection), [6] Cholesky trailing-update GEMM launches
 * count (as a double), [7] reserved.  After a distributed-storage ILMM logpdf ("partition_ilmm" = 2) the slots [4], [5], [7]
 * hold BYTES instead: the matrix rows this rank stores, its exchange / window workspace, the whole packed matrix.  With the option
 * "ozaki_time" = 1, [7] is the summed CUDA-event time (ms) of the int8 trailing-update launches since the previous query and [5] the
 * number of 128^3 tile products they covered (serial launches, i.e. "streams" = 1, make the sum a duration). */
int lmm_ctx_last_timings(lmm_ctx* ctx, double out_ms[8]);

/* ---- multi-GPU: one process (and one context) per GPU; latents are block-sharded over ranks --- */
/* (no counterpart in the reference: it is single-process; SURVEY.md §8e) */
int lmm_comm_unique_id(void* out_128_bytes);
int lmm_comm_init(lmm_ctx* ctx, const void* unique_id_128_bytes, int nranks, int rank);
/* Without NCCL (tests on CPU-only hosts, gloo plumbing): declare the shard only; the caller
 * reduces `lml_terms` / partial back-projections itself. */
int lmm_comm_set_shard(lmm_ctx* ctx, int nranks, int rank);

/* ---- Orthogonal(U, S): src/orthogonal_matrix.jl:21-23 (_validate) ----------------------------- */
/* U is p x m column-major.  Host-side check `isapprox(U'U, I)`; returns LMM_E_NOT_ORTHOGONAL. */
int lmm_orthogonal_validate(const double* U, int p, int m);

/* ---- OILMM: src/oilmm.jl -------------------------------------------------------------------- */
/* logpdf(fx::FiniteGP{<:OILMM}, y)  src/oilmm.jl:79-93 (+ project :20-30, regulariser :101-113).
 * out_dim is fx.x.out_dim (checked against p: src/ilmm.jl:52).  lml_terms (nullable) receives
 * the m per-latent terms followed by the regulariser (m+1 doubles). */
int lmm_oilmm_logpdf(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                     const double* U, const double* S, int p, double sigma2, const double* y,
                     int out_dim, double* out_logpdf, double* lml_terms, int* info_latent);

/* posterior(fx::FiniteGP{<:OILMM}, y)  src/oilmm.jl:116-134.  One factorisation per latent is
 * shared with the logpdf when out_logpdf != NULL (the reference factorises twice). */
int lmm_oilmm_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N,
                        int D, const double* U, const double* S, int p, double sigma2,
                        const double* y, int out_dim, lmm_post** out_post, double* out_logpdf,
                        double* lml_terms, int* info_latent);

/* mean_and_var(fx::FiniteGP{<:OILMM}) on *prior* latents  src/oilmm.jl:57-76.  mean/var are
 * p*Ns by outputs. */
int lmm_oilmm_prior_mean_and_var(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* xs,
                                 int Ns, int D, const double* U, const double* S, int p,
                                 double sigma2, int out_dim, double* mean, double* var);

/* rand(rng, fx::FiniteGP{<:OILMM}) on prior latents  src/oilmm.jl:40-54.  z_latent: m*N standard
 * normals (latent-major, the order Julia's rng is consumed in); z_noise: p*N. */
int lmm_oilmm_rand(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                   const double* U, const double* S, int p, double sigma2, int out_dim,
                   const double* z_latent, const double* z_noise, double* out, int* info_latent);

/* Hyper-parameter sweep (BASELINE config 5): logpdf for n_sweep inverse-lengthscale settings
 * applied to every latent (multiplying each latent's own inv_lengthscale); the projection and
 * regulariser are shared, factors are streamed through one arena. out: n_sweep doubles. */
int lmm_oilmm_logpdf_sweep(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N,
                           int D, const double* U, const double* S, int p, double sigma2,
                           const double* y, int out_dim, const double* inv_lengthscale_scales,
                           int n_sweep, double* out_logpdfs, int* info_latent);

/* rrule of logpdf (SURVEY.md §8f-1; `Zygote.gradient(logpdf, fx, y)` at test/oilmm.jl:31-32,
 * test/independent_mogp.jl:65-66 needs a ChainRulesCore.rrule around the opaque ccall): value and
 * gradients w.r.t. each latent's (variance, inv_lengthscale, mean_const) -- grad_latents is m x 3
 * row-major --, the observation noise σ², y (p*N by outputs) and the mixing matrix fields U (p x m
 * column-major, the unconstrained Euclidean gradient of the reference's expressions) and S (m).
 * grad_ard (m x D row-major) receives the gradient w.r.t. each latent's ARD multipliers (zeros for latents without an
 * ARDTransform).  All outputs nullable.  G_i = (α_i α_i' - C_i^{-1})/2 comes from a batched potri on the tensor pipe. */
int lmm_oilmm_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N,
                          int D, const double* U, const double* S, int p, double sigma2,
                          const double* y, int out_dim, double* out_logpdf, double* grad_latents,
                          double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_U, double* grad_S,
                          int* info_latent);
int lmm_imogp_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D,
                          double sigma2, const double* y, int out_dim, double* out_logpdf,
                          double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y,
                          int* info_latent);

/* The same rrules for every latent the value path accepts (KernelSum / KernelProduct of up to LMM_MAX_TERMS terms,
 * PeriodicKernel, RationalQuadraticKernel), with the gradient w.r.t. the hyper-parameters of each term.  grad_terms
 * (required) receives m x LMM_MAX_TERMS x LMM_GRAD_TERM_STRIDE doubles: term t of latent i starts at
 * (i*LMM_MAX_TERMS + t)*LMM_GRAD_TERM_STRIDE and holds d/d variance, d/d inv_lengthscale, d/d param (α / r) and
 * d/d ard[0..LMM_MAX_ARD); term 0 is the descriptor's own fields, terms 1.. are `extra[]`.  Slots of absent terms, the
 * `param` slot of kinds without a shape parameter and the ARD slots of terms without an ARDTransform (or k >= D) are 0.
 * grad_latents[:, 0:2] and grad_ard hold term 0's values (for single-kernel latents exactly what lmm_*_logpdf_grad
 * returns), grad_latents[:, 2] the mean gradient; every other output is that of lmm_*_logpdf_grad.  With a communicator
 * grad_terms is summed over the ranks like grad_ard. */
#define LMM_GRAD_TERM_STRIDE (3 + LMM_MAX_ARD)
int lmm_oilmm_logpdf_grad_terms(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N,
                                int D, const double* U, const double* S, int p, double sigma2,
                                const double* y, int out_dim, double* out_logpdf, double* grad_latents,
                                double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_U,
                                double* grad_S, double* grad_terms, int* info_latent);
int lmm_imogp_logpdf_grad_terms(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D,
                                double sigma2, const double* y, int out_dim, double* out_logpdf,
                                double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y,
                                double* grad_terms, int* info_latent);

/* Leave-one-input-out cross-validation (Rasmussen & Williams §5.4.2): out_loo = Σ_i log p(y_i | y_{-i}) where y_i is all p
 * outputs at input x_i -- the closed form of N refits, at the cost of a factorisation plus one N³/3 TRSM per latent for
 * the value, about twice the logpdf gradient's cost with a gradient.  For an OILMM it is Σ_l (GP LOO of latent l on the
 * projected data, noise σ²/S_l) + the regulariser logpdf adds.  loo_mean / loo_var (p*N by outputs) are the LOO predictive
 * marginals: what mean_and_var(posterior(f(x_{-i}, σ²), y_{-i})(x_i, σ²)) returns at each x_i.  The gradient outputs use the
 * layouts of lmm_oilmm_logpdf_grad_terms (grad_latents m x 3: term 0's variance and inv_lengthscale, mean_const; grad_ard
 * m x D; grad_terms m x LMM_MAX_TERMS x LMM_GRAD_TERM_STRIDE; grad_U / grad_S the Euclidean gradient) for every latent the
 * value path accepts.  Every output is nullable; with every gradient pointer NULL only the value path runs.  A NaN in y,
 * m > p and a non-positive σ² return LMM_E_ARG; a failed factorisation reports its pivot and info_latent as the logpdf
 * gradient does. */
int lmm_oilmm_loo(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                  const double* U, const double* S, int p, double sigma2, const double* y, int out_dim,
                  double* out_loo, double* loo_mean, double* loo_var, double* grad_latents, double* grad_ard,
                  double* grad_sigma2, double* grad_y, double* grad_U, double* grad_S, double* grad_terms,
                  int* info_latent);
int lmm_imogp_loo(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D, double sigma2,
                  const double* y, int out_dim, double* out_loo, double* loo_mean, double* loo_var,
                  double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_terms,
                  int* info_latent);

/* ---- posterior handle: the OILMM/ILMM/IndependentMOGP whose latents are PosteriorGPs -------- */
/* mean_and_var(post(x*, σ²))  src/oilmm.jl:57-76 on PosteriorGP latents (AbstractGPs posterior
 * mean/var); for an IndependentMOGP posterior: src/independent_mogp.jl:50-57; ILMM: src/ilmm.jl:122-129. */
int lmm_post_mean_and_var(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean,
                          double* var);
/* mean_and_var(get_latent_gp(post).fs[i](x*, σ²)): ONE PosteriorGP latent (global index i, resident on this rank)
 * evaluated on its own -- the per-latent call src/oilmm.jl:61 makes; AbstractGPs FiniteGP{<:PosteriorGP}:
 * mean = m_i + K(x*,x) α_i, var = k(x*,x*) - colsumsq(C.U'^{-1} K(x,x*)) + σ².  mean / var: Ns doubles. */
int lmm_post_latent_mean_and_var(lmm_post* post, int i, const double* xs, int Ns, double sigma2,
                                 double* mean, double* var);
/* mean_and_cov(post(x*, σ²)) / cov: dense (p Ns) x (p Ns) column-major output, by outputs
 * (src/ilmm.jl:132-139,147; src/independent_mogp.jl:60-63 + Σy).  mean is nullable. */
int lmm_post_mean_and_cov(lmm_post* post, const double* xs, int Ns, double sigma2, double* mean,
                          double* cov);
/* mean_and_cov(fx) on PRIOR latents mixed by H (p x m column-major; pass U*sqrt(S) for an OILMM,
 * the identity for an IndependentMOGP): C = (H ⊗ I)(blockdiag K_a + latent_jitter I)(H ⊗ I)' + σ² I.
 * latent_jitter is the FiniteGP default noise 1e-18 for ILMM/OILMM (src/ilmm.jl:115), 0 for an
 * IndependentMOGP. */
int lmm_prior_mean_and_cov(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* xs, int Ns,
                           int D, const double* H, int p, double sigma2, double latent_jitter,
                           int out_dim, double* mean, double* cov);
/* posterior(post(x2, σ²), y2): sequential conditioning of an OILMM / IndependentMOGP / general-ILMM
 * posterior (src/oilmm.jl:116-134 / src/independent_mogp.jl:119-126 / src/ilmm.jl:184-198 with PosteriorGP
 * latents).  Returns a new handle over the union of the inputs; the old handle stays valid.  Per-latent posteriors extend
 * the old factor by a block-Cholesky update (cost O(N² N₂), see option "condition_update"); a joint (general-ILMM) posterior
 * re-factorises the union. */
int lmm_post_condition(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys,
                       lmm_post** out_post, int* info_latent);
/* logpdf(post(x*, σ²), y*)  (test/oilmm.jl:84): OILMM logpdf with PosteriorGP latents. */
int lmm_post_logpdf(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys,
                    double* out_logpdf, int* info_latent);
/* rrule of logpdf(post(x*, σ²), y*) (`gradient(logpdf, po, y_test)` at test/oilmm.jl:32, test/ilmm.jl:32,
 * test/independent_mogp.jl:66): value and gradients w.r.t. σ² and y* (p*Ns by outputs); the posterior's
 * own data (α, C, x) and kernel hyper-parameters are held fixed.  All outputs nullable. */
int lmm_post_logpdf_grad(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys,
                         double* out_logpdf, double* grad_sigma2, double* grad_y, int* info_latent);
/* The same logpdf differentiated through the conditioning as well: logpdf(posterior(f(x, σ²), y)(x*, σ*²), y*) w.r.t.
 * the latents' hyper-parameters and means, the training σ² and y, σ*², y*, and (OILMM) U and S -- held-out / forecast
 * likelihood and the conditional likelihood of new data given old.  Per-latent posteriors only (OILMM, IndependentMOGP,
 * also the OILMM handles of lmm_oilmm_masked_posterior, whose y_train is the p x n_observed_inputs block); joint and
 * sequentially conditioned handles return LMM_E_UNSUPPORTED.  y_train (required) is the p*N data the handle was
 * conditioned on: T y_train - m must reproduce the handle's δ to 1e-12 (norm-relative), else LMM_E_ARG.
 * out_logpdf, grad_sigma2 (σ*²) and grad_y (y*, p*Ns) are what lmm_post_logpdf_grad returns, bit for bit.  grad_latents
 * (m x 3: term 0's variance and inv_lengthscale, mean_const), grad_ard (m x D) and grad_terms (m x LMM_MAX_TERMS x
 * LMM_GRAD_TERM_STRIDE) use the layouts of lmm_oilmm_logpdf_grad_terms; grad_train_sigma2 is d/dσ², grad_train_y p*N by
 * outputs; grad_U (p x m column-major) and grad_S (m) are the Euclidean gradient, as lmm_oilmm_logpdf_grad returns them,
 * and must be NULL for an IndependentMOGP handle (LMM_E_ARG).  Every output is nullable.  The handle is not changed. */
int lmm_post_logpdf_grad_full(lmm_post* post, const double* xs, int Ns, double sigma2, const double* ys,
                              const double* y_train, double* out_logpdf, double* grad_sigma2, double* grad_y,
                              double* grad_latents, double* grad_ard, double* grad_terms,
                              double* grad_train_sigma2, double* grad_train_y, double* grad_U, double* grad_S,
                              int* info_latent);
/* rand(rng, post(x*, σ²))  src/oilmm.jl:40-54 with PosteriorGP latents. */
int lmm_post_rand(lmm_post* post, const double* xs, int Ns, double sigma2, const double* z_latent,
                  const double* z_noise, double* out, int* info_latent);
/* PosteriorGP field access (α, C, δ) for latent i (global index): L is N x N column-major lower
 * (upper part zero); any of L / alpha / delta may be NULL.  Returns LMM_E_ARG if latent i is
 * not resident on this rank. */
int lmm_post_export(lmm_post* post, int i, double* L, double* alpha, double* delta);
int lmm_post_info(lmm_post* post, int* kind, int* m, int* p, int* N, int* D, int64_t* device_bytes);
/* Serialisable posterior (SURVEY.md §8f-3): the handle's metadata followed by its device arrays verbatim
 * (tiled factors, α, δ, inputs), little-endian Float64.  A loaded handle answers every lmm_post_* call
 * bit-identically to the saved one; no recomputation.  Each rank saves / loads its own shard. */
int lmm_post_save(lmm_post* post, const char* path);
int lmm_post_load(lmm_ctx* ctx, const char* path, lmm_post** out_post);
int lmm_post_free(lmm_post* post);

/* ---- IndependentMOGP: src/independent_mogp.jl ---------------------------------------------- */
/* logpdf src/independent_mogp.jl:74-80 (by outputs; by-features callers permute with
 * lmm_reorder_indices first, :222-229). */
int lmm_imogp_logpdf(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D,
                     double sigma2, const double* y, int out_dim, double* out_logpdf,
                     double* lml_terms, int* info_latent);
/* posterior src/independent_mogp.jl:119-126. */
int lmm_imogp_posterior(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D,
                        double sigma2, const double* y, int out_dim, lmm_post** out_post,
                        double* out_logpdf, int* info_latent);
/* IndependentMOGP with non-isotropic observation noise (AbstractGPs generic FiniteGP path; the
 * reference's fast methods dispatch on Σy::Diagonal{<:Real,<:Fill} only, src/independent_mogp.jl:44-46;
 * test/independent_mogp.jl:72-75 exercises `f(x_train_mo, Σy)` with a dense Σy).
 * LMM_NOISE_DIAG: Sigma_y is the m*N vector of per-observation variances (by outputs) -- the latents
 * stay independent; LMM_NOISE_DENSE: Sigma_y is (mN x mN) column-major -- one joint factor of
 * blockdiag(K_a) + Σy, the returned handle behaves like an ILMM posterior with identity mixing.
 * out_post / out_logpdf nullable (not both). */
#define LMM_NOISE_DIAG 1
#define LMM_NOISE_DENSE 2
int lmm_imogp_posterior_noise(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D,
                              const double* Sigma_y, int noise_kind, const double* y, int out_dim,
                              lmm_post** out_post, double* out_logpdf, int* info_latent);
/* rand src/independent_mogp.jl:83-86. */
int lmm_imogp_rand(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* x, int N, int D,
                   double sigma2, int out_dim, const double* z, double* out, int* info_latent);
/* cov(f::IndependentMOGP, x, y): prior cross-covariance, dense (m*Na) x (m*Nb) column-major block
 * diagonal, both inputs by outputs  src/independent_mogp.jl:66-71 (by-features variants :188-215
 * permute rows / columns with lmm_reorder_indices). */
int lmm_imogp_cross_cov(lmm_ctx* ctx, const lmm_gp_desc* fs, int m, const double* xa, int Na,
                        const double* xb, int Nb, int D, double* out);
/* indices_which_reorder_{outputs_to_features,features_to_outputs}  src/independent_mogp.jl:135-145
 * (0-based; direction 0 = outputs->features, 1 = features->outputs). */
int lmm_reorder_indices(int N, int p, int direction, int64_t* out);

/* ---- ILMM with a general mixing matrix: src/ilmm.jl ------------------------------------------ */
#define LMM_ILMM_FORM_PROJECTED 0 /* the reference's (mN x mN) form, incl. the 1e-9 jitter :63 */
#define LMM_ILMM_FORM_DENSE 1     /* H K H' + σ²I, pN x pN (test oracle form, test/ilmm.jl:5)  */
/* logpdf src/ilmm.jl:150-163 (+ project :61-68, regulariser :171-181).  H is p x m column-major. */
int lmm_ilmm_logpdf(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                    const double* H, int p, double sigma2, const double* y, int out_dim, int form,
                    double* out_logpdf, int* info);
/* posterior src/ilmm.jl:184-198 (projected form; joint (mN) factor). */
int lmm_ilmm_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N,
                       int D, const double* H, int p, double sigma2, const double* y, int out_dim,
                       lmm_post** out_post, double* out_logpdf, int* info);
/* mean_and_var on prior latents src/ilmm.jl:122-129. */
int lmm_ilmm_prior_mean_and_var(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* xs,
                                int Ns, int D, const double* H, int p, double sigma2, int out_dim,
                                double* mean, double* var);
/* rand src/ilmm.jl:78-87 (latent jitter 1e-12). */
int lmm_ilmm_rand(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                  const double* H, int p, double sigma2, int out_dim, const double* z_latent,
                  const double* z_noise, double* out, int* info_latent);

/* rrule of the general-ILMM logpdf (SURVEY.md §8f-1; `gradient(logpdf, ilmmx, y_train)` at
 * test/ilmm.jl:31): value and gradients of the projected form src/ilmm.jl:150-163 (through `project`
 * :61-68 and `regulariser` :171-181) w.r.t. each latent's (variance, inv_lengthscale, mean_const) --
 * grad_latents m x 3 row-major --, σ², y (p*N by outputs) and the dense mixing matrix H (p x m
 * column-major).  All outputs nullable.  G = (αα' - C^{-1})/2 over the joint (mN x mN) matrix comes
 * from a potri on the tensor pipe; the chain through T, ΣT is host arithmetic on m x p matrices. */
int lmm_ilmm_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                         const double* H, int p, double sigma2, const double* y, int out_dim,
                         double* out_logpdf, double* grad_latents, double* grad_ard, double* grad_sigma2,
                         double* grad_y, double* grad_H, int* info);
/* The same for every latent the value path accepts, with per-term gradients in grad_terms (layout of
 * lmm_oilmm_logpdf_grad_terms above). */
int lmm_ilmm_logpdf_grad_terms(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                               const double* H, int p, double sigma2, const double* y, int out_dim,
                               double* out_logpdf, double* grad_latents, double* grad_ard, double* grad_sigma2,
                               double* grad_y, double* grad_H, double* grad_terms, int* info);

/* Heterotopic / missing-data ILMM (SURVEY.md §8f-4; unsupported in the reference, examples/oilmm_and_ilmm.ipynb:112).
 * Entries of y (host memory) that are NaN are unobserved; exact inference on the observed entries of the dense model
 * y ~ N((H ⊗ I) m, Σ_l (h_l h_l') ⊗ K_l + σ² I) -- the model the reference's tests use as the ILMM's ground truth
 * (test/ilmm.jl:5).  Pass U*sqrt(S) as H for an OILMM.  The returned handle answers lmm_post_mean_and_var,
 * lmm_post_mean_and_cov (all p outputs at x*), lmm_post_rand (AbstractGPs' generic FiniteGP rand on the dense model:
 * mean + chol(C + σ²I) z with ONE vector z_latent of p*Ns standard normals, z_noise ignored), lmm_post_save / lmm_post_load,
 * lmm_post_info and lmm_post_free.  out_post / out_logpdf nullable (not both); n_observed nullable. */
int lmm_ilmm_masked_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                              const double* H, int p, double sigma2, const double* y, int out_dim,
                              lmm_post** out_post, double* out_logpdf, int* n_observed, int* info);
/* Heterotopic OILMM whose mask is PER INPUT: at every input either all p outputs are observed or all are NaN (whole time
 * steps missing).  Conditioning on the observed entries is then the ordinary OILMM (src/oilmm.jl:79-93, 116-134) on the
 * observed inputs -- the projection stays exact and the latents independent, O(m N_obs³) instead of the dense model's
 * O((p N)³) -- and the handle is a full OILMM posterior (every lmm_post_* call).  A mask that is not per-input returns
 * LMM_E_UNSUPPORTED: use lmm_ilmm_masked_posterior.  out_post / out_logpdf nullable (not both). */
int lmm_oilmm_masked_posterior(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                               const double* U, const double* S, int p, double sigma2, const double* y, int out_dim,
                               lmm_post** out_post, double* out_logpdf, int* n_observed_inputs, int* info_latent);
/* rrule of the missing-data logpdf of the dense model (lmm_ilmm_masked_posterior's value).  NaN entries of y are
 * unobserved; grad_y is 0 there.  grad_terms nullable: NULL rejects composite / periodic latents, as lmm_*_logpdf_grad.
 * Outputs as lmm_ilmm_logpdf_grad_terms: grad_latents m x 3 (term 0's variance and inv_lengthscale, mean_const), grad_ard
 * m x D, grad_H p x m column-major, grad_y p*N by outputs; all nullable.  Workspace ≈ 12 n_observed² bytes (the factor and
 * the square X of its potri); with a communicator every rank computes the whole, replicated result. */
int lmm_ilmm_masked_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                                const double* H, int p, double sigma2, const double* y, int out_dim, double* out_logpdf,
                                double* grad_latents, double* grad_ard, double* grad_sigma2, double* grad_y, double* grad_H,
                                double* grad_terms, int* n_observed, int* info);
/* Per-input mask (whole inputs missing): the OILMM gradient (lmm_oilmm_logpdf_grad[_terms]) on the observed inputs; grad_y
 * scattered back to p*N with 0 at missing inputs.  A mask that is not per-input returns LMM_E_UNSUPPORTED. */
int lmm_oilmm_masked_logpdf_grad(lmm_ctx* ctx, const lmm_gp_desc* latents, int m, const double* x, int N, int D,
                                 const double* U, const double* S, int p, double sigma2, const double* y, int out_dim,
                                 double* out_logpdf, double* grad_latents, double* grad_ard, double* grad_sigma2,
                                 double* grad_y, double* grad_U, double* grad_S, double* grad_terms,
                                 int* n_observed_inputs, int* info_latent);

/* ---- batched blocked Cholesky primitive: the `cholesky(Symmetric(C))` / dpotrf call site ---- */
/* A: batch matrices, each N x N column-major (lower triangle read).  L_out (nullable): same
 * shape, lower factor with zero upper part.  logdet_out (nullable): batch doubles = 2 Σ log L_jj.
 * info (nullable): batch ints, 0 or 1-based failing pivot.  Returns max(info). */
int lmm_potrf_batched(lmm_ctx* ctx, const double* A, int N, int batch, double* L_out,
                      double* logdet_out, int* info);
/* AbstractGPs generic FiniteGP verbs on an explicit mean (n) and covariance (n x n column-major, lower read):
 * logpdf(fx, y) when y / out_logpdf are given, rand(rng, fx) = mean + C.U' z when z / out_sample are given
 * (either pair nullable).  Serves FiniteGPs outside the fast paths, e.g. a posterior evaluated under a vector
 * or dense Σy (test/independent_mogp.jl:120-133); the dense factor and solves run on the device. */
int lmm_mvn_logpdf_rand(lmm_ctx* ctx, const double* mean, const double* cov, int n, const double* y,
                        double* out_logpdf, const double* z, double* out_sample, int* info);
/* Same factorisation run on synthetic SPD matrices generated on the device (kernel-matrix build
 * of `desc` at x plus `noise` on the diagonal), nothing copied back but logdet: the kernel-level
 * benchmark used for roofline numbers.  out_ms receives the CUDA-event time of the factorisation
 * alone (kernel-matrix build excluded). */
int lmm_potrf_bench(lmm_ctx* ctx, const lmm_gp_desc* desc, const double* x, int N, int D,
                    double noise, int batch, double* logdet_out, double* out_ms_kmat,
                    double* out_ms_chol);

#ifdef __cplusplus
}
#endif
#endif /* LMM_H_ */
