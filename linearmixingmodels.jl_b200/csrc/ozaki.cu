// Integer-slice (Ozaki-scheme) FP64 trailing update on the int8 tensor cores (tcgen05.mma kind::i8, TMEM accumulators) -- the
// one route past the native FP64 pipe (DMMA: 37 TFLOP/s) the batched Cholesky already saturates (VERDICT r01 next #10).
// OPTIONAL ("ozaki" = 6 / 7 / 8 digit planes of "ozaki_bits" = 7 / 8 bits; default 0 = DMMA, which stays the reference path).
// Replaces, for the WIDE left-looking update of a block column only, the dsyrk/dgemm LAPACK's dpotrf makes under
// `cholesky(Symmetric(C))` (src/oilmm.jl:90,128 via AbstractGPs):
//     C(I,J) -= sum_{k < s0} L(I,k) L(J,k)'         (128 x 128 tiles, K = 128 per k-tile)
// and the same update of the prediction sweep X <- X L^{-T} (K10; rectangular left operand).
//
// Every finished row i of L is written as  L(i,k) = 2^E_i * 2^-6 * sum_{t < S} q_t(i,k) R^-t  with int8 digits and ONE exponent per
// row of the whole matrix: |L(i,k)| <= sqrt(A_ii) < 2^E_i (row i of L has 2-norm sqrt(A_ii)), so E_i is known from the diagonal
// before the factorisation starts and all k-tiles of a row share it -- integer partial sums can then be accumulated over the
// whole K range.  Two radices: R = 128 (digits |q_t| <= 64 from round-to-nearest remainders) and R = 256 (balanced digits in
// [-128, 127] from one rounding to a 64-bit integer and exact carries; the top plane keeps |q_0| <= 65).  Extraction is exact.  Then
//     L(i,:) . L(j,:) = 2^(E_i+E_j-12) * sum_d R^-d * [ sum_{t+u=d} sum_k q_t(i,k) q_u(j,k) ]          d = 0 .. S-1
// where every bracket is an EXACT int32 sum on the tensor cores (at most S pairs per d: S * K * max|q|^2 < 2^31, checked on the
// host: K <= 65535 columns for 8 planes of 7 bits, 18724 for 7 planes of 8 bits) and the dropped terms (t + u >= S) are below
// R^-(S-1) * 2^-13 * K of the row scales: 8 x 7 bits truncates at 2^-56, 7 x 8 bits at 2^-55 -- the normwise bound
// |dC| <= c eps |L||L|' of an FP64 GEMM, with the fixed-point grid relative to the row norms (measured factor error 2e-14 / 1e-13).
// S(S+1)/2 int8 MMAs (36 / 28) replace one FP64 tile product: 28 * 4 * 71 clk = 8.0 k clk against 32.8 k clk of DMMA
// (profiles/r02_i8_mma.jsonl: M = 128, N = 128, K = 32 issues every 71 clk).
//
// Kernel (one CTA = one 128 x 128 output tile, 11 warps): warps 0-7 = epilogue (the C tile lives in their registers from the
// first instruction to the last), warp 8 = producer (1-D TMA bulk copies of digit planes into an mbarrier ring), warps 9 and 10 =
// MMA issuers (one thread each, even / odd stages, issue loops unrolled at compile time; plane-major order with the A operand
// kept in the collector).  TMEM holds four 128-column int32 accumulators (all 512 columns), one per d, so the K range is swept
// twice: pass A for d = 0..3 (planes 0..3 of both operands; 6 stages of 32 KB), pass B for d = 4..S-1 (all planes; S = 7: 4 stages
// of 56 KB); after each pass the epilogue converts (exact int32 -> double), combines by Horner in 1/R, scales by the row / column
// exponents and subtracts from the registers; one store at the end.
// What bounded the earlier generations, in the order it was found (profiles/r02_ozaki.md): run-time loops in the issuing thread;
// a load-after-wait epilogue; and the issuer's per-stage hand-shake (wait, fence, commit: ~450 clk), which does not overlap with
// its own MMAs -- switching the MMAs, the TMA stream and the epilogue off one by one showed time = hand-shakes + MMAs, whatever the
// operand stream did; two issuers hide one's hand-shake behind the other's MMAs (16 latents of N = 16384: 236 -> 189 ms).
// HBM layout of the sliced tile (I,k) (S * 16 KB, at sym_tile_index(I,k) * S * 16384 bytes): [K quarter kq][plane t][4096 B], the
// 4096 B being the canonical K-major no-swizzle UMMA operand of 128 rows x 32 K-bytes: [16-byte K chunk (2)][row (128)][16 B]
// (core matrix = 8 rows x 16 B contiguous; LBO = 2048, SBO = 128) -- a bulk copy lands it in shared memory ready for the MMA.
// Exact zeros skipped, bit for bit: (1) the tile envelope -- a CTA starts at k-tile max(env[I], env[J]), below which one operand
// is 0.0 in FP64; (2) the digit planes -- entries far below their row scale round to zero digits on the fixed-point grid (SE factors at
// about 9 lengthscales, against 37.6 for the FP64 envelope).  The slice kernel records per tile the first plane tp with a nonzero
// digit (S: none, and then writes no planes); k-tile k adds exactly 0 to every accumulator d < tp(I,k) + tp(J,k), so pass A walks
// only the k-tiles with tp(I,k) + tp(J,k) <= 3, pass B those with the sum <= S - 1, and a CTA with no pass-B member leaves before
// its barriers, tensor memory or C tile exist.  For the headline SE workload this keeps about 5 % of the envelope's tile products.
// Measurements, kernel generations, what was tried and dropped (CTA pairs, A operand from tensor memory): profiles/r02_ozaki.md.
#include "common.cuh"
#include "kernels.h"
#include "ozaki_slice.cuh"

namespace lmm {

constexpr int OZ_RING_BYTES = 224 * 1024;      // stage = the planes one pass needs of one K quarter of both operands: pass A 2 x 4 x 4 KB
                                               // (6 stages), pass B 2 x S x 4 KB (S = 7: 56 KB, 4 stages; S = 8: 64 KB, 3 stages)
// Stages of a pass.  An EVEN count lets two issuing threads alternate (each owns every other stage); an odd one falls back to one.
__host__ __device__ constexpr int oz_stages(int planes) {
  return OZ_RING_BYTES / (2 * planes * OZ_QB) >= 6 ? 6 : (OZ_RING_BYTES / (2 * planes * OZ_QB) >= 4 ? 4 : OZ_RING_BYTES / (2 * planes * OZ_QB));
}
constexpr size_t OZ_SMEM = (size_t)OZ_RING_BYTES + 2048;  // + alignment slack, barriers, column scales, k-tile masks (231 424 of the 232 448 B a CTA may have)
// Words of one k-tile member mask (bit k - kb: k-tile k takes part in the pass).  The host's exact-int32 bound keeps K at most 682
// k-tiles (6 planes of 7 bits); longer K ranges run without the digit-plane filter.  The masks and two quarter counts take the
// last 200 B of the 2048 after the ring; the carve-up before them ends at 127 B alignment + 256 B barriers + 1024 B column scales.
constexpr int OZ_KMASK_WORDS = 24;

__device__ __forceinline__ uint32_t oz_s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void oz_mb_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(oz_s32(bar)), "r"(count));
}
__device__ __forceinline__ void oz_mb_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(oz_s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void oz_mb_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(oz_s32(bar)) : "memory");
}
__device__ __forceinline__ void oz_mb_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(oz_s32(bar)), "r"(parity)
        : "memory");
    if (!done && ++spins > (1u << 28)) __trap();  // never hang the GPU on a protocol bug
  }
}
// The same wait for the 256 epilogue threads, which sit out a whole MMA pass (tens to hundreds of microseconds): back off between
// polls.  A tight try_wait loop of 8 warps showed up as 80 % of all warp samples in ncu and takes shared-memory / issue bandwidth
// from the tensor core's operand reads and the TMA fills.
__device__ __forceinline__ void oz_mb_wait_relaxed(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0, spins = 0, ns = 64;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(oz_s32(bar)), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(ns);
    if (ns < 1024) ns <<= 1;
    if (++spins > (1u << 24)) __trap();
  }
}
__device__ __forceinline__ void oz_bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(oz_s32(dst)), "l"(src),
               "r"(bytes), "r"(oz_s32(bar))
               : "memory");
}
// instruction descriptor of tcgen05.mma kind::i8: D = S32 (2 @ bit 4), A / B signed int8 (1 @ bits 7 / 10), both K-major,
// N >> 3 @ bit 17, M >> 4 @ bit 24
constexpr uint32_t OZ_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
// shared-memory matrix descriptor: start address >> 4, LBO >> 4 @ 16 (between the two 16-byte K chunks of one MMA), SBO >> 4 @ 32
// (between 8-row groups), descriptor version 1 @ 46, no swizzle
__device__ __forceinline__ uint64_t oz_sdesc(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(2048 >> 4) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void oz_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(OZ_IDESC), "r"(accumulate)
      : "memory");
}
// The same MMA with the A operand kept in / taken from the tensor core's collector buffer: consecutive MMAs that share A (one digit
// plane of the left operand against several planes of the right one) read it from shared memory once (SASS: A_KEEP / A_REUSE).
// mode 0: plain, 1: fill (read A, keep it), 2: use (reuse, keep), 3: lastuse (reuse, release)
__device__ __forceinline__ void oz_mma_coll(int mode, uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  if (mode == 1)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8.collector::a::fill [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
                 "l"(adesc), "l"(bdesc), "r"(OZ_IDESC), "r"(accumulate)
                 : "memory");
  else if (mode == 2)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8.collector::a::use [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
                 "l"(adesc), "l"(bdesc), "r"(OZ_IDESC), "r"(accumulate)
                 : "memory");
  else if (mode == 3)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8.collector::a::lastuse [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
                 "l"(adesc), "l"(bdesc), "r"(OZ_IDESC), "r"(accumulate)
                 : "memory");
  else
    oz_mma(tmem_d, adesc, bdesc, accumulate);
}
__device__ __forceinline__ void oz_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(oz_s32(bar)) : "memory");
}
__device__ __forceinline__ double oz_i2d(uint32_t v) {  // exact int32 -> double: 2^52 + 2^31 + v as a bit pattern, one DADD
  return __hiloint2double(0x43300000, (int)(v ^ 0x80000000u)) - 4503601774854144.0;
}

// The MMAs of one K quarter (K = 32) of one pass, fully unrolled: the issuing thread must not spend more than the ~71 clk an MMA
// takes on loop bookkeeping and descriptor arithmetic (slice t of a stage is 4096 B = 256 descriptor units further on).
// PASS 0: d = 0 .. min(S,4)-1 over the slices 0..3; PASS 1: d = 4 .. S-1 over all S slices.  first: the accumulators start here.
template <int S, int PASS>
__device__ __forceinline__ void oz_issue_quarter(uint32_t tmem, uint64_t a0, uint64_t b0, bool first) {
  constexpr int NS = PASS ? S : (S < 4 ? S : 4);
  constexpr int DLO = PASS ? 4 : 0, DHI = PASS ? S - 1 : NS - 1;
  // plane t of the left operand against every plane u of the right one with DLO <= t + u <= DHI: t-major, so that consecutive
  // MMAs share A (collector reuse) and never write the same accumulator back to back (d = t + u changes with u).  Measured
  // (tools/microbench/i8_mma.cu): 64.0 clk per MMA in this order against 71 with the accumulator-major one.
#pragma unroll
  for (int t = 0; t < NS; ++t) {
    const int ulo = DLO - t > 0 ? DLO - t : 0, uhi = DHI - t < NS - 1 ? DHI - t : NS - 1;
#pragma unroll
    for (int u = ulo; u <= uhi; ++u) {
      const int mode = uhi == ulo ? 0 : (u == ulo ? 1 : (u == uhi ? 3 : 2));
      // every accumulator of a pass is first written by plane t = 0 (u = d), so "first" only concerns t = 0
      oz_mma_coll(mode, tmem + (uint32_t)(t + u - DLO) * 128u, a0 + (uint64_t)(t * 256), b0 + (uint64_t)(u * 256), (first && t == 0) ? 0u : 1u);
    }
  }
}

// Epilogue, 8 warps: warp w owns the TMEM lane quadrant w % 4 (tile rows 32 (w % 4) .. + 31, one per lane) and the column half
// w / 4 (64 columns).  A thread keeps its 64 values of C(I,J) in REGISTERS for the whole kernel: they are loaded when the kernel
// starts (the loads complete behind the MMA phase -- a load-after-wait epilogue was latency-bound: 16 dependent L2 round trips
// per pass held the tensor pipe at 63 %), both passes subtract into them, and they are stored once at the end.
constexpr int OZ_THREADS = 352;  // warps 0-7: epilogue, warp 8: producer, warps 9 and 10: MMA issuers (even / odd stages)
__device__ __forceinline__ void oz_epi_load(const double* Ctile, int r, int ch, double (&c)[64]) {
#pragma unroll
  for (int gq = 0; gq < 16; ++gq) {
    const double2* p = reinterpret_cast<const double2*>(Ctile + tile_elem(r, 64 * ch + 4 * gq));
    const double2 x0 = p[0], x1 = p[1];
    c[4 * gq + 0] = x0.x; c[4 * gq + 1] = x0.y; c[4 * gq + 2] = x1.x; c[4 * gq + 3] = x1.y;
  }
}
__device__ __forceinline__ void oz_epi_store(double* Ctile, int r, int ch, const double (&c)[64]) {
#pragma unroll
  for (int gq = 0; gq < 16; ++gq) {
    double2* p = reinterpret_cast<double2*>(Ctile + tile_elem(r, 64 * ch + 4 * gq));
    p[0] = make_double2(c[4 * gq + 0], c[4 * gq + 1]);
    p[1] = make_double2(c[4 * gq + 2], c[4 * gq + 3]);
  }
}
// One pass: the ND int32 accumulators -> exact doubles, Horner in 2^-7, row / column scales, c -= result.
template <int ND, int BITS>
__device__ __forceinline__ void oz_epi_pass(uint32_t tmem, int quad, int ch, double ps, const double* colscale, double (&c)[64]) {
  constexpr double RINV = BITS == 8 ? 0.00390625 : 0.0078125;  // 1 / radix
#pragma unroll
  for (int c0 = 0; c0 < 64; c0 += 4) {
    uint32_t v[ND][4];
#pragma unroll
    for (int a = 0; a < ND; ++a) {
      const uint32_t taddr = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(a * 128 + 64 * ch + c0);
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                   : "=r"(v[a][0]), "=r"(v[a][1]), "=r"(v[a][2]), "=r"(v[a][3])
                   : "r"(taddr)
                   : "memory");
    }
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double acc = oz_i2d(v[ND - 1][j]);
#pragma unroll
      for (int a = ND - 2; a >= 0; --a) acc = fma(acc, RINV, oz_i2d(v[a][j]));
      c[c0 + j] = fma(-acc, ps * colscale[64 * ch + c0 + j], c[c0 + j]);
    }
  }
}
template <int S, int BITS>
__device__ __forceinline__ void oz_epi_both(uint32_t tmem, int quad, int ch, int pass, double rs, const double* colscale, double (&c)[64]) {
  constexpr int NDA = S < 4 ? S : 4, NDB = S > 4 ? S - 4 : 1;
  constexpr double R4 = BITS == 8 ? 2.3283064365386962890625e-10 : 3.7252902984619140625e-09;  // radix^-4: pass B starts at d = 4
  if (pass == 0) oz_epi_pass<NDA, BITS>(tmem, quad, ch, rs, colscale, c);
  else oz_epi_pass<NDB, BITS>(tmem, quad, ch, rs * R4, colscale, c);
}

struct OzakiArgs {
  const uint8_t* slices;      // sliced factor [batch][sym_tiles][S * 16384]
  size_t slice_batch_stride;  // bytes
  const double* scale;        // [batch][npad]: 2^(E_row - 6)
  size_t scale_batch_stride;  // doubles
  TileOperand C;
  int i0, j0, k1;             // tile (I, J) = (i0 + blockIdx.y, j0 + blockIdx.x); k-tiles [0, k1)
  int S;                      // slices (6, 7 or 8)
  // left operand from a RECTANGULAR sliced matrix X (prediction: X L^{-T} sweep) instead of the factor itself; null = the factor
  const uint8_t* a_slices;    // [batch][ntr * a_ntc tiles][S * 16384]
  size_t a_batch_stride;      // bytes
  int a_ntc;                  // tiles per row of X
  const double* a_scale;      // [batch][ntr * 128]
  size_t a_scale_stride;
  const int* env;             // nullable (factor only): tile envelope [batch][env_stride]; tile (I,J) sums k in [max(env[I], env[J]), k1)
  int env_stride;
  const uint8_t* fp;          // nullable (factor only, k1 - kb <= 32 OZ_KMASK_WORDS): first nonzero digit plane per tile [batch][fp_stride]
  size_t fp_stride;
};

template <int S, int BITS>
__global__ void __launch_bounds__(OZ_THREADS, 1) ozaki_update_kernel(OzakiArgs g) {
  extern __shared__ __align__(1024) uint8_t oz_smem_raw[];
  const int J = g.j0 + blockIdx.x, I = g.i0 + blockIdx.y, b = blockIdx.z;
  if (!g.a_slices && I < J) return;
  // first k-tile: the products below it have an all-zero operand (outside the envelope).  Decided from blockIdx only, so the whole
  // CTA leaves together -- before any barrier or tensor memory exists.
  int kb = 0;
  if (g.env) {
    const int* e = g.env + (size_t)b * g.env_stride;
    kb = max(e[I], e[J]);
    if (kb >= g.k1) return;
  }
  // 1024-aligned carve-up: stages, then barriers
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(oz_smem_raw) + 127) & ~(uintptr_t)127);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)OZ_RING_BYTES);
  // each pass has its own ring geometry and its own barriers: [pass][full 0..5 | empty 0..5]
  uint64_t* acc_full = bars + 24;              // MMAs of the current pass complete
  uint64_t* acc_empty = acc_full + 1;          // epilogue of pass A has drained TMEM
  uint64_t* init_done = acc_empty + 1;         // [2]: the issuer of the first quarter (first member k-tile) has issued it (the accumulators of the pass are initialised)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 3);
  double* colscale = reinterpret_cast<double*>(bars + 32);  // [128]
  // at the fixed end of the dynamic region (constant addresses: the epilogue, which holds its C tile in registers, has no register
  // to spare for a pointer): K quarters per pass (4 per member, read where needed), member k-tiles of pass A / pass B
  int* nquarters = reinterpret_cast<int*>(oz_smem_raw + OZ_SMEM - 8);
  uint32_t* kmask = reinterpret_cast<uint32_t*>(oz_smem_raw + OZ_SMEM - 8 - 8 * OZ_KMASK_WORDS);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int nsA = S < 4 ? S : 4;
  // Member k-tiles of each pass.  Planes 0 .. tp - 1 of a tile whose first nonzero plane is tp are zero, so the product of k-tile k
  // adds exactly 0 to every accumulator d < tp(I,k) + tp(J,k): pass A (d <= nsA - 1) needs tp(I,k) + tp(J,k) <= nsA - 1, pass B
  // (d <= S - 1) the sum <= S - 1.  Without fp every k-tile of [kb, k1) is a member.
  const int nk = g.k1 - kb;
  int nmA = nk, nmB = nk;
  if (g.fp) {
    const uint8_t* fpb = g.fp + (size_t)b * g.fp_stride;
    const uint8_t *tI = fpb + sym_tile_index(I, kb), *tJ = fpb + sym_tile_index(J, kb);
    for (int w = warp; w * 32 < nk; w += OZ_THREADS / 32) {
      const int k = w * 32 + lane;
      const int sum = k < nk ? (int)tI[k] + (int)tJ[k] : 2 * S;
      const uint32_t mA = __ballot_sync(0xffffffffu, sum <= nsA - 1), mB = __ballot_sync(0xffffffffu, sum <= S - 1);
      if (lane == 0) {
        kmask[w] = mA;
        kmask[OZ_KMASK_WORDS + w] = mB;
      }
    }
    __syncthreads();
    nmA = nmB = 0;
    for (int w = 0; w * 32 < nk; ++w) {
      nmA += __popc(kmask[w]);
      nmB += __popc(kmask[OZ_KMASK_WORDS + w]);
    }
    // every product of the tile adds exactly zero: the whole CTA leaves together, before any barrier or tensor memory exists, and
    // C(I,J) is neither read nor written
    if ((S > 4 ? nmB : nmA) == 0) return;
  }
  if (tid == 0) {
    nquarters[0] = 4 * nmA;  // a multiple of 4: both issuers get half of a pass
    nquarters[1] = 4 * nmB;
    for (int s = 0; s < 24; ++s) oz_mb_init(&bars[s], 1);
    oz_mb_init(acc_full, 2);
    oz_mb_init(&init_done[0], 1);
    oz_mb_init(&init_done[1], 1);
    oz_mb_init(acc_empty, 256);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(oz_s32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid < 128) colscale[tid] = g.scale[(size_t)b * g.scale_batch_stride + (size_t)J * TILE + tid];
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;
  const size_t tile_bytes = (size_t)S * 16384;

  if (warp == 8) {
    // ===== producer: per K quarter one bulk copy of the needed slices of A(I,k) and one of B(J,k)
    if (lane == 0) {
      const uint8_t* Abase = g.a_slices ? g.a_slices + (size_t)b * g.a_batch_stride + (size_t)I * g.a_ntc * tile_bytes
                                        : g.slices + (size_t)b * g.slice_batch_stride + sym_tile_index(I, kb) * tile_bytes;
      const uint8_t* Bbase = g.slices + (size_t)b * g.slice_batch_stride + sym_tile_index(J, kb) * tile_bytes;
      for (int pass = 0; pass < 2; ++pass) {
        const int ns = pass ? S : nsA;
        if (pass && S <= 4) break;
        const int nst = pass ? oz_stages(S) : oz_stages(S < 4 ? S : 4);
        const uint32_t half = (uint32_t)ns * OZ_QB, bytes = half;
        uint64_t* full = bars + 12 * pass;
        uint64_t* empty = full + 6;
        if (pass) oz_mb_wait(acc_full, 0);  // every MMA of pass A has read its stage: the ring can change geometry
        const int nq = nquarters[pass];
        const uint32_t* mask = kmask + (pass ? OZ_KMASK_WORDS : 0);
        int mw = 0, k = 0;  // member walk: word, k-tile offset from kb
        uint32_t mbits = g.fp ? mask[0] : 0u;
        for (int kq = 0; kq < nq; ++kq) {
          if ((kq & 3) == 0) {  // next member k-tile
            if (g.fp) {
              while (!mbits) mbits = mask[++mw];
              k = 32 * mw + __ffs(mbits) - 1;
              mbits &= mbits - 1;
            } else {
              k = kq >> 2;
            }
          }
          const int s = kq % nst;
          oz_mb_wait(&empty[s], ((kq / nst) & 1) ^ 1);
          uint8_t* st = smem + (size_t)s * (2 * half);
          oz_mb_expect_tx(&full[s], 2 * bytes);
          const size_t off = (size_t)k * tile_bytes + (size_t)(kq & 3) * S * OZ_QB;
          oz_bulk_load(st, Abase + off, bytes, &full[s]);
          oz_bulk_load(st + half, Bbase + off, bytes, &full[s]);
        }
      }
    }
  } else if (warp == 9 || warp == 10) {
    // ===== MMA issuers: accumulator d - dlo at TMEM columns (d - dlo) * 128.  TWO issuing threads, one for the even and one for the
    // odd K quarters: the per-stage hand-shake of an issuer (wait for the stage, fence, commit: ~450 clk, measured with the MMAs
    // switched off) does not overlap with its own MMAs -- with one issuer the tensor pipe idled that long after every stage
    // (66 % of peak whatever the operand stream did); with two, one issues while the other shakes hands.  int32 accumulation
    // commutes, so the interleaving of the two streams is irrelevant EXCEPT for the first quarter (kq = 0: the first quarter of the
    // first member k-tile), whose MMAs initialise the accumulators: the odd issuer starts a pass only after the even one has issued it (init_done).  Each issuer commits its own
    // stages; acc_full completes when both have committed their last one.  A pass without members (pass A when every member of pass B
    // has tp(I,k) + tp(J,k) >= 4) issues nothing: both issuers arrive on acc_full directly, and the odd one must not wait for init_done.
    if (lane == 0) {
      const int who = warp - 9;
      for (int pass = 0; pass < 2; ++pass) {
        if (pass && S <= 4) break;
        const int nst = pass ? oz_stages(S) : oz_stages(S < 4 ? S : 4);
        const uint32_t half = (uint32_t)(pass ? S : (S < 4 ? S : 4)) * OZ_QB;
        uint64_t* full = bars + 12 * pass;
        uint64_t* empty = full + 6;
        // two issuers only with an even stage count: each then owns every other stage of the ring, so neither can run a whole
        // barrier phase ahead of the other on a shared stage (with 3 stages the odd issuer's second quarter is the even one's
        // first stage: its parity wait would pass before that stage has ever been filled)
        const bool dual = (nst & 1) == 0;
        if (who == 1 && !dual) {
          if (pass) oz_mb_wait(acc_full, 0);  // (its arrival must count for THIS pass's phase of the barrier)
          oz_mb_arrive(acc_full);
          continue;
        }
        if (pass) {
          oz_mb_wait(acc_empty, 0);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        const int nq = nquarters[pass];
        if (nq == 0) {
          oz_mb_arrive(acc_full);
          continue;
        }
        if (who == 1) oz_mb_wait(&init_done[pass], 0);
        for (int kq = who; kq < nq; kq += (dual ? 2 : 1)) {
          const int s = kq % nst;
          oz_mb_wait(&full[s], (kq / nst) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sa = oz_s32(smem + (size_t)s * (2 * half));
          const uint64_t a0 = oz_sdesc(sa), b0 = oz_sdesc(sa + half);
          if (pass) oz_issue_quarter<S, 1>(tmem, a0, b0, kq == 0);
          else oz_issue_quarter<S, 0>(tmem, a0, b0, kq == 0);
          oz_commit(&empty[s]);  // the stage is free once these MMAs have read it
          if (kq == 0) oz_mb_arrive(&init_done[pass]);
        }
        oz_commit(acc_full);
      }
    }
  } else {
    // ===== epilogue (warps 0-7): C(I,J) lives in registers from here to the end
    const int quad = warp & 3, ch = warp >> 2, r = quad * 32 + lane;
    const double rs = g.a_slices ? g.a_scale[(size_t)b * g.a_scale_stride + (size_t)I * TILE + r]
                                 : g.scale[(size_t)b * g.scale_batch_stride + (size_t)I * TILE + r];
    double* Ctile = g.C.tile(b, I, J);
    double c[64];
    oz_epi_load(Ctile, r, ch, c);
    for (int pass = 0; pass < 2; ++pass) {
      if (pass && S <= 4) break;
      oz_mb_wait_relaxed(acc_full, (uint32_t)pass);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // a pass without members left TMEM unwritten and would subtract exact zeros: skip it (c - 0 = c, -0.0 included).  Only pass A
      // can be one: a CTA without members in pass B has left at the top.
      if (pass || nquarters[0] > 0) oz_epi_both<S, BITS>(tmem, quad, ch, pass, rs, colscale, c);
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      if (pass == 0) oz_mb_arrive(acc_empty);
    }
    oz_epi_store(Ctile, r, ch, c);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// A CTA-PAIR variant (tcgen05 cta_group::2, M = 256: each SM reads its own 128 rows of A and only half of B per MMA, which lifts the
// shared-memory cap -- tools/microbench/i8_mma.cu measures 64.0 clk per MMA for the pair against 71 for one CTA) was built, passed
// the same tests and was REMOVED: with the stage hand-shake across two CTAs (relay of the peer's `full` barrier, multicast
// commits) and the same 3-stage depth in pass B it reached 56-63 % tensor-pipe activity and 308-343 ms where this kernel needs
// 287 ms (16 latents, N = 16384; profiles/r02_ozaki.md).  One more thing learnt there: a kernel that uses cta_group::2 only
// launches when the pair is adjacent in x (cluster (2,1,1)); (1,2,1) fails with cudaErrorInvalidClusterSize.

// ---- row exponents from the diagonal of the matrix that is about to be factored: scale = 2^(E - 6), 2^E > sqrt(A_ii)
__global__ void __launch_bounds__(128) ozaki_scale_kernel(TiledSym L, double* __restrict__ scale, size_t scale_batch_stride) {
  const int I = blockIdx.x, b = blockIdx.y, r = threadIdx.x;
  const double a = L.tile(b, I, I)[tile_elem(r, r)];
  int e = 0;
  if (a > 0.0 && a < 1e300) e = ilogb(sqrt(a)) + 1;
  scale[(size_t)b * scale_batch_stride + (size_t)I * TILE + r] = scalbn(1.0, e - 6);
}

// ---- slice the finished tiles (I, k), I in [i0, i0 + gridDim.y), k in [k0, k0 + gridDim.x): 256 threads, thread = (row, 16 columns)
// out_ntc = 0: the factor (packed-lower tile order, tiles with k > I skipped); > 0: a rectangular matrix with out_ntc tiles per row
// fp (nullable, factor only): fp[b][sym_tile_index(I, k)] = the first plane with a nonzero digit, S when all digits are zero -- such a
// tile's planes are not written (the update never reads them).  A digit of plane t is nonzero iff some entry survives the rounding
// to the grid of plane t; all of an entry's digits are zero iff it rounds to 0 on the finest grid, R^(S-1) (both radices).
__global__ void __launch_bounds__(256) ozaki_slice_kernel(TileOperand L, const double* __restrict__ scale, size_t scale_batch_stride,
                                                          uint8_t* __restrict__ slices, size_t slice_batch_stride, int i0, int k0, int S, int bits,
                                                          int out_ntc, const int* __restrict__ env, int env_stride, uint8_t* __restrict__ fp,
                                                          size_t fp_stride) {
  const int k = k0 + blockIdx.x, I = i0 + blockIdx.y, b = blockIdx.z;
  if (!out_ntc && k > I) return;
  if (env && k < env[(size_t)b * env_stride + I]) return;  // outside the envelope: zero, and never read by the update
  oz_slice_tile(L.tile(b, I, k), scale + (size_t)b * scale_batch_stride + (size_t)I * TILE,
                slices + (size_t)b * slice_batch_stride + (out_ntc ? (size_t)I * out_ntc + k : sym_tile_index(I, k)) * ((size_t)S * 16384), S, bits,
                fp ? fp + (size_t)b * fp_stride + sym_tile_index(I, k) : nullptr);
}

cudaError_t launch_ozaki_scales(cudaStream_t st, TiledSym L, int batch, double* scale, size_t scale_batch_stride) {
  ozaki_scale_kernel<<<dim3((unsigned)L.nt, (unsigned)batch), 128, 0, st>>>(L, scale, scale_batch_stride);
  return cudaGetLastError();
}
cudaError_t launch_ozaki_slice(cudaStream_t st, TiledSym L, const DigitPlanes& p, int i0, int nrows, int k0, int ncols, int batch,
                               const int* env) {
  if (nrows <= 0 || ncols <= 0 || batch <= 0) return cudaSuccess;
  ozaki_slice_kernel<<<dim3((unsigned)ncols, (unsigned)nrows, (unsigned)batch), 256, 0, st>>>(operand(L), p.scale, p.scale_stride, p.slices,
                                                                                            p.slice_stride, i0, k0, p.S, p.bits, 0, env, L.nt,
                                                                                            p.fp, p.fp_stride);
  return cudaGetLastError();
}
cudaError_t launch_ozaki_slice_rect(cudaStream_t st, TiledRect X, const DigitPlanes& xp, int k0, int ncols, int batch) {
  if (X.ntr <= 0 || ncols <= 0 || batch <= 0) return cudaSuccess;
  ozaki_slice_kernel<<<dim3((unsigned)ncols, (unsigned)X.ntr, (unsigned)batch), 256, 0, st>>>(operand(X), xp.scale, xp.scale_stride, xp.slices,
                                                                                             xp.slice_stride, 0, k0, xp.S, xp.bits, X.ntc, nullptr, 0,
                                                                                             nullptr, 0);
  return cudaGetLastError();
}

// ---- row scales for the prediction sweep X <- X L^{-T}.  Rows of the finished factor: 2^E > ||L(i,:)||_2 (one pass over the row panel);
// rows of X = K(x*,x) L^{-T}: ||X(r,:)||^2 <= k(x*,x*), the prior variance (LatentParams.kdiag).
__global__ void __launch_bounds__(128) ozaki_factor_scale_kernel(TiledSym L, double* __restrict__ scale, size_t scale_batch_stride) {
  const int I = blockIdx.x, b = blockIdx.y, r = threadIdx.x;
  double s = 0.0;
  for (int J = 0; J <= I; ++J) {
    const double* t = L.tile(b, I, J);
    for (int c4 = 0; c4 < 32; ++c4) {
      const double2* p = reinterpret_cast<const double2*>(t + (size_t)c4 * 512 + 4 * r);
      const double2 a = p[0], c = p[1];
      s = fma(a.x, a.x, s); s = fma(a.y, a.y, s); s = fma(c.x, c.x, s); s = fma(c.y, c.y, s);
    }
  }
  int e = 0;
  if (s > 0.0 && s < 1e300) e = ilogb(sqrt(s) * 1.0000001) + 1;
  scale[(size_t)b * scale_batch_stride + (size_t)I * TILE + r] = scalbn(1.0, e - 6);
}
__global__ void __launch_bounds__(128) ozaki_const_scale_kernel(const LatentParams* __restrict__ params, double* __restrict__ scale,
                                                                size_t scale_batch_stride) {
  const int R = blockIdx.x, b = blockIdx.y, r = threadIdx.x;
  const double v = params[b].kdiag;
  int e = 0;
  if (v > 0.0 && v < 1e300) e = ilogb(sqrt(v) * 1.0000001) + 1;
  scale[(size_t)b * scale_batch_stride + (size_t)R * TILE + r] = scalbn(1.0, e - 6);
}
cudaError_t launch_ozaki_factor_scales(cudaStream_t st, TiledSym L, int batch, double* scale, size_t scale_batch_stride) {
  ozaki_factor_scale_kernel<<<dim3((unsigned)L.nt, (unsigned)batch), 128, 0, st>>>(L, scale, scale_batch_stride);
  return cudaGetLastError();
}
cudaError_t launch_ozaki_const_scales(cudaStream_t st, const LatentParams* params, int ntr, int batch, double* scale, size_t scale_batch_stride) {
  ozaki_const_scale_kernel<<<dim3((unsigned)ntr, (unsigned)batch), 128, 0, st>>>(params, scale, scale_batch_stride);
  return cudaGetLastError();
}
template <int S, int BITS>
static cudaError_t oz_launch(cudaStream_t st, dim3 grid, const OzakiArgs& a) {
  static bool configured_dev[64] = {false};  // function attributes are per device (and per instantiation)
  int dev = 0;
  cudaGetDevice(&dev);
  bool& configured = configured_dev[dev & 63];
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(ozaki_update_kernel<S, BITS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OZ_SMEM);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  ozaki_update_kernel<S, BITS><<<grid, OZ_THREADS, OZ_SMEM, st>>>(a);
  return cudaGetLastError();
}
cudaError_t oz_dispatch(cudaStream_t st, dim3 grid, const OzakiArgs& a, int S, int bits);

cudaError_t launch_ozaki_update(cudaStream_t st, TiledSym L, const DigitPlanes& p, int i0, int nrows, int j0, int ncols, int k1, int batch,
                                const int* env) {
  if (nrows <= 0 || ncols <= 0 || batch <= 0 || k1 <= 0) return cudaSuccess;
  const uint8_t* first_plane = k1 > 32 * OZ_KMASK_WORDS ? nullptr : p.fp;  // the member masks cover at most this many k-tiles
  OzakiArgs a{p.slices, p.slice_stride, p.scale, p.scale_stride, operand(L), i0, j0, k1, p.S, nullptr, 0, 0, nullptr, 0, env, L.nt,
              first_plane, p.fp_stride};
  const dim3 grid((unsigned)ncols, (unsigned)nrows, (unsigned)batch);
  return oz_dispatch(st, grid, a, p.S, p.bits);
}
// X(R, J) -= sum_{k < k1} X(R,k) L(J,k)' for all tile rows R of the rectangular X and J in [j0, j0 + ncols): the wide update of the
// prediction sweep X <- X L^{-T}, left operand from the sliced finished columns of X (xp), right operand from the sliced factor (lp).
cudaError_t launch_ozaki_update_rect(cudaStream_t st, TiledRect X, const DigitPlanes& xp, const DigitPlanes& lp, int j0, int ncols, int k1,
                                     int batch) {
  if (X.ntr <= 0 || ncols <= 0 || batch <= 0 || k1 <= 0) return cudaSuccess;
  OzakiArgs a{lp.slices, lp.slice_stride, lp.scale, lp.scale_stride, operand(X), 0, j0, k1, lp.S, xp.slices, xp.slice_stride, X.ntc, xp.scale,
              xp.scale_stride, nullptr, 0, nullptr, 0};
  const dim3 grid((unsigned)ncols, (unsigned)X.ntr, (unsigned)batch);
  return oz_dispatch(st, grid, a, lp.S, lp.bits);
}
cudaError_t oz_dispatch(cudaStream_t st, dim3 grid, const OzakiArgs& a, int S, int bits) {
  if (bits == 8) {
    if (S == 7) return oz_launch<7, 8>(st, grid, a);
    if (S == 6) return oz_launch<6, 8>(st, grid, a);
    if (S == 8) return oz_launch<8, 8>(st, grid, a);
    return cudaErrorInvalidValue;
  }
  if (S == 8) return oz_launch<8, 7>(st, grid, a);
  if (S == 7) return oz_launch<7, 7>(st, grid, a);
  if (S == 6) return oz_launch<6, 7>(st, grid, a);
  return cudaErrorInvalidValue;
}

}  // namespace lmm
