// Batched blocked Cholesky schedules and TRSM sweeps (K6 / K10 of SURVEY.md §2.3) on top of the tile kernels, and the
// `cholesky(Symmetric(C))` primitives of the C ABI.
#include "host_internal.h"

namespace lmm_host {

// ---- batched blocked Cholesky (left-looking over blocks of `outer_block` tile columns) -------
// For every block column [s0, s1): one wide trailing update against all previous columns
// (K = s0 tiles, output written once), then per tile column: narrow update inside the block,
// diagonal-tile factor (+ inverse, logdet, info), panel TRSM as a GEMM with the inverse.
// jstart > 0 EXTENDS a factor (block-Cholesky update, AbstractGPs' sequential conditioning): the tile rows < jstart of L
// and W(J), J < jstart, are already final; only the tile rows >= jstart are computed -- for the columns J < jstart that
// is L(I,J) = (A(I,J) - sum_{k<J} L(I,k) L(J,k)') W(J)' (no diagonal-tile step), from column jstart on the ordinary
// factorisation of the Schur complement.  Cost O(N² N₂) instead of O((N + N₂)³).
// Counters of the fused panel-chain kernel (potrf.cu: chain_column_kernel): `batch` blocks of chain_counter_ints(nt) ints in
// a context-owned buffer, zeroed on `st` (every column of a factorisation uses its own entries).
static cudaError_t chain_counters(lmm_ctx* ctx, cudaStream_t st, int nt, int batch, int** out) {
  const size_t need = (size_t)batch * chain_counter_ints(nt) * sizeof(int);
  if (ctx->chain_cnt_bytes < need) {
    if (ctx->chain_cnt) cudaFree(ctx->chain_cnt);
    ctx->chain_cnt = nullptr;
    ctx->chain_cnt_bytes = 0;
    cudaError_t e = cudaMalloc(&ctx->chain_cnt, need);
    if (e != cudaSuccess) return e;
    ctx->chain_cnt_bytes = need;
  }
  *out = (int*)ctx->chain_cnt;
  return cudaMemsetAsync(ctx->chain_cnt, 0, need, st);
}

// Tiles of the TRSM of column jj below which a column's panel chain runs as ONE fused launch (chain_column_kernel: sliced,
// shared-memory-free GEMM roles at one CTA per SM) instead of TMA-pipelined launches per operation.
constexpr int CHAIN_MAX_TILES = 96;

// Enveloped factors of at least this many tile rows take block width 1 under the int8 update (see chol_factor_stream).
constexpr int OZ_WIDTH1_MIN_NT = 64;

// Workspace of the optional integer-slice (Ozaki) trailing update for the latents [0, batch) of one chol_factor_stream call.
struct OzWs {
  uint8_t* slices;
  size_t slice_stride;  // bytes per latent
  double* scale;
  size_t scale_stride;  // doubles per latent
  uint8_t* fp;          // first digit plane with a nonzero digit of each sliced tile (S: all zero), written by the slice kernel
  size_t fp_stride;     // bytes per latent (sym_tiles)
  int S, min_k, bits;  // digit planes, smallest K (k-tiles) the int8 update takes, bits per digit (7: radix 128, 8: radix 256)
};

// Tile envelope (env_h: host copy, [batch][nt]; L(I,k) = 0 for k < env[b][I]): the last tile row >= r0 that some latent of the
// batch has inside its envelope for the columns < lim (env[b][I] < lim); r0 - 1 when there is none.  Grids end there; the rows
// up to it that a latent does not need return at the top of the kernel.
static int env_last_row(const int* env_h, int nt, int batch, int r0, int lim) {
  int last = r0 - 1;
  for (int b = 0; b < batch; ++b)
    for (int I = nt - 1; I > last; --I)
      if (env_h[(size_t)b * nt + I] < lim) {
        last = I;
        break;
      }
  return last;
}

cudaError_t chol_factor_stream(lmm_ctx* ctx, cudaStream_t st, TiledSym L, double* W, size_t wstride, int batch, double* logdet,
                               int* info, int jstart = 0, int* counters = nullptr, const OzWs* oz = nullptr, const int* env_d = nullptr,
                               const int* env_h = nullptr) {
  const int nt = L.nt;
  if (jstart != 0 || !env_h) env_d = env_h = nullptr;
  // tile rows of a launch whose first row is r0: all of them, or up to the last one inside some latent's envelope (see above)
  auto rows = [&](int r0, int lim) { return (env_h ? env_last_row(env_h, nt, batch, r0, lim) + 1 : nt) - r0; };
  int ob = ctx->outer_block;
  if (oz && (jstart != 0 || nt <= ob || nt < oz->min_k + 1)) oz = nullptr;  // no wide update this scheme would take
  if (oz) {
    // narrow blocks: the in-block updates stay on DMMA, so the narrower the block the less of the work is left at the FP64 rate
    // (measured at 16 / 8 latents of N = 16384, final kernel: ob = 4: 286.8 / 147.5 ms, ob = 2 with min_k = 4: 275.5 / 143.1,
    // ob = 1: 274.8 / 147.1, ob = 3: 281.8 / 144.7; with the first kernel generation: 323 ms at ob = 8, 340 at 12).
    // Large enveloped factors take width 1: every update of column J by k < J then runs in the int8 kernel, whose digit-plane
    // filter drops most of the banded products, instead of the in-block DMMA update that multiplies all of them (C4, 64 latents:
    // 97 109 DMMA tile products at width 2, tools/bench_chol_phases.py --model-only; Cholesky stage at 64 latents, width 2 -> 1:
    // N = 16384 57.0 -> 43.0 ms, 8192 25.2 -> 20.2, 4096 10.2 -> 8.5, 2048 3.75 -> 3.49, profiles/r10_chol_phases_*.json).
    // Factors below OZ_WIDTH1_MIN_NT tile rows keep width 2, the schedule (and tile-product count) the int8 path has been checked
    // with at those sizes; the rule is conservative, not a measured crossover.  No fused panel chain (jj + 1 < s1) at width 1:
    // the last columns' TRSMs take the direct kernels once their grids are small.
    if (!ctx->outer_block_user) ob = env_h && nt >= OZ_WIDTH1_MIN_NT ? 1 : 2;
    cudaError_t eo = launch_ozaki_scales(st, L, batch, oz->scale, oz->scale_stride);  // reads the diagonal BEFORE it is factored
    if (eo != cudaSuccess) return eo;
    ++ctx->launches;
  }
  GemmArgs g{};
  g.A = operand(L);
  g.B = operand(L);
  g.C = operand(L);
  g.W = W;
  g.w_batch_stride = wstride;
  g.sym = 1;
  g.env = env_d;
  g.env_stride = nt;
  cudaError_t e;
  bool factored_ahead = false;  // diagonal tile jj was factored by the previous column's fused chain launch
  for (int s0 = 0; s0 < nt; s0 += ob) {
    const int s1 = (s0 + ob < nt) ? s0 + ob : nt;
    unsigned long long sliced = 0;  // bit jj - s0: the digit planes of column jj below the block are written
    if (s0 > 0) {
      const int r0 = s0 > jstart ? s0 : jstart;  // first tile row that still has to be computed
      const int nr = rows(r0, s0);  // tile (I, J) has products with two nonzero operands iff env[I] < s0 and env[J] < s0
      g.i0 = r0; g.j0 = s0; g.k0 = 0; g.k1 = s0;
      e = cudaSuccess;
      // exact int32 accumulation: (pairs per accumulator <= S) * K * (largest digit)^2 < 2^31
      if (oz && s0 >= oz->min_k && (long long)s0 * TILE * oz->S * (oz->bits == 8 ? 16384 : 4096) < (1ll << 31)) {
        if (nr > 0) {
          cudaEvent_t ev0 = nullptr, ev1 = nullptr;
          if (ctx->ozaki_time && cudaEventCreate(&ev0) == cudaSuccess && cudaEventCreate(&ev1) == cudaSuccess) cudaEventRecord(ev0, st);
          e = launch_ozaki_update(st, L, oz->slices, oz->slice_stride, oz->scale, oz->scale_stride, r0, nr, s0, s1 - s0, s0, batch, oz->S, oz->bits,
                                  env_d, oz->fp, oz->fp_stride);
          if (ev0 && ev1) {
            cudaEventRecord(ev1, st);
            ctx->oz_events.push_back(ev0);
            ctx->oz_events.push_back(ev1);
            // 128^3 tile products in this launch's envelope: tiles (I, J), I >= J, times their k-tiles (s0, or from the later envelope
            // on).  Nominal: the kernel skips the k-tiles whose digit products are all zero (first_plane), which no host count sees.
            double tp = 0.0;
            for (int J = s0; J < s1; ++J)
              for (int I = J > r0 ? J : r0; I < r0 + nr; ++I) {
                if (!env_h) {
                  tp += (double)s0 * batch;
                  continue;
                }
                for (int b = 0; b < batch; ++b) {
                  const int* eb = env_h + (size_t)b * nt;
                  const int kb = eb[I] > eb[J] ? eb[I] : eb[J];
                  if (kb < s0) tp += (double)(s0 - kb);
                }
              }
            ctx->oz_tile_products += tp;
          }
        }
      } else if (nr > 0) {
        e = launch_gemm(st, GEMM_UPDATE, g, s1 - s0, nr, batch, (long long)(s1 - s0) * (nt - r0) * batch);
      }
      if (e != cudaSuccess) return e;
      if (nr > 0) {
        ++ctx->launches;
        ctx->timings[6] += 1;
      }
    }
    for (int jj = s0; jj < s1; ++jj) {
      const int r0 = jj > jstart ? jj : jstart;
      if (!factored_ahead) {
        const int nr = jj > s0 ? rows(r0, jj) : 0;
        if (nr > 0) {
          g.i0 = r0; g.j0 = jj; g.k0 = s0; g.k1 = jj;
          if ((e = launch_gemm(st, GEMM_UPDATE, g, 1, nr, batch, (long long)(nt - r0) * batch)) != cudaSuccess) return e;
          ++ctx->launches;
          ctx->timings[6] += 1;
        }
        if (jj >= jstart) {
          if ((e = launch_potrf_tile(st, L, W, wstride, jj, batch, logdet, info)) != cudaSuccess) return e;
          ++ctx->launches;
        }
      }
      factored_ahead = false;
      const int t0 = jj + 1 > jstart ? jj + 1 : jstart;  // rows of column jj below the diagonal tile that are not final yet
      if (t0 >= nt) continue;
      // small grid, not at a block boundary, nothing above jstart involved: TRSM(jj) + update(jj+1) + potrf(jj+1) in one launch
      if (counters && ctx->chain_fused && jj + 1 < s1 && jj >= jstart && (long long)(nt - 1 - jj) * batch <= CHAIN_MAX_TILES) {
        if ((e = launch_chain_column(st, L, W, wstride, jj, s0, jj + 2, 1, batch, logdet, info, counters, env_d)) != cudaSuccess) return e;
        ++ctx->launches;
        factored_ahead = true;
        continue;
      }
      const int nr = rows(t0, jj + 1);
      if (nr <= 0) {
        sliced |= 1ull << (jj - s0);  // no tile of the column below the block is inside the envelope
        continue;
      }
      g.i0 = t0; g.j0 = jj;
      const long long sel = (long long)(nt - t0) * batch;
      if (oz && ctx->trsm_slice && !gemm_takes_direct(sel)) {
        // the TRSM writes the digit planes of the tiles below the block itself (rows in [t0, s1) are updated again in the block)
        const TrsmSliceArgs sa{oz->scale, oz->scale_stride, oz->slices, oz->slice_stride, oz->fp, oz->fp_stride, oz->S, oz->bits, s1};
        if ((e = launch_trsm_slice(st, g, nr, batch, sa)) != cudaSuccess) return e;
        sliced |= 1ull << (jj - s0);
      } else if ((e = launch_gemm(st, GEMM_TRSM, g, 1, nr, batch, sel)) != cudaSuccess) {
        return e;
      }
      ++ctx->launches;
    }
    const int ns = oz && s1 < nt ? rows(s1, s1) : 0;
    // the block column is final: digit planes of its tiles below the block, for the later wide updates -- for the runs of columns
    // whose TRSM did not write them (direct kernels, fused chain)
    for (int c0 = s0; ns > 0 && c0 < s1;) {
      if (sliced >> (c0 - s0) & 1) {
        ++c0;
        continue;
      }
      int c1 = c0 + 1;
      while (c1 < s1 && !(sliced >> (c1 - s0) & 1)) ++c1;
      if ((e = launch_ozaki_slice(st, L, oz->scale, oz->scale_stride, oz->slices, oz->slice_stride, s1, ns, c0, c1 - c0, batch, oz->S, oz->bits,
                                  env_d, oz->fp, oz->fp_stride)) != cudaSuccess)
        return e;
      ++ctx->launches;
      c0 = c1;
    }
  }
  return cudaSuccess;
}

// Grow the context's Ozaki workspace for up to `batch` latents of nt tile rows; returns how many latents fit (0: none -- stay on
// DMMA).  One cudaMemGetInfo / cudaMalloc when the shape grows, nothing afterwards.
static int ozaki_workspace(lmm_ctx* ctx, int nt, int batch, OzWs& ws) {
  const size_t per_slices = sym_tiles(nt) * (size_t)ctx->ozaki * 16384, per_scale = (size_t)nt * TILE;
  size_t have = per_slices ? ctx->oz_slices_bytes / per_slices : 0;
  if (have < (size_t)batch) {
    cudaStreamSynchronize(ctx->stream);  // the old buffer may still be in use by work queued earlier
    if (ctx->oz_slices) cudaFree(ctx->oz_slices);
    ctx->oz_slices = nullptr;
    ctx->oz_slices_bytes = 0;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return 0;
    const size_t reserve = (size_t)6 << 30;  // leave room for the caller's later allocations (solves, predictions)
    size_t fit = free_b > reserve ? (free_b - reserve) / per_slices : 0;
    if (fit > (size_t)batch) fit = (size_t)batch;
    if (fit == 0) return 0;
    if (cudaMalloc(&ctx->oz_slices, fit * per_slices) != cudaSuccess) {
      cudaGetLastError();
      return 0;
    }
    ctx->oz_slices_bytes = fit * per_slices;
    have = fit;
  }
  if (have > (size_t)batch) have = (size_t)batch;
  if (ctx->oz_scale_bytes < have * per_scale * sizeof(double)) {
    cudaStreamSynchronize(ctx->stream);
    if (ctx->oz_scale) cudaFree(ctx->oz_scale);
    ctx->oz_scale = nullptr;
    ctx->oz_scale_bytes = 0;
    if (cudaMalloc(&ctx->oz_scale, have * per_scale * sizeof(double)) != cudaSuccess) {
      cudaGetLastError();
      return 0;
    }
    ctx->oz_scale_bytes = have * per_scale * sizeof(double);
  }
  const size_t per_fp = sym_tiles(nt);
  if (ctx->oz_fp_bytes < have * per_fp) {
    cudaStreamSynchronize(ctx->stream);
    if (ctx->oz_fp) cudaFree(ctx->oz_fp);
    ctx->oz_fp = nullptr;
    ctx->oz_fp_bytes = 0;
    if (cudaMalloc(&ctx->oz_fp, have * per_fp) != cudaSuccess) {
      cudaGetLastError();
      return 0;
    }
    ctx->oz_fp_bytes = have * per_fp;
  }
  ws = OzWs{(uint8_t*)ctx->oz_slices, per_slices, ctx->oz_scale, per_scale, ctx->oz_fp, per_fp, ctx->ozaki, ctx->ozaki_min_k, ctx->ozaki_bits};
  return (int)have;
}

// Trailing update of the columns >= s2 (tile rows first_row, first_row + row_step, ... < nt) by the k-tiles [k0, k1): ONE
// launch.  (Chunking it into launches of <= 132 CTAs, to keep a few SMs free for the panel chain on the other stream, was
// measured and is much slower -- N=16384: 48 -> 68 ms, N=8192: 8.5 -> 10.3 ms: every launch boundary costs a pipeline
// fill and a tail, while a single launch keeps the block scheduler streaming CTAs.)
cudaError_t launch_trailing(lmm_ctx* ctx, cudaStream_t st, GemmArgs g, int s2, int nt, int first_row, int row_step, int k0, int k1,
                            int batch) {
  const int nrows = first_row >= nt ? 0 : (nt - 1 - first_row) / row_step + 1;
  if (nrows <= 0) return cudaSuccess;
  g.i0 = first_row; g.j0 = s2; g.k0 = k0; g.k1 = k1; g.row_step = row_step;
  cudaError_t e = launch_gemm(st, GEMM_UPDATE, g, nt - s2, nrows, batch);
  if (e != cudaSuccess) return e;
  ++ctx->launches;
  ctx->timings[6] += 1;
  return cudaSuccess;
}

// Right-looking block schedule with look-ahead (small batches: nothing else can hide the panel latency).  After block
// column kb is factored on the high-priority panel stream X, its update of the NEXT block column runs on X (so the next
// panel can start at once) while its update of everything further right runs as one large GEMM on the low-priority
// stream Y:
//   X: [wait Y(kb-2)] update(kb-1 -> kb), panel(kb)            Y: [wait X(kb)] update(kb -> kb+2 .. end)
// The Y launches have thousands of tiles (no tail effect, unlike the wide left-looking update of one block
// column) and keep every SM busy while the latency-bound panel steps run beside them; each C tile is
// read-modify-written once per block column of L (K = `ob` tiles per launch).
// Panel chain on X, per tile column jj of block [s0, s1): with "chain_fused" (default) ONE launch --
//   inside the block:      TRSM(jj) + update(column jj+1 by k in [s0, jj]) + potrf(jj+1)
//   at the block boundary: [wait Y(kb-1)]  TRSM(s1-1) + update(columns [s1, s2) by k in [s0, s1)) + potrf(s1)
// (chain_column_kernel: the critical tiles (jj+1, jj) -> (jj+1, jj+1) -> diagonal factorisation come first, everything else
// runs beside the factorisation); without it three launches per column chained by programmatic dependent launch.
cudaError_t chol_factor_rightlooking(lmm_ctx* ctx, TiledSym L, double* W, size_t wstride, int batch, double* logdet, int* info) {
  const int nt = L.nt;
  // the panel chain is the critical path: narrow blocks for small matrices, wider ones (fewer read-modify-write
  // passes over the trailing matrix) once the trailing GEMMs dominate (measured: tools/bench_batch1.py)
  // Fused chain launches pay off while the chain IS the run time (measured, profiles/r02_panel_chain.md: N = 1024 -13 %,
  // 2048 -4 %, 4096 -2 %); from N = 8192 on the trailing GEMMs of the other stream set the time and the sliced, one-CTA-per-SM
  // roles of the fused kernel only take SMs away from them (+10 %), so larger matrices keep one launch per operation
  // ("chain_fused" = 2 forces the fused kernel everywhere).
  // Larger factors fuse only their TAIL: once at most CHAIN_TAIL_ROWS tile rows are left below the column the trailing GEMMs
  // are small again and the chain is what remains.
  constexpr int CHAIN_TAIL_ROWS = 31;
  const bool fused_all = ctx->chain_fused == 2 || (ctx->chain_fused == 1 && nt <= 32);
  auto use_fused = [&](int jj) { return fused_all || (ctx->chain_fused == 1 && (long long)(nt - 1 - jj) * batch <= CHAIN_TAIL_ROWS); };
  const bool fused = ctx->chain_fused != 0;  // some column may take the fused launch: counters needed
  const int ob = ctx->outer_block_user ? ctx->outer_block : fused_all ? (nt <= 112 ? 3 : 4) : (nt <= 32 ? 1 : nt <= 48 ? 2 : nt <= 112 ? 3 : 4);
  const int nblk = (nt + ob - 1) / ob;
  cudaError_t e;
  while ((int)ctx->blk_ev.size() < 2 * nblk + 2) {
    cudaEvent_t ev;
    if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return e;
    ctx->blk_ev.push_back(ev);
  }
  cudaStream_t X = ctx->panel_stream, Y = ctx->update_stream;
  cudaEvent_t* evX = ctx->blk_ev.data();          // panel(b) done on X
  cudaEvent_t* evY = ctx->blk_ev.data() + nblk;   // trailing update from block b done on Y
  GemmArgs g{};
  g.A = operand(L); g.B = operand(L); g.C = operand(L);
  g.W = W; g.w_batch_stride = wstride; g.sym = 1;
  int* counters = nullptr;
  if (fused && (e = chain_counters(ctx, ctx->stream, nt, batch, &counters)) != cudaSuccess) return e;
  if ((e = cudaEventRecord(ctx->ev_fork, ctx->stream)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(X, ctx->ev_fork, 0)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(Y, ctx->ev_fork, 0)) != cudaSuccess) return e;
  bool factored_ahead = false;  // the block's first diagonal tile was factored by the previous block's boundary launch
  for (int b = 0; b < nblk; ++b) {
    const int s0 = b * ob, s1 = (s0 + ob < nt) ? s0 + ob : nt;
    const int s2 = (s1 + ob < nt) ? s1 + ob : nt;  // end of the next block
    if (b >= 1 && !factored_ahead) {
      // every earlier update of this block column (Y launches up to b-2) must have landed
      if (b >= 2 && (e = cudaStreamWaitEvent(X, evY[b - 2], 0)) != cudaSuccess) return e;
      g.k0 = s0 - ob; g.k1 = s0; g.i0 = s0; g.j0 = s0;
      if ((e = launch_gemm(X, GEMM_UPDATE, g, s1 - s0, nt - s0, batch)) != cudaSuccess) return e;
      ++ctx->launches;
      ctx->timings[6] += 1;
    }
    for (int jj = s0; jj < s1; ++jj) {
      if (!factored_ahead) {
        if (jj > s0) {
          g.k0 = s0; g.k1 = jj; g.i0 = jj; g.j0 = jj;
          if ((e = launch_gemm(X, GEMM_UPDATE, g, 1, nt - jj, batch)) != cudaSuccess) return e;
          ++ctx->launches;
        }
        if ((e = launch_potrf_tile(X, L, W, wstride, jj, batch, logdet, info)) != cudaSuccess) return e;
        ++ctx->launches;
      }
      factored_ahead = false;
      if (jj + 1 >= nt) continue;
      if (use_fused(jj)) {
        int c_end = jj + 2;
        if (jj + 1 == s1) {  // block boundary: the launch also carries the panel stream's update of the whole next block
          if (b >= 1 && (e = cudaStreamWaitEvent(X, evY[b - 1], 0)) != cudaSuccess) return e;  // Y(b-1) writes the columns >= s1
          c_end = s2;
        }
        if ((e = launch_chain_column(X, L, W, wstride, jj, s0, c_end, 1, batch, logdet, info, counters)) != cudaSuccess) return e;
        ++ctx->launches;
        factored_ahead = true;
      } else {
        g.i0 = jj + 1; g.j0 = jj;
        if ((e = launch_gemm(X, GEMM_TRSM, g, 1, nt - jj - 1, batch)) != cudaSuccess) return e;
        ++ctx->launches;
      }
    }
    if ((e = cudaEventRecord(evX[b], X)) != cudaSuccess) return e;
    if (s1 + ob < nt) {  // first column of block b+2
      if ((e = cudaStreamWaitEvent(Y, evX[b], 0)) != cudaSuccess) return e;
      if ((e = launch_trailing(ctx, Y, g, s1 + ob, nt, s1 + ob, 1, s0, s1, batch)) != cudaSuccess) return e;
    }
    if ((e = cudaEventRecord(evY[b], Y)) != cudaSuccess) return e;
  }
  if ((e = cudaStreamWaitEvent(ctx->stream, evX[nblk - 1], 0)) != cudaSuccess) return e;
  if ((e = cudaEventRecord(ctx->ev_join[0], Y)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0)) != cudaSuccess) return e;
  return cudaSuccess;
}

// Row-cyclic multi-GPU factorisation of ONE large matrix (north star: "ILMM runs on one GPU unless its blocked
// Cholesky is explicitly row-cyclic partitioned").  Every rank holds the whole packed-lower matrix and runs the same
// right-looking schedule; rank r owns the tile rows I = r (mod G) of the TRAILING matrix and applies the updates to
// those rows only.  Before block column b is factored its tiles are exchanged (pack own rows -> ncclAllGather over
// NVLink -> unpack the others' rows); the latency-bound panel (diagonal-tile factor, TRSM-as-GEMM of all rows, 2-3 %
// of the flops) is then computed redundantly by every rank, so the finished columns of L are complete everywhere and
// nothing downstream (solves, predictions, logdet) needs a collective.  Per block: one all-gather of (nt - s0) * ob
// tiles; the trailing GEMMs -- 97 % of the work -- are split G ways.
cudaError_t chol_factor_rowcyclic(lmm_ctx* ctx, TiledSym L, double* W, size_t wstride, double* logdet, int* info) {
  const int nt = L.nt, G = ctx->nranks, me = ctx->rank;
  const int ob = ctx->outer_block_user ? ctx->outer_block : (nt <= 72 ? 2 : nt <= 112 ? 3 : 4);
  const int nblk = (nt + ob - 1) / ob;
  cudaError_t e;
  while ((int)ctx->blk_ev.size() < 2 * nblk + 2) {
    cudaEvent_t ev;
    if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return e;
    ctx->blk_ev.push_back(ev);
  }
  // exchange buffers: [send: slots*ob tiles][recv: G*slots*ob tiles], sized for the first (largest) exchange
  const int max_slots = (nt + G - 1) / G;
  const size_t send_elems = (size_t)max_slots * ob * TT, need = (send_elems * (size_t)(G + 1)) * sizeof(double);
  if (ctx->xbuf_bytes < need) {
    if (ctx->xbuf) cudaFree(ctx->xbuf);
    ctx->xbuf = nullptr;
    ctx->xbuf_bytes = 0;
    if ((e = cudaMalloc(&ctx->xbuf, need)) != cudaSuccess) return e;
    ctx->xbuf_bytes = need;
  }
  double* sendb = (double*)ctx->xbuf;
  double* recvb = sendb + send_elems;
  cudaStream_t X = ctx->panel_stream, Y = ctx->update_stream;
  cudaEvent_t* evX = ctx->blk_ev.data();
  cudaEvent_t* evY = ctx->blk_ev.data() + nblk;
  GemmArgs g{};
  g.A = operand(L); g.B = operand(L); g.C = operand(L);
  g.W = W; g.w_batch_stride = wstride; g.sym = 1;
  auto first_own = [&](int s) { return s + (((me - s % G) % G) + G) % G; };
  auto own_count = [&](int s) { const int f = first_own(s); return f >= nt ? 0 : (nt - 1 - f) / G + 1; };
  int* counters = nullptr;
  if (ctx->chain_fused && (e = chain_counters(ctx, ctx->stream, nt, 1, &counters)) != cudaSuccess) return e;
  if ((e = cudaEventRecord(ctx->ev_fork, ctx->stream)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(X, ctx->ev_fork, 0)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(Y, ctx->ev_fork, 0)) != cudaSuccess) return e;
  for (int b = 0; b < nblk; ++b) {
    const int s0 = b * ob, s1 = (s0 + ob < nt) ? s0 + ob : nt;
    if (b >= 1) {
      if (b >= 2 && (e = cudaStreamWaitEvent(X, evY[b - 2], 0)) != cudaSuccess) return e;
      // own rows of block column b: update with block b-1 ...
      const int cnt = own_count(s0);
      if (cnt > 0) {
        g.row_step = G; g.i0 = first_own(s0); g.j0 = s0; g.k0 = s0 - ob; g.k1 = s0;
        if ((e = launch_gemm(X, GEMM_UPDATE, g, s1 - s0, cnt, 1)) != cudaSuccess) return e;
        ++ctx->launches;
        ctx->timings[6] += 1;
      }
      // ... then exchange the block column so that every rank can factor it
      const int slots = (nt - s0 + G - 1) / G;
      if ((e = launch_rowcyclic_pack(X, L, s0, s1, s0, nt, G, me, slots, sendb)) != cudaSuccess) return e;
      const size_t cntel = (size_t)slots * (s1 - s0) * TT;
      if (nccl_api().AllGather(sendb, recvb, cntel, NCCL_DOUBLE, ctx->comm_small ? ctx->comm_small : ctx->comm, X) != 0) {
        ctx->dist_error = 1;
        return cudaErrorUnknown;
      }
      if ((e = launch_rowcyclic_unpack(X, L, s0, s1, s0, nt, G, me, slots, recvb)) != cudaSuccess) return e;
      ctx->launches += 2;
    }
    g.row_step = 1;
    bool factored_ahead = false;
    for (int jj = s0; jj < s1; ++jj) {  // the panel: every rank, all rows
      if (!factored_ahead) {
        if (jj > s0) {
          g.i0 = jj; g.j0 = jj; g.k0 = s0; g.k1 = jj;
          if ((e = launch_gemm(X, GEMM_UPDATE, g, 1, nt - jj, 1)) != cudaSuccess) return e;
          ++ctx->launches;
        }
        if ((e = launch_potrf_tile(X, L, W, wstride, jj, 1, logdet, info)) != cudaSuccess) return e;
        ++ctx->launches;
      }
      factored_ahead = false;
      if (jj + 1 >= nt) continue;
      if (counters && jj + 1 < s1 && (ctx->chain_fused == 2 || nt - 1 - jj <= 40)) {
        // inside a block the redundant panel chain is one fused launch per column (the chain is what bounds this schedule) once
        // the column is short enough for the sliced roles (above ~40 tiles the TMA-pipelined TRSM launch is the faster one)
        if ((e = launch_chain_column(X, L, W, wstride, jj, s0, jj + 2, 1, 1, logdet, info, counters)) != cudaSuccess) return e;
        ++ctx->launches;
        factored_ahead = true;
      } else {
        g.i0 = jj + 1; g.j0 = jj;
        if ((e = launch_gemm(X, GEMM_TRSM, g, 1, nt - jj - 1, 1)) != cudaSuccess) return e;
        ++ctx->launches;
      }
    }
    if ((e = cudaEventRecord(evX[b], X)) != cudaSuccess) return e;
    const int s2 = s1 + ob;
    const int cnt2 = s2 < nt ? own_count(s2) : 0;
    if (cnt2 > 0) {
      if ((e = cudaStreamWaitEvent(Y, evX[b], 0)) != cudaSuccess) return e;
      if ((e = launch_trailing(ctx, Y, g, s2, nt, first_own(s2), G, s0, s1, 1)) != cudaSuccess) return e;
    }
    if ((e = cudaEventRecord(evY[b], Y)) != cudaSuccess) return e;
  }
  if ((e = cudaStreamWaitEvent(ctx->stream, evX[nblk - 1], 0)) != cudaSuccess) return e;
  if ((e = cudaEventRecord(ctx->ev_join[0], Y)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0)) != cudaSuccess) return e;
  return cudaSuccess;
}

// Row-cyclic factorisation with DISTRIBUTED STORAGE (VERDICT r01 next #8): rank r holds only the tile rows I = r (mod G) of
// the matrix (`Lown`, cyclic-packed: 1/G of the matrix) plus two block-column windows `P` (all rows x ob tile columns).  Per
// block column b = [s0, s1):
//   X: [wait Y(b-2)]  own rows of block column b  -=  P(b-1) P(b-1)'           (the look-ahead update, operands from the window)
//      pack own rows -> ncclAllGather -> unpack into the window P(b) -- every rank now holds the whole block column
//      panel on P(b), redundantly on every rank (diagonal tile, TRSM-as-GEMM, in-block updates; <= one wave of tiles, so the
//      redundancy costs no time); own rows of the finished window -> Lown (the distributed factor)
//   Y: [wait X(b)]    own rows of the columns >= s1 + ob  -=  P(b) P(b)'       (97 % of the flops, split G ways)
// Both operands of every trailing update come from the window, so a finished column of L is never needed from another
// rank again and the all-gather of block b+1 (on X) runs beside the trailing update of block b (on Y); the two windows
// alternate.  `nrows` may exceed the `nc` columns that are factored: the extra tile row (the right-hand side, launch_rhs_row)
// receives the panel TRSMs and ends up as z = L^{-1} rhs -- the forward solve needs no distributed sweep; its segments
// are copied into `zvec` (on every rank) as the windows finish.  logdet / info / W(J) are computed by every rank.
// Per rank: cyc_tiles(nrows) + (3 + 1/G) * nrows * ob tiles instead of sym_tiles(nrows).
size_t rowcyclic_dist_workspace_tiles(int nrows, int G, int ob) {
  const size_t slots = (size_t)(nrows + G - 1) / G;
  return slots * ob * (size_t)(G + 1) + 2 * (size_t)nrows * ob;
}
int rowcyclic_dist_block(const lmm_ctx* ctx, int nc) { return ctx->outer_block_user ? ctx->outer_block : (nc <= 72 ? 2 : nc <= 112 ? 3 : 4); }

cudaError_t chol_factor_rowcyclic_dist(lmm_ctx* ctx, TiledSym Lown, int nrows, int nc, double* W, size_t wstride, double* logdet, int* info,
                                       double* zvec) {
  const int G = ctx->nranks, me = ctx->rank;
  const int ob = rowcyclic_dist_block(ctx, nc);
  const int nblk = (nc + ob - 1) / ob;
  cudaError_t e;
  while ((int)ctx->blk_ev.size() < 2 * nblk + 2) {
    cudaEvent_t ev;
    if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return e;
    ctx->blk_ev.push_back(ev);
  }
  const int max_slots = (nrows + G - 1) / G;
  const size_t send_elems = (size_t)max_slots * ob * TT, win_elems = (size_t)nrows * ob * TT;
  const size_t need = rowcyclic_dist_workspace_tiles(nrows, G, ob) * TT * sizeof(double);
  if (ctx->xbuf_bytes < need) {
    if (ctx->xbuf) cudaFree(ctx->xbuf);
    ctx->xbuf = nullptr;
    ctx->xbuf_bytes = 0;
    if ((e = cudaMalloc(&ctx->xbuf, need)) != cudaSuccess) return e;
    ctx->xbuf_bytes = need;
  }
  double* sendb = (double*)ctx->xbuf;
  double* recvb = sendb + send_elems;
  double* win[2] = {recvb + send_elems * (size_t)G, recvb + send_elems * (size_t)G + win_elems};
  cudaStream_t X = ctx->panel_stream, Y = ctx->update_stream;
  cudaEvent_t* evX = ctx->blk_ev.data();
  cudaEvent_t* evY = ctx->blk_ev.data() + nblk;
  auto first_own = [&](int s) { return s + (((me - s % G) % G) + G) % G; };
  auto own_count = [&](int s) { const int f = first_own(s); return f >= nrows ? 0 : (nrows - 1 - f) / G + 1; };
  auto window = [&](int b) {  // block column b as a TiledSym: rows >= b*ob, tile columns [b*ob, b*ob + ob)
    TiledSym P{win[b & 1], nrows, 0};
    P.ntc = ob; P.row0 = b * ob; P.col0 = b * ob;
    return P;
  };
  int* counters = nullptr;
  if (ctx->chain_fused && (e = chain_counters(ctx, ctx->stream, nrows, 1, &counters)) != cudaSuccess) return e;
  if ((e = cudaEventRecord(ctx->ev_fork, ctx->stream)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(X, ctx->ev_fork, 0)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(Y, ctx->ev_fork, 0)) != cudaSuccess) return e;
  GemmArgs g{};
  g.W = W; g.w_batch_stride = wstride; g.sym = 1;
  for (int b = 0; b < nblk; ++b) {
    const int s0 = b * ob, s1 = (s0 + ob < nc) ? s0 + ob : nc;
    const TiledSym P = window(b);
    if (b >= 1) {
      if (b >= 2 && (e = cudaStreamWaitEvent(X, evY[b - 2], 0)) != cudaSuccess) return e;  // Y(b-2): last writer of these columns, last reader of this window
      const int cnt = own_count(s0);
      if (cnt > 0) {
        const TiledSym Pp = window(b - 1);
        g.A = operand(Pp); g.B = operand(Pp); g.C = operand(Lown);
        g.row_step = G; g.i0 = first_own(s0); g.j0 = s0; g.k0 = s0 - ob; g.k1 = s0;
        if ((e = launch_gemm(X, GEMM_UPDATE, g, s1 - s0, cnt, 1)) != cudaSuccess) return e;
        ++ctx->launches;
        ctx->timings[6] += 1;
      }
    }
    // exchange: every rank receives the whole block column into its window
    const int slots = (nrows - s0 + G - 1) / G;
    if ((e = launch_rowcyclic_pack(X, Lown, s0, s0 + ob, s0, nrows, G, me, slots, sendb)) != cudaSuccess) return e;
    if (nccl_api().AllGather(sendb, recvb, (size_t)slots * ob * TT, NCCL_DOUBLE, ctx->comm_small ? ctx->comm_small : ctx->comm, X) != 0) {
      ctx->dist_error = 1;
      return cudaErrorUnknown;
    }
    if ((e = launch_rowcyclic_unpack(X, P, s0, s0 + ob, s0, nrows, G, -1, slots, recvb)) != cudaSuccess) return e;
    ctx->launches += 2;
    // the panel, on the window: every rank, all rows
    g.A = operand(P); g.B = operand(P); g.C = operand(P);
    g.row_step = 1;
    bool factored_ahead = false;
    for (int jj = s0; jj < s1; ++jj) {
      if (!factored_ahead) {
        if (jj > s0) {
          g.i0 = jj; g.j0 = jj; g.k0 = s0; g.k1 = jj;
          if ((e = launch_gemm(X, GEMM_UPDATE, g, 1, nrows - jj, 1)) != cudaSuccess) return e;
          ++ctx->launches;
        }
        if ((e = launch_potrf_tile(X, P, W, wstride, jj, 1, logdet, info)) != cudaSuccess) return e;
        ++ctx->launches;
      }
      factored_ahead = false;
      if (jj + 1 >= nrows) continue;
      if (counters && jj + 1 < s1 && (ctx->chain_fused == 2 || nrows - 1 - jj <= 40)) {
        if ((e = launch_chain_column(X, P, W, wstride, jj, s0, jj + 2, 1, 1, logdet, info, counters)) != cudaSuccess) return e;
        ++ctx->launches;
        factored_ahead = true;
      } else {
        g.i0 = jj + 1; g.j0 = jj;
        if ((e = launch_gemm(X, GEMM_TRSM, g, 1, nrows - jj - 1, 1)) != cudaSuccess) return e;
        ++ctx->launches;
      }
    }
    if ((e = cudaEventRecord(evX[b], X)) != cudaSuccess) return e;
    // trailing update of the own rows right of the NEXT block column (which X updates itself before its exchange)
    const int s2 = s1 + ob;
    if (s2 < nc) {
      const int f2 = first_own(s2), cnt2 = own_count(s2);
      if (cnt2 > 0) {
        if ((e = cudaStreamWaitEvent(Y, evX[b], 0)) != cudaSuccess) return e;
        GemmArgs t = g;
        t.A = operand(P); t.B = operand(P); t.C = operand(Lown);
        t.i0 = f2; t.j0 = s2; t.k0 = s0; t.k1 = s1; t.row_step = G;
        if ((e = launch_gemm(Y, GEMM_UPDATE, t, nc - s2, cnt2, 1)) != cudaSuccess) return e;
        ++ctx->launches;
        ctx->timings[6] += 1;
      }
    }
    if ((e = cudaEventRecord(evY[b], Y)) != cudaSuccess) return e;
    // off the critical path (X, after the event the trailing update waits for): the finished rows go home, z is collected
    if ((e = launch_tile_rows_copy(X, Lown, P, s0, s1, first_own(s0), G, nrows)) != cudaSuccess) return e;
    ++ctx->launches;
    if (zvec && nrows > nc) {
      if ((e = launch_rhs_row_extract(X, P, nc, s0, s1, zvec)) != cudaSuccess) return e;
      ++ctx->launches;
    }
  }
  if ((e = cudaEventRecord(ctx->ev_join[1], X)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(ctx->stream, ctx->ev_join[1], 0)) != cudaSuccess) return e;
  if ((e = cudaEventRecord(ctx->ev_join[0], Y)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0)) != cudaSuccess) return e;
  return cudaSuccess;
}

// Fork the batch into latent groups on separate streams (joined back into ctx->stream).  jstart > 0: extend a factor whose
// tile rows < jstart are final (see chol_factor_stream).
static bool use_rowcyclic(const lmm_ctx* ctx, int nt, int batch) {
  return ctx->partition_ilmm && ctx->partition_now && batch == 1 && ctx->comm && ctx->nranks > 1 && nt >= 2 * ctx->nranks && nccl_api().AllGather;
}
static bool use_rightlooking(const lmm_ctx* ctx, int nt, int batch) {
  // (with the integer-slice update on, a LARGE single factor is faster on the batched left-looking schedule: its wide updates run
  // at 2-3x the DMMA rate, which outweighs the exposed panel chain -- "ozaki_single_nt" tile rows and up)
  // (measured, 7 planes of 8 bits: N = 16384: 45.9 -> 33.1 ms, two factors 88.9 -> 44.4 ms; N = 8192: 7.1 -> 8.6 ms, two: 12.6 -> 8.7 ms)
  const bool oz_single = ctx->ozaki && ctx->ozaki_single_nt > 0 && nt >= (batch == 1 ? ctx->ozaki_single_nt : ctx->ozaki_single_nt * 2 / 3);
  return ctx->lookahead && batch <= 2 && nt >= 12 && !oz_single;
}

bool chol_takes_envelope(const lmm_ctx* ctx, int nt, int batch) { return !use_rowcyclic(ctx, nt, batch) && !use_rightlooking(ctx, nt, batch); }

cudaError_t chol_factor(lmm_ctx* ctx, TiledSym L, double* W, size_t wstride, int batch, double* logdet, int* info, int jstart,
                        const int* env_d, const int* env_h) {
  const int G = ctx->ngroups < batch ? ctx->ngroups : batch;
  if (!env_d || !env_h) env_d = env_h = nullptr;
  auto env_at = [&](const int* e, int b0) { return e ? e + (size_t)b0 * L.nt : nullptr; };
  if (jstart == 0) {  // the look-ahead / partitioned schedules factor from scratch only
    if (env_d && !chol_takes_envelope(ctx, L.nt, batch)) {
      // they read every tile: write the zeros a kernel-matrix build inside the envelope left out (a chunk of the batch that the
      // integer-slice workspace split off can land here)
      cudaError_t ez = launch_kmat_zero(ctx->stream, L, batch, env_d);
      if (ez != cudaSuccess) return ez;
      ++ctx->launches;
      env_d = env_h = nullptr;
    }
    if (use_rowcyclic(ctx, L.nt, batch)) return chol_factor_rowcyclic(ctx, L, W, wstride, logdet, info);
    if (use_rightlooking(ctx, L.nt, batch)) return chol_factor_rightlooking(ctx, L, W, wstride, batch, logdet, info);
  }
  cudaError_t e;
  // optional integer-slice trailing update: workspace for as many latents as fit; a larger batch is factored in chunks
  OzWs ozws{};
  const OzWs* oz = nullptr;
  if (ctx->ozaki && jstart == 0 && L.nt > ctx->outer_block && L.nt > ctx->ozaki_min_k && L.ntc == 0 && L.cyc_G == 0) {
    const int fit = ozaki_workspace(ctx, L.nt, batch, ozws);
    if (fit > 0) {
      oz = &ozws;
      if (fit < batch) {
        for (int c0 = 0; c0 < batch; c0 += fit) {
          const int cb = batch - c0 < fit ? batch - c0 : fit;
          TiledSym Lc{L.base + (size_t)c0 * L.batch_stride, L.nt, L.batch_stride};
          if ((e = chol_factor(ctx, Lc, W + (size_t)c0 * wstride, wstride, cb, logdet + c0, info + c0, 0, env_at(env_d, c0), env_at(env_h, c0))) !=
              cudaSuccess)
            return e;
        }
        return cudaSuccess;
      }
    }
  }
  auto oz_at = [&](int b0, OzWs& tmp) -> const OzWs* {
    if (!oz) return nullptr;
    tmp = *oz;
    tmp.slices += (size_t)b0 * oz->slice_stride;
    tmp.scale += (size_t)b0 * oz->scale_stride;
    tmp.fp += (size_t)b0 * oz->fp_stride;
    return &tmp;
  };
  // small grids (few latents x few tile rows, e.g. the reference's notebook shape: 20 latents, 5 tile columns): ONE stream,
  // one fused launch per tile column -- stream groups would only multiply the launches
  int* counters = nullptr;
  const bool chain_all = ctx->chain_fused && (long long)(L.nt - 1) * batch <= CHAIN_MAX_TILES && L.nt > 1;
  if (ctx->chain_fused && L.nt > 1 && (e = chain_counters(ctx, ctx->stream, L.nt, batch, &counters)) != cudaSuccess) return e;
  if (G <= 1 || L.nt <= 1 || chain_all)
    return chol_factor_stream(ctx, ctx->stream, L, W, wstride, batch, logdet, info, jstart, counters, oz, env_d, env_h);
  if ((e = cudaEventRecord(ctx->ev_fork, ctx->stream)) != cudaSuccess) return e;
  for (int gi = 0; gi < G; ++gi) {
    const int b0 = (int)((int64_t)batch * gi / G), b1 = (int)((int64_t)batch * (gi + 1) / G);
    cudaStream_t st = ctx->gstream[gi];
    if ((e = cudaStreamWaitEvent(st, ctx->ev_fork, 0)) != cudaSuccess) return e;
    TiledSym Lg{L.base + (size_t)b0 * L.batch_stride, L.nt, L.batch_stride};
    OzWs oztmp{};
    if ((e = chol_factor_stream(ctx, st, Lg, W + (size_t)b0 * wstride, wstride, b1 - b0, logdet + b0, info + b0, jstart,
                                counters ? counters + (size_t)b0 * chain_counter_ints(L.nt) : nullptr, oz_at(b0, oztmp), env_at(env_d, b0),
                                env_at(env_h, b0))) != cudaSuccess)
      return e;
    if ((e = cudaEventRecord(ctx->ev_join[gi], st)) != cudaSuccess) return e;
    if ((e = cudaStreamWaitEvent(ctx->stream, ctx->ev_join[gi], 0)) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// Workspace of the integer-slice path of the prediction sweep for the latents [0, batch) of one trsm_right_lt_stream call: digit planes
// and row scales of the finished factor (right operand) and of the finished columns of X (left operand).
struct OzPred {
  uint8_t* lsl; size_t lsl_stride; double* lsc; size_t lsc_stride;
  uint8_t* xsl; size_t xsl_stride; double* xsc; size_t xsc_stride;
  const LatentParams* params;  // kdiag = k(x*, x*) bounds the squared row norms of X = K(x*,x) L^{-T}
  int S, bits, min_k;
};

// X <- X L^{-T} for a rectangular tiled X (rows = e.g. test points): the same update/TRSM sweep
// with X's tile rows appended under the factor.  With `oz` the wide updates (K = s0 k-tiles against all finished columns) run as
// integer-slice products on the int8 tensor cores, exactly as in chol_factor_stream: the factor is sliced once up front (row scales =
// row 2-norms of L), every finished block column of X right after its TRSM (row scales from the prior variance).
cudaError_t trsm_right_lt_stream(lmm_ctx* ctx, cudaStream_t st, TiledRect X, TiledSym L, const double* W, size_t wstride, int batch,
                                 const OzPred* oz = nullptr) {
  const int nt = L.nt;
  int ob = ctx->outer_block;
  cudaError_t e;
  if (oz && nt <= 8) oz = nullptr;
  if (oz) {
    if (!ctx->outer_block_user) ob = 2;
    if ((e = launch_ozaki_factor_scales(st, L, batch, oz->lsc, oz->lsc_stride)) != cudaSuccess) return e;
    if ((e = launch_ozaki_slice(st, L, oz->lsc, oz->lsc_stride, oz->lsl, oz->lsl_stride, 1, nt - 1, 0, nt - 1, batch, oz->S, oz->bits)) != cudaSuccess) return e;
    if ((e = launch_ozaki_const_scales(st, oz->params, X.ntr, batch, oz->xsc, oz->xsc_stride)) != cudaSuccess) return e;
    ctx->launches += 3;
  }
  GemmArgs g{};
  g.A = operand(X);
  g.B = operand(L);
  g.C = operand(X);
  g.W = W;
  g.w_batch_stride = wstride;
  g.sym = 0;
  g.i0 = 0;
  for (int s0 = 0; s0 < nt; s0 += ob) {
    const int s1 = (s0 + ob < nt) ? s0 + ob : nt;
    if (s0 > 0) {
      g.j0 = s0; g.k0 = 0; g.k1 = s0;
      if (oz && s0 >= oz->min_k && (long long)s0 * TILE * oz->S * (oz->bits == 8 ? 16384 : 4096) < (1ll << 31))
        e = launch_ozaki_update_rect(st, X, oz->xsl, oz->xsl_stride, oz->xsc, oz->xsc_stride, oz->lsl, oz->lsl_stride, oz->lsc, oz->lsc_stride, s0,
                                     s1 - s0, s0, batch, oz->S, oz->bits);
      else
        e = launch_gemm(st, GEMM_UPDATE, g, s1 - s0, X.ntr, batch);
      if (e != cudaSuccess) return e;
      ++ctx->launches;
    }
    for (int jj = s0; jj < s1; ++jj) {
      if (jj > s0) {
        g.j0 = jj; g.k0 = s0; g.k1 = jj;
        if ((e = launch_gemm(st, GEMM_UPDATE, g, 1, X.ntr, batch)) != cudaSuccess) return e;
        ++ctx->launches;
      }
      g.j0 = jj;
      if ((e = launch_gemm(st, GEMM_TRSM, g, 1, X.ntr, batch)) != cudaSuccess) return e;
      ++ctx->launches;
    }
    if (oz && s1 < nt) {  // the block column of X is final: its digit planes, for the later wide updates
      if ((e = launch_ozaki_slice_rect(st, X, oz->xsc, oz->xsc_stride, oz->xsl, oz->xsl_stride, s0, s1 - s0, batch, oz->S, oz->bits)) != cudaSuccess) return e;
      ++ctx->launches;
    }
  }
  return cudaSuccess;
}

// `xbound` (device, one LatentParams per latent of the batch; nullable): kdiag bounds the squared row norms of the result -- what the
// integer-slice path needs to fix the row scales of X in advance.  Without it, or with the option off, every update runs on DMMA.
cudaError_t trsm_right_lt(lmm_ctx* ctx, TiledRect X, TiledSym L, const double* W, size_t wstride, int batch, const LatentParams* xbound) {
  const int G = ctx->ngroups < batch ? ctx->ngroups : batch;
  OzPred oz{};
  bool use_oz = false;
  if (ctx->ozaki && xbound && L.nt > 8 && L.ntc == 0 && L.cyc_G == 0) {
    OzWs ws{};
    if (ozaki_workspace(ctx, L.nt, batch, ws) >= batch) {
      const size_t per_x = (size_t)X.ntr * X.ntc * ctx->ozaki * 16384, per_xs = (size_t)X.ntr * TILE;
      const size_t need = (size_t)batch * (per_x + per_xs * sizeof(double));
      if (ctx->oz_x_bytes < need) {
        cudaStreamSynchronize(ctx->stream);
        if (ctx->oz_x) cudaFree(ctx->oz_x);
        ctx->oz_x = nullptr;
        ctx->oz_x_bytes = 0;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && free_b > need + ((size_t)4 << 30) && cudaMalloc(&ctx->oz_x, need) == cudaSuccess)
          ctx->oz_x_bytes = need;
        else
          cudaGetLastError();
      }
      if (ctx->oz_x_bytes >= need) {
        use_oz = true;
        oz = OzPred{ws.slices, ws.slice_stride, ws.scale, ws.scale_stride, (uint8_t*)ctx->oz_x, per_x,
                    (double*)((uint8_t*)ctx->oz_x + (size_t)batch * per_x), per_xs, xbound, ws.S, ws.bits, ws.min_k};
      }
    }
  }
  auto oz_at = [&](int b0, OzPred& tmp) -> const OzPred* {
    if (!use_oz) return nullptr;
    tmp = oz;
    tmp.lsl += (size_t)b0 * oz.lsl_stride; tmp.lsc += (size_t)b0 * oz.lsc_stride;
    tmp.xsl += (size_t)b0 * oz.xsl_stride; tmp.xsc += (size_t)b0 * oz.xsc_stride;
    tmp.params += b0;
    return &tmp;
  };
  OzPred t0{};
  if (G <= 1) return trsm_right_lt_stream(ctx, ctx->stream, X, L, W, wstride, batch, oz_at(0, t0));
  cudaError_t e;
  if ((e = cudaEventRecord(ctx->ev_fork, ctx->stream)) != cudaSuccess) return e;
  for (int gi = 0; gi < G; ++gi) {
    const int b0 = (int)((int64_t)batch * gi / G), b1 = (int)((int64_t)batch * (gi + 1) / G);
    cudaStream_t st = ctx->gstream[gi];
    if ((e = cudaStreamWaitEvent(st, ctx->ev_fork, 0)) != cudaSuccess) return e;
    TiledRect Xg{X.base + (size_t)b0 * X.batch_stride, X.ntr, X.ntc, X.batch_stride};
    TiledSym Lg{L.base + (size_t)b0 * L.batch_stride, L.nt, L.batch_stride};
    OzPred tg{};
    if ((e = trsm_right_lt_stream(ctx, st, Xg, Lg, W + (size_t)b0 * wstride, wstride, b1 - b0, oz_at(b0, tg))) != cudaSuccess) return e;
    if ((e = cudaEventRecord(ctx->ev_join[gi], st)) != cudaSuccess) return e;
    if ((e = cudaStreamWaitEvent(ctx->stream, ctx->ev_join[gi], 0)) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// X <- X L^{-T} for an upper-triangular X given as full rectangular tiles (zero tiles skipped).
cudaError_t trsm_right_lt_upper(lmm_ctx* ctx, cudaStream_t st, TiledRect X, TiledSym L, const double* W, size_t wstride, int batch) {
  const int nt = L.nt, ob = ctx->outer_block;
  GemmArgs g{};
  g.A = operand(X); g.B = operand(L); g.C = operand(X);
  g.W = W; g.w_batch_stride = wstride;
  g.sym = 0; g.upper = 1; g.k_from_row = 1; g.i0 = 0;
  cudaError_t e;
  for (int s0 = 0; s0 < nt; s0 += ob) {
    const int s1 = (s0 + ob < nt) ? s0 + ob : nt;
    if (s0 > 0) {
      g.j0 = s0; g.k0 = 0; g.k1 = s0;
      if ((e = launch_gemm(st, GEMM_UPDATE, g, s1 - s0, s0, batch)) != cudaSuccess) return e;  // rows < s0 have k < s0 terms
      ++ctx->launches;
    }
    for (int jj = s0; jj < s1; ++jj) {
      if (jj > s0) {
        g.j0 = jj; g.k0 = s0; g.k1 = jj;
        if ((e = launch_gemm(st, GEMM_UPDATE, g, 1, jj, batch)) != cudaSuccess) return e;
        ++ctx->launches;
      }
      g.j0 = jj;
      if ((e = launch_gemm(st, GEMM_TRSM, g, 1, jj + 1, batch)) != cudaSuccess) return e;
      ++ctx->launches;
    }
  }
  return cudaSuccess;
}

}  // namespace lmm_host

// ------------------------------------------------------------------------------------------------
// Batched Cholesky primitive
// ------------------------------------------------------------------------------------------------
extern "C" int lmm_potrf_batched(lmm_ctx* ctx, const double* A, int N, int batch, double* L_out, double* logdet_out, int* info) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!A || N <= 0 || batch <= 0) return ctx->fail(LMM_E_ARG, "null pointer or non-positive size");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  const int nt = ntiles(N);
  DevBuf b_A, b_L, b_W, b_logdet, b_info;
  const double* dA = A;
  if (!is_device_ptr(A)) {
    CU(b_A.alloc(ctx, (size_t)batch * N * N * sizeof(double)));
    CU(copy_in(ctx, b_A.as<double>(), A, (size_t)batch * N * N));
    dA = b_A.as<double>();
  }
  CU(b_L.alloc(ctx, (size_t)batch * sym_tiles(nt) * TT * sizeof(double)));
  CU(b_W.alloc(ctx, (size_t)batch * nt * TT * sizeof(double)));
  CU(b_logdet.alloc(ctx, (size_t)batch * sizeof(double)));
  CU(b_info.alloc(ctx, (size_t)batch * sizeof(int)));
  CU(cudaMemsetAsync(b_logdet.p, 0, (size_t)batch * sizeof(double), st));
  CU(cudaMemsetAsync(b_info.p, 0, (size_t)batch * sizeof(int), st));
  TiledSym L{b_L.as<double>(), nt, sym_tiles(nt) * TT};
  CU(launch_tile_from_dense(st, L, batch, dA, N));
  ++ctx->launches;
  CU(cudaEventRecord(ctx->ev[0], st));
  {
    PartitionScope scope(ctx);
    CU(chol_factor(ctx, L, b_W.as<double>(), (size_t)nt * TT, batch, b_logdet.as<double>(), b_info.as<int>()));
  }
  CU(cudaEventRecord(ctx->ev[1], st));
  std::vector<int> hinfo(batch, 0);
  CU(copy_out(ctx, hinfo.data(), b_info.p, (size_t)batch * sizeof(int)));
  if (logdet_out) CU(copy_out(ctx, logdet_out, b_logdet.p, (size_t)batch * sizeof(double)));
  if (L_out) {
    DevBuf dense;
    CU(dense.alloc(ctx, (size_t)N * N * sizeof(double)));
    for (int b = 0; b < batch; ++b) {
      CU(cudaMemsetAsync(dense.p, 0, (size_t)N * N * sizeof(double), st));
      CU(launch_untile_lower(st, L, b, dense.as<double>(), N));
      ++ctx->launches;
      CU(copy_out(ctx, L_out + (size_t)b * N * N, dense.p, (size_t)N * N * sizeof(double)));
      CU(cudaStreamSynchronize(st));
    }
  }
  CU(cudaStreamSynchronize(st));
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
  ctx->timings[0] = ms;
  ctx->timings[2] = ms;
  int worst = 0;
  for (int b = 0; b < batch; ++b) {
    int v = hinfo[b] > N ? N : hinfo[b];
    if (info) info[b] = v;
    if (v > worst) worst = v;
  }
  return worst;
}

extern "C" int lmm_potrf_bench(lmm_ctx* ctx, const lmm_gp_desc* desc, const double* x, int N, int D, double noise, int batch,
                               double* logdet_out, double* out_ms_kmat, double* out_ms_chol) {
  if (!ctx) return LMM_E_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (!desc || !x || N <= 0 || D <= 0 || batch <= 0) return ctx->fail(LMM_E_ARG, "null pointer or non-positive size");
  int rc = check_descs(ctx, desc, 1, D);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (double& t : ctx->timings) t = 0.0;
  const int nt = ntiles(N);
  const size_t npad = (size_t)nt * TILE;
  DevBuf b_x, b_L, b_W, b_logdet, b_info, b_params;
  CU(b_x.alloc(ctx, npad * D * sizeof(double)));
  CU(cudaMemsetAsync(b_x.p, 0, npad * D * sizeof(double), st));
  CU(copy_in(ctx, b_x.as<double>(), x, (size_t)N * D));
  std::vector<LatentParams> hp(batch);
  for (int b = 0; b < batch; ++b) {
    set_params(hp[b], *desc, noise, 1.0, D);
  }
  CU(b_params.alloc(ctx, hp.size() * sizeof(LatentParams)));
  CU(cudaMemcpyAsync(b_params.p, hp.data(), hp.size() * sizeof(LatentParams), cudaMemcpyHostToDevice, st));
  CU(b_L.alloc(ctx, (size_t)batch * sym_tiles(nt) * TT * sizeof(double)));
  CU(b_W.alloc(ctx, (size_t)batch * nt * TT * sizeof(double)));
  CU(b_logdet.alloc(ctx, (size_t)batch * sizeof(double)));
  CU(b_info.alloc(ctx, (size_t)batch * sizeof(int)));
  CU(cudaMemsetAsync(b_logdet.p, 0, (size_t)batch * sizeof(double), st));
  CU(cudaMemsetAsync(b_info.p, 0, (size_t)batch * sizeof(int), st));
  TiledSym L{b_L.as<double>(), nt, sym_tiles(nt) * TT};
  CU(cudaEventRecord(ctx->ev[0], st));
  CU(launch_kmat_sym(st, L, batch, b_x.as<double>(), N, D, b_params.as<LatentParams>(), ctx->distance_form));
  ++ctx->launches;
  CU(cudaEventRecord(ctx->ev[1], st));
  {
    PartitionScope scope(ctx);
    CU(chol_factor(ctx, L, b_W.as<double>(), (size_t)nt * TT, batch, b_logdet.as<double>(), b_info.as<int>()));
  }
  CU(cudaEventRecord(ctx->ev[2], st));
  std::vector<int> hinfo(batch, 0);
  CU(copy_out(ctx, hinfo.data(), b_info.p, (size_t)batch * sizeof(int)));
  if (logdet_out) CU(copy_out(ctx, logdet_out, b_logdet.p, (size_t)batch * sizeof(double)));
  CU(cudaStreamSynchronize(st));
  float a = 0, c = 0;
  cudaEventElapsedTime(&a, ctx->ev[0], ctx->ev[1]);
  cudaEventElapsedTime(&c, ctx->ev[1], ctx->ev[2]);
  if (out_ms_kmat) *out_ms_kmat = a;
  if (out_ms_chol) *out_ms_chol = c;
  ctx->timings[0] = a + c; ctx->timings[1] = a; ctx->timings[2] = c;
  int worst = 0;
  for (int b = 0; b < batch; ++b) {
    int v = hinfo[b] > N ? N : hinfo[b];
    if (v > worst) worst = v;
  }
  return worst;
}
