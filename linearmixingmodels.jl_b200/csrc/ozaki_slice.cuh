// Digit planes of one finished factor tile (csrc/ozaki.cu: the integer-slice trailing update reads them).  Included by ozaki.cu
// (ozaki_slice_kernel) and gemm.cu (the panel TRSM that slices the tiles it has just finished).
#pragma once
#include "common.cuh"

namespace lmm {

constexpr int OZ_QB = 4096;  // bytes of one slice of one K quarter (128 rows x 32 K-bytes)

// One tile, 256 threads (the whole CTA): `tile` in the tile layout (global or shared memory), `scale` the 128 row scales of its tile
// row, `out` its S * 16384 bytes of digit planes, `fp` (nullable) its first-plane byte.  Shared by the slice kernel and the panel
// TRSM that writes the planes of the tiles it has just finished (gemm.cu), so both produce the same bytes.
__device__ __forceinline__ void oz_slice_tile(const double* tile, const double* __restrict__ scale, uint8_t* __restrict__ out, int S, int bits,
                              uint8_t* __restrict__ fp) {
  __shared__ uint32_t nz_planes;  // bit t: plane t has a nonzero digit
  if (fp) {
    // all-zero tile?  X = round(y R^(S-1)) == 0 for every entry (the radix-256 rule below: X itself; radix 128: the round-to-nearest
    // remainders of |y R^t| <= 1/2 are y R^(t+1), exact, so every digit is zero iff |y R^(S-1)| <= 1/2, i.e. rint gives 0)
    const double fine = __longlong_as_double((long long)(1023 + (bits == 8 ? 8 : 7) * (S - 1)) << 52);  // R^(S-1), exact
    bool any = false;
    for (int it = threadIdx.x; it < 1024; it += 256) {
      const int r = it & 127, c16 = it >> 7;
      const double inv = 1.0 / scale[r];
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        const double2* p = reinterpret_cast<const double2*>(tile + (size_t)(4 * c16 + gq) * 512 + 4 * r);
        const double2 a = p[0], c = p[1];
        any |= (__double2ll_rn(a.x * inv * fine) | __double2ll_rn(a.y * inv * fine) | __double2ll_rn(c.x * inv * fine) |
                __double2ll_rn(c.y * inv * fine)) != 0;
      }
    }
    if (threadIdx.x == 0) nz_planes = 0;
    if (!__syncthreads_or(any)) {
      if (threadIdx.x == 0) *fp = (uint8_t)S;
      return;
    }
  }
  uint32_t nz = 0;  // this thread's planes with a nonzero digit
  for (int it = threadIdx.x; it < 1024; it += 256) {
    const int r = it & 127, c16 = it >> 7;  // 16 columns c16*16 .. +15 of row r
    const double inv = 1.0 / scale[r];  // 2^(6 - E): exact
    double y[16];
#pragma unroll
    for (int gq = 0; gq < 4; ++gq) {
      const double2* p = reinterpret_cast<const double2*>(tile + (size_t)(4 * c16 + gq) * 512 + 4 * r);
      const double2 a = p[0], c = p[1];
      y[4 * gq + 0] = a.x * inv; y[4 * gq + 1] = a.y * inv; y[4 * gq + 2] = c.x * inv; y[4 * gq + 3] = c.y * inv;
    }
    uint8_t* dst = out + (size_t)(c16 >> 1) * S * OZ_QB + (size_t)(c16 & 1) * 2048 + (size_t)r * 16;
    if (bits == 8) {
      // radix 256, digits in [-128, 127]: X = round(y * 256^(S-1)) as a 64-bit integer (|X| <= 2^(6 + 8 (S-1)) < 2^63), balanced digits
      // from the bottom with exact carries, the top plane keeps what is left (|q_0| <= 65)
      uint32_t w[8][4] = {};
      const double up = __longlong_as_double((long long)(1023 + 8 * (S - 1)) << 52);  // 256^(S-1), exact
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        long long X = __double2ll_rn(y[e] * up);
#pragma unroll
        for (int t = 7; t >= 1; --t) {  // (static plane indices: w stays in registers)
          if (t < S) {
            const long long q = ((X + 128) & 255) - 128;
            X = (X - q) >> 8;
            w[t][e >> 2] |= ((uint32_t)q & 0xFFu) << (8 * (e & 3));
          }
        }
        w[0][e >> 2] |= ((uint32_t)X & 0xFFu) << (8 * (e & 3));
      }
#pragma unroll
      for (int t = 0; t < 8; ++t)
        if (t < S) {
          *reinterpret_cast<uint4*>(dst + (size_t)t * OZ_QB) = make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
          if (w[t][0] | w[t][1] | w[t][2] | w[t][3]) nz |= 1u << t;
        }
      continue;
    }
    for (int t = 0; t < S; ++t) {
      uint32_t w[4];
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        uint32_t pk = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          // round to nearest by the 1.5 * 2^52 shift: the low word of t is the digit in two's complement, t - M the digit as a
          // double (two DADDs instead of a rounding and a conversion instruction); |v| <= 64 (1 + few eps), so no clamp is needed
          double& v = y[4 * gq + j];
          const double t = v + 6755399441055744.0;
          v = (v - (t - 6755399441055744.0)) * 128.0;
          pk |= ((uint32_t)__double2loint(t) & 0xFFu) << (8 * j);
        }
        w[gq] = pk;
      }
      *reinterpret_cast<uint4*>(dst + (size_t)t * OZ_QB) = make_uint4(w[0], w[1], w[2], w[3]);
      if (w[0] | w[1] | w[2] | w[3]) nz |= 1u << t;
    }
  }
  if (fp) {
    if (nz) atomicOr(&nz_planes, nz);
    __syncthreads();
    if (threadIdx.x == 0) *fp = (uint8_t)(nz_planes ? __ffs(nz_planes) - 1 : S);
  }
}

}  // namespace lmm
