// bf16 two-term split operands for tcgen05 (v = hi + mid, residual <= 2^-17 |v|): row writers for the 128-B-swizzled
// UMMA tiles and the multi-product MMA issue helpers shared by the update (update_tc.cu) and value (values_tc.cu) kernels.
#pragma once
#include "tc.cuh"

namespace aur {

// the two bf16 halves of a packed pair, negated, as fp32: adding them takes both residuals with one FADD2
__device__ __forceinline__ float2 neg_bf16x2(unsigned int w) {
  return make_float2(-__uint_as_float(w << 16), -__uint_as_float(w & 0xFFFF0000u));
}

// 8 fp32 values (4 pairs) -> one 16-B chunk of bf16 hi and one of bf16 mid (v - hi), chunk `c` of row `r` (128-B swizzle)
__device__ __forceinline__ void store_split_chunk(unsigned char* tile_hi, unsigned char* tile_mid, int r, int c, const float2* v) {
  unsigned int hi[4], mid[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    __nv_bfloat162 h = __float22bfloat162_rn(v[e]);
    const unsigned int hw = *reinterpret_cast<unsigned int*>(&h);
    hi[e] = hw;
    __nv_bfloat162 m = __float22bfloat162_rn(__fadd2_rn(v[e], neg_bf16x2(hw)));
    mid[e] = *reinterpret_cast<unsigned int*>(&m);
  }
  const int off = r * 128 + ((c ^ (r & 7)) << 4);
  *reinterpret_cast<uint4*>(tile_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<uint4*>(tile_mid + off) = make_uint4(mid[0], mid[1], mid[2], mid[3]);
}

// three-term variant (v = hi + mid + lo, residual <= 2^-25 |v|: fp32-equivalent operands)
__device__ __forceinline__ void store_split3_chunk(unsigned char* tile_hi, unsigned char* tile_mid, unsigned char* tile_lo, int r, int c,
                                                   const float2* v) {
  unsigned int hi[4], mid[4], lo[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    __nv_bfloat162 h = __float22bfloat162_rn(v[e]);
    const unsigned int hw = *reinterpret_cast<unsigned int*>(&h);
    const float2 rs = __fadd2_rn(v[e], neg_bf16x2(hw));
    __nv_bfloat162 m = __float22bfloat162_rn(rs);
    const unsigned int mw = *reinterpret_cast<unsigned int*>(&m);
    __nv_bfloat162 l = __float22bfloat162_rn(__fadd2_rn(rs, neg_bf16x2(mw)));
    hi[e] = hw; mid[e] = mw; lo[e] = *reinterpret_cast<unsigned int*>(&l);
  }
  const int off = r * 128 + ((c ^ (r & 7)) << 4);
  *reinterpret_cast<uint4*>(tile_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<uint4*>(tile_mid + off) = make_uint4(mid[0], mid[1], mid[2], mid[3]);
  *reinterpret_cast<uint4*>(tile_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// three-product split MMA: D (+)= A_hi B_hi + A_hi B_mid + A_mid B_hi over `ksteps` steps of K = 16
__device__ __forceinline__ void mma_split(uint32_t d, uint64_t a_hi, uint64_t a_mid, uint64_t b_hi, uint64_t b_mid, uint32_t idesc,
                                          int ksteps, uint32_t a_step, uint32_t b_step, bool accumulate) {
  for (int k = 0; k < ksteps; ++k)
    tc::mma_f16(d, a_hi + (uint64_t)(a_step * k), b_hi + (uint64_t)(b_step * k), idesc, (accumulate || k > 0) ? 1u : 0u);
  for (int k = 0; k < ksteps; ++k) tc::mma_f16(d, a_hi + (uint64_t)(a_step * k), b_mid + (uint64_t)(b_step * k), idesc, 1u);
  for (int k = 0; k < ksteps; ++k) tc::mma_f16(d, a_mid + (uint64_t)(a_step * k), b_hi + (uint64_t)(b_step * k), idesc, 1u);
}
// four-product variant (adds mid*mid): ~2^-17 relative per product, used where the result is compared at 1e-5
__device__ __forceinline__ void mma_split4(uint32_t d, uint64_t a_hi, uint64_t a_mid, uint64_t b_hi, uint64_t b_mid, uint32_t idesc,
                                           int ksteps, uint32_t a_step, uint32_t b_step, bool accumulate) {
  mma_split(d, a_hi, a_mid, b_hi, b_mid, idesc, ksteps, a_step, b_step, accumulate);
  for (int k = 0; k < ksteps; ++k) tc::mma_f16(d, a_mid + (uint64_t)(a_step * k), b_mid + (uint64_t)(b_step * k), idesc, 1u);
}

// six products of three-term operands (everything above 2^-25): fp32-equivalent contraction
__device__ __forceinline__ void mma_split6(uint32_t d, const uint64_t (&a)[3], const uint64_t (&b)[3], uint32_t idesc, int ksteps,
                                           uint32_t a_step, uint32_t b_step, bool accumulate = false) {
  const int pa[6] = {0, 0, 1, 1, 0, 2}, pb[6] = {0, 1, 0, 1, 2, 0};
  for (int p = 0; p < 6; ++p)
    for (int k = 0; k < ksteps; ++k)
      tc::mma_f16(d, a[pa[p]] + (uint64_t)(a_step * k), b[pb[p]] + (uint64_t)(b_step * k), idesc, (accumulate || p > 0 || k > 0) ? 1u : 0u);
}

}  // namespace aur
