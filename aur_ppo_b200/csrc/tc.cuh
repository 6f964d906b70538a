// tcgen05 / TMEM / TMA building blocks (sm_100a): PTX wrappers, shared-memory matrix descriptors,
// instruction descriptors, tensor-map creation.  Used by the tensor-core GEMM / implicit-GEMM
// convolution kernels of the equivariant encoder path (row X).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"

namespace aur {
namespace tc {

// ---- TMEM allocation (one full warp executes these) ---------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  // hand the allocation permit back right away: a co-resident CTA's tcgen05.alloc waits for it otherwise
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// make generic-proxy smem writes visible to the async proxy (UMMA / TMA reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout) --------------
// K-major operand, SWIZZLE_128B: rows of 128 bytes (64 bf16 / 32 tf32), 8-row groups of 1024 B.
__device__ __forceinline__ uint64_t smem_desc_k_sw128(const void* smem_ptr) {
  const uint32_t addr = smem_u32(smem_ptr);
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);   // start address, 16-B units
  d |= (uint64_t)1 << 16;                  // leading byte offset (ignored for swizzled K-major) = 1
  d |= (uint64_t)(1024 >> 4) << 32;        // stride byte offset: 8 rows x 128 B
  d |= (uint64_t)1 << 46;                  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                  // SWIZZLE_128B
  return d;
}
// MN-major operand, SWIZZLE_128B: the contiguous dimension is M/N (64 bf16 = 128 B per row),
// 8 K-rows of 128 B form one 1024-B swizzle atom; atoms along MN are `lbo_bytes` apart,
// groups of 8 along K are `sbo_bytes` apart.
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(const void* smem_ptr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  const uint32_t addr = smem_u32(smem_ptr);
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// ---- instruction descriptor (cute::UMMA::InstrDescriptor), fp32 accumulate ------------------
enum : uint32_t { FMT_F16 = 0, FMT_BF16 = 1, FMT_TF32 = 2 };
__host__ __device__ constexpr uint32_t instr_desc(uint32_t fmt, uint32_t M, uint32_t N, uint32_t a_mn_major, uint32_t b_mn_major) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (a_mn_major << 15) | (b_mn_major << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when complete (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- TMEM -> registers: 32 lanes x 32 columns of fp32 per warp -------------------------------
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 lanes x 16 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 32 lanes x 8 columns, split issue / wait so several loads overlap
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// the same as 4 column pairs (column 2 i -> v[i].x, 2 i + 1 -> v[i].y), for packed fp32x2 arithmetic
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, float2* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM, 32 lanes x 8 columns
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
               "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float2* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(__float_as_uint(v[0].x)), "r"(__float_as_uint(v[0].y)), "r"(__float_as_uint(v[1].x)), "r"(__float_as_uint(v[1].y)),
               "r"(__float_as_uint(v[2].x)), "r"(__float_as_uint(v[2].y)), "r"(__float_as_uint(v[3].x)), "r"(__float_as_uint(v[3].y))
               : "memory");
}
// one column: a 32-bit word per lane
__device__ __forceinline__ void tmem_st1(uint32_t taddr, float v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(__float_as_uint(v)) : "memory");
}
__device__ __forceinline__ float tmem_ld1(uint32_t taddr) {
  uint32_t r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  return __uint_as_float(r);
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- TMA tensor loads (tile mode), completion on an mbarrier ---------------------------------
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
          smem_u32(smem_dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(
          smem_u32(smem_dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// ---- host: tensor-map encode through the driver entry point (no -lcuda link dependency) ------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn();
// rank-R tiled map over `base` with dims[0] the contiguous dimension; strides in BYTES for dims 1..R-1;
// 128-B swizzle (box[0] * elem_bytes must be 128).
int make_tensor_map(CUtensorMap* out, CUtensorMapDataType dt, int rank, const void* base, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box);


// ---- operand precision of the row-X tensor-core entry points (aur_tc_set_precision) -------------------------------
// 1 plane : bf16 operands (fast mode, below the reference's fp32 arithmetic).
// 2 planes: every bf16 tensor is a stack [2][...] of a HI plane bf16(v) and a MID plane bf16(v - hi), |v - hi - mid| <=
//           2^-18 |v|; contractions issue hi*hi + hi*mid + mid*hi with fp32 accumulation in TMEM (3x the MMA work):
//           ~3e-5 relative through the seven-layer encoders.
// 3 planes: a third LO plane bf16(v - hi - mid) (3 x 8 = 24 mantissa bits: all of fp32) and six products hi*hi + hi*mid +
//           mid*hi + mid*mid + hi*lo + lo*hi (everything above 2^-24 of the product): fp32-equivalent, 6x the MMA work.
// The planes are walked as extra K steps of the same pipelines: plane index = outermost TMA coordinate.
int tc_planes();
__host__ __device__ __forceinline__ int tc_terms(int planes) { return planes == 1 ? 1 : (planes == 2 ? 3 : 6); }
// K-step term -> (plane of the first operand, plane of the second): 0 (0,0)  1 (0,1)  2 (1,0)  3 (1,1)  4 (0,2)  5 (2,0)
__host__ __device__ __forceinline__ int term_plane_a(int t) { return (t == 2 || t == 3) ? 1 : (t == 5 ? 2 : 0); }
__host__ __device__ __forceinline__ int term_plane_b(int t) { return (t == 1 || t == 3) ? 1 : (t == 4 ? 2 : 0); }
#ifdef __CUDACC__
__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& mid) {
  hi = __float2bfloat16_rn(v);
  mid = __float2bfloat16_rn(v - __bfloat162float(hi));
}
// v -> plane p of nplanes planes at dst[p * plane_stride] (successive bf16 roundings of the remainder)
__device__ __forceinline__ void store_planes(__nv_bfloat16* dst, size_t plane_stride, int nplanes, float v) {
  for (int p = 0; p < nplanes; ++p) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    dst[(size_t)p * plane_stride] = h;
    v -= __bfloat162float(h);
  }
}
// 8 consecutive values -> one 16-byte store per plane
__device__ __forceinline__ void store8_planes(__nv_bfloat16* dst, size_t plane_stride, int nplanes, const float* v) {
  float r[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) r[i] = v[i];
  for (int p = 0; p < nplanes; ++p) {
    uint4 pk;
    unsigned int* w = reinterpret_cast<unsigned int*>(&pk);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 t = __floats2bfloat162_rn(r[2 * j], r[2 * j + 1]);
      w[j] = *reinterpret_cast<const unsigned int*>(&t);
      r[2 * j] -= __low2float(t);
      r[2 * j + 1] -= __high2float(t);
    }
    *reinterpret_cast<uint4*>(dst + (size_t)p * plane_stride) = pk;
  }
}
// sum of the planes of one element
__device__ __forceinline__ float load_planes(const __nv_bfloat16* src, size_t plane_stride, int nplanes) {
  float v = 0.0f;
  for (int p = nplanes - 1; p >= 0; --p) v += __bfloat162float(src[(size_t)p * plane_stride]);
  return v;
}
#endif

}  // namespace tc
}  // namespace aur
