// Batched critic forward on tensor cores: values[i] = critic(obs[i]) for a whole [T*N] observation buffer.
// In the reference the critic is evaluated inside the rollout loop (actor_critic.evaluate, ppo.py:105, and
// policy.value, ppo.py:161), but a value never feeds back into the trajectory (only the actor's action does),
// so the fused rollout kernel keeps just the actor + physics on its sequential path and the T*N values are one
// embarrassingly parallel pass over the observation rows it has just written (contiguous, no gather).
//
// Same scheme as update_tc.cu's forward (hidden 64 or 128): CTA = 128 samples x 2 feature halves, first layer in registers, h1 rows
// written as a THREE-term bf16 split (hi + mid + lo, fp32-equivalent: values are compared with the reference at
// 2e-6) into 128-B-swizzled tiles, z2 = h1 W2^T on tcgen05 as six products with fp32 accumulation in TMEM, tanh +
// 64->1 head from TMEM lanes.
// Three CTAs per SM (75 KB of shared memory each) cover each other's MMA round trip.  HBM: 16 + 4 B per sample.
#include "tc_split.cuh"
#include "policy.cuh"

namespace aur {

constexpr int VT_S = 128, VT_THREADS = 256;
constexpr int VT_TILE = VT_S * 128;              // one K atom of the h1 tile: 128 samples x 64 features
// H = 64: three CTAs per SM (75 KB each).  H = 128 (`--hidden_dim 128`): two K atoms per tile, W2 128 rows: 195 KB, one CTA per SM.
template <int H>
struct VtCfg {
  static constexpr int KA = H / 64, WTILE = H * 128, FPT = H / 2;       // FPT: features per thread (two threads per sample)
  static constexpr int O_H1 = 0;                                        // [hi, mid, lo][atom]
  static constexpr int O_W2 = O_H1 + 3 * KA * VT_TILE;                  // [hi, mid, lo][atom]
  static constexpr int O_SMALL = O_W2 + 3 * KA * WTILE;                 // W1^T [4][H], b1 [H], b2 [H], W3 [H], b3
  static constexpr int S_W1T = 0, S_B1 = 4 * H, S_B2 = 5 * H, S_W3 = 6 * H, S_B3 = 7 * H, S_N = 7 * H + 4;
  static constexpr int O_BAR = O_SMALL + S_N * 4;
  static constexpr size_t SMEM = O_BAR + 16 + 1024;
  static constexpr int CTAS = H == 64 ? 3 : 1;
};
static_assert(3 * (VtCfg<64>::SMEM + 1024) <= 233472, "three CTAs per SM");
static_assert(VtCfg<128>::SMEM <= 232448, "one CTA per SM");

// POP: population form, grid (x, K): the rows are T segments per member of n_member rows each, segment (t, k) at rows
// (t * K + k) * n_member ..; CTA (x, k) walks member k's tiles (at most 128 rows of one segment) with member k's critic
// (critic + k * pop_P).  A value depends on its own row only, so it is the single run's whatever the tiling.
template <int H, bool POP = false>
__global__ void __launch_bounds__(VT_THREADS, VtCfg<H>::CTAS) critic_values_tc_kernel(const float* __restrict__ critic, int obs_dim,
                                                                                      const float* __restrict__ obs, long long M,
                                                                                      float* __restrict__ out, int pop_K,
                                                                                      long long n_member, long long pop_P) {
  using Cfg = VtCfg<H>;
  if constexpr (POP) critic += (long long)blockIdx.y * pop_P;
  constexpr int KA = Cfg::KA, FPT = Cfg::FPT;
  constexpr int VS_W1T = Cfg::S_W1T, VS_B1 = Cfg::S_B1, VS_B2 = Cfg::S_B2, VS_W3 = Cfg::S_W3, VS_B3 = Cfg::S_B3;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* h1t[3] = {base + Cfg::O_H1, base + Cfg::O_H1 + KA * VT_TILE, base + Cfg::O_H1 + 2 * KA * VT_TILE};
  unsigned char* w2t[3] = {base + Cfg::O_W2, base + Cfg::O_W2 + KA * Cfg::WTILE, base + Cfg::O_W2 + 2 * KA * Cfg::WTILE};
  float* sw = reinterpret_cast<float*>(base + Cfg::O_SMALL);
  uint64_t* bar = reinterpret_cast<uint64_t*>(base + Cfg::O_BAR);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(base + Cfg::O_BAR + 8);
  const int tid = threadIdx.x, warp = tid >> 5, s = tid & 127, half = tid >> 7, f0 = FPT * half;

  if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  if (warp == 0) tc::tmem_alloc(tslot, H);
  {
    const float* gb1 = critic + H * obs_dim;
    const float* gW2 = gb1 + H;
    const float* gb2 = gW2 + H * H;
    const float* gW3 = gb2 + H;
    for (int e = tid; e < 4 * H; e += VT_THREADS) {
      const int c = e / H, j = e - c * H;
      sw[VS_W1T + e] = c < obs_dim ? TANH_PRESCALE * critic[j * obs_dim + c] : 0.0f;      // tanh argument scale folded in
    }
    for (int e = tid; e < H; e += VT_THREADS) { sw[VS_B1 + e] = TANH_PRESCALE * gb1[e]; sw[VS_B2 + e] = TANH_PRESCALE * gb2[e]; sw[VS_W3 + e] = gW3[e]; }
    if (tid == 0) sw[VS_B3] = gW3[H];
#pragma unroll 1
    for (int e = tid; e < H * (H / 8); e += VT_THREADS) {
      const int j = e % H, ch = e / H;
      float2 v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = make_float2(gW2[j * H + 8 * ch + 2 * q], gW2[j * H + 8 * ch + 2 * q + 1]);
      const int o = (ch >> 3) * Cfg::WTILE;
      store_split3_chunk(w2t[0] + o, w2t[1] + o, w2t[2] + o, j, ch & 7, v);
    }
  }
  tc::fence_proxy_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tm_z = *tslot;
  const uint32_t lane_base = (uint32_t)(32 * (warp & 3)) << 16;
  constexpr uint32_t ID_FWD = tc::instr_desc(tc::FMT_BF16, 128, H, 0, 0);
  const bool vec = obs_dim == 4 && (reinterpret_cast<uintptr_t>(obs) & 15) == 0;

  // POP: member-local tiles, tps per segment
  const long long tps = POP ? (n_member + VT_S - 1) / VT_S : 1;
  const long long ntiles = POP ? (M / ((long long)pop_K * n_member)) * tps : (M + VT_S - 1) / VT_S;
  auto tile_row = [&](long long tile, bool& ok) -> long long {
    if constexpr (POP) {
      const long long t = tile / tps, r = (tile - t * tps) * VT_S + s;
      ok = tile < ntiles && r < n_member;
      return (t * pop_K + blockIdx.y) * n_member + r;
    } else {
      const long long row = tile * VT_S + s;
      ok = tile < ntiles && row < M;
      return row;
    }
  };
  auto load_obs = [&](long long tile, float (&x)[POL_IN_PAD]) {
    bool ok;
    const long long row = tile_row(tile, ok);
    if (ok && vec) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(obs) + row);
      x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
    } else {
#pragma unroll
      for (int c = 0; c < POL_IN_PAD; ++c) x[c] = (ok && c < obs_dim) ? __ldg(obs + row * obs_dim + c) : 0.0f;
    }
  };
  float xn[POL_IN_PAD];
  load_obs(blockIdx.x, xn);
  uint32_t it = 0;
#pragma unroll 1
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    // ---- first layer -> operand rows (8-feature chunks)
#pragma unroll
    for (int c = 0; c < FPT / 8; ++c) {
      float2 hv[4];
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const int f = f0 + 8 * c + 4 * g;
        const float4 b = lds4(sw + VS_B1 + f);
        float2 a01 = make_float2(b.x, b.y), a23 = make_float2(b.z, b.w);
#pragma unroll
        for (int cc = 0; cc < POL_IN_PAD; ++cc) {
          const float4 w = lds4(sw + VS_W1T + cc * H + f);
          const float2 xx = make_float2(xn[cc], xn[cc]);
          a01 = __ffma2_rn(make_float2(w.x, w.y), xx, a01);
          a23 = __ffma2_rn(make_float2(w.z, w.w), xx, a23);
        }
        hv[2 * g] = tanh_prescaled2(a01);
        hv[2 * g + 1] = tanh_prescaled2(a23);
      }
      const int ch = (FPT / 8) * half + c, o = (ch >> 3) * VT_TILE;
      store_split3_chunk(h1t[0] + o, h1t[1] + o, h1t[2] + o, s, ch & 7, hv);
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    if (tid == 0) {
      tc::fence_after_sync();
#pragma unroll
      for (int ka = 0; ka < KA; ++ka) {
        const uint64_t da[3] = {tc::smem_desc_k_sw128(h1t[0] + ka * VT_TILE), tc::smem_desc_k_sw128(h1t[1] + ka * VT_TILE),
                                tc::smem_desc_k_sw128(h1t[2] + ka * VT_TILE)};
        const uint64_t db[3] = {tc::smem_desc_k_sw128(w2t[0] + ka * Cfg::WTILE), tc::smem_desc_k_sw128(w2t[1] + ka * Cfg::WTILE),
                                tc::smem_desc_k_sw128(w2t[2] + ka * Cfg::WTILE)};
        mma_split6(tm_z, da, db, ID_FWD, 4, 2, 2, ka > 0);
      }
      tc::mma_commit(bar);
    }
    load_obs(tile + gridDim.x, xn);                  // next tile's rows, in flight across the MMA round trip
    mbar_wait(bar, it & 1u);
    tc::fence_after_sync();
    float2 p01 = make_float2(0.0f, 0.0f);            // even / odd features
    const float2 prescale2 = make_float2(TANH_PRESCALE, TANH_PRESCALE);
#pragma unroll
    for (int q = 0; q < FPT / 32; ++q) {
      float z[32];
      tc::tmem_ld32(tm_z + lane_base + f0 + 32 * q, z);
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const float4 b = lds4(sw + VS_B2 + f0 + 32 * q + 4 * g), w = lds4(sw + VS_W3 + f0 + 32 * q + 4 * g);
        p01 = __ffma2_rn(make_float2(w.x, w.y), tanh_prescaled2(__ffma2_rn(make_float2(z[4 * g], z[4 * g + 1]), prescale2, make_float2(b.x, b.y))), p01);
        p01 = __ffma2_rn(make_float2(w.z, w.w), tanh_prescaled2(__ffma2_rn(make_float2(z[4 * g + 2], z[4 * g + 3]), prescale2, make_float2(b.z, b.w))), p01);
      }
    }
    const float p0 = p01.x, p1 = p01.y;
    // the upper half hands its head partial over through a TMEM column of its own (already consumed) z range
    if (half == 1) { tc::tmem_st1(tm_z + lane_base + FPT, p0 + p1); tc::tmem_wait_st(); }
    tc::fence_before_sync();
    __syncthreads();                                  // head partials visible; the h1 tile is free again
    if (half == 0) {
      tc::fence_after_sync();
      const float other = tc::tmem_ld1(tm_z + lane_base + FPT);
      bool ok;
      const long long row = tile_row(tile, ok);
      if (ok) out[row] = ((p0 + p1) + other) + sw[VS_B3];
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tm_z, H);
}

// values of M observation rows with the critic of a (hidden 64 or 128, 2 layers) policy; `critic` points at the critic's
// first parameter inside the flat buffer
template <int H>
static int launch_values(const float* critic, int obs_dim, const float* obs, long long M, float* out, cudaStream_t s) {
  using Cfg = VtCfg<H>;
  static DeviceOnce attr;
  if (attr.first()) {
    AUR_CUDA_OK(cudaFuncSetAttribute(critic_values_tc_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
    AUR_CUDA_OK(cudaFuncSetAttribute(critic_values_tc_kernel<H>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr.done();
  }
  const long long ntiles = (M + VT_S - 1) / VT_S;
  long long grid = (long long)Cfg::CTAS * sm_count();
  if (grid > ntiles) grid = ntiles;
  critic_values_tc_kernel<H><<<(unsigned)grid, VT_THREADS, Cfg::SMEM, s>>>(critic, obs_dim, obs, M, out, 1, 0, 0);
  AUR_LAUNCH_OK("critic_values_tc_kernel");
  return 0;
}
int launch_critic_values_tc(const float* critic, int obs_dim, int hidden, const float* obs, long long M, float* out, cudaStream_t s) {
  if (M <= 0) return 0;
  return hidden == 128 ? launch_values<128>(critic, obs_dim, obs, M, out, s) : launch_values<64>(critic, obs_dim, obs, M, out, s);
}

// population values (aur_pop_rollout): M = segs * K * n_member rows, member k's critic at critic + k * P; about as many CTAs in
// all as the single-run pass
int launch_critic_values_tc_pop(const float* critic, int obs_dim, const float* obs, long long segs, int K, long long n_member,
                                long long P, float* out, cudaStream_t s) {
  using Cfg = VtCfg<64>;
  static DeviceOnce attr;
  if (attr.first()) {
    AUR_CUDA_OK(cudaFuncSetAttribute(critic_values_tc_kernel<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
    AUR_CUDA_OK(cudaFuncSetAttribute(critic_values_tc_kernel<64, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr.done();
  }
  const long long ntiles = segs * ((n_member + VT_S - 1) / VT_S);      // per member
  long long gx = ((long long)Cfg::CTAS * sm_count() + K - 1) / K;
  if (gx > ntiles) gx = ntiles;
  critic_values_tc_kernel<64, true><<<dim3((unsigned)gx, (unsigned)K), VT_THREADS, Cfg::SMEM, s>>>(
      critic, obs_dim, obs, segs * K * n_member, out, K, n_member, P);
  AUR_LAUNCH_OK("critic_values_tc_kernel (population)");
  return 0;
}

}  // namespace aur
