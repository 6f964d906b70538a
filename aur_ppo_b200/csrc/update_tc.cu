// Tensor-core implementation of the fused PPO minibatch update (row U, src/ppo.py:220-267).
//
// Every contraction over a 64-wide feature axis or over the samples of a tile runs on tcgen05 with fp32
// accumulation in TMEM:
//   forward        z2[s][j]  = sum_i h1[s][i] W2[j][i]
//   backward-data  dh1[s][i] = sum_j dz2[s][j] W2[j][i]
//   weight grad    dW2[j][i] = sum_s dz2[s][j] h1[s][i]
//   bias / input   db2[j] = sum_s dz2[s][j],  db1[j] = sum_s dz1[s][j],  dW1[j][c] = sum_s dz1[s][j] x[s][c]
// Operands are bf16 two-term splits (v = hi + mid, residual <= 2^-17 |v|) and three products are issued per
// contraction (hi*hi + hi*mid + mid*hi), so a product is exact to ~1e-5 relative: the reference's 1e-4 bar on
// losses and gradients holds (tests/test_update_gpu.py).
//
// The actor and the critic are independent MLPs with separable losses: a CTA trains ONE net (blockIdx picks
// it), two CTAs of 256 threads are resident per SM (one of each net when the grid is 2 x #SM), so one CTA's
// barrier / MMA waits are covered by the other's arithmetic.  A CTA walks tiles of 128 samples.  Thread =
// (sample s, feature half): two threads share a sample, each owning 32 of the 64 hidden features, and the
// per-sample state stays in registers.  TMEM lane s is sample s: every accumulator row comes back to the
// threads that own the sample (tcgen05.ld 32x32b, 32 columns per thread).  The operand rows are written by
// their owners straight into the 128-B-swizzled UMMA layout; the SAME tiles serve as K-major A operands
// (forward / backward-data) and as MN-major A/B operands of the contractions over samples, whose accumulators
// (dW2 64x64, [db2], [db1 | dW1]) live in TMEM for the whole kernel.  The bias and first-layer gradients use a
// 16-column K-major "aux" tile [1, x0..x3].  Only dW3 / db3 (out_dim <= 4 columns) stay SIMT, staged through
// shared memory warp by warp.
//
// Pipeline per tile t (two elected threads issue the MMA batches, mbarriers track them):
//   wait bwd/wgrad(t-1) | store dz1(t-1), h1(t) (+ fp32 copy in TMEM), aux(t) | issue fwd(t), aux_w1(t-1)
//   (h1(t) itself was computed at the end of iteration t-1, ahead of that wait)
//   gather(t+1) and index(t+2) loads | wait fwd(t) | h2, head, loss | wait aux_w1(t-1) | store dz2(t)
//   issue bwd(t), wgrad(t), aux_b2(t) | warp-local dW3 passes (overlap the MMAs)
#include "tc_split.cuh"
#include "update.cuh"

namespace aur {

constexpr int T2_S = 128;                   // samples per tile
constexpr int T2_LD = T2_S + 4;             // fp32 staging row stride
constexpr int T2_TILE = T2_S * 128;         // operand tile: 128 rows x 128 B
constexpr int T2_WTILE = 64 * 128;          // W2 tile: 64 rows x 128 B
constexpr int T2_AUXT = 2 * 8 * 128;        // aux tile: [sample block 2][n 8][64 samples] bf16, K-major
constexpr int T2_SW = 768;                  // small-weight floats
// shared memory map (bytes, from a 1024-aligned base)
constexpr int O2_H1 = 0;                                // [hi][mid]
constexpr int O2_DZ = O2_H1 + 2 * T2_TILE;              // [hi][mid]
constexpr int O2_W2 = O2_DZ + 2 * T2_TILE;              // [hi][mid]   (follows dz mid: see the M = 128 note below)
constexpr int O2_AUX = O2_W2 + 2 * T2_WTILE;            // [buffer 2][hi, mid]
constexpr int O2_SMALL = O2_AUX + 4 * T2_AUXT;          // fp32 small weights (also what the aux tiles' unused rows 8..15 over-read)
constexpr int T2_STAGE_BYTES = 16 * 8 * 36 * 4;         // 16 warp patches of [8][36] floats; also head exchange / epilogue scratch
constexpr int O2_STAGE = O2_SMALL + T2_SW * 4;
constexpr int O2_DOUT = O2_STAGE + T2_STAGE_BYTES;      // fp32 [4][T2_LD]: dout
constexpr int O2_BAR = O2_DOUT + 4 * T2_LD * 4;         // mbarriers + tmem slot
constexpr int T2_SMEM_USED = O2_BAR + 128;
constexpr size_t T2_SMEM = T2_SMEM_USED + 1024;
static_assert(2 * (T2_SMEM + 1024) <= 233472, "two CTAs per SM");

// small-weight block (floats): W1^T [4][64] (zero rows >= obs_dim), b1 [64], b2 [64], W3 [4][64], b3 [4]
constexpr int S2_W1T = 0, S2_B1 = 256, S2_B2 = 320, S2_W3 = 384, S2_B3 = 640, S2_NC = 644, S2_ST = 660;   // S2_NC: Normal constants [3][4], then advantage mean / std + 1e-8; S2_ST: statistics slots [4 warps][9]
constexpr int S2_PC = 700;                  // population form: the member's clip, clip_lo, clip_hi, ent_c, vf_c
enum { BAR_FWD = 0, BAR_AUX = 1, BAR_WG = 2, BAR_FIN = 3 };
constexpr int T2_TMEM_COLS = 256;           // z / dh 64 (never live together) | dW2 64 | db2 16 | [db1 dW1] 16 | h1 (fp32 copy) 64

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// d * (1 - h^2) for a pair of features: the gradient through tanh, h = tanh output (FFMA2 + FMUL2)
__device__ __forceinline__ float2 tanh_grad2(float2 d, float2 h) {
  return __fmul2_rn(d, __ffma2_rn(make_float2(-h.x, -h.y), h, make_float2(1.0f, 1.0f)));
}

struct T2Ptrs {
  unsigned char* base;
  __device__ __forceinline__ unsigned char* h1(int part) const { return base + O2_H1 + part * T2_TILE; }
  __device__ __forceinline__ unsigned char* dz(int part) const { return base + O2_DZ + part * T2_TILE; }
  __device__ __forceinline__ unsigned char* w2(int part) const { return base + O2_W2 + part * T2_WTILE; }
  __device__ __forceinline__ unsigned char* aux(int buf, int part) const { return base + O2_AUX + (buf * 2 + part) * T2_AUXT; }
  __device__ __forceinline__ float* small_w() const { return reinterpret_cast<float*>(base + O2_SMALL); }
  __device__ __forceinline__ float* stage() const { return reinterpret_cast<float*>(base + O2_STAGE); }
  __device__ __forceinline__ float* sdout() const { return reinterpret_cast<float*>(base + O2_DOUT); }
  __device__ __forceinline__ uint64_t* bar(int i) const { return reinterpret_cast<uint64_t*>(base + O2_BAR) + i; }
  __device__ __forceinline__ uint32_t* tmem_slot() const { return reinterpret_cast<uint32_t*>(base + O2_BAR + 96); }
};

// byte offset of element (n < 8, s) of an aux tile (K-major, 128-B swizzle): row n holds 64 samples of one block.
// The MMA reads N = 16 rows; rows 8..15 fall 1 KB further (the next block / tile / the small weights behind the aux
// region) and only reach accumulator columns 8..15, which nobody reads.
__device__ __forceinline__ int aux_off(int n, int s) {
  return (s >> 6) * 1024 + n * 128 + (((((s & 63) >> 3) ^ n)) << 4) + (s & 7) * 2;
}

// Contractions over the 128 samples of a tile (K = 8 steps of 16 rows) with only 64 output rows (features): the A
// descriptor's second 64-row atom is the MID tile (LBO = one tile), so one M = 128 MMA yields hi^T B in accumulator
// rows 0..63 and mid^T B in rows 64..127; two passes (B_hi, B_mid) give all four split products and the epilogue
// adds the two row blocks.  b_step / b_block: 16-B units per K step inside / across the 64-sample blocks of B.
// b_mid_pass = false skips the second pass (B's mid part is known to be zero where it matters: the ones column).
__device__ __forceinline__ void mma_over_samples(uint32_t d, uint64_t a_himid, uint64_t b_hi, uint64_t b_mid, uint32_t idesc,
                                                 uint32_t b_step, uint32_t b_block, bool accumulate, bool b_mid_pass = true) {
  for (int k = 0; k < 8; ++k)
    tc::mma_f16(d, a_himid + (uint64_t)(128 * k), b_hi + (uint64_t)((k & 3) * b_step + (k >> 2) * b_block), idesc,
                (accumulate || k > 0) ? 1u : 0u);
  if (!b_mid_pass) return;
  for (int k = 0; k < 8; ++k)
    tc::mma_f16(d, a_himid + (uint64_t)(128 * k), b_mid + (uint64_t)((k & 3) * b_step + (k >> 2) * b_block), idesc, 1u);
}

// TPS = threads per sample (2 or 4): each owns FPT = 64 / TPS hidden features of its sample.
// AOUT = act_dim (1 .. POL_OUT_MAX), the actor's head width; the critic's is 1.  A compile-time width leaves no dead head
// columns or width tests in the loops.  Adjacent features go through packed fp32x2 ops (FFMA2 / FADD2 / FMUL2) as float2
// pairs; every lane rounds as the scalar op it replaces, in the same order, so the results are those of scalar code.
// POP: member blockIdx.y of a population (ppo_grad_tc_kernel<TPS, true>): its parameters, index list, moments and partial rows
// are offset by pop's strides, its coefficients come from pop.hp and live in shared memory (S2_PC); the argument block itself is
// never modified, so it stays in the constant bank.
template <bool ACTOR, int TPS, bool POP, int AOUT>
__device__ __forceinline__ void tc_update_net(const UpdDev& a, const PopUpd& pop, unsigned char* smem_base, int cta, int ncta) {
  constexpr int THREADS = 128 * TPS, FPT = 64 / TPS, CPT = FPT / 8, FP2 = FPT / 2;
  T2Ptrs P;
  P.base = smem_base;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int s = tid & 127, half = tid >> 7, f0 = FPT * half;      // `half`: which feature slice of the sample (0 .. TPS-1)
  const int obs_dim = a.obs_dim;
  constexpr int A = AOUT, OUT = ACTOR ? A : 1;
  const int64_t gA = net_param_count(obs_dim, UPD_H, 2, A), gC = net_param_count(obs_dim, UPD_H, 2, 1);

  // ---- one-time setup: barriers, TMEM, weights, aux tiles
  if (tid == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(P.bar(i), 1);
    mbar_fence_init();
  }
  if (warp == 0) tc::tmem_alloc(P.tmem_slot(), T2_TMEM_COLS);
  float* sw = P.small_w();
  {
    const float* g = (POP ? a.params + blockIdx.y * pop.P : a.params) + (ACTOR ? 0 : gA);
    const float* gb1 = g + 64 * obs_dim;
    const float* gW2 = gb1 + 64;
    const float* gb2 = gW2 + 4096;
    const float* gW3 = gb2 + 64;
    const float* gb3 = gW3 + OUT * 64;
    if (tid < 256) {
      const int c = tid >> 6, j = tid & 63;
      sw[S2_W1T + tid] = c < obs_dim ? TANH_PRESCALE * g[j * obs_dim + c] : 0.0f;     // tanh argument scale folded in
      sw[S2_W3 + tid] = tid < OUT * 64 ? gW3[tid] : 0.0f;
    }
    if (tid < 64) { sw[S2_B1 + tid] = TANH_PRESCALE * gb1[tid]; sw[S2_B2 + tid] = TANH_PRESCALE * gb2[tid]; }
    if (tid < 4) sw[S2_B3 + tid] = tid < OUT ? gb3[tid] : 0.0f;
    {                                                  // W2 row j, 512 / THREADS chunks per thread (block only 4-byte aligned)
      constexpr int CW = 512 / THREADS;
      const int j = tid & 63, cq = tid >> 6;
#pragma unroll 1
      for (int c = CW * cq; c < CW * cq + CW; ++c) {
        float2 v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = make_float2(gW2[j * 64 + 8 * c + 2 * e], gW2[j * 64 + 8 * c + 2 * e + 1]);
        store_split_chunk(P.w2(0), P.w2(1), j, c, v);
      }
    }
  }
  {                                                    // aux tiles + pad: zero, then the row of ones (n = 0)
    uint4* ax = reinterpret_cast<uint4*>(P.aux(0, 0));
    for (int e = tid; e < (4 * T2_AUXT) / 16; e += THREADS) ax[e] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();
  if (tid < 256) *reinterpret_cast<unsigned short*>(P.aux(tid >> 7, 0) + aux_off(0, tid & 127)) = 0x3F80;

  if (ACTOR && a.continuous && tid == 0) {
    const NormalConsts nc = normal_consts((POP ? a.params + blockIdx.y * pop.P : a.params) + gA + gC, A);
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) { sw[S2_NC + k] = nc.std[k]; sw[S2_NC + 4 + k] = nc.inv2var[k]; sw[S2_NC + 8 + k] = nc.log_scale[k]; }
  }
  if constexpr (POP) {
    if (ACTOR && a.norm_adv && tid == 32) {
      const double* mom = a.moments + blockIdx.y * pop.mom_stride;
      adv_norm_from_moments(mom[0], mom[1], mom[2], sw[S2_NC + 12], sw[S2_NC + 13]);
    }
    if (tid == 64) {                                   // exactly as aur_ppo_update_grad derives them from its float arguments
      const aur_pop_hparams& h = pop.hp[blockIdx.y];
      const float clip = (float)h.clip_coeff;
      sw[S2_PC] = clip; sw[S2_PC + 1] = (float)(1.0 - (double)clip); sw[S2_PC + 2] = (float)(1.0 + (double)clip);
      sw[S2_PC + 3] = (float)h.entropy_coeff; sw[S2_PC + 4] = (float)h.value_coeff;
    }
  } else {
    if (ACTOR && a.norm_adv && tid == 32) adv_norm_consts(a, sw[S2_NC + 12], sw[S2_NC + 13]);   // (waits for the peers' moments when data-parallel)
  }
  tc::fence_proxy_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *P.tmem_slot();
  const float adv_mean = (ACTOR && a.norm_adv) ? sw[S2_NC + 12] : 0.0f, adv_den = (ACTOR && a.norm_adv) ? sw[S2_NC + 13] : 1.0f;
  const uint32_t tm_z = tmem, tm_dh = tmem, tm_w = tmem + 64, tm_b2 = tmem + 128, tm_w1 = tmem + 144, tm_h1 = tmem + 160;
  const uint32_t lane_base = (uint32_t)(32 * (warp & 3)) << 16;

  constexpr uint32_t ID_FWD = tc::instr_desc(tc::FMT_BF16, 128, 64, 0, 0);
  constexpr uint32_t ID_BWD = tc::instr_desc(tc::FMT_BF16, 128, 64, 0, 1);
  constexpr uint32_t ID_WG = tc::instr_desc(tc::FMT_BF16, 128, 64, 1, 1);
  constexpr uint32_t ID_AUX = tc::instr_desc(tc::FMT_BF16, 128, 16, 1, 0);

  float* stg = P.stage();
  float* sdo = P.sdout();

  // accumulators that stay in registers for the whole kernel
  float acc_w3[CPT][POL_OUT_MAX];      // dW3[k][f0 + 8 p + (lane & 7)] over samples 8 (lane >> 3) .. + 7 of this warp
#pragma unroll
  for (int r = 0; r < CPT; ++r)
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) acc_w3[r][k] = 0.0f;
  float acc_b3 = 0.0f;
  constexpr int NST = ACTOR ? 9 : 1;   // actor: policy loss, entropy, old kl, kl, clipfrac, d logstd[4]; critic: value loss
  // statistics: per-thread registers (TPS 2) or, to stay inside 64 registers (TPS 4), one smem slot per loss warp that its
  // lane 0 owns (warp sums added tile by tile: still a fixed order)
  constexpr bool ST_REGS = TPS == 2;
  float st[ST_REGS ? NST : 1];
#pragma unroll
  for (int i = 0; i < (ST_REGS ? NST : 1); ++i) st[i] = 0.0f;
  float* sst = sw + S2_ST + (warp & 3) * 9;
  if (!ST_REGS && tid < 36) sw[S2_ST + tid] = 0.0f;
  auto stat_add = [&](int i, float v) {
    if (ST_REGS) st[ST_REGS ? i : 0] += v;
    else { const float w = warp_sum(v); if ((tid & 31) == 0) sst[i] += w; }
  };

  const long long ntiles = (a.m_local + T2_S - 1) / T2_S;
  const bool any = (long long)cta < ntiles;
  const bool obs_vec = obs_dim == 4 && (reinterpret_cast<uintptr_t>(a.obs) & 15) == 0;
  // gather pipeline: row index two tiles ahead, observation one tile ahead (row < 0: no sample)
  // (kept as the raw 32-bit load result; widened one iteration later, so nothing waits on the load here)
  auto fetch_row = [&](long long tile) -> int {
    const long long gi = tile * T2_S + s;
    if (tile >= ntiles || gi >= a.m_local) return -1;
    if constexpr (POP) return __ldg(a.idx + blockIdx.y * pop.idx_stride + gi);
    return a.idx ? __ldg(a.idx + gi) : (int)gi;
  };
  const long long row_off = (POP || a.idx) ? 0 : a.idx_offset;
  // the member's coefficients (POP: from shared memory), else the argument block's
  auto c_clip = [&]() -> float { if constexpr (POP) return sw[S2_PC]; else return a.clip; };
  auto c_clip_lo = [&]() -> float { if constexpr (POP) return sw[S2_PC + 1]; else return a.clip_lo; };
  auto c_clip_hi = [&]() -> float { if constexpr (POP) return sw[S2_PC + 2]; else return a.clip_hi; };
  auto c_ent = [&]() -> float { if constexpr (POP) return sw[S2_PC + 3]; else return a.ent_c; };
  auto c_vf = [&]() -> float { if constexpr (POP) return sw[S2_PC + 4]; else return a.vf_c; };
  float xn[POL_IN_PAD];
  const float4* rec = ACTOR ? a.rec_actor : a.rec_critic;      // packed records: one 32-B sector per sample
  auto fetch_obs = [&](long long row) {
    if (row >= 0 && rec) {
      const float4 v = __ldg(rec + 2 * row);
      xn[0] = v.x; xn[1] = v.y; xn[2] = v.z; xn[3] = v.w;
      return;
    }
    if (row >= 0 && obs_vec) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(a.obs) + row);
      xn[0] = v.x; xn[1] = v.y; xn[2] = v.z; xn[3] = v.w;
    } else {
#pragma unroll
      for (int c = 0; c < POL_IN_PAD; ++c) xn[c] = (row >= 0 && c < obs_dim) ? __ldg(a.obs + row * obs_dim + c) : 0.0f;
    }
    if (row >= 0 && half == 0) {
      if (ACTOR) { prefetch_l2(a.logprobs + row); prefetch_l2(a.advantages + row); prefetch_l2(a.actions + row * (a.continuous ? A : 1)); }
      else { prefetch_l2(a.returns + row); prefetch_l2(a.values + row); }
    }
  };
  int rownn = fetch_row((long long)cta + ncta);
  long long rown;
  { const int r0 = fetch_row(cta); rown = r0 < 0 ? -1 : row_off + r0; }
  fetch_obs(rown);

  // first layer of one tile: this thread's FPT features from the prefetched observation
  auto first_layer = [&](float2 (&hv)[FP2]) {
#pragma unroll
    for (int g = 0; g < FPT / 4; ++g) {
      const int f = f0 + 4 * g;
      const float4 b = lds4(sw + S2_B1 + f);
      float2 a01 = make_float2(b.x, b.y), a23 = make_float2(b.z, b.w);
#pragma unroll
      for (int cc = 0; cc < POL_IN_PAD; ++cc) {
        const float4 w = lds4(sw + S2_W1T + cc * 64 + f);
        const float2 xx = make_float2(xn[cc], xn[cc]);
        a01 = __ffma2_rn(make_float2(w.x, w.y), xx, a01);
        a23 = __ffma2_rn(make_float2(w.z, w.w), xx, a23);
      }
      hv[2 * g] = tanh_prescaled2(a01);
      hv[2 * g + 1] = tanh_prescaled2(a23);
    }
  };
  // TPS 2 computes the next tile's first layer ahead of the MMA wait and carries it across the loop edge; TPS 4 has
  // no registers for that (and twice the warps to cover the wait): it computes it right before storing
  constexpr bool H1_AHEAD = TPS == 2;
  float2 h1n[FP2];
  if (H1_AHEAD) first_layer(h1n);

  uint32_t it = 0;
#pragma unroll 1
  for (long long tile = cta; tile < ntiles; tile += ncta, ++it) {
    const uint32_t ph = it & 1u;
    float x[POL_IN_PAD];
#pragma unroll
    for (int c = 0; c < POL_IN_PAD; ++c) x[c] = xn[c];
    const long long row = rown;
    const bool valid = row >= 0;
    // ---- backward of the previous tile (dz1 = dh1 * (1 - h1^2), h1 kept as an fp32 copy in TMEM) in 8-feature
    // chunks straight into the operand tile, then this tile's first layer (computed an iteration ago, ahead of this
    // wait).  bwd + wgrad + aux_b2 of t-1 have retired once BAR_WG flips: dh is ready, the dz / h1 tiles are free.
    if (it > 0) {
      mbar_wait(P.bar(BAR_WG), ph ^ 1u);
      tc::fence_after_sync();
#pragma unroll
      for (int c = 0; c < CPT; ++c) {
        const uint32_t col = lane_base + (uint32_t)(f0 + 8 * c);
        float2 d[4], hp[4];
        tc::tmem_ld8_nowait(tm_dh + col, d);
        tc::tmem_ld8_nowait(tm_h1 + col, hp);
        tc::tmem_wait_ld();
#pragma unroll
        for (int e = 0; e < 4; ++e) d[e] = tanh_grad2(d[e], hp[e]);
        store_split_chunk(P.dz(0), P.dz(1), s, CPT * half + c, d);
      }
    }
    if (!H1_AHEAD) first_layer(h1n);
#pragma unroll
    for (int c = 0; c < CPT; ++c) {
      store_split_chunk(P.h1(0), P.h1(1), s, CPT * half + c, h1n + 4 * c);
      tc::tmem_st8(tm_h1 + lane_base + (uint32_t)(f0 + 8 * c), h1n + 4 * c);
    }
    tc::tmem_wait_st();
    {
      // aux(t): x columns, 4 / TPS per thread of the sample group
      unsigned char* ah = P.aux(ph, 0);
      unsigned char* am = P.aux(ph, 1);
      constexpr int XC = 4 / TPS;
#pragma unroll
      for (int cc = 0; cc < XC; ++cc) {
        const int c = XC * half + cc;
        float xv = x[0];
#pragma unroll
        for (int q = 1; q < POL_IN_PAD; ++q) xv = c == q ? x[q] : xv;
        const __nv_bfloat16 hb = __float2bfloat16_rn(xv);
        const __nv_bfloat16 mb = __float2bfloat16_rn(xv - __bfloat162float(hb));
        const int off = aux_off(1 + c, s);
        *reinterpret_cast<unsigned short*>(ah + off) = __bfloat16_as_ushort(hb);
        *reinterpret_cast<unsigned short*>(am + off) = __bfloat16_as_ushort(mb);
      }
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    if (tid == 128) {                                  // a thread that idles through the loss issues this batch
      tc::fence_after_sync();
      mma_split(tm_z, tc::smem_desc_k_sw128(P.h1(0)), tc::smem_desc_k_sw128(P.h1(1)), tc::smem_desc_k_sw128(P.w2(0)),
                tc::smem_desc_k_sw128(P.w2(1)), ID_FWD, 4, 2, 2, false);
      tc::mma_commit(P.bar(BAR_FWD));
      if (it > 0)
        mma_over_samples(tm_w1, tc::smem_desc_mn_sw128(P.dz(0), T2_TILE, 1024), tc::smem_desc_k_sw128(P.aux(ph ^ 1u, 0)),
                         tc::smem_desc_k_sw128(P.aux(ph ^ 1u, 1)), ID_AUX, 2, 64, it > 1);
      tc::mma_commit(P.bar(BAR_AUX));
    }
    // ---- gather: observation of tile t+1 (its row index arrived an iteration ago), row index of tile t+2
    rown = rownn < 0 ? -1 : row_off + rownn;
    rownn = fetch_row(tile + 2LL * ncta);
    fetch_obs(rown);
    // per-sample scalars of this tile (L2 hits: prefetched one tile ago), in flight across the second layer
    float e0 = 0.0f, e1 = 0.0f, e2 = 0.0f, e3 = 0.0f;
    if (half == 0 && valid) {
      if (rec) {                                       // second half of the record: same sector as the observation
        const float4 v = __ldg(rec + 2 * row + 1);
        if (ACTOR) { e2 = v.x; e0 = v.y; e1 = v.z; e3 = v.w; }
        else { e0 = v.x; e1 = v.y; }
      } else if (ACTOR) {
        e0 = __ldg(a.logprobs + row); e1 = __ldg(a.advantages + row);
        e2 = __ldg(a.actions + row * (a.continuous ? A : 1));
      } else {
        e0 = __ldg(a.returns + row); e1 = __ldg(a.values + row);
      }
    }
    // ---- second layer, head, loss
    mbar_wait(P.bar(BAR_FWD), ph);
    tc::fence_after_sync();
    float2 h2[FP2];
#pragma unroll
    for (int c = 0; c < CPT; ++c) tc::tmem_ld8_nowait(tm_z + lane_base + (uint32_t)(f0 + 8 * c), h2 + 4 * c);
    tc::tmem_wait_ld();                                // one round trip for all CPT chunks (their registers are h2 anyway)
    const float2 prescale2 = make_float2(TANH_PRESCALE, TANH_PRESCALE);
#pragma unroll
    for (int g = 0; g < FPT / 4; ++g) {
      const float4 b = lds4(sw + S2_B2 + f0 + 4 * g);
      h2[2 * g] = tanh_prescaled2(__ffma2_rn(h2[2 * g], prescale2, make_float2(b.x, b.y)));
      h2[2 * g + 1] = tanh_prescaled2(__ffma2_rn(h2[2 * g + 1], prescale2, make_float2(b.z, b.w)));
    }
    float outp[POL_OUT_MAX];             // this half's share of the head pre-activations
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) {
      outp[k] = 0.0f;
      if (k < OUT) {
        float2 p01 = make_float2(0.0f, 0.0f);        // even / odd features
#pragma unroll
        for (int g = 0; g < FPT / 4; ++g) {
          const float4 w = lds4(sw + S2_W3 + k * 64 + f0 + 4 * g);
          p01 = __ffma2_rn(make_float2(w.x, w.y), h2[2 * g], p01);
          p01 = __ffma2_rn(make_float2(w.z, w.w), h2[2 * g + 1], p01);
        }
        outp[k] = p01.x + p01.y;
        if (half > 0) stg[((half - 1) * POL_OUT_MAX + k) * T2_LD + s] = outp[k];     // head exchange: [slice - 1][k][sample]
      }
    }
    if (TPS == 4) {                                    // park h2 in its (consumed) z columns across the loss: registers
#pragma unroll
      for (int c = 0; c < CPT; ++c) tc::tmem_st8(tm_z + lane_base + (uint32_t)(f0 + 8 * c), h2 + 4 * c);
      tc::tmem_wait_st();
    }
    __syncthreads();
    if (half == 0) {
      float out[POL_OUT_MAX], dout[POL_OUT_MAX];
      float sv[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};     // this sample's statistic terms
#pragma unroll
      for (int k = 0; k < POL_OUT_MAX; ++k) {
        float o = outp[k];
#pragma unroll
        for (int q = 1; q < TPS; ++q) o += stg[((q - 1) * POL_OUT_MAX + k) * T2_LD + s];
        out[k] = k < OUT ? o + sw[S2_B3 + k] : 0.0f;
        dout[k] = 0.0f;
      }
      if (valid) {
        if (ACTOR) {
          const float oldlp = e0, adv = e1;
          float newlogp, entropy, dlp[POL_OUT_MAX], dH[POL_OUT_MAX];
          float g_ls[POL_OUT_MAX] = {0.f, 0.f, 0.f, 0.f};
          if (!a.continuous) {
            float m = out[0];
#pragma unroll
            for (int k = 1; k < POL_OUT_MAX; ++k) if (k < OUT) m = fmaxf(m, out[k]);
            float se = 0.0f;
#pragma unroll
            for (int k = 0; k < POL_OUT_MAX; ++k) if (k < OUT) se += expf(out[k] - m);
            const float lse = m + logf(se);
            const int act = (int)e2;
            float lp[POL_OUT_MAX], pr[POL_OUT_MAX];
            entropy = 0.0f; newlogp = 0.0f;
#pragma unroll
            for (int k = 0; k < POL_OUT_MAX; ++k) {
              lp[k] = out[k] - lse;
              pr[k] = k < OUT ? expf(lp[k]) : 0.0f;
              if (k < OUT) entropy -= pr[k] * lp[k];
              if (k == act) newlogp = lp[k];
            }
#pragma unroll
            for (int k = 0; k < POL_OUT_MAX; ++k) {
              dlp[k] = (k == act ? 1.0f : 0.0f) - pr[k];
              dH[k] = k < OUT ? -pr[k] * (lp[k] + entropy) : 0.0f;
            }
          } else {
            NormalConsts nc;
#pragma unroll
            for (int k = 0; k < POL_OUT_MAX; ++k) { nc.std[k] = sw[S2_NC + k]; nc.inv2var[k] = sw[S2_NC + 4 + k]; nc.log_scale[k] = sw[S2_NC + 8 + k]; }
            float act[POL_OUT_MAX];
            act[0] = e2;
#pragma unroll
            for (int k = 1; k < POL_OUT_MAX; ++k) act[k] = k < OUT ? (rec ? (k == 1 ? e3 : 0.0f) : __ldg(a.actions + row * OUT + k)) : 0.0f;
            normal_logp(out, act, OUT, nc, newlogp, entropy);
#pragma unroll
            for (int k = 0; k < POL_OUT_MAX; ++k) {
              const float d = act[k] - out[k], var = nc.std[k] * nc.std[k];
              dlp[k] = k < OUT ? d / var : 0.0f;
              dH[k] = 0.0f;
              g_ls[k] = k < OUT ? d * d / var - 1.0f : 0.0f;
            }
          }
          const float logr = newlogp - oldlp, ratio = expf(logr);
          const float advn = a.norm_adv ? (adv - adv_mean) / adv_den : adv;
          const float l1 = -advn * ratio, l2 = -advn * fminf(fmaxf(ratio, c_clip_lo()), c_clip_hi());
          const float w1 = l1 > l2 ? 1.0f : (l1 == l2 ? 0.5f : 0.0f);
          const float inr = (ratio >= c_clip_lo() && ratio <= c_clip_hi()) ? 1.0f : 0.0f;
          const float g_logp = -advn * (w1 + (1.0f - w1) * inr) * ratio * a.inv_m;
          const float g_H = -c_ent() * a.inv_m;
#pragma unroll
          for (int k = 0; k < POL_OUT_MAX; ++k) dout[k] = g_logp * dlp[k] + g_H * dH[k];
          if (a.continuous) {
#pragma unroll
            for (int k = 0; k < POL_OUT_MAX; ++k) if (k < OUT) sv[5 + k] = g_logp * g_ls[k] + g_H;
          }
          sv[0] = fmaxf(l1, l2); sv[1] = entropy; sv[2] = -logr; sv[3] = (ratio - 1.0f) - logr;
          sv[4] = fabsf(ratio - 1.0f) > c_clip() ? 1.0f : 0.0f;
        } else {
          const float R = e0, vold = e1, v = out[0];
          if (a.clip_vloss) {
            const float du = v - R, vu = du * du;
            const float d = v - vold, vc = vold + fminf(fmaxf(d, -c_clip()), c_clip());
            const float dc = vc - R, lc = dc * dc;
            const float w1 = vu > lc ? 1.0f : (vu == lc ? 0.5f : 0.0f);
            const float inr = (d >= -c_clip() && d <= c_clip()) ? 1.0f : 0.0f;
            dout[0] = (w1 * du + (1.0f - w1) * dc * inr) * c_vf() * a.inv_m;
            sv[0] = 0.5f * fmaxf(vu, lc);
          } else {
            const float d = v - vold;
            dout[0] = d * c_vf() * a.inv_m;
            sv[0] = 0.5f * d * d;
          }
        }
      }
#pragma unroll
      for (int k = 0; k < POL_OUT_MAX; ++k) sdo[k * T2_LD + s] = dout[k];
#pragma unroll
      for (int i = 0; i < NST; ++i) {
        if (ACTOR && i >= 5 && !a.continuous) break;
        stat_add(i, sv[i]);
      }
    }
    __syncthreads();
    if (TPS == 4) {
#pragma unroll
      for (int c = 0; c < CPT; ++c) tc::tmem_ld8_nowait(tm_z + lane_base + (uint32_t)(f0 + 8 * c), h2 + 4 * c);
      tc::tmem_wait_ld();
    }
    float dout[POL_OUT_MAX];
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) dout[k] = sdo[k * T2_LD + s];
    // ---- dz2 = (W3^T dout) * (1 - h2^2): operand rows of the backward MMAs (the dz tiles are free once aux_w1(t-1) retired)
    mbar_wait(P.bar(BAR_AUX), ph);
#pragma unroll
    for (int c = 0; c < CPT; ++c) {
      float2 dz2[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) dz2[e] = make_float2(0.0f, 0.0f);
#pragma unroll
      for (int k = 0; k < OUT; ++k) {
        const float4 wa = lds4(sw + S2_W3 + k * 64 + f0 + 8 * c), wb = lds4(sw + S2_W3 + k * 64 + f0 + 8 * c + 4);
        const float2 dk = make_float2(dout[k], dout[k]);
        dz2[0] = __ffma2_rn(make_float2(wa.x, wa.y), dk, dz2[0]); dz2[1] = __ffma2_rn(make_float2(wa.z, wa.w), dk, dz2[1]);
        dz2[2] = __ffma2_rn(make_float2(wb.x, wb.y), dk, dz2[2]); dz2[3] = __ffma2_rn(make_float2(wb.z, wb.w), dk, dz2[3]);
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) dz2[e] = tanh_grad2(dz2[e], h2[4 * c + e]);
      store_split_chunk(P.dz(0), P.dz(1), s, CPT * half + c, dz2);
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    if (tid == 160) {
      tc::fence_after_sync();
      mma_split(tm_dh, tc::smem_desc_k_sw128(P.dz(0)), tc::smem_desc_k_sw128(P.dz(1)), tc::smem_desc_mn_sw128(P.w2(0), 8192, 1024),
                tc::smem_desc_mn_sw128(P.w2(1), 8192, 1024), ID_BWD, 4, 2, 128, false);
      // D_w[j][i] (+)= sum_s dz2[s][j] h1[s][i], K = 128 samples = 8 steps of 16 rows
      mma_over_samples(tm_w, tc::smem_desc_mn_sw128(P.dz(0), T2_TILE, 1024), tc::smem_desc_mn_sw128(P.h1(0), T2_TILE, 1024),
                       tc::smem_desc_mn_sw128(P.h1(1), T2_TILE, 1024), ID_WG, 128, 512, it > 0);
      // db2 only needs the ones column of the aux tile, whose mid part is zero: one pass
      mma_over_samples(tm_b2, tc::smem_desc_mn_sw128(P.dz(0), T2_TILE, 1024), tc::smem_desc_k_sw128(P.aux(ph, 0)),
                       tc::smem_desc_k_sw128(P.aux(ph, 1)), ID_AUX, 2, 64, it > 0, false);
      tc::mma_commit(P.bar(BAR_WG));
    }
    // ---- dW3[k][j] += sum_s dout[s][k] h2[s][j], db3[k] += sum_s dout[s][k], warp-local (overlaps the MMAs):
    // a warp transposes its 32 samples x 8 features through a private smem patch ([8][36] floats, conflict-free
    // both ways), lane = (feature jj, sample octet qd) then sums 8 samples; 4 passes, no CTA barrier.
    {
      // TPS 2: two patches per warp, the stores of pass p+1 are issued before the loads of pass p (one __syncwarp per
      // pass instead of a store -> sync -> load -> sync chain); TPS 4 has room for one patch per warp
      constexpr int NPATCH = TPS == 2 ? 2 : 1;
      float* patch0 = stg + warp * (NPATCH * 8 * 36);
      const int lane = tid & 31, jj = lane & 7, qd = lane >> 3;
      const float* dbase = sdo + 32 * (warp & 3) + 8 * qd;
      auto put = [&](int p) {
        float* patch = patch0 + (p % NPATCH) * (8 * 36);
#pragma unroll
        for (int j = 0; j < 4; ++j) { patch[2 * j * 36 + lane] = h2[4 * p + j].x; patch[(2 * j + 1) * 36 + lane] = h2[4 * p + j].y; }
      };
      // this octet's dout, loaded once for all passes (TPS 2; TPS 4 has no registers to spare and reloads it per pass)
      constexpr int KD = TPS == 2 ? OUT : 1;
      float4 dva[KD], dvb[KD];
#pragma unroll
      for (int k = 0; k < KD; ++k) { dva[k] = lds4(dbase + k * T2_LD); dvb[k] = lds4(dbase + k * T2_LD + 4); }
      put(0);
      __syncwarp();
#pragma unroll
      for (int p = 0; p < CPT; ++p) {
        if (NPATCH == 2 && p + 1 < CPT) put(p + 1);
        const float* patch = patch0 + (p % NPATCH) * (8 * 36);
        const float4 ha = lds4(patch + jj * 36 + 8 * qd), hb = lds4(patch + jj * 36 + 8 * qd + 4);
#pragma unroll
        for (int k = 0; k < POL_OUT_MAX; ++k) {
          if (k < OUT) {
            const float4 da = TPS == 2 ? dva[k < KD ? k : 0] : lds4(dbase + k * T2_LD), db = TPS == 2 ? dvb[k < KD ? k : 0] : lds4(dbase + k * T2_LD + 4);
            float2 s01 = __fmul2_rn(make_float2(ha.x, ha.y), make_float2(da.x, da.y));      // even / odd samples
            s01 = __ffma2_rn(make_float2(ha.z, ha.w), make_float2(da.z, da.w), s01);
            s01 = __ffma2_rn(make_float2(hb.x, hb.y), make_float2(db.x, db.y), s01);
            s01 = __ffma2_rn(make_float2(hb.z, hb.w), make_float2(db.z, db.w), s01);
            acc_w3[p][k] += s01.x + s01.y;
            if (p == 0 && half == 0 && jj == k) acc_b3 += ((da.x + da.y) + (da.z + da.w)) + ((db.x + db.y) + (db.z + db.w));
          }
        }
        __syncwarp();
        if (NPATCH == 1 && p + 1 < CPT) { put(p + 1); __syncwarp(); }
      }
    }
    // ---- first layer of the next tile (its observation was requested right after this tile's forward MMAs)
    if (H1_AHEAD) first_layer(h1n);
  }

  // ---- tail: first-layer gradients of the last tile
  if (any) {
    const uint32_t ph = (it - 1u) & 1u;
    mbar_wait(P.bar(BAR_WG), ph);
    tc::fence_after_sync();
#pragma unroll
    for (int c = 0; c < CPT; ++c) {
      const uint32_t col = lane_base + (uint32_t)(f0 + 8 * c);
      float2 d[4], hp[4];
      tc::tmem_ld8_nowait(tm_dh + col, d);
      tc::tmem_ld8_nowait(tm_h1 + col, hp);
      tc::tmem_wait_ld();
#pragma unroll
      for (int e = 0; e < 4; ++e) d[e] = tanh_grad2(d[e], hp[e]);
      store_split_chunk(P.dz(0), P.dz(1), s, CPT * half + c, d);
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    if (tid == 128) {
      tc::fence_after_sync();
      mma_over_samples(tm_w1, tc::smem_desc_mn_sw128(P.dz(0), T2_TILE, 1024), tc::smem_desc_k_sw128(P.aux(ph, 0)),
                       tc::smem_desc_k_sw128(P.aux(ph, 1)), ID_AUX, 2, 64, it > 1);
      tc::mma_commit(P.bar(BAR_FIN));
    }
    mbar_wait(P.bar(BAR_FIN), 0);
    tc::fence_after_sync();
  }
  __syncthreads();

  // ---- epilogue: this CTA's partial sums in the net's flat parameter order
  float* part = (POP ? a.partials + blockIdx.y * pop.part_stride : a.partials) + ((size_t)(ACTOR ? 0 : 1) * ncta + cta) * UPD_PSTRIDE;
  const int oB1 = 64 * obs_dim, oW2 = oB1 + 64, oB2 = oW2 + 4096, oW3 = oB2 + 64, oB3 = oW3 + OUT * 64, oLS = oB3 + OUT;
  {
    // TMEM accumulators: rows 0..63 (hi^T B) + rows 64..127 (mid^T B) = feature j; thread (row, slice) reads FPT columns
    float v[FPT];
    uint32_t u[16];
#pragma unroll
    for (int i = 0; i < FPT; ++i) v[i] = 0.0f;
#pragma unroll
    for (int i = 0; i < 16; ++i) u[i] = 0u;
    if (any) {
#pragma unroll
      for (int c = 0; c < CPT; ++c) {
        float vc[8];
        tc::tmem_ld8_nowait(tm_w + lane_base + (uint32_t)(f0 + 8 * c), vc);
        tc::tmem_wait_ld();
#pragma unroll
        for (int e = 0; e < 8; ++e) v[8 * c + e] = vc[e];
      }
      if (half < 2) tc::tmem_ld16((half == 0 ? tm_b2 : tm_w1) + lane_base, u);
    }
    if (s >= 64) {
#pragma unroll
      for (int i = 0; i < FPT; ++i) stg[(s - 64) * 65 + f0 + i] = v[i];
      if (half == 0) sdo[s - 64] = __uint_as_float(u[0]);
      else if (half == 1) {
#pragma unroll
        for (int c = 0; c < 5; ++c) sdo[64 + (s - 64) * 5 + c] = __uint_as_float(u[c]);
      }
    }
    __syncthreads();
    if (s < 64) {
      const int j = s;
#pragma unroll
      for (int i = 0; i < FPT; ++i) part[oW2 + j * 64 + f0 + i] = v[i] + stg[j * 65 + f0 + i];
      if (half == 0) part[oB2 + j] = __uint_as_float(u[0]) + sdo[j];
      else if (half == 1) {
        part[oB1 + j] = __uint_as_float(u[0]) + sdo[64 + j * 5];
#pragma unroll
        for (int c = 0; c < POL_IN_PAD; ++c)
          if (c < obs_dim) part[j * obs_dim + c] = __uint_as_float(u[1 + c]) + sdo[64 + j * 5 + 1 + c];
      }
    }
    __syncthreads();
  }
  {
    // SIMT accumulators: dW3 / db3 summed over the 8 sample slices, statistics over the warps of half 0
    float* red = stg;   // dW3 [feature octet (f0 / 8 + p)][k][warp & 3][qd][jj] (4096), db3 [k][warp & 3][qd] (64), stats [9][4]
    const int lane = tid & 31, jj = lane & 7, qd = lane >> 3, wq = warp & 3;
#pragma unroll
    for (int p = 0; p < CPT; ++p)
#pragma unroll
      for (int k = 0; k < POL_OUT_MAX; ++k) red[((((half * CPT + p) * 4 + k) * 4 + wq) * 4 + qd) * 8 + jj] = acc_w3[p][k];
    if (half == 0 && jj < POL_OUT_MAX) red[4096 + (jj * 4 + wq) * 4 + qd] = acc_b3;
    if (half == 0) {
#pragma unroll
      for (int i = 0; i < NST; ++i) {
        if (ST_REGS) {
          const float v = warp_sum(st[ST_REGS ? i : 0]);
          if (lane == 0) red[4160 + i * 4 + wq] = v;
        } else if (lane == 0) {
          red[4160 + i * 4 + wq] = sst[i];
        }
      }
    }
    __syncthreads();
    if (tid < 256) {
      const int f = tid & 63, k = tid >> 6;
      if (k < OUT) {
        const float* q = red + (((f >> 3) * 4 + k) * 16) * 8 + (f & 7);
        float sum = 0.0f;
#pragma unroll
        for (int c = 0; c < 16; ++c) sum += q[c * 8];
        part[oW3 + k * 64 + f] = sum;
      }
      if (tid < OUT) {
        float sum = 0.0f;
#pragma unroll
        for (int c = 0; c < 16; ++c) sum += red[4096 + tid * 16 + c];
        part[oB3 + tid] = sum;
      }
      if (tid < NST) {
        const float* q = red + 4160 + tid * 4;
        const float sum = (q[0] + q[1]) + (q[2] + q[3]);
        float* stat = part + UPD_STAT_OFF;
        if (ACTOR) {
          if (tid == 0) stat[AUR_STAT_POLICY_LOSS] = sum;
          if (tid == 1) stat[AUR_STAT_ENTROPY] = sum;
          if (tid == 2) stat[AUR_STAT_OLD_APPROX_KL] = sum;
          if (tid == 3) stat[AUR_STAT_APPROX_KL] = sum;
          if (tid == 4) stat[AUR_STAT_CLIPFRAC] = sum;
          if (tid >= 5 && a.continuous && tid - 5 < OUT) part[oLS + tid - 5] = sum;
        } else {
          stat[AUR_STAT_VALUE_LOSS] = sum;
        }
      }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, T2_TMEM_COLS);
}

// POP: population form (aur_pop_update_grad), grid (2 c, K): member k = blockIdx.y trains with its own parameters, index
// list, advantage moments, coefficients and partial rows; an inactive member (target_kl) does nothing.
template <int TPS, bool POP, int AOUT>
__global__ void __launch_bounds__(128 * TPS, 2) ppo_grad_tc_kernel(UpdDev a, PopUpd pop) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
  const int ncta = gridDim.x >> 1;                     // CTAs per net; blockIdx < ncta: actor, else critic
  if constexpr (POP) {
    if (!pop.active[blockIdx.y]) return;               // the whole CTA: a member stopped by its target_kl
  }
  if ((int)blockIdx.x < ncta) tc_update_net<true, TPS, POP, AOUT>(a, pop, base, blockIdx.x, ncta);
  else tc_update_net<false, TPS, POP, AOUT>(a, pop, base, blockIdx.x - ncta, ncta);
}

size_t ppo_grad_tc_smem_bytes() { return T2_SMEM; }

template <int TPS, bool POP, int AOUT>
static int tc_attrs() {
  AUR_CUDA_OK(cudaFuncSetAttribute(ppo_grad_tc_kernel<TPS, POP, AOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T2_SMEM));
  // two CTAs per SM need the full shared-memory carve-out
  AUR_CUDA_OK(cudaFuncSetAttribute(ppo_grad_tc_kernel<TPS, POP, AOUT>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                   cudaSharedmemCarveoutMaxShared));
  return 0;
}

// one launch of the instantiation for act_dim (1 .. POL_OUT_MAX, checked by the caller)
template <int TPS, bool POP>
static int launch_tc(const UpdDev& d, const PopUpd& pop, dim3 grid, cudaStream_t s) {
  static DeviceOnce attr;
  if (attr.first()) {
    int rc;
    if ((rc = tc_attrs<TPS, POP, 1>()) || (rc = tc_attrs<TPS, POP, 2>()) || (rc = tc_attrs<TPS, POP, 3>()) ||
        (rc = tc_attrs<TPS, POP, 4>()))
      return rc;
    attr.done();
  }
  static_assert(POL_OUT_MAX == 4, "one instantiation per act_dim");
  switch (d.act_dim) {
    case 1: ppo_grad_tc_kernel<TPS, POP, 1><<<grid, 128 * TPS, T2_SMEM, s>>>(d, pop); break;
    case 2: ppo_grad_tc_kernel<TPS, POP, 2><<<grid, 128 * TPS, T2_SMEM, s>>>(d, pop); break;
    case 3: ppo_grad_tc_kernel<TPS, POP, 3><<<grid, 128 * TPS, T2_SMEM, s>>>(d, pop); break;
    default: ppo_grad_tc_kernel<TPS, POP, 4><<<grid, 128 * TPS, T2_SMEM, s>>>(d, pop); break;
  }
  return 0;
}

// gx = CTAs per net (partials are [2][gx][UPD_PSTRIDE]); the grid is 2 * gx.  tps = threads per sample (2 or 4).
int launch_ppo_grad_tc(const UpdDev& d, int gx, int tps, cudaStream_t s) {
  const int rc = tps == 4 ? launch_tc<4, false>(d, PopUpd{}, dim3(2 * gx), s) : launch_tc<2, false>(d, PopUpd{}, dim3(2 * gx), s);
  if (rc) return rc;
  AUR_LAUNCH_OK("ppo_grad_tc_kernel");
  return 0;
}

// population form: gx CTAs per net and member, K members (two threads per sample)
int launch_ppo_grad_tc_pop(const UpdDev& d, const PopUpd& pop, int gx, int K, cudaStream_t s) {
  const int rc = launch_tc<2, true>(d, pop, dim3(2 * gx, K), s);
  if (rc) return rc;
  AUR_LAUNCH_OK("ppo_grad_tc_kernel (population)");
  return 0;
}

}  // namespace aur
