// Fused rollout with the actor's hidden layer on tensor cores (rows R, Ec, Ep, Ev, M, D; hidden 64 or 128, 2 layers).
// Same contract as rollout_kernel (rollout.cu): T env steps x N envs in one launch, env state in registers, fp64
// physics bit-identical to the checker, Philox sampling keyed by the global env id.  The difference is where the
// 64x64 layer of the actor runs: a CTA owns 128 envs (thread = env = TMEM lane), every step the threads write their
// h1 row as a bf16 hi/mid split into a 128-B-swizzled tile, ONE tcgen05 MMA batch (four split products, fp32
// accumulate in TMEM) produces z2 for all 128 envs, and each thread reads its row back (tcgen05.ld 32x32b) for tanh,
// head, sampling and the env step.  Four CTAs per SM (52 KB of shared memory, 64 TMEM columns each) interleave
// their per-step MMA round trips.  The critic is not evaluated here (critic_values_tc_kernel does all T*N values).
#include <stdlib.h>

#include "envs.cuh"
#include "tc_split.cuh"

namespace aur {

constexpr int RT_S = 128;
constexpr int RT_TILE = RT_S * 128;               // one K atom of the h1 tile: 128 envs x 64 features (128-B rows)
// H = 64: four CTAs per SM (52 KB, 64 TMEM columns each).  H = 128 (`--hidden_dim 128`): the operand tiles are two K atoms wide
// and W2 has 128 rows - 131 KB, one CTA per SM, 128 TMEM columns; still 30x the runtime-width SIMT kernel.
template <int H>
struct RtCfg {
  static constexpr int KA = H / 64;                           // K atoms (64 features each)
  static constexpr int WTILE = H * 128;                       // one K atom of W2: H rows x 128 B
  static constexpr int O_H1 = 0;                              // [hi, mid][atom]
  static constexpr int O_W2 = O_H1 + 2 * KA * RT_TILE;        // [hi, mid][atom]
  static constexpr int O_SMALL = O_W2 + 2 * KA * WTILE;       // fp32: W1^T [4][H] and b1, b2 pre-scaled for tanh, W3 [4][H], b3 [4], logstd [4]
  static constexpr int S_W1T = 0, S_B1 = 4 * H, S_B2 = 5 * H, S_W3 = 6 * H, S_B3 = 10 * H, S_LS = 10 * H + 4, S_N = 10 * H + 8;
  static constexpr int O_BAR = O_SMALL + S_N * 4;
  static constexpr size_t SMEM = O_BAR + 64 + 1024;
  static constexpr int CTAS = H == 64 ? 4 : (H == 0 ? 4 : 1);
};

// H = 0: the actor's outputs come from outside (a.ext_logits [N][4], rollout_wide.cu computes them layer by layer for the widths
// whose W2 does not fit shared memory); the kernel is then only the per-step env / sampling / bookkeeping part, launched once
// per step (a.T = 1, a.t0 = step) with the env state round-tripping through its global arrays.
// POP: population form (aur_pop_rollout), grid (ceil(n_member / 128), K): the CTA's member is blockIdx.y, its envs are the
// member-local indices blockIdx.x * 128 + tid < n_member, stored in the population's columns k * n_member + local; the
// weights, the Philox key and the episode-log row are the member's, the Philox counters and logged env ids member-local.
template <class ENV, int H, bool POP = false>
__global__ void __launch_bounds__(RT_S, RtCfg<H>::CTAS) rollout_tc_kernel(RolloutDev a) {
  using Cfg = RtCfg<H>;
  static_assert(!POP || H == 64, "populations run the 64-wide kernel");
  constexpr bool EXT = H == 0;
  constexpr int KA = Cfg::KA;
  constexpr int RS_W1T = Cfg::S_W1T, RS_B1 = Cfg::S_B1, RS_B2 = Cfg::S_B2, RS_W3 = Cfg::S_W3, RS_B3 = Cfg::S_B3, RS_LS = Cfg::S_LS;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* h1t[2] = {base + Cfg::O_H1, base + Cfg::O_H1 + KA * RT_TILE};
  unsigned char* w2t[2] = {base + Cfg::O_W2, base + Cfg::O_W2 + KA * Cfg::WTILE};
  float* sw = reinterpret_cast<float*>(base + Cfg::O_SMALL);
  uint64_t* bar = reinterpret_cast<uint64_t*>(base + Cfg::O_BAR);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(base + Cfg::O_BAR + 32);
  const int tid = threadIdx.x, warp = tid >> 5;
  constexpr bool PEND = ENV::CONT;
  const int A = a.act_dim, obs_dim = a.obs_dim;

  uint32_t tm_z = 0;
  if constexpr (!EXT) {
  if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  if (warp == 0) tc::tmem_alloc(tslot, H);
  {
    const float* g = POP ? a.params + (long long)blockIdx.y * a.pop_P : a.params;   // the actor comes first in the flat buffer
    const float* gb1 = g + H * obs_dim;
    const float* gW2 = gb1 + H;
    const float* gb2 = gW2 + H * H;
    const float* gW3 = gb2 + H;
    const float* gb3 = gW3 + A * H;
    for (int e = tid; e < 4 * H; e += RT_S) {
      const int c = e / H, j = e - c * H;
      sw[RS_W1T + e] = c < obs_dim ? TANH_PRESCALE * g[j * obs_dim + c] : 0.0f;
      sw[RS_W3 + e] = e < A * H ? gW3[e] : 0.0f;
    }
    for (int e = tid; e < H; e += RT_S) { sw[RS_B1 + e] = TANH_PRESCALE * gb1[e]; sw[RS_B2 + e] = TANH_PRESCALE * gb2[e]; }
    if (tid < 4) {
      sw[RS_B3 + tid] = tid < A ? gb3[tid] : 0.0f;
      const int64_t gA = net_param_count(obs_dim, H, 2, A), gC = net_param_count(obs_dim, H, 2, 1);
      sw[RS_LS + tid] = (a.continuous && tid < A) ? g[gA + gC + tid] : 0.0f;
    }
#pragma unroll 1
    for (int e = tid; e < H * (H / 8); e += RT_S) {         // W2 row j, 8-feature chunk ch -> K atom ch / 8
      const int j = e % H, ch = e / H;
      float2 v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = make_float2(gW2[j * H + 8 * ch + 2 * q], gW2[j * H + 8 * ch + 2 * q + 1]);
      store_split_chunk(w2t[0] + (ch >> 3) * Cfg::WTILE, w2t[1] + (ch >> 3) * Cfg::WTILE, j, ch & 7, v);
    }
  }
  tc::fence_proxy_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  tm_z = *tslot;
  }
  const uint32_t lane_base = (uint32_t)(32 * warp) << 16;
  constexpr uint32_t ID_FWD = tc::instr_desc(tc::FMT_BF16, 128, H, 0, 0);

  const long long N = a.N;
  const long long n_loc = (long long)blockIdx.x * RT_S + tid;         // member-local env index (POP), else the column
  const long long n = POP ? (long long)blockIdx.y * a.n_member + n_loc : n_loc;
  const bool live = POP ? n_loc < a.n_member : n < N;
  const long long m0 = live ? n : 0;
  ENV env;
  NormState nm;
  float obs[POL_IN_PAD];
  Pcg64 rng;                                     // reset stream in registers: a reset costs no global round trip
  rng.load(a.env.pcg, N, m0);
  env.load(a.env.phys, N, m0);
  int elapsed = a.env.elapsed[m0], ep_len = a.env.ep_length[m0];
  float ep_ret = a.env.ep_return[m0], done_prev = a.next_done[m0];
#pragma unroll
  for (int k = 0; k < POL_IN_PAD; ++k) obs[k] = k < ENV::OBS ? a.next_obs[m0 * ENV::OBS + k] : 0.0f;
  if constexpr (PEND) { if (a.wrappers) nm.load(a.env.norm, N, m0); }
  NormalConsts nc;
  if (a.continuous) {
    if constexpr (EXT) nc = normal_consts(a.params + net_param_count(obs_dim, a.hid, a.nl, A) + net_param_count(obs_dim, a.hid, a.nl, 1), A);
    else nc = normal_consts(sw + RS_LS, A);
  }

  for (int tt = 0; tt < a.T; ++tt) {
    const int t = a.t0 + tt;
    const size_t o = (size_t)t * (size_t)N + (size_t)n;
    // ---- buffer.states[t] = next_obs; buffer.terminals[t] = next_done (ppo.py:203-204)
    if (live) {
      if constexpr (ENV::OBS == 4) {
        *reinterpret_cast<float4*>(a.obs_buf + o * 4) = make_float4(obs[0], obs[1], obs[2], obs[3]);
      } else {
#pragma unroll
        for (int k = 0; k < ENV::OBS; ++k) a.obs_buf[o * ENV::OBS + k] = obs[k];
      }
      a.done_buf[o] = done_prev;
    }
    // ---- actor, first layer: this env's h1 row straight into the operand tile (8-feature chunks)
    if constexpr (!EXT) {
#pragma unroll
    for (int c = 0; c < H / 8; ++c) {
      float2 hv[4];
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const int f = 8 * c + 4 * g;
        const float4 b = lds4(sw + RS_B1 + f);
        float2 a01 = make_float2(b.x, b.y), a23 = make_float2(b.z, b.w);
#pragma unroll
        for (int cc = 0; cc < POL_IN_PAD; ++cc) {
          const float4 w = lds4(sw + RS_W1T + cc * H + f);
          const float2 xx = make_float2(obs[cc], obs[cc]);
          a01 = __ffma2_rn(make_float2(w.x, w.y), xx, a01);
          a23 = __ffma2_rn(make_float2(w.z, w.w), xx, a23);
        }
        hv[2 * g] = tanh_prescaled2(a01);
        hv[2 * g + 1] = tanh_prescaled2(a23);
      }
      store_split_chunk(h1t[0] + (c >> 3) * RT_TILE, h1t[1] + (c >> 3) * RT_TILE, tid, c & 7, hv);
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();                               // also: every thread has read last step's z2 out of TMEM
    if (tid == 0) {
      tc::fence_after_sync();
#pragma unroll
      for (int ka = 0; ka < KA; ++ka)
        mma_split4(tm_z, tc::smem_desc_k_sw128(h1t[0] + ka * RT_TILE), tc::smem_desc_k_sw128(h1t[1] + ka * RT_TILE),
                   tc::smem_desc_k_sw128(w2t[0] + ka * Cfg::WTILE), tc::smem_desc_k_sw128(w2t[1] + ka * Cfg::WTILE), ID_FWD, 4, 2, 2,
                   ka > 0);
      tc::mma_commit(bar);
    }
    }
    // the step's random numbers do not depend on the logits: draw them while the MMAs run
    const uint64_t gid = a.env_id0 + (uint64_t)(POP ? n_loc : n), gstep = a.step0 + (uint64_t)t;
    Philox rnd;
    rnd.c[0] = rnd.c[1] = rnd.c[2] = rnd.c[3] = 0u;
    if (a.actions_in == nullptr) {
      const uint64_t seed = POP ? a.pop_seeds[blockIdx.y] : a.seed;
      rnd = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)gstep, (uint32_t)(gstep >> 32), (uint32_t)seed,
                          (uint32_t)(seed >> 32));
    }
    float head[POL_OUT_MAX];
    if constexpr (EXT) {
      const float4 lg = live ? __ldg(reinterpret_cast<const float4*>(a.ext_logits) + n) : make_float4(0.f, 0.f, 0.f, 0.f);
      head[0] = lg.x; head[1] = lg.y; head[2] = lg.z; head[3] = lg.w;
    } else {
    mbar_wait(bar, (uint32_t)tt & 1u);
    tc::fence_after_sync();
    // ---- second layer activation + head from this env's TMEM lane
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) head[k] = sw[RS_B3 + k];
#pragma unroll
    for (int c = 0; c < H / 16; ++c) {
      uint32_t zr[16];
      tc::tmem_ld16(tm_z + lane_base + 16 * c, zr);
      float h2[16];
      const float2 prescale2 = make_float2(TANH_PRESCALE, TANH_PRESCALE);
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const float4 b = lds4(sw + RS_B2 + 16 * c + 4 * g);
        const float2 t01 = tanh_prescaled2(__ffma2_rn(make_float2(__uint_as_float(zr[4 * g]), __uint_as_float(zr[4 * g + 1])),
                                                      prescale2, make_float2(b.x, b.y)));
        const float2 t23 = tanh_prescaled2(__ffma2_rn(make_float2(__uint_as_float(zr[4 * g + 2]), __uint_as_float(zr[4 * g + 3])),
                                                      prescale2, make_float2(b.z, b.w)));
        h2[4 * g] = t01.x; h2[4 * g + 1] = t01.y; h2[4 * g + 2] = t23.x; h2[4 * g + 3] = t23.y;
      }
#pragma unroll
      for (int k = 0; k < POL_OUT_MAX; ++k) {
        if (k < A) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const float4 w = lds4(sw + RS_W3 + k * H + 16 * c + 4 * g);
            head[k] = fmaf(w.x, h2[4 * g], head[k]); head[k] = fmaf(w.y, h2[4 * g + 1], head[k]);
            head[k] = fmaf(w.z, h2[4 * g + 2], head[k]); head[k] = fmaf(w.w, h2[4 * g + 3], head[k]);
          }
        }
      }
    }
    }
    if (!live) continue;
    // ---- distribution, env step, bookkeeping: as rollout_kernel (rollout.cu)
    float logp, entropy, reward32;
    bool terminated;
    double reward;
    if constexpr (!PEND) {
      int action;
      const bool sample = a.actions_in == nullptr;
      float u = 0.0f;
      if (sample) { u = u01_24(rnd.c[0]); action = 0; }
      else action = (int)a.actions_in[o];
      categorical(head, A, sample, u, action, logp, entropy);
      a.act_buf[o] = (float)action;
      reward = env.step(action, terminated);
    } else {
      float act[POL_OUT_MAX] = {0.f, 0.f, 0.f, 0.f};
      if (a.actions_in == nullptr) {
        float z[POL_OUT_MAX];
        normal4(rnd, z);
#pragma unroll
        for (int k = 0; k < POL_OUT_MAX; ++k) act[k] = fmaf(nc.std[k], z[k], head[k]);
      } else {
        for (int k = 0; k < A; ++k) act[k] = a.actions_in[o * A + k];
      }
      normal_logp(head, act, A, nc, logp, entropy);
      for (int k = 0; k < A; ++k) a.act_buf[o * A + k] = act[k];
      reward = env.step(act[0], a.wrappers != 0, terminated);
    }
    a.logp_buf[o] = logp;
    // ---- TimeLimit, RecordEpisodeStatistics (raw reward, fp32 accumulator)
    elapsed += 1;
    const bool truncated = elapsed >= ENV::LIMIT;
    ep_ret = __fadd_rn(ep_ret, (float)reward);
    ep_len += 1;
    const bool finished = terminated || truncated;
    if constexpr (PEND) {
      float raw[3];
      env.raw_obs(raw);
      if (a.wrappers) {
        nm.obs(raw, obs);
        reward = nm.reward(reward, finished, a.gamma);
      } else {
        obs[0] = raw[0]; obs[1] = raw[1]; obs[2] = raw[2]; obs[3] = 0.0f;
      }
    } else {
      env.raw_obs(obs);
    }
    reward32 = (float)reward;                        // torch.tensor(reward) fp64 -> fp32 buffer (ppo.py:111)
    a.rew_buf[o] = reward32;
    if (finished) {
      // ---- SyncVectorEnv autoreset: the returned obs is the RESET obs; `done` keeps `terminated`
      if constexpr (POP) {                           // the member's row of the episode log, member-local env index
        aur_episode_log lg = a.log;
        if (lg.first_finished) lg.first_finished += (size_t)blockIdx.y * a.T;
        if (lg.totals) lg.totals += 3 * (size_t)blockIdx.y;
        log_episode(lg, t, n_loc, (int)gstep, (int)gid, ep_ret, ep_len);
      } else {
        log_episode(a.log, t, n, (int)gstep, (int)gid, ep_ret, ep_len);
      }
      env.reset(rng);
      elapsed = 0; ep_ret = 0.0f; ep_len = 0;
      if constexpr (PEND) {
        float raw[3];
        env.raw_obs(raw);
        if (a.wrappers) nm.obs(raw, obs);
        else { obs[0] = raw[0]; obs[1] = raw[1]; obs[2] = raw[2]; obs[3] = 0.0f; }
      } else {
        env.raw_obs(obs);
      }
    }
    done_prev = terminated ? 1.0f : 0.0f;            // ppo.py:110 keeps `terminated`, drops `truncated`
  }

  if (live) {
    rng.store(a.env.pcg, N, n);
    env.store(a.env.phys, N, n);
    a.env.elapsed[n] = elapsed; a.env.ep_return[n] = ep_ret; a.env.ep_length[n] = ep_len;
    a.next_done[n] = done_prev;
#pragma unroll
    for (int k = 0; k < ENV::OBS; ++k) a.next_obs[n * ENV::OBS + k] = obs[k];
    if constexpr (PEND) { if (a.wrappers) nm.store(a.env.norm, N, n); }
  }
  if constexpr (!EXT) {
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tm_z, H);
  }
}

// 1 = tensor-core rollout (default for hidden 64 / 2 layers), 0 = SIMT rollout_kernel; AUR_ROLLOUT_IMPL=simt|tc
static int g_rollout_impl = -1;
int rollout_impl() {
  if (g_rollout_impl < 0) {
    const char* e = getenv("AUR_ROLLOUT_IMPL");
    g_rollout_impl = e ? ((e[0] == 's' || e[0] == '0') ? 0 : 1) : 1;
  }
  return g_rollout_impl;
}
void set_rollout_impl(int impl) { g_rollout_impl = impl; }

template <class ENV, int H, bool POP = false>
static int rollout_tc_attrs() {
  AUR_CUDA_OK(cudaFuncSetAttribute(rollout_tc_kernel<ENV, H, POP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RtCfg<H>::SMEM));
  AUR_CUDA_OK(cudaFuncSetAttribute(rollout_tc_kernel<ENV, H, POP>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  return 0;
}

// population rollout (aur_pop_rollout): every member's envs in one launch, grid (ceil(n_member / 128), K)
int launch_rollout_tc_pop(const RolloutDev& d, int env_kind, int K, cudaStream_t s) {
  static DeviceOnce attr;
  if (attr.first()) {
    int rc;
    if ((rc = rollout_tc_attrs<CartPole, 64, true>()) || (rc = rollout_tc_attrs<Pendulum, 64, true>()) ||
        (rc = rollout_tc_attrs<MountainCar, 64, true>()))
      return rc;
    attr.done();
  }
  const dim3 grid((unsigned)((d.n_member + RT_S - 1) / RT_S), (unsigned)K);
  constexpr size_t SM = RtCfg<64>::SMEM;
  if (env_kind == AUR_ENV_PENDULUM) rollout_tc_kernel<Pendulum, 64, true><<<grid, RT_S, SM, s>>>(d);
  else if (env_kind == AUR_ENV_MOUNTAINCAR) rollout_tc_kernel<MountainCar, 64, true><<<grid, RT_S, SM, s>>>(d);
  else rollout_tc_kernel<CartPole, 64, true><<<grid, RT_S, SM, s>>>(d);
  AUR_LAUNCH_OK("rollout_tc_kernel (population)");
  return 0;
}

// one env step of all N envs from externally computed actor outputs (d.ext_logits, d.t0; d.T = 1)
int launch_rollout_step_ext(const RolloutDev& d, int env_kind, cudaStream_t s) {
  const unsigned grid = (unsigned)((d.N + RT_S - 1) / RT_S);
  if (env_kind == AUR_ENV_PENDULUM) rollout_tc_kernel<Pendulum, 0><<<grid, RT_S, 0, s>>>(d);
  else if (env_kind == AUR_ENV_MOUNTAINCAR) rollout_tc_kernel<MountainCar, 0><<<grid, RT_S, 0, s>>>(d);
  else rollout_tc_kernel<CartPole, 0><<<grid, RT_S, 0, s>>>(d);
  AUR_LAUNCH_OK("rollout_tc_kernel (external actor)");
  return 0;
}

// hidden = 64 or 128 (two layers, widths <= 4)
int launch_rollout_tc(const RolloutDev& d, int env_kind, int hidden, cudaStream_t s) {
  static DeviceOnce attr;
  if (attr.first()) {
    int rc;
    if ((rc = rollout_tc_attrs<CartPole, 64>()) || (rc = rollout_tc_attrs<Pendulum, 64>()) || (rc = rollout_tc_attrs<MountainCar, 64>()) ||
        (rc = rollout_tc_attrs<CartPole, 128>()) || (rc = rollout_tc_attrs<Pendulum, 128>()) || (rc = rollout_tc_attrs<MountainCar, 128>()))
      return rc;
    attr.done();
  }
  const unsigned grid = (unsigned)((d.N + RT_S - 1) / RT_S);
  if (hidden == 128) {
    constexpr size_t SM = RtCfg<128>::SMEM;
    if (env_kind == AUR_ENV_PENDULUM) rollout_tc_kernel<Pendulum, 128><<<grid, RT_S, SM, s>>>(d);
    else if (env_kind == AUR_ENV_MOUNTAINCAR) rollout_tc_kernel<MountainCar, 128><<<grid, RT_S, SM, s>>>(d);
    else rollout_tc_kernel<CartPole, 128><<<grid, RT_S, SM, s>>>(d);
  } else {
    constexpr size_t SM = RtCfg<64>::SMEM;
    if (env_kind == AUR_ENV_PENDULUM) rollout_tc_kernel<Pendulum, 64><<<grid, RT_S, SM, s>>>(d);
    else if (env_kind == AUR_ENV_MOUNTAINCAR) rollout_tc_kernel<MountainCar, 64><<<grid, RT_S, SM, s>>>(d);
    else rollout_tc_kernel<CartPole, 64><<<grid, RT_S, SM, s>>>(d);
  }
  AUR_LAUNCH_OK("rollout_tc_kernel");
  return 0;
}

}  // namespace aur

extern "C" int aur_rollout_set_impl(int impl) {
  if (impl != 0 && impl != 1) { aur::set_error("aur_rollout_set_impl: impl must be 0 (simt) or 1 (tensor core)"); return AUR_ERR_ARG; }
  aur::set_rollout_impl(impl);
  return 0;
}
extern "C" int aur_rollout_get_impl(void) { return aur::rollout_impl(); }
