// Fused rollout: T env steps x N envs in one persistent kernel (rows R, Ec, Ep, Ev, M, D of the
// scope table).  Replaces src/ppo.py:201-205 + rewards_to_go (src/ppo.py:103-123) and the gym
// pieces it drives (CartPole-v1 / Pendulum-v1 physics, TimeLimit, RecordEpisodeStatistics,
// SyncVectorEnv autoreset, the continuous wrapper stack of src/ppo.py:92-97).
//
// One env per thread (E envs per thread for the small-register discrete config), env state in
// registers for all T steps, fp64 physics with one rounding per gym operation (--fmad=false),
// deterministic double-double sin/cos (det_sincos.h), PCG64 reset streams identical to NumPy's,
// policy MLPs from shared memory (policy.cuh), Philox4x32-10 sampling keyed by the GLOBAL env id.
// Per step each env writes 36 B (CartPole) into the [T,N] buffers, coalesced across the warp.
#include "envs.cuh"

namespace aur {

int launch_critic_values_tc(const float* critic, int obs_dim, int hidden, const float* obs, long long M, float* out, cudaStream_t s);
int launch_rollout_tc(const RolloutDev& d, int env_kind, int hidden, cudaStream_t s);
int rollout_impl();
bool rollout_wide_eligible(const aur_policy_desc& p, int env_kind);      // rollout_wide.cu: layer-wise actor on tensor cores
int launch_rollout_wide(const RolloutDev& d, const aur_policy_desc& p, int env_kind, cudaStream_t s);

// ENV: CartPole or Pendulum.  E envs per thread (env n = base + e * nthreads_total keeps warps coalesced).
// CRITIC = false: the values are filled afterwards by critic_values_tc_kernel (values_tc.cu) from the observation rows.
template <class ENV, int HID, int E, bool CRITIC>
__global__ void __launch_bounds__(256, 1) rollout_kernel(RolloutDev a) {
  extern __shared__ __align__(16) float smem[];
  const float *sActor, *sCritic, *sLogstd;
  float* scratch;
  bool vec_critic = true;
  if constexpr (HID == 0) {
    load_policy_dyn(smem, a, sActor, sCritic, sLogstd, scratch, vec_critic);
  } else {
    load_policy_smem<HID>(smem, a, sActor, sCritic, sLogstd);
    const int policy_floats = net_smem_floats(HID, a.nl, a.act_dim) + net_smem_floats(HID, a.nl, 1) + 4;
    scratch = smem + policy_floats + threadIdx.x;   // [HID][blockDim] column (NL >= 3 only)
  }
  __syncthreads();

  constexpr bool PEND = ENV::CONT;            // continuous env: Normal policy, optional wrapper stack
  constexpr int INP = ENV::OBS > POL_IN_PAD ? 8 : POL_IN_PAD;     // observation registers per env (Acrobot: 6 -> 8)
  static_assert(HID == 0 || INP == POL_IN_PAD, "observations wider than 4 run the runtime-width policy path");
  const long long N = a.N;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long base = (long long)blockIdx.x * blockDim.x + threadIdx.x;

  ENV env[E];
  NormStateT<ENV::OBS> nm[PEND ? E : 1];
  float obs[E][INP];
  float done_prev[E], ep_ret[E];
  int elapsed[E], ep_len[E];
  bool live[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const long long n = base + e * stride;
    live[e] = n < N;
    const long long m = live[e] ? n : 0;
    env[e].load(a.env.phys, N, m);
    elapsed[e] = a.env.elapsed[m]; ep_ret[e] = a.env.ep_return[m]; ep_len[e] = a.env.ep_length[m];
    done_prev[e] = a.next_done[m];
#pragma unroll
    for (int k = 0; k < INP; ++k) obs[e][k] = k < ENV::OBS ? a.next_obs[m * ENV::OBS + k] : 0.0f;
    if constexpr (PEND) { if (a.wrappers) nm[e].load(a.env.norm, N, m); }
  }
  NormalConsts nc;
  if (a.continuous) nc = normal_consts(sLogstd, a.act_dim);

  for (int t = 0; t < a.T; ++t) {
    // ---- buffer.states[t] = next_obs; buffer.terminals[t] = next_done (ppo.py:203-204)
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const long long n = base + e * stride;
      if (live[e]) {
        const size_t o = (size_t)t * (size_t)N + (size_t)n;
        if constexpr (ENV::OBS == 4) {
          *reinterpret_cast<float4*>(a.obs_buf + o * 4) = make_float4(obs[e][0], obs[e][1], obs[e][2], obs[e][3]);
        } else {
#pragma unroll
          for (int k = 0; k < ENV::OBS; ++k) a.obs_buf[o * ENV::OBS + k] = obs[e][k];
        }
        a.done_buf[o] = done_prev[e];
      }
    }
    // ---- policy.evaluate(next_obs) (ppo.py:105): actor head, critic value
    float head[E][POL_OUT_MAX], value[E];
#pragma unroll 1
    for (int net = 0; net < (CRITIC ? 2 : 1); ++net) {
      float o[E][POL_OUT_MAX];
      policy_net_forward<HID, E, INP>(a, net == 0 ? sActor : sCritic, net == 0 || vec_critic, net == 0 ? a.act_dim : 1, obs, o, scratch);
#pragma unroll
      for (int e = 0; e < E; ++e) {
        if (net == 0) {
#pragma unroll
          for (int k = 0; k < POL_OUT_MAX; ++k) head[e][k] = o[e][k];
        } else {
          value[e] = o[e][0];
        }
      }
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const long long n = base + e * stride;
      if (!live[e]) continue;
      const size_t o = (size_t)t * (size_t)N + (size_t)n;
      const uint64_t gid = a.env_id0 + (uint64_t)n, gstep = a.step0 + (uint64_t)t;
      float logp, entropy, reward32;
      bool terminated;
      double reward;
      if constexpr (!PEND) {
        // ---- Categorical sample / replay, env.step
        int action;
        const bool sample = a.actions_in == nullptr;
        float u = 0.0f;
        if (sample) {
          const Philox r = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)gstep, (uint32_t)(gstep >> 32),
                                         (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
          u = u01_24(r.c[0]);
          action = 0;
        } else {
          action = (int)a.actions_in[o];
        }
        categorical(head[e], a.act_dim, sample, u, action, logp, entropy);
        a.act_buf[o] = (float)action;
        reward = env[e].step(action, terminated);
      } else {
        float act[POL_OUT_MAX] = {0.f, 0.f, 0.f, 0.f};
        if (a.actions_in == nullptr) {
          const Philox r = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)gstep, (uint32_t)(gstep >> 32),
                                         (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
          float z[POL_OUT_MAX];
          normal4(r, z);
#pragma unroll
          for (int k = 0; k < POL_OUT_MAX; ++k) act[k] = fmaf(nc.std[k], z[k], head[e][k]);
        } else {
          for (int k = 0; k < a.act_dim; ++k) act[k] = a.actions_in[o * a.act_dim + k];
        }
        normal_logp(head[e], act, a.act_dim, nc, logp, entropy);
        for (int k = 0; k < a.act_dim; ++k) a.act_buf[o * a.act_dim + k] = act[k];
        reward = env[e].step(act[0], a.wrappers != 0, terminated);
      }
      a.logp_buf[o] = logp;
      if (CRITIC) a.val_buf[o] = value[e];
      // ---- TimeLimit, RecordEpisodeStatistics (raw reward, fp32 accumulator)
      elapsed[e] += 1;
      const bool truncated = elapsed[e] >= ENV::LIMIT;
      ep_ret[e] = __fadd_rn(ep_ret[e], (float)reward);
      ep_len[e] += 1;
      const bool finished = terminated || truncated;
      if constexpr (PEND) {
        // wrappers see the stepped observation before SyncVectorEnv autoresets
        float raw[ENV::OBS];
        env[e].raw_obs(raw);
        if (a.wrappers) {
          nm[PEND ? e : 0].obs(raw, obs[e]);
          reward = nm[PEND ? e : 0].reward(reward, finished, a.gamma);
        } else {
#pragma unroll
          for (int k = 0; k < POL_IN_PAD; ++k) obs[e][k] = k < ENV::OBS ? raw[k < ENV::OBS ? k : 0] : 0.0f;
        }
      } else {
        env[e].raw_obs(obs[e]);
      }
      reward32 = (float)reward;                      // torch.tensor(reward) fp64 -> fp32 buffer (ppo.py:111)
      a.rew_buf[o] = reward32;
      if (finished) {
        // ---- SyncVectorEnv autoreset: the returned obs is the RESET obs; `done` keeps `terminated`
        log_episode(a.log, t, n, (int)gstep, (int)gid, ep_ret[e], ep_len[e]);
        Pcg64 rng;
        rng.load(a.env.pcg, N, n);
        env[e].reset(rng);
        rng.store(a.env.pcg, N, n);
        elapsed[e] = 0; ep_ret[e] = 0.0f; ep_len[e] = 0;
        if constexpr (PEND) {
          float raw[ENV::OBS];
          env[e].raw_obs(raw);
          if (a.wrappers) nm[PEND ? e : 0].obs(raw, obs[e]);
          else {
#pragma unroll
            for (int k = 0; k < POL_IN_PAD; ++k) obs[e][k] = k < ENV::OBS ? raw[k < ENV::OBS ? k : 0] : 0.0f;
          }
        } else {
          env[e].raw_obs(obs[e]);
        }
      }
      done_prev[e] = terminated ? 1.0f : 0.0f;       // ppo.py:110 keeps `terminated`, drops `truncated`
    }
  }

  // ---- write back: next_obs / next_done / env state, and critic(next_obs) for GAE (ppo.py:161)
  if (CRITIC && a.next_value) {
    float o[E][POL_OUT_MAX];
    policy_net_forward<HID, E, INP>(a, sCritic, vec_critic, 1, obs, o, scratch);
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const long long n = base + e * stride;
      if (live[e]) a.next_value[n] = o[e][0];
    }
  }
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const long long n = base + e * stride;
    if (!live[e]) continue;
    env[e].store(a.env.phys, N, n);
    a.env.elapsed[n] = elapsed[e]; a.env.ep_return[n] = ep_ret[e]; a.env.ep_length[n] = ep_len[e];
    a.next_done[n] = done_prev[e];
#pragma unroll
    for (int k = 0; k < ENV::OBS; ++k) a.next_obs[n * ENV::OBS + k] = obs[e][k];
    if constexpr (PEND) { if (a.wrappers) nm[e].store(a.env.norm, N, n); }
  }
}

// envs.reset(seed=list) (ppo.py:188)
template <class ENV>
__global__ void env_reset_kernel(long long N, int wrappers, aur_env_state st, float* obs_out, float* done_out) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  Pcg64 rng;
  rng.load(st.pcg, N, n);
  ENV env;
  env.reset(rng);
  rng.store(st.pcg, N, n);
  env.store(st.phys, N, n);
  st.elapsed[n] = 0; st.ep_return[n] = 0.0f; st.ep_length[n] = 0;
  float obs[ENV::OBS > POL_IN_PAD ? 8 : POL_IN_PAD];
  if constexpr (ENV::CONT) {
    float raw[ENV::OBS];
    env.raw_obs(raw);
    if (wrappers) {
      NormStateT<ENV::OBS> nm;
      nm.init();
      nm.obs(raw, obs);
      nm.store(st.norm, N, n);
    } else {
      for (int k = 0; k < ENV::OBS; ++k) obs[k] = raw[k];
    }
  } else {
    env.raw_obs(obs);
  }
  for (int k = 0; k < ENV::OBS; ++k) obs_out[n * ENV::OBS + k] = obs[k];
  if (done_out) done_out[n] = 0.0f;
}

// actor_critic.evaluate / value on a batch (models/actor_critic.py:31-51), no grad
template <int HID>
__global__ void __launch_bounds__(256, 1) policy_evaluate_kernel(RolloutDev a, long long B, const float* obs_in,
                                                                 uint64_t row0, uint64_t step, float* act_out,
                                                                 float* logp_out, float* ent_out, float* val_out) {
  extern __shared__ __align__(16) float smem[];
  const float *sActor, *sCritic, *sLogstd;
  load_policy_smem<HID>(smem, a, sActor, sCritic, sLogstd);
  const int policy_floats = net_smem_floats(HID, a.nl, a.act_dim) + net_smem_floats(HID, a.nl, 1) + 4;
  float* scratch = smem + policy_floats + threadIdx.x;
  __syncthreads();
  NormalConsts nc;
  if (a.continuous) nc = normal_consts(sLogstd, a.act_dim);
  for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    float x[1][POL_IN_PAD];
    for (int k = 0; k < POL_IN_PAD; ++k) x[0][k] = k < a.obs_dim ? obs_in[b * a.obs_dim + k] : 0.0f;
    float head[1][POL_OUT_MAX], v[1][POL_OUT_MAX];
    mlp_forward<HID, 1>(sActor, a.nl, a.act_dim, x, head, scratch, blockDim.x);
    mlp_forward<HID, 1>(sCritic, a.nl, 1, x, v, scratch, blockDim.x);
    float logp, entropy;
    const uint64_t gid = row0 + (uint64_t)b;
    if (!a.continuous) {
      int action = 0;
      const bool sample = a.actions_in == nullptr && !a.greedy;
      float u = 0.0f;
      if (a.greedy) {                                       // first maximum, like torch.argmax
        const auto& lg = head[0];
        for (int k = 1; k < a.act_dim; ++k) if (lg[k] > lg[action]) action = k;
      } else if (sample) {
        const Philox r = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)step, (uint32_t)(step >> 32),
                                       (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
        u = u01_24(r.c[0]);
      } else {
        action = (int)a.actions_in[b];
      }
      categorical(head[0], a.act_dim, sample, u, action, logp, entropy);
      if (act_out) act_out[b] = (float)action;
    } else {
      float act[POL_OUT_MAX] = {0.f, 0.f, 0.f, 0.f};
      if (a.greedy) {
        for (int k = 0; k < POL_OUT_MAX; ++k) act[k] = head[0][k];
      } else if (a.actions_in == nullptr) {
        const Philox r = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)step, (uint32_t)(step >> 32),
                                       (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
        float z[POL_OUT_MAX];
        normal4(r, z);
        for (int k = 0; k < POL_OUT_MAX; ++k) act[k] = fmaf(nc.std[k], z[k], head[0][k]);
      } else {
        for (int k = 0; k < a.act_dim; ++k) act[k] = a.actions_in[b * a.act_dim + k];
      }
      normal_logp(head[0], act, a.act_dim, nc, logp, entropy);
      if (act_out) for (int k = 0; k < a.act_dim; ++k) act_out[b * a.act_dim + k] = act[k];
    }
    if (logp_out) logp_out[b] = logp;
    if (ent_out) ent_out[b] = entropy;
    if (val_out) val_out[b] = v[0][0];
  }
}

// the same for runtime hidden widths and observation / action widths up to 8 (e.g. the reference's shipped
// actor_critic_2.pt: state 8, 4 actions): mlp_forward_dyn, one sample per thread
constexpr int DYN_IO = 8;
__global__ void __launch_bounds__(128, 1) policy_evaluate_dyn_kernel(RolloutDev a, long long B, const float* obs_in,
                                                                     uint64_t row0, uint64_t step, float* act_out,
                                                                     float* logp_out, float* ent_out, float* val_out) {
  extern __shared__ __align__(16) float smem[];
  const float *sActor, *sCritic, *sLogstd;
  float* scratch;
  bool vec_critic = true;
  load_policy_dyn(smem, a, sActor, sCritic, sLogstd, scratch, vec_critic);
  __syncthreads();
  NormalConstsT<DYN_IO> nc;
  if (a.continuous) nc = normal_consts<DYN_IO>(sLogstd, a.act_dim);
  for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
    float x[DYN_IO], head[DYN_IO], v[DYN_IO];
#pragma unroll
    for (int k = 0; k < DYN_IO; ++k) x[k] = k < a.obs_dim ? obs_in[b * a.obs_dim + k] : 0.0f;
    mlp_forward_dyn<true, DYN_IO, DYN_IO>(sActor, a.obs_dim, a.hid, a.nl, a.act_dim, x, head, scratch, blockDim.x);
    if (vec_critic) mlp_forward_dyn<true, DYN_IO, DYN_IO>(sCritic, a.obs_dim, a.hid, a.nl, 1, x, v, scratch, blockDim.x);
    else mlp_forward_dyn<false, DYN_IO, DYN_IO>(sCritic, a.obs_dim, a.hid, a.nl, 1, x, v, scratch, blockDim.x);
    float logp, entropy;
    const uint64_t gid = row0 + (uint64_t)b;
    if (!a.continuous) {
      int action = 0;
      const bool sample = a.actions_in == nullptr && !a.greedy;
      float u = 0.0f;
      if (a.greedy) {                                       // first maximum, like torch.argmax
        const auto& lg = head;
        for (int k = 1; k < a.act_dim; ++k) if (lg[k] > lg[action]) action = k;
      } else if (sample) {
        const Philox r = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)step, (uint32_t)(step >> 32),
                                       (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
        u = u01_24(r.c[0]);
      } else {
        action = (int)a.actions_in[b];
      }
      categorical(head, a.act_dim, sample, u, action, logp, entropy);
      if (act_out) act_out[b] = (float)action;
    } else {
      float act[DYN_IO];
#pragma unroll
      for (int k = 0; k < DYN_IO; ++k) act[k] = 0.0f;
      if (a.greedy) {
#pragma unroll
        for (int k = 0; k < DYN_IO; ++k) act[k] = k < a.act_dim ? head[k] : 0.0f;
      } else if (a.actions_in == nullptr) {
        // dims 0..3 from the Philox block the 4-wide kernels use, dims 4..7 from a second block (counter word 3 ^ 1 << 24)
#pragma unroll
        for (int blk = 0; blk < 2; ++blk) {
          if (blk * 4 < a.act_dim) {
            const Philox r = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)step,
                                           (uint32_t)(step >> 32) ^ ((uint32_t)blk << 24), (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
            float z[POL_OUT_MAX];
            normal4(r, z);
#pragma unroll
            for (int k = 0; k < 4; ++k) act[blk * 4 + k] = fmaf(nc.std[blk * 4 + k], z[k], head[blk * 4 + k]);
          }
        }
      } else {
        for (int k = 0; k < a.act_dim; ++k) act[k] = a.actions_in[b * a.act_dim + k];
      }
      normal_logp(head, act, a.act_dim, nc, logp, entropy);
      if (act_out) for (int k = 0; k < a.act_dim; ++k) act_out[b * a.act_dim + k] = act[k];
    }
    if (logp_out) logp_out[b] = logp;
    if (ent_out) ent_out[b] = entropy;
    if (val_out) val_out[b] = v[0];
  }
}

__global__ void sincos_kernel(long long n, const double* x, double* s, double* c) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) aur_sincos(x[i], &s[i], &c[i]);
}

static bool is_compiled_width(const aur_policy_desc& p) {
  return p.hidden_dim == 64 && p.obs_dim >= 1 && p.obs_dim <= POL_IN_PAD && p.act_dim >= 1 && p.act_dim <= POL_OUT_MAX;
}
// 64 hidden units and widths <= 4 run the register-resident kernels; everything else the runtime-width path
static int check_policy(const aur_policy_desc& p, const char* who, int io_max) {
  if (p.num_layers < 1 || p.num_layers > 16) { set_error("%s: num_layers %d outside 1..16", who, p.num_layers); return AUR_ERR_UNSUPPORTED; }
  if (is_compiled_width(p)) return 0;
  if (p.hidden_dim < 4 || p.hidden_dim > 256 || (p.hidden_dim & 3)) {
    set_error("%s: hidden_dim %d outside the compiled range (multiples of 4 in 4..256); no fallback", who, p.hidden_dim);
    return AUR_ERR_UNSUPPORTED;
  }
  if (p.obs_dim < 1 || p.obs_dim > io_max) { set_error("%s: obs_dim %d outside 1..%d", who, p.obs_dim, io_max); return AUR_ERR_UNSUPPORTED; }
  if (p.act_dim < 1 || p.act_dim > io_max) { set_error("%s: act_dim %d outside 1..%d", who, p.act_dim, io_max); return AUR_ERR_UNSUPPORTED; }
  return 0;
}
// runtime-width launch shape: keep the nets in shared memory when they fit beside the activation columns, shrinking the
// block down to 64 threads first; else read them from global memory.  Returns the smem bytes, sets block / in_smem.
static size_t dyn_launch_shape(const aur_policy_desc& p, int& block, int& in_smem) {
  const size_t pf = (size_t)dyn_policy_smem_floats(p.obs_dim, p.hidden_dim, p.num_layers, p.act_dim);
  const size_t limit = 226 * 1024;      // 227 KB is the per-CTA maximum on sm_100; 64 hidden-128 columns + both nets need 204 KB
  for (int b = block; b >= 64; b -= 32) {
    const size_t need = (pf + (size_t)2 * p.hidden_dim * b) * sizeof(float);
    if (need <= limit) { block = b; in_smem = 1; return need; }
  }
  in_smem = 0;
  for (int b = block; b >= 32; b -= 32) {
    const size_t need = (size_t)2 * p.hidden_dim * b * sizeof(float);
    if (need <= limit) { block = b; return need; }
  }
  block = 32;
  return (size_t)2 * p.hidden_dim * 32 * sizeof(float);
}

static size_t policy_smem_bytes(const aur_policy_desc& p, int threads, bool need_scratch) {
  size_t f = net_smem_floats(p.hidden_dim, p.num_layers, p.act_dim) + net_smem_floats(p.hidden_dim, p.num_layers, 1) + 4;
  if (need_scratch) f += (size_t)p.hidden_dim * threads;
  return f * sizeof(float);
}

// the 64-wide kernels keep BOTH nets in shared memory (register-resident activations): deep policies (e.g. the reference's
// shipped 10-layer checkpoint, 328 KB of weights) take the runtime-shape path, which can read the weights from global / L1
static bool fits_compiled_kernel(const aur_policy_desc& p) {
  return is_compiled_width(p) && policy_smem_bytes(p, 256, p.num_layers >= 3) <= (size_t)227 * 1024;
}

template <class K>
static int launch_cfg(K kernel, size_t smem) {
  if (smem > 227 * 1024) { set_error("policy does not fit shared memory (%zu B); no fallback", smem); return AUR_ERR_UNSUPPORTED; }
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute");
  return 0;
}

static int round_up(int v, int m) { return (v + m - 1) / m * m; }

}  // namespace aur

extern "C" int64_t aur_policy_param_count(const aur_policy_desc* d) {
  if (!d) return AUR_ERR_ARG;
  return aur::policy_param_count(*d);
}

extern "C" int aur_sincos_f64(int64_t n, const double* x, double* s, double* c, void* stream) {
  using namespace aur;
  if (n < 0 || (n > 0 && (!x || !s || !c))) { set_error("aur_sincos_f64: bad arguments"); return AUR_ERR_ARG; }
  if (n == 0) return 0;
  sincos_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((long long)n, x, s, c);
  AUR_LAUNCH_OK("sincos_kernel");
  return 0;
}

extern "C" int aur_env_reset(int32_t env_kind, int64_t N, int32_t wrappers, const aur_env_state* st, float* obs_out,
                             float* done_out, void* stream) {
  using namespace aur;
  if (!st || N < 0 || !obs_out) { set_error("aur_env_reset: bad arguments"); return AUR_ERR_ARG; }
  if (N == 0) return 0;
  if (!st->phys || !st->pcg || !st->elapsed || !st->ep_return || !st->ep_length) { set_error("aur_env_reset: null env state array"); return AUR_ERR_ARG; }
  const unsigned grid = (unsigned)((N + 127) / 128);
  cudaStream_t s = (cudaStream_t)stream;
  if (env_kind == AUR_ENV_CARTPOLE) {
    env_reset_kernel<CartPole><<<grid, 128, 0, s>>>((long long)N, 0, *st, obs_out, done_out);
  } else if (env_kind == AUR_ENV_MOUNTAINCAR) {
    env_reset_kernel<MountainCar><<<grid, 128, 0, s>>>((long long)N, 0, *st, obs_out, done_out);
  } else if (env_kind == AUR_ENV_ACROBOT) {
    env_reset_kernel<Acrobot><<<grid, 128, 0, s>>>((long long)N, 0, *st, obs_out, done_out);
  } else if (env_kind == AUR_ENV_MOUNTAINCAR_CONT) {
    if (wrappers && !st->norm) { set_error("aur_env_reset: wrappers need env.norm"); return AUR_ERR_ARG; }
    env_reset_kernel<MountainCarContinuous><<<grid, 128, 0, s>>>((long long)N, wrappers, *st, obs_out, done_out);
  } else if (env_kind == AUR_ENV_PENDULUM) {
    if (wrappers && !st->norm) { set_error("aur_env_reset: wrappers need env.norm"); return AUR_ERR_ARG; }
    env_reset_kernel<Pendulum><<<grid, 128, 0, s>>>((long long)N, wrappers, *st, obs_out, done_out);
  } else {
    set_error("aur_env_reset: unknown env_kind %d", env_kind); return AUR_ERR_UNSUPPORTED;
  }
  AUR_LAUNCH_OK("env_reset_kernel");
  return 0;
}

static aur::RolloutDev to_dev(const aur_rollout_args& a) {
  aur::RolloutDev d;
  d.N = a.N; d.T = a.T; d.wrappers = a.wrappers;
  d.obs_dim = a.policy.obs_dim; d.act_dim = a.policy.act_dim; d.nl = a.policy.num_layers; d.continuous = a.policy.continuous;
  d.hid = a.policy.hidden_dim; d.dyn_smem = 0;
  d.params = a.params; d.env = a.env;
  d.obs_buf = a.obs_buf; d.act_buf = a.act_buf; d.logp_buf = a.logp_buf; d.val_buf = a.val_buf; d.rew_buf = a.rew_buf;
  d.done_buf = a.done_buf; d.next_obs = a.next_obs; d.next_done = a.next_done; d.next_value = a.next_value;
  d.t0 = 0; d.ext_logits = nullptr;
  d.n_member = 0; d.pop_P = 0; d.pop_seeds = nullptr;
  d.actions_in = a.actions_in; d.seed = a.seed; d.step0 = a.step0; d.env_id0 = a.env_id0; d.log = a.log; d.gamma = a.gamma;
  return d;
}

extern "C" int aur_rollout(const aur_rollout_args* args, void* stream) {
  using namespace aur;
  if (!args) { set_error("aur_rollout: null args"); return AUR_ERR_ARG; }
  const aur_rollout_args& a = *args;
  if (a.N < 0 || a.T < 0) { set_error("aur_rollout: negative N or T"); return AUR_ERR_ARG; }
  if (a.N == 0 || a.T == 0) return 0;
  int rc = check_policy(a.policy, "aur_rollout", DYN_IO);
  if (rc) return rc;
  if (!a.params || !a.obs_buf || !a.act_buf || !a.logp_buf || !a.val_buf || !a.rew_buf || !a.done_buf || !a.next_obs ||
      !a.next_done || !a.env.phys || !a.env.pcg || !a.env.elapsed || !a.env.ep_return || !a.env.ep_length) {
    set_error("aur_rollout: null buffer"); return AUR_ERR_ARG;
  }
  const bool pend = a.env_kind == AUR_ENV_PENDULUM;
  if (a.env_kind == AUR_ENV_CARTPOLE) {
    if (a.policy.continuous || a.policy.obs_dim != 4 || a.policy.act_dim != 2) { set_error("aur_rollout: CartPole needs obs 4, 2 discrete actions"); return AUR_ERR_ARG; }
  } else if (a.env_kind == AUR_ENV_MOUNTAINCAR) {
    if (a.policy.continuous || a.policy.obs_dim != 2 || a.policy.act_dim != 3) { set_error("aur_rollout: MountainCar needs obs 2, 3 discrete actions"); return AUR_ERR_ARG; }
  } else if (a.env_kind == AUR_ENV_MOUNTAINCAR_CONT) {
    if (!a.policy.continuous || a.policy.obs_dim != 2 || a.policy.act_dim != 1) { set_error("aur_rollout: MountainCarContinuous needs obs 2, 1 continuous action"); return AUR_ERR_ARG; }
    if (a.wrappers && !a.env.norm) { set_error("aur_rollout: wrappers need env.norm"); return AUR_ERR_ARG; }
  } else if (a.env_kind == AUR_ENV_ACROBOT) {
    if (a.policy.continuous || a.policy.obs_dim != 6 || a.policy.act_dim != 3) { set_error("aur_rollout: Acrobot needs obs 6, 3 discrete actions"); return AUR_ERR_ARG; }
  } else if (pend) {
    if (!a.policy.continuous || a.policy.obs_dim != 3 || a.policy.act_dim != 1) { set_error("aur_rollout: Pendulum needs obs 3, 1 continuous action"); return AUR_ERR_ARG; }
    if (a.wrappers && !a.env.norm) { set_error("aur_rollout: wrappers need env.norm"); return AUR_ERR_ARG; }
  } else {
    set_error("aur_rollout: unknown env_kind %d", a.env_kind); return AUR_ERR_UNSUPPORTED;
  }
  RolloutDev d = to_dev(a);
  cudaStream_t s = (cudaStream_t)stream;
  const int sms = sm_count();
  // `--hidden_dim 128` (two layers, widths <= 4) on the envs the tensor-core rollout knows: the same two kernels as the
  // 64-wide headline shape, operand tiles two K atoms wide
  if (a.policy.hidden_dim == 128 && a.policy.num_layers == 2 && a.policy.obs_dim <= POL_IN_PAD && a.policy.act_dim <= POL_OUT_MAX &&
      rollout_impl() == 1 && (a.env_kind == AUR_ENV_CARTPOLE || pend || a.env_kind == AUR_ENV_MOUNTAINCAR)) {
    if ((rc = launch_rollout_tc(d, a.env_kind, 128, s))) return rc;
    const float* critic = a.params + net_param_count(a.policy.obs_dim, 128, 2, a.policy.act_dim);
    if ((rc = launch_critic_values_tc(critic, a.policy.obs_dim, 128, a.obs_buf, (long long)a.T * a.N, a.val_buf, s))) return rc;
    if (a.next_value && (rc = launch_critic_values_tc(critic, a.policy.obs_dim, 128, a.next_obs, a.N, a.next_value, s))) return rc;
    return 0;
  }
  // the other wide shapes (256 units; 128 units with more layers): the actor layer by layer over all envs each step
  if (rollout_impl() == 1 && rollout_wide_eligible(a.policy, a.env_kind)) return launch_rollout_wide(d, a.policy, a.env_kind, s);
  if (!fits_compiled_kernel(a.policy)) {
    // runtime-width policy: one env per thread, both nets in the sequential kernel
    if (((uintptr_t)a.params & 15) != 0) { set_error("aur_rollout: params must be 16-byte aligned"); return AUR_ERR_ARG; }
    int block = round_up((int)((a.N + sms - 1) / sms < 256 ? (a.N + sms - 1) / sms : 256), 32);
    if (block < 64) block = 64;
    const size_t smem = dyn_launch_shape(a.policy, block, d.dyn_smem);
    const long long grid = (a.N + block - 1) / block;
#define AUR_LAUNCH_DYN(ENVT)                                                             \
  do {                                                                                   \
    if ((rc = launch_cfg(rollout_kernel<ENVT, 0, 1, true>, smem))) return rc;            \
    rollout_kernel<ENVT, 0, 1, true><<<(unsigned)grid, block, smem, s>>>(d);             \
  } while (0)
    if (pend) AUR_LAUNCH_DYN(Pendulum);
    else if (a.env_kind == AUR_ENV_MOUNTAINCAR) AUR_LAUNCH_DYN(MountainCar);
    else if (a.env_kind == AUR_ENV_ACROBOT) AUR_LAUNCH_DYN(Acrobot);
    else if (a.env_kind == AUR_ENV_MOUNTAINCAR_CONT) AUR_LAUNCH_DYN(MountainCarContinuous);
    else AUR_LAUNCH_DYN(CartPole);
#undef AUR_LAUNCH_DYN
    AUR_LAUNCH_OK("rollout_kernel (runtime width)");
    return 0;
  }
  const bool two = a.env_kind == AUR_ENV_CARTPOLE && a.policy.num_layers <= 2 && a.N >= 2LL * 32 * sms;   // E = 2 needs enough envs to fill the chip
  const long long threads_needed = two ? (a.N + 1) / 2 : a.N;
  int block = round_up((int)((threads_needed + sms - 1) / sms < 256 ? (threads_needed + sms - 1) / sms : 256), 32);
  if (block < 64) block = 64;
  const long long grid = (threads_needed + block - 1) / block;
  const size_t smem = policy_smem_bytes(a.policy, block, a.policy.num_layers >= 3);
  // hidden 64 / 2 layers: the critic leaves the sequential kernel and runs as one batched tensor-core pass afterwards
  const bool split_critic = a.policy.num_layers == 2;
#define AUR_LAUNCH_ROLLOUT(ENVT, EE)                                                                   \
  do {                                                                                                 \
    if (split_critic) {                                                                                \
      if ((rc = launch_cfg(rollout_kernel<ENVT, 64, EE, false>, smem))) return rc;                     \
      rollout_kernel<ENVT, 64, EE, false><<<(unsigned)grid, block, smem, s>>>(d);                      \
    } else {                                                                                           \
      if ((rc = launch_cfg(rollout_kernel<ENVT, 64, EE, true>, smem))) return rc;                      \
      rollout_kernel<ENVT, 64, EE, true><<<(unsigned)grid, block, smem, s>>>(d);                       \
    }                                                                                                  \
  } while (0)
  const bool mcar = a.env_kind == AUR_ENV_MOUNTAINCAR, mcc = a.env_kind == AUR_ENV_MOUNTAINCAR_CONT;
  if (split_critic && rollout_impl() == 1 && !mcc) {
    if ((rc = launch_rollout_tc(d, a.env_kind, 64, s))) return rc;     // actor hidden layer on tcgen05 (rollout_tc.cu)
  } else {
    if (pend) AUR_LAUNCH_ROLLOUT(Pendulum, 1);
    else if (mcc) AUR_LAUNCH_ROLLOUT(MountainCarContinuous, 1);
    else if (mcar) AUR_LAUNCH_ROLLOUT(MountainCar, 1);
    else if (two) AUR_LAUNCH_ROLLOUT(CartPole, 2);
    else AUR_LAUNCH_ROLLOUT(CartPole, 1);
    AUR_LAUNCH_OK("rollout_kernel");
  }
#undef AUR_LAUNCH_ROLLOUT
  if (split_critic) {
    const float* critic = a.params + net_param_count(a.policy.obs_dim, 64, 2, a.policy.act_dim);
    if ((rc = launch_critic_values_tc(critic, a.policy.obs_dim, 64, a.obs_buf, (long long)a.T * a.N, a.val_buf, s))) return rc;
    if (a.next_value && (rc = launch_critic_values_tc(critic, a.policy.obs_dim, 64, a.next_obs, a.N, a.next_value, s))) return rc;
  }
  return 0;
}

namespace aur {
int check_pop(const aur_pop_desc* pop, const char* who);                    // update.cu
int check_pop_policy(const aur_policy_desc& p, const char* who);
int launch_rollout_tc_pop(const RolloutDev& d, int env_kind, int K, cudaStream_t s);   // rollout_tc.cu
int launch_critic_values_tc_pop(const float* critic, int obs_dim, const float* obs, long long segs, int K, long long n_member,
                                long long P, float* out, cudaStream_t s);   // values_tc.cu
}  // namespace aur

extern "C" int aur_pop_rollout(const aur_pop_desc* pop, const aur_rollout_args* args, void* stream) {
  using namespace aur;
  int rc = check_pop(pop, "aur_pop_rollout");
  if (rc) return rc;
  if (!args) { set_error("aur_pop_rollout: null args"); return AUR_ERR_ARG; }
  const aur_rollout_args& a = *args;
  if ((rc = check_pop_policy(a.policy, "aur_pop_rollout"))) return rc;
  const int ek = a.env_kind;
  if (ek != AUR_ENV_CARTPOLE && ek != AUR_ENV_PENDULUM && ek != AUR_ENV_MOUNTAINCAR) {
    set_error("aur_pop_rollout: env_kind %d has no population kernel (CartPole-v1, Pendulum-v1, MountainCar-v0); no fallback", ek);
    return AUR_ERR_UNSUPPORTED;
  }
  const bool cont = ek == AUR_ENV_PENDULUM;
  const int want_obs = ek == AUR_ENV_CARTPOLE ? 4 : (cont ? 3 : 2), want_act = ek == AUR_ENV_CARTPOLE ? 2 : (cont ? 1 : 3);
  if ((a.policy.continuous != 0) != cont || a.policy.obs_dim != want_obs || a.policy.act_dim != want_act) {
    set_error("aur_pop_rollout: env_kind %d needs obs %d, %d %s actions", ek, want_obs, want_act, cont ? "continuous" : "discrete");
    return AUR_ERR_ARG;
  }
  if (a.T < 1 || a.N != (int64_t)pop->K * pop->n_member) {
    set_error("aur_pop_rollout: need T >= 1 and N = K * n_member (got T %d, N %lld, K %d, n_member %lld)", a.T, (long long)a.N, pop->K,
              (long long)pop->n_member);
    return AUR_ERR_ARG;
  }
  if (!a.params || !a.obs_buf || !a.act_buf || !a.logp_buf || !a.val_buf || !a.rew_buf || !a.done_buf || !a.next_obs ||
      !a.next_done || !a.env.phys || !a.env.pcg || !a.env.elapsed || !a.env.ep_return || !a.env.ep_length ||
      (cont && a.wrappers && !a.env.norm) || a.log.entries || a.log.count) {
    set_error("aur_pop_rollout: null buffer, wrappers without env.norm, or a full episode log (not supported for populations)");
    return AUR_ERR_ARG;
  }
  RolloutDev d = to_dev(a);
  d.n_member = pop->n_member; d.pop_seeds = pop->seeds; d.pop_P = policy_param_count(a.policy);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = launch_rollout_tc_pop(d, ek, pop->K, s))) return rc;
  const float* critic = a.params + net_param_count(a.policy.obs_dim, 64, 2, a.policy.act_dim);
  if ((rc = launch_critic_values_tc_pop(critic, a.policy.obs_dim, a.obs_buf, a.T, pop->K, pop->n_member, d.pop_P, a.val_buf, s))) return rc;
  if (a.next_value &&
      (rc = launch_critic_values_tc_pop(critic, a.policy.obs_dim, a.next_obs, 1, pop->K, pop->n_member, d.pop_P, a.next_value, s)))
    return rc;
  return 0;
}

extern "C" int aur_policy_evaluate(const aur_policy_desc* desc, const float* params, int64_t B, const float* obs,
                                   const float* actions_in, uint64_t seed, uint64_t row0, uint64_t step,
                                   float* actions_out, float* logp_out, float* entropy_out, float* value_out,
                                   void* stream) {
  return aur_policy_act(desc, params, B, obs, actions_in, 0, seed, row0, step, actions_out, logp_out, entropy_out, value_out, stream);
}

extern "C" int aur_policy_act(const aur_policy_desc* desc, const float* params, int64_t B, const float* obs,
                              const float* actions_in, int32_t greedy, uint64_t seed, uint64_t row0, uint64_t step,
                              float* actions_out, float* logp_out, float* entropy_out, float* value_out, void* stream) {
  using namespace aur;
  if (!desc || !params || B < 0 || (B > 0 && !obs)) { set_error("aur_policy_evaluate: bad arguments"); return AUR_ERR_ARG; }
  if (greedy && actions_in) { set_error("aur_policy_act: greedy and actions_in are mutually exclusive"); return AUR_ERR_ARG; }
  if (B == 0) return 0;
  int rc = check_policy(*desc, "aur_policy_evaluate", DYN_IO);
  if (rc) return rc;
  RolloutDev d{};
  d.obs_dim = desc->obs_dim; d.act_dim = desc->act_dim; d.nl = desc->num_layers; d.continuous = desc->continuous;
  d.hid = desc->hidden_dim; d.dyn_smem = 0;
  d.params = params; d.actions_in = actions_in; d.seed = seed; d.greedy = greedy ? 1 : 0;
  if (!fits_compiled_kernel(*desc)) {
    if (((uintptr_t)params & 15) != 0) { set_error("aur_policy_evaluate: params must be 16-byte aligned"); return AUR_ERR_ARG; }
    int block = 128;
    const size_t smem = dyn_launch_shape(*desc, block, d.dyn_smem);
    long long grid = (B + block - 1) / block;
    if (grid > 4LL * sm_count()) grid = 4LL * sm_count();
    if ((rc = launch_cfg(policy_evaluate_dyn_kernel, smem))) return rc;
    policy_evaluate_dyn_kernel<<<(unsigned)grid, block, smem, (cudaStream_t)stream>>>(d, (long long)B, obs, row0, step, actions_out,
                                                                                    logp_out, entropy_out, value_out);
    AUR_LAUNCH_OK("policy_evaluate_dyn_kernel");
    return 0;
  }
  const int block = 128;
  long long grid = (B + block - 1) / block;
  if (grid > 4LL * sm_count()) grid = 4LL * sm_count();
  const size_t smem = policy_smem_bytes(*desc, block, desc->num_layers >= 3);
  if ((rc = launch_cfg(policy_evaluate_kernel<64>, smem))) return rc;
  policy_evaluate_kernel<64><<<(unsigned)grid, block, smem, (cudaStream_t)stream>>>(d, (long long)B, obs, row0, step,
                                                                                  actions_out, logp_out, entropy_out, value_out);
  AUR_LAUNCH_OK("policy_evaluate_kernel");
  return 0;
}
