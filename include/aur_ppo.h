/* aur_ppo.h -- C ABI of libaurppo.so, the sm_100a implementation of the PPO hot
 * path of biirving/aur_ppo (rollout step -> GAE -> minibatch update).
 *
 * The reference has no FFI of its own: its boundary is the Python surface
 * (src/run_ppo.py:14-41 flags, `ppo(params).train()` src/ppo.py:44,169,
 * `actor_critic.evaluate/value` src/models/actor_critic.py:31-51).  Each entry
 * point below replaces the stock-PyTorch/gym code at the cited reference lines;
 * aur_ppo_b200/ (the Python host mirror) binds them with ctypes, and
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.
 *   - All data pointers are DEVICE pointers into caller-owned memory (torch
 *     tensors); `stream` is a cudaStream_t passed as void* (NULL = default).
 *     The caller sets the current CUDA device before calling.
 *   - Return 0 on success, <0 on error: AUR_ERR_ARG (bad argument),
 *     AUR_ERR_UNSUPPORTED (shape outside the compiled kernels -- there is NO
 *     CPU or library fallback), or -(1000 + cudaError_t).  aur_last_error()
 *     gives a thread-local human-readable message.
 *   - Nothing is allocated that the caller must free; functions are
 *     re-entrant per (device, stream) and launch asynchronously.
 */
#ifndef AUR_PPO_H
#define AUR_PPO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AUR_ABI_VERSION 3   /* 2: operand-plane precision modes, aur_update_args.mom_index / mom_seq, library-owned tickets;
                               3: aur_ppo_update_set_wide (layer-wise tensor-core update for hidden 128 / 256) */
#define AUR_ERR_ARG (-1)
#define AUR_ERR_UNSUPPORTED (-2)

#define AUR_ENV_CARTPOLE 0 /* gym CartPole-v1 */
#define AUR_ENV_PENDULUM 1 /* gym Pendulum-v1 */
#define AUR_ENV_MOUNTAINCAR 2 /* gym MountainCar-v0 (discrete, 3 actions, obs 2) */
#define AUR_ENV_MOUNTAINCAR_CONT 4 /* gym MountainCarContinuous-v0 (1 continuous action, obs 2, 999 steps) */
#define AUR_ENV_ACROBOT 3     /* gym Acrobot-v1 (discrete, 3 actions, obs 6; runtime-width policy path) */

int aur_abi_version(void);
const char* aur_last_error(void);
/* number of this library's kernels launched by the calling thread since the last reset */
int64_t aur_launch_count(void);
void aur_launch_count_reset(void);

/* ---------------------------------------------------------------- GAE ----
 * Replaces ppo.advantages -> run_gae (src/ppo.py:125-142, use_gae != 0) or
 * normal_advantage (src/ppo.py:145-157, use_gae == 0): the reverse scan over
 * the [T,N] rollout buffers with done masking, then returns = adv + values
 * (GAE) / adv = returns - values (Monte-Carlo).
 *
 *   rewards, values, terminals : [T,N] fp32 row-major (torch_buffer layout,
 *                                src/ppo.py:26-29); terminals[t] is the done
 *                                flag that arrived WITH obs[t] (ppo.py:204)
 *   next_value, next_done      : [N] fp32 (critic(next_obs), ppo.py:161)
 *   adv_out, ret_out           : [T,N] fp32
 *   gamma, gae_lambda          : Python floats of the reference; converted
 *                                exactly as torch does for tensor*scalar
 *                                ((float)gamma, (float)(gamma*gae_lambda))
 * Arithmetic is fp32, sequential in t, one rounding per reference operation
 * (no FMA contraction): results are bit-identical to the reference's torch
 * CPU loop.  T >= 1, N >= 1; N == 0 or T == 0 is a no-op returning 0. */
int aur_gae_f32(int32_t T, int64_t N, const float* rewards, const float* values, const float* terminals,
                const float* next_value, const float* next_done, double gamma, double gae_lambda,
                int32_t use_gae, float* adv_out, float* ret_out, void* stream);

/* Which kernel aur_gae_f32 would pick for this shape/alignment: 1 = bulk-async
 * (TMA 1-D) pipelined kernel, 0 = plain column kernel.  For tests/bench. */
int aur_gae_kernel_kind(int32_t T, int64_t N, const float* rewards, const float* values, const float* terminals,
                        const float* adv_out, const float* ret_out);

/* ------------------------------------------------------------- policy ----
 * The reference's actor_critic (src/models/actor_critic.py:8-26): two
 * independent MLPs Linear(obs,H)-Tanh-[Linear(H,H)-Tanh]*(num_layers-1)-
 * Linear(H,out) (src/nets/nets.py:19-53), out = act_dim for the actor and 1
 * for the critic, plus actor_logstd[act_dim] when continuous.
 *
 * Flat parameter buffer (fp32), the order every kernel reads and Adam updates:
 *   actor : W0[H,obs] b0[H]  W1[H,H] b1[H] ... Wout[act,H] bout[act]
 *   critic: W0[H,obs] b0[H]  W1[H,H] b1[H] ... Wout[1,H]   bout[1]
 *   actor_logstd[act]                       (continuous only)
 * every W row-major [out,in] exactly as torch.nn.Linear.weight. */
typedef struct {
  int32_t obs_dim;     /* 1..8 (4 CartPole, 3 Pendulum, 6 Acrobot); widths <= 4 with 64 hidden units run the specialised kernels */
  int32_t act_dim;     /* number of discrete actions, or action dimensions if continuous; 1..8 */
  int32_t hidden_dim;  /* multiples of 4 in 4..256; 64 (the reference default) runs the register / tcgen05 kernels,
                          other widths the runtime-width forward and the shape-generic update kernel */
  int32_t num_layers;  /* number of hidden layers (the reference's num_layers), 1..16; the update keeps all layers of a
                          sample tile in shared memory, which bounds hidden_dim * num_layers (AUR_ERR_UNSUPPORTED beyond) */
  int32_t continuous;  /* 0 Categorical, 1 diagonal Normal with state-independent std */
} aur_policy_desc;

int64_t aur_policy_param_count(const aur_policy_desc* desc);

/* Replaces actor_critic.evaluate / .value (src/models/actor_critic.py:31-51) for a
 * batch of B observations, no grad: obs [B,obs_dim]; actions_in nullable
 * ([B] action index as fp32 if discrete, [B,act_dim] if continuous) -- when NULL
 * actions are sampled from the Philox stream (seed, row0 + b, step);
 * outputs (each nullable): actions [B(,act_dim)] fp32, logp [B], entropy [B], value [B]. */
int aur_policy_evaluate(const aur_policy_desc* desc, const float* params, int64_t B, const float* obs,
                        const float* actions_in, uint64_t seed, uint64_t row0, uint64_t step, float* actions_out,
                        float* logp_out, float* entropy_out, float* value_out, void* stream);

/* The same with a `greedy` switch for checkpoint evaluation (src/test.py:17-61 plays a saved policy; its
 * `agent.act(state)` samples, greedy != 0 takes torch.argmax of the logits / the Normal mean instead).
 * greedy and actions_in are mutually exclusive. */
int aur_policy_act(const aur_policy_desc* desc, const float* params, int64_t B, const float* obs,
                   const float* actions_in, int32_t greedy, uint64_t seed, uint64_t row0, uint64_t step,
                   float* actions_out, float* logp_out, float* entropy_out, float* value_out, void* stream);

/* ---------------------------------------------------------------- envs ----
 * Device-resident vector env: replaces gym.vector.SyncVectorEnv over the
 * make_env thunks (src/ppo.py:66-68,85-99): gym CartPole-v1 / Pendulum-v1
 * dynamics in fp64, TimeLimit (500 / 200), RecordEpisodeStatistics, autoreset,
 * and -- when `wrappers` -- the continuous stack ClipAction, NormalizeObservation,
 * clip +-10, NormalizeReward(gamma), clip +-10 (src/ppo.py:92-97), per env.
 * All arrays are struct-of-arrays over the N envs this GPU owns. */
typedef struct {
  double* phys;       /* [S][N] fp64: CartPole x, x_dot, theta, theta_dot; Pendulum theta, theta_dot; MountainCar position, velocity; Acrobot theta1, theta2, dtheta1, dtheta2 */
  uint64_t* pcg;      /* [4][N] PCG64 state_hi, state_lo, inc_hi, inc_lo (np.random.PCG64(SeedSequence(seed_i))) */
  int32_t* elapsed;   /* [N] TimeLimit step counter */
  float* ep_return;   /* [N] RecordEpisodeStatistics accumulator (fp32 as in gym) */
  int32_t* ep_length; /* [N] */
  double* norm;       /* [2 D + 5][N] or NULL (D = obs_dim; Pendulum: 11 rows): obs mean[D], var[D], count; return-rms mean, var, count; return acc */
} aur_env_state;

typedef struct {
  int32_t step;   /* global step index (step0 + t) at which the episode ended */
  int32_t env;    /* global env id */
  float ret;      /* info["episode"]["r"] */
  int32_t len;    /* info["episode"]["l"] */
} aur_episode;

typedef struct {
  aur_episode* entries; /* [capacity] or NULL: full log of finished episodes (tests, small runs) */
  uint32_t* count;      /* device counter of finished episodes (may exceed capacity; extras are dropped) */
  uint32_t capacity;
  uint32_t _pad;
  /* [T] or NULL, caller-initialised to all ones: per rollout step, the FIRST finished env in env
   * order -- what the reference logs (ppo.py:114-122 breaks after the first final_info item).
   * Packed (local_env << 42) | (length << 32) | float_bits(return), merged with atomicMin (length < 1024). */
  unsigned long long* first_finished;
  double* totals;       /* [3] or NULL: += episodes, sum of returns, sum of lengths */
} aur_episode_log;

/* envs.reset(seed=[...]) (src/ppo.py:188): `st.pcg` must already hold each env's seeded PCG64
 * state; draws the initial state from it, zeroes counters / wrapper statistics and writes the
 * first observation [N,obs_dim] and next_done = 0 [N]. */
int aur_env_reset(int32_t env_kind, int64_t N, int32_t wrappers, const aur_env_state* st, float* obs_out,
                  float* done_out, void* stream);

/* ------------------------------------------------------------- rollout ----
 * Replaces the rollout loop src/ppo.py:201-205 + rewards_to_go src/ppo.py:103-123 for T
 * steps over the N envs of this GPU in ONE kernel: per step store obs/done, run both MLPs,
 * sample (or take actions_in), store action/logp/value, step the env in fp64, store the
 * reward, autoreset.  Buffers are the reference's torch_buffer (src/ppo.py:20-29):
 *   obs_buf [T,N,obs_dim], act_buf [T,N] (discrete, fp32 index) or [T,N,act_dim],
 *   logp_buf / val_buf / rew_buf / done_buf [T,N]; done_buf[t] is the flag that arrived
 *   with obs[t] (ppo.py:204) and carries `terminated` only (ppo.py:110 drops `truncated`).
 * next_obs [N,obs_dim] and next_done [N] are in/out; next_value [N] (nullable) receives
 * critic(next_obs) after the last step (ppo.py:161).
 * Sampling: Philox4x32-10, key = seed, counter = (env_id0 + n, step0 + t): independent of how
 * envs are sharded over GPUs.  actions_in (nullable, same layout as act_buf) replays given
 * actions instead (parity mode). */
typedef struct {
  int32_t env_kind;
  int32_t wrappers;
  int64_t N;
  int32_t T;
  int32_t _pad;
  aur_policy_desc policy;
  const float* params;
  aur_env_state env;
  float* obs_buf;
  float* act_buf;
  float* logp_buf;
  float* val_buf;
  float* rew_buf;
  float* done_buf;
  float* next_obs;
  float* next_done;
  float* next_value;
  const float* actions_in;
  uint64_t seed;
  uint64_t step0;
  uint64_t env_id0;
  aur_episode_log log;
  double gamma; /* NormalizeReward discount (the wrapper's own default 0.99) */
} aur_rollout_args;

int aur_rollout(const aur_rollout_args* args, void* stream);

/* Kernel behind aur_rollout: 1 (default) = tensor cores - hidden 64 or 128 with 2 layers: the fused rollout_tc_kernel (actor
 * hidden layer on tcgen05) followed by the batched tensor-core value pass; hidden 256, or 128 with more layers (obs_dim <= 4,
 * act_dim <= 4, CartPole / Pendulum / MountainCar): the actor layer by layer over all envs every step (rollout_wide.cu), which
 * keeps its activation scratch (about 1.1 GB at 256 units) in a library-owned, grow-only allocation per (device, stream) because
 * this entry point has no workspace argument - make the first call of a shape outside a CUDA-graph capture;
 * 0 = SIMT rollout_kernel (also the path of every other width / depth).  AUR_ROLLOUT_IMPL=simt|tc sets the initial choice. */
int aur_rollout_set_impl(int impl);
int aur_rollout_get_impl(void);

/* -------------------------------------------------------------- update ----
 * Replaces one minibatch step of src/ppo.py:220-269: gather of the shuffled indices,
 * actor_critic.evaluate with grad, ratio / KL / clip-fraction diagnostics, minibatch
 * advantage normalisation (unbiased std + 1e-8), clipped surrogate, clipped value loss,
 * entropy bonus, backward, clip_grad_norm_(all params), Adam(eps=1e-5).
 *
 * Split in phases so that the one exchange of a data-parallel run (an allreduce of the
 * packed gradient buffer, and of the three advantage moments) sits between them:
 *   aur_ppo_adv_moments   sum / sum of squares / count of advantages[idx]      (fp64)
 *   aur_ppo_update_grad   gather + forward + loss + backward, reduced over the minibatch
 *                         into grads_out = [P gradient sums | 16 statistic sums]
 *   aur_ppo_update_apply  grad-norm clip + Adam on the flat parameter buffer, statistics
 * The actor and the critic are independent MLPs with separable losses, so half of the
 * CTAs train each net.  Gradients are reduced in a fixed order (deterministic). */
/* Data-parallel context (one process per GPU, ranks of ONE node): the exchange area of every rank, mapped into
 * this process with aur_dp_alloc / aur_dp_open.  With world > 1 the update kernels do the gradient all-reduce
 * themselves over NVLink peer memory: aur_ppo_adv_moments_dp pushes the local advantage moments to every rank,
 * aur_ppo_update_grad waits for them inside the gradient kernel and pushes its packed [grads | stats] sums,
 * aur_ppo_update_apply_dp gathers the world's sums in rank order (bit-identical on every rank) and applies
 * clip + Adam.  seq is the 1-based minibatch counter, the same on every rank.  NULL / world <= 1: single GPU.
 * This replaces the per-minibatch allreduce a multi-GPU port of ppo.py:266-269 would issue. */
#define AUR_DP_MAX_RANKS 16
#define AUR_DP_HANDLE_BYTES 64
typedef struct {
  int32_t world, rank;
  void* peer[AUR_DP_MAX_RANKS];   /* peer[r]: exchange area of rank r (peer[rank] = own allocation) */
} aur_dp_ctx;
int64_t aur_dp_area_bytes(const aur_policy_desc* desc);
int aur_dp_alloc(int64_t bytes, void** area_out, void* ipc_handle_out /* AUR_DP_HANDLE_BYTES */);
int aur_dp_open(const void* ipc_handle, void** area_out);
int aur_dp_close(void* area);
int aur_dp_free(void* area);
int aur_dp_status(const void* area, void* stream);   /* 0 ok, 1 = a kernel timed out waiting for a peer */
/* Time this rank's kernels spent waiting for peers since the last reset, measured on the device: out6 (host) = {spin ns on
 * gradient flags summed over the spinning threads, number of spins, the same two for moment flags, WALL ns the clip + Adam
 * kernels stood still until every peer's gradients had arrived, number of those launches}; reset != 0 zeroes the counters.
 * Synchronises `stream`. */
int aur_dp_wait_stats(void* area, uint64_t* out6, int32_t reset, void* stream);

typedef struct {
  aur_policy_desc policy;
  int32_t norm_adv;          /* ppo.py:238 */
  int32_t clip_vloss;        /* ppo.py:250; 0 reproduces the reference's b_values quirk (ppo.py:261) */
  int32_t mom_index;         /* which entry of an aur_ppo_adv_moments_multi launch this minibatch is (with dp + mom_seq) */
  int64_t m_local;           /* samples of this GPU's share of the minibatch */
  int64_t m_total;           /* samples of the whole minibatch (means divide by this) */
  const int32_t* idx;        /* [m_local] row indices into the flattened buffers, or NULL: idx_offset + i */
  int64_t idx_offset;
  const float* obs;          /* b_obs        [B,obs_dim]            (ppo.py:33) */
  const float* actions;      /* b_actions    [B] or [B,act_dim]     (ppo.py:35) */
  const float* logprobs;     /* b_logprobs   [B] */
  const float* advantages;   /* b_advantages [B] */
  const float* returns;      /* b_returns    [B] */
  const float* values;       /* b_values     [B] */
  const float* params;       /* flat parameter buffer */
  float clip_coeff, entropy_coeff, value_coeff, _pad2;
  const double* adv_moments; /* [3] device: sum, sum of squares, count over the WHOLE minibatch; NULL iff !norm_adv */
  float* workspace;          /* >= aur_ppo_update_workspace_bytes(); contents need NOT be initialised (the last-CTA tickets of
                                the reductions live in a library-owned allocation per (device, stream)) */
  float* grads_out;          /* [P + 16] */
  const aur_dp_ctx* dp;      /* NULL: single GPU */
  uint32_t dp_seq;
  uint32_t mom_seq;          /* != 0: the advantage moments were exchanged AHEAD by aur_ppo_adv_moments_multi(mom_seq): the
                                gradient kernel reads entry mom_index of that exchange instead of waiting for a per-minibatch one */
  const float* rec_actor;    /* optional: [B,8] records of aur_ppo_pack_records (both or neither); the kernel then */
  const float* rec_critic;   /* gathers one 32-byte sector per sample and net instead of one per array */
} aur_update_args;

#define AUR_STAT_POLICY_LOSS 0   /* sums over samples; aur_ppo_update_apply turns them into means */
#define AUR_STAT_VALUE_LOSS 1
#define AUR_STAT_ENTROPY 2
#define AUR_STAT_OLD_APPROX_KL 3
#define AUR_STAT_APPROX_KL 4
#define AUR_STAT_CLIPFRAC 5
#define AUR_STAT_GRAD_NORM 6     /* written by aur_ppo_update_apply (pre-clip total norm) */
#define AUR_STAT_LOSS 7          /* policy - ent_c * entropy + vf_c * value */
#define AUR_NUM_STATS 16

/* Replaces `np.random.shuffle(b_inds)` (ppo.py:214-215): out[i] = pi(i), pi a keyed pseudo-random bijection of
 * [0, n), n < 2^31 (Feistel network + cycle walking; keys from Philox4x32-10(seed, stream_id)).  Use a new
 * stream_id per epoch (and per rank).  Restated bit for bit in oracle/ppo_ref.py::feistel_shuffle. */
int aur_shuffle_indices(int64_t n, uint64_t seed, uint64_t stream_id, int32_t* out, void* stream);

/* Optional gather-friendly copy of the flattened batch (ppo.py:208-212 `b_obs ... b_values`): two [B,8] fp32 record
 * arrays, 32-byte aligned.  actor: obs[0..3] | action[0], logprob, advantage, action[1];  critic: obs[0..3] | return,
 * value, 0, 0.  action_width = 1 (discrete index or one continuous dim) or 2.  Pass them in aur_update_args. */
int aur_ppo_pack_records(int64_t B, int32_t obs_dim, int32_t action_width, const float* obs, const float* actions,
                         const float* logprobs, const float* advantages, const float* returns, const float* values,
                         float* rec_actor, float* rec_critic, void* stream);

int64_t aur_ppo_update_workspace_bytes(const aur_policy_desc* desc);

int aur_ppo_adv_moments(int64_t m, const int32_t* idx, int64_t idx_offset, const float* advantages,
                        double* moments_out, float* workspace, void* stream);

int aur_ppo_adv_moments_dp(int64_t m, const int32_t* idx, int64_t idx_offset, const float* advantages,
                           double* moments_out, float* workspace, const aur_dp_ctx* dp, uint32_t seq, void* stream);

/* Advantage moments of ALL the minibatches of an iteration in one launch: the permutations of every epoch do not depend
 * on the parameters, so they (and these moments) can be produced right after GAE.  idx: n_mb consecutive index lists of m
 * rows each (idx_stride apart).  moments_out [n_mb][3] (sum, sum of squares, count).  Data-parallel: the local moments of
 * all n_mb minibatches are pushed to every rank once, under the iteration counter mom_seq (1-based, the same on every rank) -
 * one rendezvous per iteration instead of one per minibatch; aur_update_args.mom_seq / mom_index select an entry.
 * n_mb <= AUR_DP_MAX_MINIBATCHES.  Replaces `mb_advantages.mean() / .std()` of ppo.py:239 for the whole update loop. */
#define AUR_DP_MAX_MINIBATCHES 512
int aur_ppo_adv_moments_multi(int32_t n_mb, int64_t m, const int32_t* idx, int64_t idx_stride, const float* advantages,
                              double* moments_out, float* workspace, const aur_dp_ctx* dp, uint32_t mom_seq, void* stream);

int aur_ppo_update_grad(const aur_update_args* args, void* stream);

/* Kernel behind aur_ppo_update_grad for the 64 x 2 shape (widths <= 4): 1 = tcgen05 (bf16 two-term split operands,
 * fp32 TMEM accumulators; the default), 2 = the same with four threads per sample, 0 = SIMT fp32 (independent
 * implementation kept as a cross-check), 3 = the shape-generic SIMT kernel (update_generic.cu).  Every other
 * shape always runs kernel 3.  All are CUDA; there is no CPU path.  AUR_UPDATE_IMPL=simt|tc|tc4|generic sets the
 * initial choice. */
int aur_ppo_update_set_impl(int impl);
int aur_ppo_update_get_impl(void);
/* `--hidden_dim` 128 / 256 with `--num_layers` >= 2 (src/run_ppo.py:36,38; obs_dim <= 8, act_dim <= 4): 1 (default) = the
 * layer-wise tensor-core path (update_wide.cu: every H x H contraction of forward, backward-data and weight gradient is a
 * tcgen05 GEMM over two-plane bf16 operands, activations of a 262,144-sample sub-batch staged in the workspace), 0 = the
 * shape-generic SIMT kernel (kept as the cross-check).  AUR_UPDATE_WIDE=0|1 sets the initial choice. */
int aur_ppo_update_set_wide(int on);
int aur_ppo_update_get_wide(void);

/* params / adam_m / adam_v: [P] fp32 updated in place (torch.optim.Adam single-tensor math, no
 * weight decay, no amsgrad).  step is the 1-based Adam step count.  stats_out [AUR_NUM_STATS]
 * (nullable) receives the minibatch means; entropy_coeff/value_coeff only enter stats_out[LOSS]. */
int aur_ppo_update_apply(const aur_policy_desc* desc, float* params, float* grads_packed, float* adam_m,
                         float* adam_v, double lr, double beta1, double beta2, double eps, int64_t step,
                         double max_grad_norm, int64_t m_total, double entropy_coeff, double value_coeff,
                         float* stats_out, void* stream);
/* Data-parallel form: first replaces grads_packed by the sum over all ranks (gathered from the exchange area). */
int aur_ppo_update_apply_dp(const aur_policy_desc* desc, float* params, float* grads_packed, float* adam_m,
                            float* adam_v, double lr, double beta1, double beta2, double eps, int64_t step,
                            double max_grad_norm, int64_t m_total, double entropy_coeff, double value_coeff,
                            float* stats_out, const aur_dp_ctx* dp, uint32_t seq, void* stream);

/* ---------------------------------------------------------- populations ----
 * K independent PPO runs ("members") trained in shared launches on one GPU: the seed / hyper-parameter sweeps of the
 * reference (src/grid_search.sh, src/robot.sh; `--trials`, src/run_ppo.py:41) as one set of kernels instead of K processes.
 * Members share the policy shape, the env and every size (num_envs = n_member, num_steps, minibatches, epochs); each has its
 * own parameters, Adam moments, Philox / shuffle key and the hyper-parameters of aur_pop_hparams.  Member k computes exactly
 * (bit for bit) what the single-run entry points compute for a run of n_member envs with philox_seed = shuffle_seed =
 * seeds[k] started from the same parameters: the same kernels run with per-member operands, the update splits each member's
 * minibatch over min(#SM, tiles) CTAs per net exactly as a single run does, and every fp64 reduction keeps its single-run order.
 *
 * Scope: hidden 64, 2 layers, obs_dim <= 4, act_dim <= 4 (act_dim <= 2 if continuous), CartPole-v1, Pendulum-v1 (with or
 * without the wrapper stack) and MountainCar-v0, one GPU.  Anything else returns AUR_ERR_UNSUPPORTED; there is no fallback.
 * Populations always run the tensor-core kernels: aur_rollout_set_impl / aur_ppo_update_set_impl do not apply to them.
 *
 * Layout: the rollout buffers are the single-run buffers of N = K * n_member envs ([T][K * n_member], member k owns columns
 * k * n_member .. (k+1) * n_member - 1), so aur_gae_f32 and aur_ppo_pack_records run on them unchanged, as one launch each.
 * Per-member device arrays are stacked along a leading K axis (parameters [K][P], Adam moments [K][P], gradients
 * [K][P + 16], ...).  Last-CTA tickets are not used: the workspace needs no initialisation. */
typedef struct {
  int32_t K;               /* members, >= 1 */
  int32_t _pad;
  int64_t n_member;        /* envs per member, >= 1 (any value: a CTA never straddles two members) */
  const uint64_t* seeds;   /* [K] device: member k's Philox sampling key and shuffle key */
} aur_pop_desc;

/* One member's hyper-parameters (src/run_ppo.py:21-31 flags), a device table [K] written once. */
typedef struct {
  double learning_rate;    /* before the anneal factor: the step uses (float)((learning_rate * frac) / bias_correction1) */
  double entropy_coeff;
  double clip_coeff;
  double value_coeff;
  double max_grad_norm;
  double target_kl;        /* +inf: no early stop (the reference's None) */
} aur_pop_hparams;

/* Replaces the rollout loop (src/ppo.py:201-205) of every member in one launch of the fused tensor-core rollout kernel, grid
 * (ceil(n_member / 128), K), followed by the batched critic pass.  `args` is as for aur_rollout with N = K * n_member and:
 *   params       [K][P]: member k's flat parameter buffer at params + k * P
 *   seed         ignored: member k samples from Philox(key = pop->seeds[k], counter = (env_id0 + n, step0 + t)), n the
 *                member-local env index - the counters of a single run of n_member envs
 *   log          first_finished [K][T] (caller-initialised to all ones), totals [K][3] (or NULL); keys hold the member-local
 *                env index.  entries / count must be NULL.
 * Env state, next_obs / next_done / next_value and the buffers span all K * n_member columns.
 * AUR_ERR_UNSUPPORTED outside the population scope, AUR_ERR_ARG for bad pointers / sizes. */
int aur_pop_rollout(const aur_pop_desc* pop, const aur_rollout_args* args, void* stream);

/* `np.random.shuffle(b_inds)` (ppo.py:214-215) of `epochs` consecutive epochs for every member in one launch: member k's
 * epoch e is the permutation aur_shuffle_indices(T * n_member, pop->seeds[k], stream_id0 + e) of its local batch, each local
 * index j written as the GLOBAL row (j / n_member) * (K * n_member) + k * n_member + j % n_member of the population batch.
 * out: [K][epochs][T * n_member] int32.  T * n_member < 2^31, K * T * n_member < 2^31. */
int aur_pop_shuffle_indices(const aur_pop_desc* pop, int32_t T, int32_t epochs, uint64_t stream_id0, int32_t* out, void* stream);

/* aur_ppo_adv_moments_multi for every member (ppo.py:239 `mb_advantages.mean() / .std()` of the whole update loop): idx
 * [K][n_mb][m] global rows, moments_out [K][n_mb][3].  Each member is split over the CTAs a single run would use, and the
 * fp64 partials are combined in the single-run order.  Two launches, whatever K. */
int aur_pop_adv_moments_multi(const aur_pop_desc* pop, int32_t n_mb, int64_t m, const int32_t* idx, const float* advantages,
                              double* moments_out, float* workspace, void* stream);

typedef struct {
  aur_policy_desc policy;
  int32_t norm_adv;          /* ppo.py:238 */
  int32_t clip_vloss;        /* ppo.py:250 */
  int32_t mb_index;          /* minibatch j of the iteration: index list j and moments entry j of every member */
  int32_t n_mb;              /* minibatches per iteration (entries per member of idx / adv_moments) */
  int64_t m;                 /* samples per minibatch and member (means divide by this) */
  const int32_t* idx;        /* [K][n_mb][m] global rows (aur_pop_shuffle_indices) */
  const float* rec_actor;    /* [K * T * n_member][8] records of aur_ppo_pack_records over the population batch (required) */
  const float* rec_critic;
  const float* params;       /* [K][P] */
  const aur_pop_hparams* hparams;   /* [K] device */
  const double* adv_moments; /* [K][n_mb][3] (aur_pop_adv_moments_multi); NULL iff !norm_adv */
  const int32_t* active;     /* [K] device: members with 0 are skipped (target_kl, aur_pop_update_apply) */
  float* workspace;          /* >= aur_pop_update_workspace_bytes(); contents need not be initialised */
  float* grads_out;          /* [K][P + 16]: member k's [gradient sums | statistic sums] */
} aur_pop_update_args;

/* Workspace of aur_pop_adv_moments_multi / aur_pop_update_grad for K members, n_mb minibatches of m samples. */
int64_t aur_pop_update_workspace_bytes(const aur_pop_desc* pop, const aur_policy_desc* desc, int32_t n_mb, int64_t m);

/* aur_ppo_update_grad for one minibatch of every active member: gather + forward + loss + backward on the tensor cores, grid
 * (2 c, K) with c = min(#SM, ceil(m / 128)) CTAs per net (tile i on CTA i mod c, as a single run), then one fixed-order fp64
 * reduction per member that keeps the single-run quarter boundaries.  Two launches, whatever K. */
int aur_pop_update_grad(const aur_pop_desc* pop, const aur_pop_update_args* args, void* stream);

/* clip_grad_norm_ + Adam (ppo.py:266-269) for every active member, one CTA each.  Member k steps with lr = (float)(
 * (hparams[k].learning_rate * frac) / bc[s][0]), bc[s][1] = 1 - beta2^s under the sqrt, s = steps[k] + 1 its 1-based Adam step
 * (bc [bc_len][2] fp64, a host-computed table of 1 - beta1^s, 1 - beta2^s: the values aur_ppo_update_apply derives with host
 * pow), then steps[k] = s.  The caller keeps bc_len > the largest step any member can reach (at most the number of apply calls
 * made so far); a member whose next step has no table entry is NOT stepped (its parameters, moments and step count stay as
 * they are), so a short table shows as a step count that stops advancing.  stats_out [K][stats_rows][16]: row stats_row of member k receives its minibatch means.  epoch_end
 * != 0 (the last minibatch of an epoch): a member whose approx_kl exceeds hparams[k].target_kl is cleared in `active`
 * (ppo.py:271-273 `break`), so its later grad / apply work of the iteration is skipped and its step count stops.
 * params / adam_m / adam_v [K][P], grads [K][P + 16], steps [K] int64 device. */
int aur_pop_update_apply(const aur_pop_desc* pop, const aur_policy_desc* desc, const aur_pop_hparams* hparams, float* params,
                         const float* grads, float* adam_m, float* adam_v, int64_t* steps, int32_t* active, const double* bc,
                         int64_t bc_len, double frac, double beta1, double beta2, double eps, int64_t m_total,
                         float* stats_out, int32_t stats_rows, int32_t stats_row, int32_t epoch_end, void* stream);

/* ------------------------------------------------ population-based training ----
 * PBT (Jaderberg et al., 2017) between two population iterations, never inside one: the worst members copy the weights and
 * optimizer state of the best ones ("exploit"), then perturb the copied hyper-parameters ("explore").  Everything stays in
 * the population's stacked [K][...] device arrays; a round is three launches whatever K is (aur_pop_episode_fitness: one,
 * aur_pop_pbt_step: two).
 *
 * Decision rule of a round, from fitness[K] (fp64), a fraction q, factors down / up, a perturb mask over the six fields of
 * aur_pop_hparams (bit j = field j in declaration order), a 64-bit seed and the round number r (1, 2, ...):
 *   1. member k is ranked when fitness[k] is not NaN (+-inf are ranked); n_valid = the number of ranked members.
 *   2. order = the ranked members sorted by fitness, highest first; ties (-0.0 == +0.0 included) go to the lower member
 *      index.  rank[k] = k's position in order, -1 when k is not ranked.
 *   3. n_sel = floor(q * n_valid) in fp64, 0 < q <= 0.5.  n_sel == 0: the round changes nothing.
 *   4. k is a recipient when rank[k] >= n_valid - n_sel (the bottom n_sel); donors are the top n_sel.  q <= 0.5, so no
 *      member is both, and every copy runs in one pass.
 *   5. recipient k draws w = philox4x32_10(counter (k, (uint32) r, (uint32)(r >> 32), AUR_PBT_PHILOX_C3),
 *      key ((uint32) seed, (uint32)(seed >> 32))); donor = order[((uint64) w0 * n_sel) >> 32].  Every field j of the donor's
 *      aur_pop_hparams is copied; a field whose mask bit is set is then multiplied in fp64 by ((w1 >> j) & 1) ? up : down
 *      (target_kl = +inf stays +inf).
 *   6. the recipient receives the donor's parameter row, adam_m row, adam_v row and Adam step count (the bias correction
 *      continues as the donor's) and, with the continuous wrapper stack, rows 0 .. 2D + 3 of the donor's env columns of
 *      `norm` (observation mean / var / count, return-rms mean / var / count: donor column d * n_member + j -> recipient
 *      column k * n_member + j) -- what the copied policy and critic were trained against.  It keeps its own seed (Philox
 *      and shuffle key), env physics, PCG state, TimeLimit counters, episode accumulators and row 2D + 4 of `norm` (the
 *      discounted-return accumulator of its own running episodes).
 * oracle/pbt_ref.py restates steps 1-6. */
#define AUR_PBT_PHILOX_C3 0x50B7D0E5u   /* fixed fourth counter word of the recipient's draw */

/* The default fitness: fitness_out[k] = mean return of the episodes member k finished since the last call, from the delta
 * of the rollout's cumulative totals [K][3] (count, return sum, length sum; aur_pop_rollout's log.totals) against snapshot
 * [K][3] (zeros before the first call); NaN when no episode finished.  snapshot is then set to totals.  One launch.
 * totals is accumulated with fp64 atomicAdd, so for non-integer returns (Pendulum) the last bits of a sum can depend on
 * arrival order; integer-return envs (CartPole, MountainCar) are exact. */
int aur_pop_episode_fitness(const aur_pop_desc* pop, const double* totals, double* snapshot, double* fitness_out, void* stream);

typedef struct {
  const double* fitness;     /* [K] device, any metric (higher is better; NaN = not ranked) */
  double q;                  /* fraction, 0 < q <= 0.5 */
  double down, up;           /* perturb factors, finite and > 0 */
  uint32_t mask;             /* fields of aur_pop_hparams to perturb, bits 0..5 */
  uint32_t _pad;
  uint64_t seed;             /* Philox key of the draws */
  uint64_t round;            /* r = 1, 2, ...: Philox counter of the draws */
  float* params;             /* [K][P] */
  float* adam_m;             /* [K][P] */
  float* adam_v;             /* [K][P] */
  int64_t* steps;            /* [K] Adam step counts */
  aur_pop_hparams* hparams;  /* [K] */
  double* norm;              /* aur_env_state.norm [2 D + 5][norm_ld] of the K * n_member envs, or NULL without wrappers */
  int64_t norm_ld;           /* >= K * n_member when norm is given */
  int32_t* rank_out;         /* [K]: rank[k], -1 when not ranked */
  int32_t* donor_out;        /* [K]: the donor of recipient k, -1 for every other member */
  int32_t* order;            /* [K + 1] scratch: order[0 .. n_valid - 1], then order[K] = n_valid */
} aur_pop_pbt_args;

/* One PBT round (rank, then exploit / explore) on the population's device arrays, two launches.  AUR_ERR_ARG without touching
 * the device for q outside (0, 0.5], a factor <= 0 or not finite, mask bits above 5, null required pointers or a short
 * norm_ld; AUR_ERR_UNSUPPORTED for a policy outside the population scope. */
int aur_pop_pbt_step(const aur_pop_desc* pop, const aur_policy_desc* desc, const aur_pop_pbt_args* args, void* stream);

/* ------------------------------------------------ squashed Gaussian head ----
 * PPOGaussianPolicyBase.sample (src/nets/nets.py:90-105): y = tanh(action), log_prob = sum_k Normal(mean,
 * exp(log_std)).log_prob(action) - log(1 - y^2 + 1e-6) ([B], the reference keeps dim 1), tanh(mean), and the
 * unsummed Normal entropy [B,A].  action_in NULL: action = mean + std * N(0,1) from Philox(seed; row, stream_id).
 * pre_tanh_out (nullable) receives the un-squashed action.  mean / log_std / outputs: [B,A] fp32, A <= 16. */
int aur_squashed_gaussian_sample(int64_t B, int32_t A, const float* mean, const float* log_std, const float* action_in,
                                 uint64_t seed, uint64_t stream_id, float* action_out, float* logp_out, float* mean_out,
                                 float* entropy_out, float* pre_tanh_out, void* stream);

/* ------------------------------------------------------ tensor-core core ----
 * C[M,N] (fp32, row-major) = A[M,K] * B[N,K]^T with A, B bf16 row-major (K contiguous), fp32
 * accumulation in TMEM (tcgen05.mma kind::f16, TMA operand loads).  The dense-contraction core
 * of the equivariant encoder's convolutions (src/nets/equiv.py:17-59), exported for tests.
 * K must be a multiple of 8. */
int aur_tc_gemm_bf16(int64_t M, int64_t N, int64_t K, const void* A, const void* B, float* C, void* stream);

/* Operand precision of every row-X entry point below (and of aur_tc_gemm_bf16), per calling thread, like a BLAS math mode:
 *   planes = 1  bf16 operands, fp32 accumulation: the fast mode, BELOW the reference's fp32 arithmetic
 *               (src/nets/equiv.py:12-157 and src/robot_ppo.py:329-408 compute in fp32);
 *   planes = 2  every bf16 tensor argument (activations, gradients, expanded filters; inputs and outputs alike) is a stack
 *               [2][...] of two planes of the documented shape: hi = bf16(v), mid = bf16(v - hi), so v = hi + mid to
 *               2^-17 relative.  Contractions issue hi*hi + hi*mid + mid*hi on the tensor cores with fp32 accumulation
 *               (three K passes of the same pipelines): fp32-class results, north_star's 1e-4 gradient bar, 3x the MMA work.
 *               ReLU / max-pool decisions are taken on the fp32 accumulators; masks read the hi plane (hi > 0 <=> v > 0).
 * fp32 arguments (parameters, biases, gradients of parameters, GEMM outputs) are unaffected.  Returns the previous value,
 * or AUR_ERR_ARG.  Default 1. */
int aur_tc_set_precision(int planes);
int aur_tc_get_precision(void);

/* -------------------------------------------- equivariant encoder (row X) ----
 * The C4-equivariant convolutions of EquivariantEncoder128 (src/nets/equiv.py:12-62), which the
 * reference runs as e2cnn R2Conv -> cuDNN.  Activations are NHWC bf16 buffers that INCLUDE their
 * zero halo; a 3x3 layer is a valid convolution over the buffer (output H = Hb - 2). */
typedef struct {
  int32_t B, Hb, Wb, Cin, Cout;   /* input buffer [B,Hb,Wb,Cin] bf16; Cin % 64 == 0, Cout % 32 == 0 */
  int32_t epilogue;               /* 0 linear, 1 bias + ReLU, 2 bias + ReLU + 2x2 max-pool,
                                     3 linear * (relu_ref > 0): backward-data through a ReLU-only layer */
  int32_t out_Hb, out_Wb, out_off;/* output buffer [B,out_Hb,out_Wb,Cout] bf16, written at (+off,+off) */
  int32_t _pad;
  const void* in;
  const void* wmat;               /* [Cout][tap][Cin] bf16 (aur_equiv_expand_regular) */
  const float* bias;              /* [Cout] fp32 or NULL */
  void* out;
  uint8_t* pool_arg;              /* [B,Ho/2,Wo/2,Cout] arg-max (0..3) of each pool window, or NULL */
  const void* relu_ref;           /* epilogue 3: forward activation buffer [B,ref_Hb,ref_Wb,Cout], interior at +ref_off */
  int32_t ref_Hb, ref_Wb, ref_off, _pad2;
} aur_conv_args;

/* implicit-GEMM 3x3 convolution on tcgen05 (TMA halo boxes, TMEM accumulator, fused epilogue). */
int aur_conv3x3_bf16(const aur_conv_args* args, void* stream);

/* psi [Fo,Fi,4,3,3] fp32 (regular -> regular p4 filter) -> wmat [(o,r)][tap][(i,s)] bf16, optional
 * backward-data matrix wt [(i,s)][8-tap][(o,r)] bf16, optional per-channel bias from per-field bias. */
int aur_equiv_expand_regular(const float* psi, int32_t Fo, int32_t Fi, const float* bias_f, void* wmat, void* wt,
                             float* bias_ch, void* stream);

/* layer 0 (trivial -> regular, 2 -> 64 channels at 128x128) + ReLU + max-pool, direct fp32 convolution:
 * obs [B,1,128,128] fp32, state [B] fp32 (tiled second channel, robot_actor_critic.py:106-107),
 * psi [16,2,3,3], bias [16] -> interior of out [B,66,66,64] bf16 (caller zeroes the halo once). */
int aur_equiv_conv0(const float* obs, const float* state, const float* psi, const float* bias_f, int32_t B, void* out,
                    uint8_t* pool_arg, void* stream);

/* weight gradient of a 3x3 layer: dwmat[co][tap][ci] (fp32, ACCUMULATED with atomics: zero it first) +=
 * sum_q dy[q][co] * x[q + base_off + dy*Wb + dx][ci], q the flat pixel index of the haloed NHWC bf16
 * buffers (same geometry for both).  Split-K tcgen05 GEMM with MN-major operands; split_k <= 0 picks it. */
int aur_wgrad3x3_bf16(int32_t Cout, int32_t Cin, int64_t Q, const void* dy, const void* x, int32_t base_off,
                      int32_t Wb, float* dwmat, int32_t split_k, void* stream);

/* max-pool(2) + ReLU backward: dpool [B,Hp,Wp,C] bf16, forward pooled activations `act` (buffer
 * [B,aHb,aWb,C], interior at +aoff), arg [B,Hp,Wp,C] -> dy buffer [B,dHb,dWb,C] interior at +doff. */
int aur_unpool_relu_bwd(int32_t B, int32_t Hp, int32_t Wp, int32_t C, const void* dpool, const void* act, int32_t aHb,
                        int32_t aWb, int32_t aoff, const uint8_t* arg, void* dy, int32_t dHb, int32_t dWb, int32_t doff,
                        void* stream);

/* The same, also accumulating the layer's bias gradient from the values it writes: colsum_out[c / group] += sum of dy[.., c]
 * (what aur_colsum_bf16 would compute by re-reading dy).  colsum_out NULL: plain un-pool.  Needs C / 8 dividing 256. */
int aur_unpool_relu_bwd_colsum(int32_t B, int32_t Hp, int32_t Wp, int32_t C, const void* dpool, const void* act, int32_t aHb,
                               int32_t aWb, int32_t aoff, const uint8_t* arg, void* dy, int32_t dHb, int32_t dWb, int32_t doff,
                               int32_t group, float* colsum_out, void* stream);

int aur_transpose_bf16(int64_t R, int32_t C, const void* in, void* out, void* stream);   /* [R][C] -> [C][R] */

/* adjoint of aur_equiv_expand_regular: dpsi [Fo,Fi,4,3,3] += projection of dwmat [Fo*4][9][Fi*4] */
int aur_equiv_project_regular(const float* dwmat, int32_t Fo, int32_t Fi, float* dpsi, void* stream);

/* out[c / group] += sum_q in[q][c]  (bias gradients from an NHWC output-gradient buffer [Q][C]) */
int aur_colsum_bf16(int64_t Q, int32_t C, const void* in, int32_t group, float* out, void* stream);

/* layer-0 weight gradient fused with its un-pooling: dpsi [16,2,3,3] +=, dbias_f [16] += */
int aur_equiv_conv0_wgrad(const float* obs, const float* state, const void* da1, const void* a1, const uint8_t* arg, int32_t B,
                          float* scratch, float* dpsi, float* dbias_f, void* stream);

int aur_bias_relu_bf16(int64_t rows, int32_t C, const float* in, const float* bias, void* out, void* stream);
int aur_relu_mask_bf16(int64_t n, const float* g, const void* ref, void* out, void* stream); /* ref NULL: plain cast */

/* Heads + loss of the equivariant update: actor head decode (src/nets/equiv.py:86-90), Normal log-prob and
 * entropy summed over the 5 action dims (src/models/robot_actor_critic.py:115-130), critic head ReLU +
 * GroupPooling + value (src/nets/equiv.py:138-150), PPO loss seeds (src/robot_ppo.py:345-398). */
typedef struct {
  int32_t B;
  int32_t clip_vloss;
  int64_t m_total;
  const float* a_out;        /* [B,16] actor head output before bias (10 used) */
  const float* a_bias;       /* [10] */
  const float* c_pre;        /* [B,512] critic head-1 output before bias */
  const float* c_bias1;      /* [512] */
  const float* c_w2;         /* [128] */
  const float* c_b2;         /* [1] */
  const float* action;       /* [B,5] */
  const float* oldlp;
  const float* adv;
  const float* ret;
  const float* vold;
  const double* adv_moments; /* [3] or NULL */
  float clip_coeff, entropy_coeff, value_coeff, _pad;
  void* d_a_out;             /* [B,16] bf16 out */
  void* d_c_h;               /* [B,512] bf16 out */
  float* d_head;             /* [651] accumulated: a_bias 10 | c_w2 128 | c_b2 1 | c_bias1 512 */
  float* stats;              /* [8] accumulated sums */
  float* value_out;          /* [B] or NULL */
  float* logp_out;           /* [B] or NULL */
} aur_equiv_head_args;
int aur_equiv_head_loss(const aur_equiv_head_args* args, void* stream);

/* Layer 0 of the plain CNN (base_encoder's first Conv2d(2,16) + ReLU + MaxPool, src/nets/base_cnns.py:25-27) and its weight
 * gradient: the 16 output channels live in channels 0..15 of the same [B,66,66,64] bf16 buffer / [B,64,64,64] arg-max
 * buffer the equivariant layer 0 uses (the other 48 channels must be zero: allocate the buffers zeroed).
 * weight [16,2,3,3], bias [16]; scratch >= 64*18+64 floats. */
int aur_plain_conv0(const float* obs, const float* state, const float* weight, const float* bias, int32_t B, void* out,
                    uint8_t* pool_arg, void* stream);
int aur_plain_conv0_wgrad(const float* obs, const float* state, const void* da1, const void* a1, const uint8_t* arg, int32_t B,
                          float* scratch, float* dweight, float* dbias, void* stream);

/* Heads at inference: robot_actor_critic.evaluate / value (src/models/robot_actor_critic.py:57-60,104-131) on the
 * head GEMM outputs.  Actor part (a_out non-NULL): Normal(mean, exp(clamp(log_std))) log-prob and entropy summed
 * over the 5 dims, action = action_in or mean + std * N(0,1) from Philox(seed; row, stream_id), and decodeActions
 * (robot_actor_critic.py:63-82): scaled = 0.5 * (u + 1) * (hi - lo) + lo with ranges_lo_hi = host float[10]
 * {lo,hi} for p, dx, dy, dz, dtheta.  Critic part (c_pre non-NULL): ReLU + GroupPooling + 1x1 -> value [B].
 * Either part may be skipped by passing NULL.  mean_out / logstd_out [B,5] nullable. */
int aur_equiv_head_eval(int32_t B, const float* a_out, const float* a_bias, const float* c_pre, const float* c_bias1,
                        const float* c_w2, const float* c_b2, const float* action_in, uint64_t seed, uint64_t stream_id,
                        const float* ranges_lo_hi, float* unscaled_out, float* scaled_out, float* logp_out,
                        float* entropy_out, float* value_out, float* mean_out, float* logstd_out, void* stream);

/* The same for the plain CNN heads of robot_actor_critic(equivariant=False) (src/models/robot_actor_critic.py:41-51,
 * src/nets/base_cnns.py:57-84): a_out cols 0..4 = base_actor.mean_linear output before bias, log_std = the actor_logstd
 * parameter [5], critic = Linear(128,128)-ReLU-Linear(128,1) on c_pre [B,128]. */
int aur_plain_head_eval(int32_t B, const float* a_out, const float* a_bias, const float* actor_logstd, const float* c_pre,
                        const float* c_bias1, const float* c_w2, const float* c_b2, const float* action_in, uint64_t seed,
                        uint64_t stream_id, const float* ranges_lo_hi, float* unscaled_out, float* scaled_out, float* logp_out,
                        float* entropy_out, float* value_out, float* mean_out, float* logstd_out, void* stream);

/* Heads + PPO loss of the plain CNN update (robot_ppo.update, src/robot_ppo.py:345-398, on the non-equivariant model):
 * gradients wrt the two head GEMM outputs (bf16) and the small head parameters. */
typedef struct {
  int32_t B;
  int32_t clip_vloss;
  int64_t m_total;
  const float* a_out;        /* [B,16] mean_linear output before bias (5 used) */
  const float* a_bias;       /* [5] */
  const float* actor_logstd; /* [5] */
  const float* c_pre;        /* [B,128] critic.0 output before bias */
  const float* c_bias1;      /* [128] */
  const float* c_w2;         /* [128] */
  const float* c_b2;         /* [1] */
  const float* action;       /* [B,5] */
  const float* oldlp;
  const float* adv;
  const float* ret;
  const float* vold;
  const double* adv_moments; /* [3] or NULL */
  float clip_coeff, entropy_coeff, value_coeff, _pad;
  void* d_a_out;             /* [B,16] bf16 out */
  void* d_c_h;               /* [B,128] bf16 out */
  float* d_head;             /* [267] accumulated: a_bias 5 | actor_logstd 5 | c_w2 128 | c_b2 1 | c_bias1 128 */
  float* stats;              /* [8] accumulated sums */
  float* value_out;          /* [B] or NULL */
  float* logp_out;           /* [B] or NULL */
} aur_plain_head_args;
int aur_plain_head_loss(const aur_plain_head_args* args, void* stream);

int aur_sumsq_f32(int64_t n, const float* g, double* out_accum, void* stream);
/* torch.optim.Adam math on a flat buffer; clip_sumsq (nullable) = device sum of squares of the clipped group */
int aur_adam_flat(int64_t n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, double lr, double beta1,
                  double beta2, double eps, int64_t step, const double* clip_sumsq, double max_grad_norm, void* stream);

/* diagnostic: shared-window address of the first dynamic shared-memory byte of a kernel */
int aur_debug_smem_base(unsigned int* out_dev, void* stream);

/* Evaluates the deterministic fp64 sin/cos the env kernels use (csrc/det_sincos.h) on n
 * device doubles -- exported so tests can compare it with the host copy bit for bit. */
int aur_sincos_f64(int64_t n, const double* x, double* sin_out, double* cos_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AUR_PPO_H */
