// Device-side environments and their bookkeeping, shared by the rollout kernels (rollout.cu, rollout_tc.cu):
// PCG64 reset streams, gym's CartPole-v1 / Pendulum-v1 dynamics, the continuous wrapper stack's running statistics,
// the kernel argument block and the episode log.  Third-party behaviour restated from gym 0.26.2 (see DESIGN.md 5).
#pragma once
#include "det_sincos.h"
#include "policy.cuh"

namespace aur {

typedef unsigned __int128 u128;

// ---- PCG64 (setseq 128, XSL-RR) : the generator behind gym's np_random ------------------
struct Pcg64 {
  u128 state, inc;
  __device__ __forceinline__ void load(const uint64_t* pcg, long long N, long long n) {
    state = ((u128)pcg[0 * N + n] << 64) | pcg[1 * N + n];
    inc = ((u128)pcg[2 * N + n] << 64) | pcg[3 * N + n];
  }
  __device__ __forceinline__ void store(uint64_t* pcg, long long N, long long n) const {
    pcg[0 * N + n] = (uint64_t)(state >> 64);
    pcg[1 * N + n] = (uint64_t)state;
  }
  __device__ __forceinline__ double next_double() {
    const u128 MULT = ((u128)0x2360ED051FC65DA4ULL << 64) | 0x4385DF649FCCF645ULL;
    state = state * MULT + inc;
    const uint64_t hi = (uint64_t)(state >> 64), lo = (uint64_t)state;
    const uint64_t x = hi ^ lo;
    const unsigned rot = (unsigned)(hi >> 58);
    const uint64_t r = (x >> rot) | (x << ((64u - rot) & 63u));
    return (double)(r >> 11) * (1.0 / 9007199254740992.0);
  }
  // Generator.uniform(low, high) = low + (high - low) * next_double
  __device__ __forceinline__ double uniform(double low, double range) { return low + range * next_double(); }
};

// ---- RunningMeanStd.update with batch_count == 1 (gym/wrappers/normalize.py) ------------
__device__ __forceinline__ void rms_update1(double& mean, double& var, double count, double x) {
  const double delta = x - mean;
  const double tot = count + 1.0;
  const double new_mean = mean + delta * 1.0 / tot;
  const double m_a = var * count;
  const double M2 = m_a + 0.0 + delta * delta * count * 1.0 / tot;
  mean = new_mean;
  var = M2 / tot;
}
__device__ __forceinline__ double clip10(double z) { return z < -10.0 ? -10.0 : (z > 10.0 ? 10.0 : z); }

// Wrapper statistics of one env: obs mean[D], var[D], count; return-rms mean, var, count; acc -> [2 D + 5][N] in HBM.
template <int D>
struct NormStateT {
  double om[D], ov[D], oc, rm, rv, rc, racc;
  __device__ __forceinline__ void init() {
    for (int k = 0; k < D; ++k) { om[k] = 0.0; ov[k] = 1.0; }
    oc = 1e-4; rm = 0.0; rv = 1.0; rc = 1e-4; racc = 0.0;
  }
  __device__ __forceinline__ void load(const double* g, long long N, long long n) {
    for (int k = 0; k < D; ++k) { om[k] = g[k * N + n]; ov[k] = g[(D + k) * N + n]; }
    oc = g[(2 * D) * N + n]; rm = g[(2 * D + 1) * N + n]; rv = g[(2 * D + 2) * N + n]; rc = g[(2 * D + 3) * N + n];
    racc = g[(2 * D + 4) * N + n];
  }
  __device__ __forceinline__ void store(double* g, long long N, long long n) const {
    for (int k = 0; k < D; ++k) { g[k * N + n] = om[k]; g[(D + k) * N + n] = ov[k]; }
    g[(2 * D) * N + n] = oc; g[(2 * D + 1) * N + n] = rm; g[(2 * D + 2) * N + n] = rv; g[(2 * D + 3) * N + n] = rc;
    g[(2 * D + 4) * N + n] = racc;
  }
  // NormalizeObservation.normalize + clip(-10, 10), result cast to the fp32 obs buffer
  __device__ __forceinline__ void obs(const float (&raw)[D], float (&out)[POL_IN_PAD]) {
    for (int k = 0; k < D; ++k) rms_update1(om[k], ov[k], oc, (double)raw[k]);
    oc = oc + 1.0;
    for (int k = 0; k < D; ++k) out[k] = (float)clip10(((double)raw[k] - om[k]) / sqrt(ov[k] + 1e-8));
    for (int k = D; k < POL_IN_PAD; ++k) out[k] = 0.0f;
  }
  // NormalizeReward.step + clip(-10, 10)
  __device__ __forceinline__ double reward(double r, bool done, double gamma) {
    racc = racc * gamma + r;
    rms_update1(rm, rv, rc, racc);
    rc = rc + 1.0;
    double out = r / sqrt(rv + 1e-8);
    if (done) racc = 0.0;
    return clip10(out);
  }
};
using NormState = NormStateT<3>;

// ---- CartPole-v1 (gym/envs/classic_control/cartpole.py) ----------------------------------
struct CartPole {
  static constexpr int S = 4, OBS = 4, LIMIT = 500;
  static constexpr bool CONT = false;
  double x, xd, th, thd;
  __device__ __forceinline__ void load(const double* g, long long N, long long n) {
    x = g[n]; xd = g[N + n]; th = g[2 * N + n]; thd = g[3 * N + n];
  }
  __device__ __forceinline__ void store(double* g, long long N, long long n) const {
    g[n] = x; g[N + n] = xd; g[2 * N + n] = th; g[3 * N + n] = thd;
  }
  __device__ __forceinline__ void reset(Pcg64& rng) {
    x = rng.uniform(-0.05, 0.05 - (-0.05)); xd = rng.uniform(-0.05, 0.05 - (-0.05));
    th = rng.uniform(-0.05, 0.05 - (-0.05)); thd = rng.uniform(-0.05, 0.05 - (-0.05));
  }
  __device__ __forceinline__ void raw_obs(float (&o)[POL_IN_PAD]) const {
    o[0] = (float)x; o[1] = (float)xd; o[2] = (float)th; o[3] = (float)thd;
  }
  // returns reward; sets terminated
  __device__ __forceinline__ double step(int action, bool& terminated) {
    const double gravity = 9.8, masscart = 1.0, masspole = 0.1, length = 0.5, force_mag = 10.0, tau = 0.02;
    const double total_mass = masspole + masscart, polemass_length = masspole * length;
    const double theta_thr = 12 * 2 * 3.141592653589793 / 360, x_thr = 2.4;
    const double force = action == 1 ? force_mag : -force_mag;
    double sintheta, costheta;
    aur_sincos(th, &sintheta, &costheta);
    const double temp = (force + polemass_length * (thd * thd) * sintheta) / total_mass;
    const double thetaacc = (gravity * sintheta - costheta * temp) /
                            (length * (4.0 / 3.0 - masspole * (costheta * costheta) / total_mass));
    const double xacc = temp - polemass_length * thetaacc * costheta / total_mass;
    x = x + tau * xd;
    xd = xd + tau * xacc;
    th = th + tau * thd;
    thd = thd + tau * thetaacc;
    terminated = (x < -x_thr) || (x > x_thr) || (th < -theta_thr) || (th > theta_thr);
    return 1.0;
  }
};

// ---- MountainCar-v0 (gym/envs/classic_control/mountain_car.py) ------------------------------
struct MountainCar {
  static constexpr int S = 2, OBS = 2, LIMIT = 200;
  static constexpr bool CONT = false;
  double pos, vel;
  __device__ __forceinline__ void load(const double* g, long long N, long long n) { pos = g[n]; vel = g[N + n]; }
  __device__ __forceinline__ void store(double* g, long long N, long long n) const { g[n] = pos; g[N + n] = vel; }
  __device__ __forceinline__ void reset(Pcg64& rng) {
    pos = rng.uniform(-0.6, -0.4 - (-0.6));
    vel = 0.0;
  }
  __device__ __forceinline__ void raw_obs(float (&o)[POL_IN_PAD]) const { o[0] = (float)pos; o[1] = (float)vel; o[2] = 0.0f; o[3] = 0.0f; }
  __device__ __forceinline__ double step(int action, bool& terminated) {
    const double min_position = -1.2, max_position = 0.6, max_speed = 0.07, goal_position = 0.5, goal_velocity = 0.0;
    const double force = 0.001, gravity = 0.0025;
    double s3, c3;
    aur_sincos(3 * pos, &s3, &c3);
    vel = vel + ((double)(action - 1) * force + c3 * (-gravity));
    vel = vel < -max_speed ? -max_speed : (vel > max_speed ? max_speed : vel);
    pos = pos + vel;
    pos = pos < min_position ? min_position : (pos > max_position ? max_position : pos);
    if (pos == min_position && vel < 0) vel = 0;
    terminated = (pos >= goal_position) && (vel >= goal_velocity);
    return -1.0;
  }
};

// ---- Acrobot-v1 (gym/envs/classic_control/acrobot.py, "book" dynamics, no torque noise) -------------------------------
// fp64 state [theta1, theta2, dtheta1, dtheta2], one classic RK4 step of dt = 0.2 per env step with the torque carried as a
// fifth, constant component; every expression keeps the operation order of the Python source so that each fp64 operation
// rounds once (the library is compiled with --fmad=false).  reset() rounds the uniform draws to fp32 as gym does
// (`.astype(np.float32)`).  Trigonometry goes through the deterministic sin/cos shared with the CPU checker.
struct Acrobot {
  static constexpr int S = 4, OBS = 6, LIMIT = 500;
  static constexpr bool CONT = false;
  double s0, s1, s2, s3;
  __device__ __forceinline__ void load(const double* g, long long N, long long n) {
    s0 = g[n]; s1 = g[N + n]; s2 = g[2 * N + n]; s3 = g[3 * N + n];
  }
  __device__ __forceinline__ void store(double* g, long long N, long long n) const {
    g[n] = s0; g[N + n] = s1; g[2 * N + n] = s2; g[3 * N + n] = s3;
  }
  __device__ __forceinline__ void reset(Pcg64& rng) {
    s0 = (double)(float)rng.uniform(-0.1, 0.1 - (-0.1)); s1 = (double)(float)rng.uniform(-0.1, 0.1 - (-0.1));
    s2 = (double)(float)rng.uniform(-0.1, 0.1 - (-0.1)); s3 = (double)(float)rng.uniform(-0.1, 0.1 - (-0.1));
  }
  __device__ __forceinline__ void raw_obs(float (&o)[8]) const {
    double sa, ca, sb, cb;
    aur_sincos(s0, &sa, &ca);
    aur_sincos(s1, &sb, &cb);
    o[0] = (float)ca; o[1] = (float)sa; o[2] = (float)cb; o[3] = (float)sb; o[4] = (float)s2; o[5] = (float)s3;
    o[6] = 0.0f; o[7] = 0.0f;
  }
  // AcrobotEnv._dsdt: y = [theta1, theta2, dtheta1, dtheta2], a = torque -> k = d/dt of the four components
  static __device__ __forceinline__ void dsdt(const double (&y)[4], double a, double (&k)[4]) {
    const double m1 = 1.0, m2 = 1.0, l1 = 1.0, lc1 = 0.5, lc2 = 0.5, I1 = 1.0, I2 = 1.0, g = 9.8;
    const double PI = 3.141592653589793;
    const double theta1 = y[0], theta2 = y[1], dtheta1 = y[2], dtheta2 = y[3];
    double sin2, cos2, sd, c12, c1;
    aur_sincos(theta2, &sin2, &cos2);
    aur_sincos(theta1 + theta2 - PI / 2.0, &sd, &c12);
    aur_sincos(theta1 - PI / 2, &sd, &c1);
    const double d1 = m1 * (lc1 * lc1) + m2 * (l1 * l1 + lc2 * lc2 + 2 * l1 * lc2 * cos2) + I1 + I2;
    const double d2 = m2 * (lc2 * lc2 + l1 * lc2 * cos2) + I2;
    const double phi2 = m2 * lc2 * g * c12;
    const double phi1 = -m2 * l1 * lc2 * (dtheta2 * dtheta2) * sin2 - 2 * m2 * l1 * lc2 * dtheta2 * dtheta1 * sin2 +
                        (m1 * lc1 + m2 * l1) * g * c1 + phi2;
    const double ddtheta2 = (a + d2 / d1 * phi1 - m2 * l1 * lc2 * (dtheta1 * dtheta1) * sin2 - phi2) /
                            (m2 * (lc2 * lc2) + I2 - (d2 * d2) / d1);
    const double ddtheta1 = -(d2 * ddtheta2 + phi1) / d1;
    k[0] = dtheta1; k[1] = dtheta2; k[2] = ddtheta1; k[3] = ddtheta2;
  }
  __device__ __forceinline__ double step(int action, bool& terminated) {
    const double PI = 3.141592653589793, dt = 0.2 - 0, dt2 = dt / 2.0;
    const double torque = (double)(action - 1);                 // AVAIL_TORQUE = [-1., 0., +1]
    const double y0[4] = {s0, s1, s2, s3};
    double k1[4], k2[4], k3[4], k4[4], y[4];
    dsdt(y0, torque, k1);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = y0[i] + dt2 * k1[i];
    dsdt(y, torque, k2);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = y0[i] + dt2 * k2[i];
    dsdt(y, torque, k3);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = y0[i] + dt * k3[i];
    dsdt(y, torque, k4);
    double ns[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) ns[i] = y0[i] + dt / 6.0 * (k1[i] + 2 * k2[i] + 2 * k3[i] + k4[i]);
    const double diff = PI - (-PI);
#pragma unroll
    for (int i = 0; i < 2; ++i) {                               // wrap(x, -pi, pi)
      while (ns[i] > PI) ns[i] = ns[i] - diff;
      while (ns[i] < -PI) ns[i] = ns[i] + diff;
    }
    const double mv1 = 4 * PI, mv2 = 9 * PI;                    // bound(x, -MAX_VEL, MAX_VEL) = min(max(x, m), M)
    ns[2] = ns[2] < -mv1 ? -mv1 : ns[2]; ns[2] = ns[2] > mv1 ? mv1 : ns[2];
    ns[3] = ns[3] < -mv2 ? -mv2 : ns[3]; ns[3] = ns[3] > mv2 ? mv2 : ns[3];
    s0 = ns[0]; s1 = ns[1]; s2 = ns[2]; s3 = ns[3];
    double sa, ca, sb, cb;
    aur_sincos(s0, &sa, &ca);
    aur_sincos(s1 + s0, &sb, &cb);
    terminated = (-ca - cb) > 1.0;
    return terminated ? 0.0 : -1.0;
  }
};

// ---- MountainCarContinuous-v0 (gym/envs/classic_control/continuous_mountain_car.py) -----------------------------------
// The env keeps its state as a float32 array after every step (np.array([position, velocity], dtype=np.float32)) and
// computes in float64 in between (NumPy 1.24 scalar promotion: float32 scalar with a Python float -> float64), so the
// fp64 state here always holds float32-representable values except right after reset (float64 uniform draw).
struct MountainCarContinuous {
  static constexpr int S = 2, OBS = 2, LIMIT = 999;
  static constexpr bool CONT = true;
  double pos, vel;
  __device__ __forceinline__ void load(const double* g, long long N, long long n) { pos = g[n]; vel = g[N + n]; }
  __device__ __forceinline__ void store(double* g, long long N, long long n) const { g[n] = pos; g[N + n] = vel; }
  __device__ __forceinline__ void reset(Pcg64& rng) {
    pos = rng.uniform(-0.6, -0.4 - (-0.6));
    vel = 0.0;
  }
  __device__ __forceinline__ void raw_obs(float (&o)[2]) const { o[0] = (float)pos; o[1] = (float)vel; }
  __device__ __forceinline__ double step(float u_in, bool clip_action, bool& terminated) {
    const double min_position = -1.2, max_position = 0.6, max_speed = 0.07, goal_position = 0.45, goal_velocity = 0.0;
    const double power = 0.0015;
    float u = u_in;
    if (clip_action) u = u < -1.0f ? -1.0f : (u > 1.0f ? 1.0f : u);      // ClipAction wrapper (action space [-1, 1])
    const float f32 = u < -1.0f ? -1.0f : (u > 1.0f ? 1.0f : u);         // min(max(action[0], min_action), max_action)
    double s3, c3;
    aur_sincos(3 * pos, &s3, &c3);
    double velocity = vel + ((double)f32 * power - 0.0025 * c3);
    if (velocity > max_speed) velocity = max_speed;
    if (velocity < -max_speed) velocity = -max_speed;
    double position = pos + velocity;
    if (position > max_position) position = max_position;
    if (position < min_position) position = min_position;
    if (position == min_position && velocity < 0) velocity = 0;
    terminated = (position >= goal_position) && (velocity >= goal_velocity);
    double reward = 0;
    if (terminated) reward = 100.0;
    reward -= ((double)u * (double)u) * 0.1;                             // math.pow(action[0], 2) * 0.1
    pos = (double)(float)position; vel = (double)(float)velocity;
    return reward;
  }
};

// ---- Pendulum-v1 (gym/envs/classic_control/pendulum.py, g = 10) --------------------------
struct Pendulum {
  static constexpr int S = 2, OBS = 3, LIMIT = 200;
  static constexpr bool CONT = true;
  double th, thd;
  double s_th, c_th;   // sin/cos of the CURRENT theta (the obs needs them, the next step reuses sin)
  __device__ __forceinline__ void load(const double* g, long long N, long long n) {
    th = g[n]; thd = g[N + n];
    aur_sincos(th, &s_th, &c_th);
  }
  __device__ __forceinline__ void store(double* g, long long N, long long n) const { g[n] = th; g[N + n] = thd; }
  __device__ __forceinline__ void reset(Pcg64& rng) {
    const double PI = 3.141592653589793;
    th = rng.uniform(-PI, PI - (-PI));
    thd = rng.uniform(-1.0, 1.0 - (-1.0));
    aur_sincos(th, &s_th, &c_th);
  }
  __device__ __forceinline__ void raw_obs(float (&o)[3]) const { o[0] = (float)c_th; o[1] = (float)s_th; o[2] = (float)thd; }
  __device__ __forceinline__ double step(float u_in, bool clip_action, bool& terminated) {
    const double max_speed = 8.0, dt = 0.05, g = 10.0, m = 1.0, l = 1.0, PI = 3.141592653589793;
    float u = u_in;
    if (clip_action) u = u < -2.0f ? -2.0f : (u > 2.0f ? 2.0f : u);   // ClipAction wrapper
    u = u < -2.0f ? -2.0f : (u > 2.0f ? 2.0f : u);                    // np.clip(u, -max_torque, max_torque)
    const float usq = __fmul_rn(u, u);
    const double twopi = 2 * PI;
    double an = fmod(th + PI, twopi);
    if (an != 0.0 && an < 0.0) an += twopi;
    an = an - PI;
    const double costs = an * an + 0.1 * (thd * thd) + 0.001 * (double)usq;
    double newthd = thd + (3 * g / (2 * l) * s_th + 3.0 / (m * (l * l)) * (double)u) * dt;
    newthd = newthd < -max_speed ? -max_speed : (newthd > max_speed ? max_speed : newthd);
    th = th + newthd * dt;
    thd = newthd;
    aur_sincos(th, &s_th, &c_th);
    terminated = false;
    return -costs;
  }
};

struct RolloutDev {
  long long N;
  int T, wrappers;
  int obs_dim, act_dim, nl, continuous;
  int greedy;                 // policy_evaluate kernels only: 1 = arg-max action / the Normal mean instead of a sample (test.py-style evaluation)
  int hid, dyn_smem;          // runtime-width path (hidden_dim != 64): hidden units, 1 = both nets are copied to shared memory
  const float* params;
  aur_env_state env;
  float *obs_buf, *act_buf, *logp_buf, *val_buf, *rew_buf, *done_buf, *next_obs, *next_done, *next_value;
  const float* actions_in;
  uint64_t seed, step0, env_id0;
  aur_episode_log log;
  double gamma;
  int t0;                     // first step index of this launch (buffers / episode log); 0 except for the per-step launches of rollout_wide.cu
  const float* ext_logits;    // [N][4] actor outputs computed outside the kernel (rollout_tc_kernel<ENV, 0>), else nullptr
  // populations (rollout_tc_kernel<ENV, H, true>, aur_pop_rollout): N = K * n_member columns, member k = blockIdx.y owns
  // columns k * n_member ..; its parameters sit at params + k * pop_P, its Philox key is pop_seeds[k]
  long long n_member, pop_P;
  const uint64_t* pop_seeds;
};

template <int HID>
__device__ __forceinline__ void load_policy_smem(float* smem, const RolloutDev& a, const float*& sActor,
                                                 const float*& sCritic, const float*& sLogstd) {
  const int nA = net_smem_floats(HID, a.nl, a.act_dim), nC = net_smem_floats(HID, a.nl, 1);
  const int64_t gA = net_param_count(a.obs_dim, HID, a.nl, a.act_dim), gC = net_param_count(a.obs_dim, HID, a.nl, 1);
  load_net_to_smem(smem, a.params, a.obs_dim, HID, a.nl, a.act_dim, threadIdx.x, blockDim.x);
  load_net_to_smem(smem + nA, a.params + gA, a.obs_dim, HID, a.nl, 1, threadIdx.x, blockDim.x);
  if (a.continuous && threadIdx.x < POL_OUT_MAX)
    smem[nA + nC + threadIdx.x] = threadIdx.x < a.act_dim ? a.params[gA + gC + threadIdx.x] : 0.0f;
  sActor = smem; sCritic = smem + nA; sLogstd = smem + nA + nC;
}

// Runtime-width policies (rollout_kernel<ENV, 0, 1, true>, policy_evaluate_dyn_kernel): the flat nets are copied to
// 16-byte aligned shared memory when they fit (a.dyn_smem), else read in place from global memory; `scratch` is the
// calling thread's activation column ([2][hid][blockDim] floats behind the weights).
__device__ __forceinline__ void load_policy_dyn(float* smem, const RolloutDev& a, const float*& act, const float*& cri,
                                                const float*& ls, float*& scratch, bool& vec_critic) {
  const int64_t gA = net_param_count(a.obs_dim, a.hid, a.nl, a.act_dim), gC = net_param_count(a.obs_dim, a.hid, a.nl, 1);
  if (a.dyn_smem) {
    const int64_t oC = (gA + 3) & ~3LL, oL = oC + ((gC + 3) & ~3LL);
    for (int64_t i = threadIdx.x; i < gA; i += blockDim.x) smem[i] = a.params[i];
    for (int64_t i = threadIdx.x; i < gC; i += blockDim.x) smem[oC + i] = a.params[gA + i];
    if (threadIdx.x < 8) smem[oL + threadIdx.x] = (a.continuous && (int)threadIdx.x < a.act_dim) ? a.params[gA + gC + threadIdx.x] : 0.0f;
    act = smem; cri = smem + oC; ls = smem + oL;
    scratch = smem + oL + 8 + threadIdx.x;
    vec_critic = true;
  } else {
    act = a.params; cri = a.params + gA; ls = a.params + gA + gC;
    scratch = smem + threadIdx.x;
    vec_critic = (gA & 3) == 0;
  }
}
__host__ __device__ inline int64_t dyn_policy_smem_floats(int obs, int H, int NL, int act) {
  return ((net_param_count(obs, H, NL, act) + 3) & ~3LL) + ((net_param_count(obs, H, NL, 1) + 3) & ~3LL) + 8;
}

// forward of one net for E envs of a thread: compiled 64-wide path (registers) or the runtime-width path (HID == 0)
template <int HID, int E, int INP>
__device__ __forceinline__ void policy_net_forward(const RolloutDev& a, const float* __restrict__ net, bool vec, int out_dim,
                                                   const float (&x)[E][INP], float (&o)[E][POL_OUT_MAX],
                                                   float* __restrict__ scratch) {
  if constexpr (HID == 0) {
    static_assert(E == 1, "runtime-width policies run one env per thread");
    if (vec) mlp_forward_dyn<true, INP, POL_OUT_MAX>(net, a.obs_dim, a.hid, a.nl, out_dim, x[0], o[0], scratch, blockDim.x);
    else mlp_forward_dyn<false, INP, POL_OUT_MAX>(net, a.obs_dim, a.hid, a.nl, out_dim, x[0], o[0], scratch, blockDim.x);
  } else {
    static_assert(INP == POL_IN_PAD, "the register-resident 64-wide path takes at most 4 observation dims");
    mlp_forward<HID, E>(net, a.nl, out_dim, x, o, scratch, blockDim.x);
  }
}

__device__ __forceinline__ void log_episode(const aur_episode_log& log, int t, long long local_env, int step, int env,
                                            float ret, int len) {
  if (log.first_finished) {
    const unsigned long long key = ((unsigned long long)local_env << 42) | ((unsigned long long)(len & 1023) << 32) |
                                   (unsigned long long)__float_as_uint(ret);
    atomicMin(log.first_finished + t, key);
  }
  if (log.totals) {
    atomicAdd(log.totals + 0, 1.0);
    atomicAdd(log.totals + 1, (double)ret);
    atomicAdd(log.totals + 2, (double)len);
  }
  if (!log.count) return;
  const uint32_t idx = atomicAdd(log.count, 1u);
  if (log.entries && idx < log.capacity) {
    int4 v = make_int4(step, env, __float_as_int(ret), len);
    *reinterpret_cast<int4*>(&log.entries[idx]) = v;
  }
}


}  // namespace aur
