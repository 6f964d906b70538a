// Device-side actor-critic MLP forward (no grad) shared by the rollout and evaluate kernels.
// Restates nets/nets.py:19-53 (Linear-Tanh stacks) and the distribution arithmetic of
// models/actor_critic.py:34-51 (Categorical / diagonal Normal).
//
// Mapping: each thread owns E envs; the weights of one net sit in shared memory in torch's own
// [out][in] layout (first layer padded to 4 inputs), every lane of a warp reads the same weight
// (LDS.128 broadcast) and feeds packed fp32x2 FMAs (FFMA2, the full-rate fp32 path on sm_100):
// an output neuron accumulates even/odd inputs in the two halves of a float2 and adds them at
// the end.  Activations never leave registers.
#pragma once
#include "common.cuh"

namespace aur {

constexpr int POL_IN_PAD = 4;   // first-layer rows padded to 4 inputs (obs_dim <= 4)
constexpr int POL_OUT_MAX = 4;  // act_dim <= 4 compiled

__host__ __device__ inline int64_t net_param_count(int obs, int H, int NL, int out) {
  return (int64_t)H * obs + H + (int64_t)(NL - 1) * ((int64_t)H * H + H) + (int64_t)out * H + out;
}
__host__ __device__ inline int64_t policy_param_count(const aur_policy_desc& d) {
  return net_param_count(d.obs_dim, d.hidden_dim, d.num_layers, d.act_dim) +
         net_param_count(d.obs_dim, d.hidden_dim, d.num_layers, 1) + (d.continuous ? d.act_dim : 0);
}
// floats one net occupies in shared memory (padded layout)
__host__ __device__ inline int net_smem_floats(int H, int NL, int out) {
  return H * POL_IN_PAD + H + (NL - 1) * (H * H + H) + out * H + 4;
}

// Copy one net from the flat global buffer into its padded shared-memory layout.
__device__ inline void load_net_to_smem(float* __restrict__ s, const float* __restrict__ g, int obs, int H, int NL,
                                        int out, int tid, int nthreads) {
  // first layer, rows padded to POL_IN_PAD
  for (int i = tid; i < H * POL_IN_PAD; i += nthreads) {
    int j = i / POL_IN_PAD, c = i - j * POL_IN_PAD;
    s[i] = c < obs ? g[j * obs + c] : 0.0f;
  }
  const float* gp = g + H * obs;
  float* sp = s + H * POL_IN_PAD;
  const int rest = H + (NL - 1) * (H * H + H) + out * H + out;
  for (int i = tid; i < rest; i += nthreads) sp[i] = gp[i];
  for (int i = tid; i < 4 - out; i += nthreads) sp[rest + i] = 0.0f;
}

__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float2 lds2(const float* p) { return *reinterpret_cast<const float2*>(p); }

// tanh(x) = 1 - 2 / (exp(2x) + 1): 3 FMA-pipe ops + 2 MUFU, |abs err| ~ 1.5e-7, exact saturation.
__device__ __forceinline__ float tanh_fast(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  return fmaf(-2.0f, r, 1.0f);
}

// same for a pair of arguments already multiplied by 2 log2(e) (the scale folded into the producing weights / FMA), with
// packed fp32x2 add / FMA (FADD2, FFMA2): 6 instructions per pair, each lane rounding as tanh_fast does after its scaling
constexpr float TANH_PRESCALE = 2.8853900817779268f;
__device__ __forceinline__ float2 tanh_prescaled2(float2 y) {
  float2 e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(y.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(y.y));
  const float2 d = __fadd2_rn(e, make_float2(1.0f, 1.0f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.x) : "f"(d.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.y) : "f"(d.y));
  return __ffma2_rn(make_float2(-2.0f, -2.0f), r, make_float2(1.0f, 1.0f));
}

// h[e][.] = tanh(W0 x + b0)
template <int HID, int E>
__device__ __forceinline__ void mlp_first_layer(const float* __restrict__ sW0, const float* __restrict__ sB0,
                                                const float (&x)[E][POL_IN_PAD], float2 (&h)[E][HID / 2]) {
  float2 x01[E], x23[E];
#pragma unroll
  for (int e = 0; e < E; ++e) { x01[e] = make_float2(x[e][0], x[e][1]); x23[e] = make_float2(x[e][2], x[e][3]); }
#pragma unroll
  for (int jp = 0; jp < HID / 2; ++jp) {
    const float4 wa = lds4(sW0 + (2 * jp) * POL_IN_PAD), wb = lds4(sW0 + (2 * jp + 1) * POL_IN_PAD);
    const float2 b = lds2(sB0 + 2 * jp);
#pragma unroll
    for (int e = 0; e < E; ++e) {
      float2 a = __ffma2_rn(make_float2(wa.z, wa.w), x23[e], __fmul2_rn(make_float2(wa.x, wa.y), x01[e]));
      float2 c = __ffma2_rn(make_float2(wb.z, wb.w), x23[e], __fmul2_rn(make_float2(wb.x, wb.y), x01[e]));
      h[e][jp] = make_float2(tanh_fast(a.x + a.y + b.x), tanh_fast(c.x + c.y + b.y));
    }
  }
}

// z[e][jj] = b[j0+jj] + sum_i W[j0+jj][i] h[e][i], jj < 8 (pre-activation of 8 neurons)
template <int HID, int E>
__device__ __forceinline__ void mlp_hidden_block(const float* __restrict__ sW, const float* __restrict__ sB, int j0,
                                                 const float2 (&h)[E][HID / 2], float (&z)[E][8]) {
  float2 acc[E][8];
  const float* wrow = sW + j0 * HID;
#pragma unroll
  for (int i4 = 0; i4 < HID / 4; ++i4) {
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      const float4 w = lds4(wrow + jj * HID + i4 * 4);
#pragma unroll
      for (int e = 0; e < E; ++e) {
        float2 a = (i4 == 0) ? __fmul2_rn(make_float2(w.x, w.y), h[e][0])
                             : __ffma2_rn(make_float2(w.x, w.y), h[e][2 * i4], acc[e][jj]);
        acc[e][jj] = __ffma2_rn(make_float2(w.z, w.w), h[e][2 * i4 + 1], a);
      }
    }
  }
  const float4 b0 = lds4(sB + j0), b1 = lds4(sB + j0 + 4);
  const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
  for (int e = 0; e < E; ++e)
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) z[e][jj] = acc[e][jj].x + acc[e][jj].y + bb[jj];
}

// Full forward of one net.  sNet: padded smem layout (see load_net_to_smem).  scratch: per-thread
// column in shared memory ([HID][nthreads] floats) used only when NL >= 3 (E must be 1 then).
template <int HID, int E>
__device__ __forceinline__ void mlp_forward(const float* __restrict__ sNet, int NL, int out_dim,
                                            const float (&x)[E][POL_IN_PAD], float (&out)[E][POL_OUT_MAX],
                                            float* __restrict__ scratch, int scratch_stride) {
  float2 h[E][HID / 2];
  const float* p = sNet;
  mlp_first_layer<HID, E>(p, p + HID * POL_IN_PAD, x, h);
  p += HID * POL_IN_PAD + HID;
  if constexpr (E == 1) {
    // middle hidden layers (num_layers >= 3): results staged through the thread's smem column
    for (int l = 1; l < NL - 1; ++l) {
#pragma unroll 1
      for (int j0 = 0; j0 < HID; j0 += 8) {
        float z[E][8];
        mlp_hidden_block<HID, E>(p, p + HID * HID, j0, h, z);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) scratch[(j0 + jj) * scratch_stride] = tanh_fast(z[0][jj]);
      }
#pragma unroll
      for (int jp = 0; jp < HID / 2; ++jp)
        h[0][jp] = make_float2(scratch[(2 * jp) * scratch_stride], scratch[(2 * jp + 1) * scratch_stride]);
      p += HID * HID + HID;
    }
  }
  float2 o2[E][POL_OUT_MAX];
#pragma unroll
  for (int e = 0; e < E; ++e)
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) o2[e][k] = make_float2(0.0f, 0.0f);
  if (NL >= 2) {
    // last hidden layer fused with the output layer
    const float* sWo = p + HID * HID + HID;
#pragma unroll 1
    for (int j0 = 0; j0 < HID; j0 += 8) {
      float z[E][8];
      mlp_hidden_block<HID, E>(p, p + HID * HID, j0, h, z);
      float2 t[E][4];
#pragma unroll
      for (int e = 0; e < E; ++e)
#pragma unroll
        for (int q = 0; q < 4; ++q) t[e][q] = make_float2(tanh_fast(z[e][2 * q]), tanh_fast(z[e][2 * q + 1]));
#pragma unroll
      for (int k = 0; k < POL_OUT_MAX; ++k) {
        if (k < out_dim) {
          const float4 wa = lds4(sWo + k * HID + j0), wb = lds4(sWo + k * HID + j0 + 4);
#pragma unroll
          for (int e = 0; e < E; ++e) {
            float2 a = __ffma2_rn(make_float2(wa.x, wa.y), t[e][0], o2[e][k]);
            a = __ffma2_rn(make_float2(wa.z, wa.w), t[e][1], a);
            a = __ffma2_rn(make_float2(wb.x, wb.y), t[e][2], a);
            o2[e][k] = __ffma2_rn(make_float2(wb.z, wb.w), t[e][3], a);
          }
        }
      }
    }
    p = sWo;
  } else {
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) {
      if (k < out_dim) {
#pragma unroll
        for (int i4 = 0; i4 < HID / 4; ++i4) {
          const float4 w = lds4(p + k * HID + i4 * 4);
#pragma unroll
          for (int e = 0; e < E; ++e) {
            float2 a = __ffma2_rn(make_float2(w.x, w.y), h[e][2 * i4], o2[e][k]);
            o2[e][k] = __ffma2_rn(make_float2(w.z, w.w), h[e][2 * i4 + 1], a);
          }
        }
      }
    }
  }
  const float4 bo = lds4(p + out_dim * HID);
  const float bb[4] = {bo.x, bo.y, bo.z, bo.w};
#pragma unroll
  for (int e = 0; e < E; ++e)
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) out[e][k] = o2[e][k].x + o2[e][k].y + bb[k];
}

// ---- runtime-width forward (hidden_dim != 64, or observation / action widths above 4) ----------------------------
// One sample per thread.  Activations ping-pong through two per-thread columns of shared memory (col[i * stride],
// col[(H + i) * stride]); the weights are read through `net` in torch's flat [out][in] order, from shared or global
// memory, every lane of a warp at the same address (one broadcast transaction).  VEC: rows of the hidden / output
// matrices are 16-byte aligned (net base aligned and H a multiple of 4), so they load as float4.
template <bool VEC>
__device__ __forceinline__ void dyn_row4(const float* __restrict__ w, float (&v)[4]) {
  if constexpr (VEC) {
    const float4 t = *reinterpret_cast<const float4*>(w);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
    v[0] = w[0]; v[1] = w[1]; v[2] = w[2]; v[3] = w[3];
  }
}
template <bool VEC, int IN_MAX, int OUT_MAX>
__device__ inline void mlp_forward_dyn(const float* __restrict__ net, int obs_dim, int H, int NL, int out_dim,
                                       const float (&x)[IN_MAX], float (&out)[OUT_MAX], float* __restrict__ col, int stride) {
  const float* p = net;
  float* cur = col;
  float* nxt = col + (size_t)H * stride;
  for (int j = 0; j < H; ++j) {                                    // first layer: obs_dim inputs, scalar loads
    float z = p[(size_t)H * obs_dim + j];
#pragma unroll
    for (int c = 0; c < IN_MAX; ++c) if (c < obs_dim) z = fmaf(p[(size_t)j * obs_dim + c], x[c], z);
    cur[(size_t)j * stride] = tanh_fast(z);
  }
  p += (size_t)H * obs_dim + H;
  for (int l = 1; l < NL; ++l) {
    for (int j = 0; j < H; j += 4) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int i = 0; i < H; i += 4) {
        float hv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) hv[q] = cur[(size_t)(i + q) * stride];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          float w[4];
          dyn_row4<VEC>(p + (size_t)(j + jj) * H + i, w);
          acc[jj] = fmaf(w[3], hv[3], fmaf(w[2], hv[2], fmaf(w[1], hv[1], fmaf(w[0], hv[0], acc[jj]))));
        }
      }
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) nxt[(size_t)(j + jj) * stride] = tanh_fast(acc[jj] + p[(size_t)H * H + j + jj]);
    }
    float* t = cur; cur = nxt; nxt = t;
    p += (size_t)H * H + H;
  }
#pragma unroll
  for (int k = 0; k < OUT_MAX; ++k) {
    float acc = 0.0f;
    if (k < out_dim) {
      for (int i = 0; i < H; i += 4) {
        float w[4];
        dyn_row4<VEC>(p + (size_t)k * H + i, w);
        acc = fmaf(w[3], cur[(size_t)(i + 3) * stride], fmaf(w[2], cur[(size_t)(i + 2) * stride],
              fmaf(w[1], cur[(size_t)(i + 1) * stride], fmaf(w[0], cur[(size_t)i * stride], acc))));
      }
      acc += p[(size_t)out_dim * H + k];
    }
    out[k] = acc;
  }
}

// ---- distributions (models/actor_critic.py:34-51) ---------------------------------------
// Categorical(logits): normalised log-probs, then sample by inverse CDF or take `action_in`.
template <int POL_OUT_MAX>
__device__ __forceinline__ void categorical(const float (&logits)[POL_OUT_MAX], int A, bool sample, float u,
                                            int& action, float& logp, float& entropy) {
  float m = logits[0];
#pragma unroll
  for (int k = 1; k < POL_OUT_MAX; ++k) if (k < A) m = fmaxf(m, logits[k]);
  float s = 0.0f;
#pragma unroll
  for (int k = 0; k < POL_OUT_MAX; ++k) if (k < A) s += expf(logits[k] - m);
  const float lse = m + logf(s);
  float lp[POL_OUT_MAX], pr[POL_OUT_MAX];
  entropy = 0.0f;
#pragma unroll
  for (int k = 0; k < POL_OUT_MAX; ++k) {
    lp[k] = logits[k] - lse;
    pr[k] = k < A ? expf(lp[k]) : 0.0f;
    if (k < A) entropy -= pr[k] * lp[k];
  }
  if (sample) {
    // the fp32 running sum can end a few ulp below 1, under the largest u (1 - 2^-24): such a draw takes the last class
    // with nonzero probability, never one whose probability underflowed to 0
    float c = 0.0f;
    int last = 0;
    bool found = false;
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) {
      c += pr[k];
      if (k < A && pr[k] > 0.0f) last = k;
      if (k < A && !found && u < c) { action = k; found = true; }
    }
    if (!found) action = last;
  }
  logp = lp[0];
#pragma unroll
  for (int k = 1; k < POL_OUT_MAX; ++k) if (k == action) logp = lp[k];
}

template <int M>
struct NormalConstsT {   // per action dimension, from actor_logstd
  float std[M], inv2var[M], log_scale[M];
};
using NormalConsts = NormalConstsT<POL_OUT_MAX>;
template <int POL_OUT_MAX = aur::POL_OUT_MAX>
__device__ __forceinline__ NormalConstsT<POL_OUT_MAX> normal_consts(const float* logstd, int A) {
  NormalConstsT<POL_OUT_MAX> c;
#pragma unroll
  for (int k = 0; k < POL_OUT_MAX; ++k) {
    const float ls = k < A ? logstd[k] : 0.0f;
    c.std[k] = expf(ls);
    const float var = c.std[k] * c.std[k];
    c.inv2var[k] = 2.0f * var;             // kept as the divisor 2*var: torch divides
    c.log_scale[k] = logf(c.std[k]);        // torch Normal: log(exp(logstd))
  }
  return c;
}
// Normal(mean, std): log_prob summed over dims, entropy summed over dims.
template <int POL_OUT_MAX>
__device__ __forceinline__ void normal_logp(const float (&mean)[POL_OUT_MAX], const float (&act)[POL_OUT_MAX], int A,
                                            const NormalConstsT<POL_OUT_MAX>& c, float& logp, float& entropy) {
  const float LOG_SQRT_2PI = 0.91893853320467267f;
  logp = 0.0f; entropy = 0.0f;
#pragma unroll
  for (int k = 0; k < POL_OUT_MAX; ++k) {
    if (k < A) {
      const float d = act[k] - mean[k];
      logp += -(d * d) / c.inv2var[k] - c.log_scale[k] - LOG_SQRT_2PI;
      entropy += 0.5f + LOG_SQRT_2PI + c.log_scale[k];
    }
  }
}
// 4 standard normals from one Philox block (Box-Muller).
__device__ __forceinline__ void normal4(const Philox& r, float (&z)[POL_OUT_MAX]) {
  const float TWO_PI = 6.283185307179586f, S = 1.0f / 16777216.0f;
  const float u1 = ((float)(r.c[0] >> 8) + 0.5f) * S, u2 = ((float)(r.c[1] >> 8) + 0.5f) * S;
  const float u3 = ((float)(r.c[2] >> 8) + 0.5f) * S, u4 = ((float)(r.c[3] >> 8) + 0.5f) * S;
  const float ra = sqrtf(-2.0f * logf(u1)), rb = sqrtf(-2.0f * logf(u3));
  float s, c;
  sincosf(TWO_PI * u2, &s, &c); z[0] = ra * c; z[1] = ra * s;
  sincosf(TWO_PI * u4, &s, &c); z[2] = rb * c; z[3] = rb * s;
}

}  // namespace aur
