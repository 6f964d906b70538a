// Fused PPO minibatch update (row U of the scope table): replaces src/ppo.py:220-269.
//
//   adv_moments_kernel   sum / sum-of-squares of advantages[idx] in fp64 (minibatch normalisation)
//   ppo_grad_kernel      gather -> forward -> loss -> backward -> gradient reduction, one launch
//   grad_reduce_kernel   fixed-order sum of the per-CTA partials -> packed [grads | stats]
//   adam_kernel          clip_grad_norm_ + torch.optim.Adam math on the flat parameter buffer
//
// The actor and the critic are independent MLPs and the PPO loss is separable in them, so
// blockIdx.y selects the net a CTA trains.  A CTA walks tiles of 256 samples.  Per tile the
// per-sample work (forward, loss, backward-data) is thread-per-sample with weights broadcast from
// shared memory into FFMA2 (policy.cuh); the three weight-gradient contractions over the samples
// (dW3 = dout^T h2, dW2 = dz2^T h1, dW1 = dz1^T x) are CTA-level register-tiled GEMMs over
// activations staged feature-major in shared memory, their accumulators living in registers for
// the whole kernel.  This path is fp32-FMA bound (~50 kFLOP per sample vs 40 B gathered).
#include <stdlib.h>

#include "update.cuh"

namespace aur {

__device__ __forceinline__ float block_sum_256(float v, float* sred) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.0f;
  if (threadIdx.x < 8) t = sred[threadIdx.x];
  if (threadIdx.x < 32) {
    t += __shfl_xor_sync(0xffffffffu, t, 4);
    t += __shfl_xor_sync(0xffffffffu, t, 2);
    t += __shfl_xor_sync(0xffffffffu, t, 1);
  }
  return t;   // valid in thread 0
}

// Sum over 64 samples of one feature row (bias gradients): thread -> (row = tid % 64, quarter = tid / 64).
__device__ __forceinline__ float row_quarter_sum(const float* __restrict__ buf, int tid) {
  const float* p = buf + (tid & 63) * UPD_LD + (tid >> 6) * 64;
  float s = 0.0f;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const float4 v = lds4(p + 4 * q);
    s += (v.x + v.y) + (v.z + v.w);
  }
  return s;
}

// CTA-level register-tiled contraction over 64 input features for a tile of 256 samples:
//   out[n][s] = sum_k Wd[k][n] * X[k][s]      X feature-major [64][UPD_LD], Wd = weights duplicated [k][n][2]
// Thread (256 per CTA) = 8 samples x 8 outputs: samples s = sgh*64 + t*32 + sgl*4 + q (t<2, q<4), outputs
// n = ngh*32 + u*8 + ngl*2 + v (u<4, v<2); lane = ngl*8 + sgl, warp = ngh*4 + sgh.  Per k: 2 LDS.128 of X
// (8 lanes x 16 B contiguous: one wavefront each) + 4 LDS.128 of Wd (4 x 16 B contiguous) feed 32 FFMA2 whose
// two halves are two adjacent samples, so nothing is duplicated in registers.  acc[p][o]: p = sample pair
// (t*2 + q/2), o = u*2 + v.
struct GemmMap {
  int s_base, n_base;
  __device__ __forceinline__ GemmMap(int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    const int sgl = lane & 7, ngl = lane >> 3, sgh = warp & 3, ngh = warp >> 2;
    s_base = sgh * 64 + sgl * 4;          // + t*32 + q
    n_base = ngh * 32 + ngl * 2;          // + u*8 + v
  }
};
__device__ __forceinline__ void cta_gemm64(const float* __restrict__ X, const float* __restrict__ Wd, const GemmMap& gm,
                                           float2 (&acc)[4][8]) {
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[p][o] = make_float2(0.f, 0.f);
  const float* xp = X + gm.s_base;
  const float* wp = Wd + 2 * gm.n_base;
#pragma unroll 4
  for (int k = 0; k < UPD_H; ++k) {
    const float4 x0 = lds4(xp + k * UPD_LD), x1 = lds4(xp + k * UPD_LD + 32);
    const float2 xs[4] = {make_float2(x0.x, x0.y), make_float2(x0.z, x0.w), make_float2(x1.x, x1.y), make_float2(x1.z, x1.w)};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float4 w = lds4(wp + k * (2 * UPD_H) + u * 16);     // (w_n, w_n, w_n+1, w_n+1)
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        acc[p][2 * u] = __ffma2_rn(make_float2(w.x, w.y), xs[p], acc[p][2 * u]);
        acc[p][2 * u + 1] = __ffma2_rn(make_float2(w.z, w.w), xs[p], acc[p][2 * u + 1]);
      }
    }
  }
}

// KIND: 0 actor (Categorical), 1 actor (Normal), 2 critic.
template <int KIND>
__device__ void update_net(const UpdDev& a, float* smem) {
  constexpr bool ACTOR = KIND != 2;
  const int tid = threadIdx.x;
  const int OUT = ACTOR ? a.act_dim : 1;
  const int obs_dim = a.obs_dim;
  float* sW = smem;
  float* sW2d = sW + UPD_SW;             // W2 duplicated, [i][j][2]   (forward:  z2[j] = sum_i W2[j][i] h1[i])
  float* sW2Td = sW2d + UPD_WD;          // W2^T duplicated, [j][i][2] (backward: dh1[i] = sum_j W2[j][i] dz2[j])
  float* sZero = sW2Td + UPD_WD;
  float* Hs = sZero + UPD_H;
  float* B2 = Hs + UPD_H * UPD_LD;
  float* sX = B2 + UPD_H * UPD_LD;
  float* sDout = sX + 4 * UPD_LD;
  float* sRed = sDout + 4 * UPD_LD;

  // ---- weights of this net -> shared memory (padded layout + transposed copy of W2)
  const int64_t gA = net_param_count(obs_dim, UPD_H, 2, a.act_dim), gC = net_param_count(obs_dim, UPD_H, 2, 1);
  const float* gnet = ACTOR ? a.params : a.params + gA;
  load_net_to_smem(sW, gnet, obs_dim, UPD_H, 2, OUT, tid, UPD_THREADS);
  const float* sW0 = sW;
  const float* sB0 = sW + UPD_H * POL_IN_PAD;
  const float* sW2 = sB0 + UPD_H;
  const float* sB2 = sW2 + UPD_H * UPD_H;
  const float* sW3 = sB2 + UPD_H;
  const float* sB3 = sW3 + OUT * UPD_H;
  {
    const float* gW2 = gnet + UPD_H * obs_dim + UPD_H;
    for (int e = tid; e < UPD_H * UPD_H; e += UPD_THREADS) {
      const int j = e >> 6, i = e & 63;          // W2[j][i]
      const float w = gW2[e];
      *reinterpret_cast<float2*>(sW2d + (i * UPD_H + j) * 2) = make_float2(w, w);
      *reinterpret_cast<float2*>(sW2Td + (j * UPD_H + i) * 2) = make_float2(w, w);
    }
    if (tid < UPD_H) sZero[tid] = 0.0f;
  }
  NormalConsts nc;
  float logstd_g[POL_OUT_MAX] = {0.f, 0.f, 0.f, 0.f};
  if (KIND == 1) nc = normal_consts(a.params + gA + gC, a.act_dim);
  float adv_mean = 0.0f, adv_den = 1.0f;
  if (ACTOR && a.norm_adv && tid == 0) adv_norm_consts(a, sRed[0], sRed[1]);
  __syncthreads();
  if (ACTOR && a.norm_adv) { adv_mean = sRed[0]; adv_den = sRed[1]; }
  __syncthreads();

  // persistent accumulators
  float2 acc2[4][4];
#pragma unroll
  for (int jj = 0; jj < 4; ++jj)
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) acc2[jj][ii] = make_float2(0.f, 0.f);
  float acc_w3 = 0.f, acc_b3 = 0.f, acc_w1 = 0.f, acc_b2 = 0.f, acc_b1 = 0.f;
  float st0 = 0.f, st1 = 0.f, st2 = 0.f, st3 = 0.f, st4 = 0.f;   // loss, entropy, -logr, r-1-logr, clipped

  const int tj = tid >> 4, ti = tid & 15;
  const GemmMap gm(tid);
  const long long ntiles = (a.m_local + UPD_S - 1) / UPD_S;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    // ================= P1: gather, forward, loss =================
    const long long gi = tile * UPD_S + tid;
    const bool valid = gi < a.m_local;
    const long long row = valid ? (a.idx ? (long long)a.idx[gi] : a.idx_offset + gi) : 0;
    float x[1][POL_IN_PAD];
#pragma unroll
    for (int c = 0; c < POL_IN_PAD; ++c) {
      x[0][c] = (valid && c < obs_dim) ? __ldg(a.obs + row * obs_dim + c) : 0.0f;
      sX[c * UPD_LD + tid] = x[0][c];
    }
    {
      float2 h1[1][UPD_H / 2];
      mlp_first_layer<UPD_H, 1>(sW0, sB0, x, h1);
#pragma unroll
      for (int jp = 0; jp < UPD_H / 2; ++jp) {
        Hs[(2 * jp) * UPD_LD + tid] = h1[0][jp].x;
        Hs[(2 * jp + 1) * UPD_LD + tid] = h1[0][jp].y;
      }
    }
    __syncthreads();
    // ---- hidden layer 2 for the whole tile: h2 = tanh(W2 h1 + b2), CTA-level GEMM -> B2 (feature-major)
    {
      float2 acc[4][8];
      cta_gemm64(Hs, sW2d, gm, acc);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const int n = gm.n_base + u * 8 + v;
          const float b = sB2[n];
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const float2 a0 = acc[2 * t][2 * u + v], a1 = acc[2 * t + 1][2 * u + v];
            *reinterpret_cast<float4*>(B2 + n * UPD_LD + gm.s_base + t * 32) =
                make_float4(tanh_fast(a0.x + b), tanh_fast(a0.y + b), tanh_fast(a1.x + b), tanh_fast(a1.y + b));
          }
        }
    }
    __syncthreads();
    // ---- head (thread per sample): out = W3 h2 + b3
    float2 o2[POL_OUT_MAX];
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) o2[k] = make_float2(0.f, 0.f);
#pragma unroll 4
    for (int j = 0; j < UPD_H; j += 2) {
      const float2 t = make_float2(B2[j * UPD_LD + tid], B2[(j + 1) * UPD_LD + tid]);
#pragma unroll
      for (int k = 0; k < POL_OUT_MAX; ++k)
        if (k < OUT) o2[k] = __ffma2_rn(lds2(sW3 + k * UPD_H + j), t, o2[k]);
    }
    float out[POL_OUT_MAX], dout[POL_OUT_MAX];
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) { out[k] = o2[k].x + o2[k].y + (k < OUT ? sB3[k] : 0.0f); dout[k] = 0.0f; }

    if (valid) {
      if (ACTOR) {
        const float oldlp = __ldg(a.logprobs + row), adv = __ldg(a.advantages + row);
        float newlogp, entropy;
        float dlp[POL_OUT_MAX], dH[POL_OUT_MAX];     // d newlogp / d out_k , d entropy / d out_k
        if (KIND == 0) {
          float m = out[0];
#pragma unroll
          for (int k = 1; k < POL_OUT_MAX; ++k) if (k < OUT) m = fmaxf(m, out[k]);
          float se = 0.0f;
#pragma unroll
          for (int k = 0; k < POL_OUT_MAX; ++k) if (k < OUT) se += expf(out[k] - m);
          const float lse = m + logf(se);
          const int act = (int)__ldg(a.actions + row);
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
          float act[POL_OUT_MAX];
#pragma unroll
          for (int k = 0; k < POL_OUT_MAX; ++k) act[k] = k < OUT ? __ldg(a.actions + row * OUT + k) : 0.0f;
          normal_logp(out, act, OUT, nc, newlogp, entropy);
#pragma unroll
          for (int k = 0; k < POL_OUT_MAX; ++k) {
            const float d = act[k] - out[k], var = nc.std[k] * nc.std[k];
            dlp[k] = k < OUT ? d / var : 0.0f;
            dH[k] = 0.0f;
          }
        }
        const float logr = newlogp - oldlp;
        const float ratio = expf(logr);
        const float advn = a.norm_adv ? (adv - adv_mean) / adv_den : adv;
        const float l1 = -advn * ratio;
        const float l2 = -advn * fminf(fmaxf(ratio, a.clip_lo), a.clip_hi);
        const float w1 = l1 > l2 ? 1.0f : (l1 == l2 ? 0.5f : 0.0f);
        const float inr = (ratio >= a.clip_lo && ratio <= a.clip_hi) ? 1.0f : 0.0f;
        const float g_logp = -advn * (w1 + (1.0f - w1) * inr) * ratio * a.inv_m;
        const float g_H = -a.ent_c * a.inv_m;
#pragma unroll
        for (int k = 0; k < POL_OUT_MAX; ++k) dout[k] = g_logp * dlp[k] + g_H * dH[k];
        if (KIND == 1) {
#pragma unroll
          for (int k = 0; k < POL_OUT_MAX; ++k) {
            if (k < OUT) {
              const float d = out[k] - __ldg(a.actions + row * OUT + k);
              logstd_g[k] += g_logp * (d * d / (nc.std[k] * nc.std[k]) - 1.0f) + g_H;
            }
          }
        }
        st0 += fmaxf(l1, l2); st1 += entropy; st2 += -logr; st3 += (ratio - 1.0f) - logr;
        st4 += fabsf(ratio - 1.0f) > a.clip ? 1.0f : 0.0f;
      } else {
        const float R = __ldg(a.returns + row), vold = __ldg(a.values + row), v = out[0];
        if (a.clip_vloss) {
          const float du = v - R, vu = du * du;
          const float d = v - vold, vc = vold + fminf(fmaxf(d, -a.clip), a.clip);
          const float dc = vc - R, lc = dc * dc;
          const float w1 = vu > lc ? 1.0f : (vu == lc ? 0.5f : 0.0f);
          const float inr = (d >= -a.clip && d <= a.clip) ? 1.0f : 0.0f;
          dout[0] = (w1 * du + (1.0f - w1) * dc * inr) * a.vf_c * a.inv_m;
          st0 += 0.5f * fmaxf(vu, lc);
        } else {
          const float d = v - vold;                  // reference quirk ppo.py:261: b_values, not b_returns
          dout[0] = d * a.vf_c * a.inv_m;
          st0 += 0.5f * d * d;
        }
      }
    }
#pragma unroll
    for (int k = 0; k < POL_OUT_MAX; ++k) sDout[k * UPD_LD + tid] = dout[k];
    __syncthreads();

    // ================= G1: dW3 += dout^T h2, db3 += sum dout =================
    {
      const int k = tid >> 6, j = tid & 63;
      if (k < OUT) {
        const float* hp = B2 + j * UPD_LD;
        const float* dp = sDout + k * UPD_LD;
        float2 s2 = make_float2(0.f, 0.f);
#pragma unroll 8
        for (int s4 = 0; s4 < UPD_S / 4; ++s4) {
          const float4 hv = lds4(hp + 4 * s4), dv = lds4(dp + 4 * s4);
          s2 = __ffma2_rn(make_float2(hv.x, hv.y), make_float2(dv.x, dv.y), s2);
          s2 = __ffma2_rn(make_float2(hv.z, hv.w), make_float2(dv.z, dv.w), s2);
        }
        acc_w3 += s2.x + s2.y;
      }
      if (tid < OUT) {
        const float* dp = sDout + tid * UPD_LD;
        float s = 0.0f;
        for (int s4 = 0; s4 < UPD_S / 4; ++s4) { const float4 dv = lds4(dp + 4 * s4); s += (dv.x + dv.y) + (dv.z + dv.w); }
        acc_b3 += s;
      }
    }
    __syncthreads();

    // ================= P2: dz2 = (W3^T dout) * (1 - h2^2), in place over h2 =================
#pragma unroll 4
    for (int j = 0; j < UPD_H; ++j) {
      const float h2 = B2[j * UPD_LD + tid];
      float dh = 0.0f;
#pragma unroll
      for (int k = 0; k < POL_OUT_MAX; ++k) if (k < OUT) dh = fmaf(sW3[k * UPD_H + j], dout[k], dh);
      B2[j * UPD_LD + tid] = dh * fmaf(-h2, h2, 1.0f);
    }
    __syncthreads();

    // ================= G2: dW2 += dz2^T h1 (64x64 outputs, K = 256 samples), db2 =================
#pragma unroll 2
    for (int s4 = 0; s4 < UPD_S / 4; ++s4) {
      float4 av[4], bv[4];
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) av[jj] = lds4(B2 + (tj + 16 * jj) * UPD_LD + 4 * s4);
#pragma unroll
      for (int ii = 0; ii < 4; ++ii) bv[ii] = lds4(Hs + (ti + 16 * ii) * UPD_LD + 4 * s4);
#pragma unroll
      for (int jj = 0; jj < 4; ++jj)
#pragma unroll
        for (int ii = 0; ii < 4; ++ii) {
          float2 s = __ffma2_rn(make_float2(av[jj].x, av[jj].y), make_float2(bv[ii].x, bv[ii].y), acc2[jj][ii]);
          acc2[jj][ii] = __ffma2_rn(make_float2(av[jj].z, av[jj].w), make_float2(bv[ii].z, bv[ii].w), s);
        }
    }
    acc_b2 += row_quarter_sum(B2, tid);

    // ================= P3: dz1 = (W2^T dz2) * (1 - h1^2), CTA-level GEMM =================
    {
      float2 acc[4][8];
      cta_gemm64(B2, sW2Td, gm, acc);
      float4 dzv[8][2];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const int n = gm.n_base + u * 8 + v;
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const float4 hv = lds4(Hs + n * UPD_LD + gm.s_base + t * 32);
            const float2 a0 = acc[2 * t][2 * u + v], a1 = acc[2 * t + 1][2 * u + v];
            dzv[2 * u + v][t] = make_float4(a0.x * fmaf(-hv.x, hv.x, 1.0f), a0.y * fmaf(-hv.y, hv.y, 1.0f),
                                            a1.x * fmaf(-hv.z, hv.z, 1.0f), a1.y * fmaf(-hv.w, hv.w, 1.0f));
          }
        }
      __syncthreads();            // every thread is done reading h1 (G2, P3)
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const int n = gm.n_base + u * 8 + v;
#pragma unroll
          for (int t = 0; t < 2; ++t) *reinterpret_cast<float4*>(Hs + n * UPD_LD + gm.s_base + t * 32) = dzv[2 * u + v][t];
        }
    }
    __syncthreads();

    // ================= G3: dW1 += dz1^T x, db1 =================
    {
      const int c = tid >> 6, j = tid & 63;
      const float* zp = Hs + j * UPD_LD;
      const float* xp = sX + c * UPD_LD;
      float2 s2 = make_float2(0.f, 0.f);
#pragma unroll 8
      for (int s4 = 0; s4 < UPD_S / 4; ++s4) {
        const float4 zv = lds4(zp + 4 * s4), xv = lds4(xp + 4 * s4);
        s2 = __ffma2_rn(make_float2(zv.x, zv.y), make_float2(xv.x, xv.y), s2);
        s2 = __ffma2_rn(make_float2(zv.z, zv.w), make_float2(xv.z, xv.w), s2);
      }
      acc_w1 += s2.x + s2.y;
      acc_b1 += row_quarter_sum(Hs, tid);
    }
    __syncthreads();            // tile buffers free for the next tile
  }

  // ---- write this CTA's partial (the net's flat parameter order, then statistics)
  float* part = a.partials + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * UPD_PSTRIDE;
  const int oW1 = 0, oB1 = UPD_H * obs_dim, oW2 = oB1 + UPD_H, oB2 = oW2 + UPD_H * UPD_H, oW3 = oB2 + UPD_H,
            oB3 = oW3 + OUT * UPD_H, oLS = oB3 + OUT;
  {
    const int c = tid >> 6, j = tid & 63;
    if (c < obs_dim) part[oW1 + j * obs_dim + c] = acc_w1;
    if (c < OUT) part[oW3 + c * UPD_H + j] = acc_w3;
    if (tid < OUT) part[oB3 + tid] = acc_b3;
  }
#pragma unroll
  for (int jj = 0; jj < 4; ++jj)
#pragma unroll
    for (int ii = 0; ii < 4; ++ii)
      part[oW2 + (tj + 16 * jj) * UPD_H + (ti + 16 * ii)] = acc2[jj][ii].x + acc2[jj][ii].y;
  // bias row-sums: 4 quarter partials per row -> combine through shared memory
  __syncthreads();
  sRed[tid] = acc_b2;
  Hs[tid] = acc_b1;
  __syncthreads();
  if (tid < UPD_H) {
    part[oB2 + tid] = (sRed[tid] + sRed[tid + 64]) + (sRed[tid + 128] + sRed[tid + 192]);
    part[oB1 + tid] = (Hs[tid] + Hs[tid + 64]) + (Hs[tid + 128] + Hs[tid + 192]);
  }
  float* sred8 = B2;   // scratch for block sums
  float s;
  if (KIND == 1) {
    for (int k = 0; k < POL_OUT_MAX; ++k) {
      s = block_sum_256(logstd_g[k], sred8);
      if (tid == 0 && k < OUT) part[oLS + k] = s;
    }
  }
  float* stat = part + UPD_STAT_OFF;
  s = block_sum_256(st0, sred8); if (tid == 0) stat[ACTOR ? AUR_STAT_POLICY_LOSS : AUR_STAT_VALUE_LOSS] = s;
  if (ACTOR) {
    s = block_sum_256(st1, sred8); if (tid == 0) stat[AUR_STAT_ENTROPY] = s;
    s = block_sum_256(st2, sred8); if (tid == 0) stat[AUR_STAT_OLD_APPROX_KL] = s;
    s = block_sum_256(st3, sred8); if (tid == 0) stat[AUR_STAT_APPROX_KL] = s;
    s = block_sum_256(st4, sred8); if (tid == 0) stat[AUR_STAT_CLIPFRAC] = s;
  }
}

__global__ void __launch_bounds__(UPD_THREADS, 1) ppo_grad_kernel(UpdDev a) {
  extern __shared__ __align__(16) float smem[];
  if (blockIdx.y == 0) {
    if (a.continuous) update_net<1>(a, smem);
    else update_net<0>(a, smem);
  } else {
    update_net<2>(a, smem);
  }
}

// Population form of the reduction (grid.y = K): member k's ncta real partial rows at partials + k * part_stride, summed with
// the quarter boundaries of the single run's chunk_ncta rows (the rows a single run has beyond ncta are the exact zeros its
// idle CTAs write), into grads_out + k * grads_stride; inactive members are skipped.
struct PopRed {
  int chunk_ncta;
  long long part_stride, grads_stride;
  const int32_t* active;
};

// grads_out[p] = sum over CTAs of the partials, in CTA order, fp64 accumulation.
template <bool POP = false>
__global__ void grad_reduce_kernel(const float* __restrict__ partials, int ncta, int obs_dim, int act_dim, int continuous,
                                   int hidden, int nl, int pstride, float* __restrict__ grads_out, DpDev dp,
                                   unsigned int* __restrict__ ticket, PopRed pop) {
  if constexpr (POP) {
    if (!pop.active[blockIdx.y]) return;
    partials += blockIdx.y * pop.part_stride;
    grads_out += blockIdx.y * pop.grads_stride;
  }
  const int64_t nA = net_param_count(obs_dim, hidden, nl, act_dim), nC = net_param_count(obs_dim, hidden, nl, 1);
  const int64_t P = nA + nC + (continuous ? act_dim : 0);
  // four lanes per output: lane q sums its quarter of the CTA partials in CTA order (fp64), the quarters are combined as
  // (q0 + q1) + (q2 + q3) - a fixed order, so the result is bit-reproducible and the same on every rank
  const int64_t tg = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i = tg >> 2;
  const int q = (int)(tg & 3);
  const bool live = i < P + AUR_NUM_STATS;
  double s = 0.0;
  if (live) {
    int net; int64_t off;
    bool zero = false;
    if (i < nA) { net = 0; off = i; }
    else if (i < nA + nC) { net = 1; off = i - nA; }
    else if (i < P) { net = 0; off = nA + (i - nA - nC); }          // actor_logstd sits after the actor's own params
    else {
      const int sidx = (int)(i - P);
      net = (sidx == AUR_STAT_VALUE_LOSS) ? 1 : 0;
      off = (pstride - AUR_NUM_STATS) + sidx;
      zero = sidx > AUR_STAT_CLIPFRAC;
    }
    if (!zero) {
      const float* p = partials + (size_t)net * ncta * pstride + off;
      const int chunk = ((POP ? pop.chunk_ncta : ncta) + 3) >> 2;
      int c = q * chunk;
      const int c1 = min(ncta, c + chunk);
      for (; c + 8 <= c1; c += 8) {                     // 8 loads in flight
        float v8[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v8[k] = __ldcg(p + (size_t)(c + k) * pstride);
#pragma unroll
        for (int k = 0; k < 8; ++k) s += (double)v8[k];
      }
      for (; c < c1; ++c) s += (double)__ldcg(p + (size_t)c * pstride);
    }
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);              // q0 + q1 | q2 + q3 (IEEE addition is commutative: both lanes agree)
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  __shared__ float sv[64];                              // the block's 64 outputs, so that the stores below are coalesced
  if (q == 0) sv[threadIdx.x >> 2] = (float)s;
  __syncthreads();
  if (threadIdx.x < 64) {
    const int64_t o = (int64_t)blockIdx.x * 64 + threadIdx.x;
    if (o < P + AUR_NUM_STATS) {
      const float v = sv[threadIdx.x];
      grads_out[o] = v;
      if (dp.world > 1) {                                // push this rank's sums into every rank's exchange area
        const size_t slot_off = DP_OFF_GRAD + ((size_t)(dp.seq & 1u) * DP_MAX + dp.rank) * dp_grad_stride(P) * sizeof(float);
        for (int r = 0; r < dp.world; ++r) reinterpret_cast<float*>(dp.peer[r] + slot_off)[o] = v;
      }
    }
  }
  if (dp.world > 1) {                                    // the last block to finish releases the flags
    __shared__ bool last;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (last) {
      __threadfence_system();
      if ((int)threadIdx.x < dp.world)
        st_release_sys(reinterpret_cast<uint32_t*>(dp.peer[threadIdx.x] + DP_OFF_FLAG_GRAD) + dp.rank, dp.seq);
      if (threadIdx.x == 0) *ticket = 0u;
    }
  }
}

// sum / sum of squares of advantages[idx] (fp64), finalised by the last CTA to finish.
__global__ void __launch_bounds__(256) adv_moments_kernel(long long m, const int32_t* __restrict__ idx, long long idx_offset,
                                                        const float* __restrict__ adv, double* __restrict__ partial,
                                                        unsigned int* __restrict__ ticket, double* __restrict__ out, DpDev dp) {
  __shared__ double sh[2][8];
  __shared__ bool last;
  double s = 0.0, ss = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < m; i += 4 * stride) {            // four independent gathers in flight, summed in index order
    float v4[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long row = idx ? (long long)__ldg(idx + i + k * stride) : idx_offset + i + k * stride;
      v4[k] = __ldg(adv + row);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) { const double v = (double)v4[k]; s += v; ss += v * v; }
  }
  for (; i < m; i += stride) {
    const long long row = idx ? (long long)idx[i] : idx_offset + i;
    const double v = (double)__ldg(adv + row);
    s += v; ss += v * v;
  }
  s = warp_sum(s); ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = ss; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int w = 0; w < 8; ++w) { a += sh[0][w]; b += sh[1][w]; }
    partial[2 * blockIdx.x] = a; partial[2 * blockIdx.x + 1] = b;
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {                                            // block-uniform: the whole last CTA finalises, in a fixed order
    __threadfence();
    double a = 0.0, b = 0.0;
    for (unsigned c = threadIdx.x; c < gridDim.x; c += blockDim.x) { a += __ldcg(partial + 2 * c); b += __ldcg(partial + 2 * c + 1); }
    a = warp_sum(a); b = warp_sum(b);
    __syncthreads();                                     // sh[][] of the first phase has been consumed by thread 0
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = a; sh[1][threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
      a = 0.0; b = 0.0;
      for (int w = 0; w < 8; ++w) { a += sh[0][w]; b += sh[1][w]; }
      out[0] = a; out[1] = b; out[2] = (double)m;
      sh[0][0] = a; sh[1][0] = b;
      *ticket = 0u;
    }
  }
  if (dp.world > 1 && last) {                            // push the local moments to every rank, then release the flags
    __syncthreads();
    if ((int)threadIdx.x < dp.world) {
      unsigned char* area = dp.peer[threadIdx.x];
      double* rm = reinterpret_cast<double*>(area + DP_OFF_MOM) + ((size_t)(dp.seq & 1u) * DP_MAX + dp.rank) * 4;
      rm[0] = sh[0][0]; rm[1] = sh[1][0]; rm[2] = (double)m;
      __threadfence_system();
      st_release_sys(reinterpret_cast<uint32_t*>(area + DP_OFF_FLAG_MOM) + dp.rank, dp.seq);
    }
  }
}

// The same for all n_mb minibatches of an iteration at once: grid = (CTAs per minibatch, n_mb).  The last CTA of a minibatch
// finalises it (fixed order) and, data-parallel, pushes its three moments to every rank; the last minibatch to finish
// releases the flags - ONE rendezvous per iteration instead of one per minibatch.
// POP (aur_pop_adv_moments_multi): grid (cpm, n_mb, K), entry (k, y) = index list k * n_mb + y; the CTAs only write their
// partials, pop_moments_final_kernel combines them in the order of the last-CTA finalisation below.
template <bool POP = false>
__global__ void __launch_bounds__(256) adv_moments_multi_kernel(long long m, const int32_t* __restrict__ idx, long long idx_stride,
                                                              const float* __restrict__ adv, double* __restrict__ partial,
                                                              unsigned int* __restrict__ tickets, double* __restrict__ out, DpDev dp) {
  __shared__ double sh[2][8];
  __shared__ bool last, last_of_all;
  const int y = blockIdx.y;
  const long long entry = POP ? (long long)blockIdx.z * gridDim.y + y : y;
  const int32_t* my_idx = idx ? idx + entry * idx_stride : nullptr;
  const long long row0 = entry * idx_stride;
  double s = 0.0, ss = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < m; i += 4 * stride) {
    float v4[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long row = my_idx ? (long long)__ldg(my_idx + i + k * stride) : row0 + i + k * stride;
      v4[k] = __ldg(adv + row);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) { const double v = (double)v4[k]; s += v; ss += v * v; }
  }
  for (; i < m; i += stride) {
    const long long row = my_idx ? (long long)my_idx[i] : row0 + i;
    const double v = (double)__ldg(adv + row);
    s += v; ss += v * v;
  }
  s = warp_sum(s); ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = ss; }
  __syncthreads();
  double* part = partial + (size_t)entry * gridDim.x * 2;
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int w = 0; w < 8; ++w) { a += sh[0][w]; b += sh[1][w]; }
    part[2 * blockIdx.x] = a; part[2 * blockIdx.x + 1] = b;
    if constexpr (!POP) {
      __threadfence();
      last = atomicAdd(tickets + 1 + y, 1u) == gridDim.x - 1;
      last_of_all = false;
    }
  }
  if constexpr (POP) return;                             // the whole CTA: pop_moments_final_kernel finalises
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (unsigned c = 0; c < gridDim.x; ++c) { a += __ldcg(part + 2 * c); b += __ldcg(part + 2 * c + 1); }
    out[3 * y] = a; out[3 * y + 1] = b; out[3 * y + 2] = (double)m;
    tickets[1 + y] = 0u;
    if (dp.world > 1) {
      for (int r = 0; r < dp.world; ++r) {
        double* rm = reinterpret_cast<double*>(dp.peer[r] + DP_OFF_MOMX) + ((size_t)(dp.mom_seq & 1u) * DP_MAX + dp.rank) * DP_MAXMB * 4 +
                     (size_t)y * 4;
        rm[0] = a; rm[1] = b; rm[2] = (double)m;
      }
      __threadfence_system();
      last_of_all = atomicAdd(tickets, 1u) == gridDim.y - 1;
    }
  }
  __syncthreads();
  if (last_of_all) {                                     // every minibatch of this rank has been pushed: release the flags
    __threadfence_system();
    if ((int)threadIdx.x < dp.world)
      st_release_sys(reinterpret_cast<uint32_t*>(dp.peer[threadIdx.x] + DP_OFF_FLAG_MOMX) + dp.rank, dp.mom_seq);
    if (threadIdx.x == 0) tickets[0] = 0u;
  }
}

// the finalisation of adv_moments_multi_kernel<true>: entry e = (member, minibatch) sums its cpm CTA partials in CTA order
__global__ void __launch_bounds__(128) pop_moments_final_kernel(int entries, int cpm, long long m, const double* __restrict__ partial,
                                                              double* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= entries) return;
  const double* part = partial + (size_t)e * cpm * 2;
  double a = 0.0, b = 0.0;
  for (int c = 0; c < cpm; ++c) { a += __ldcg(part + 2 * c); b += __ldcg(part + 2 * c + 1); }
  out[3 * e] = a; out[3 * e + 1] = b; out[3 * e + 2] = (double)m;
}

// clip_grad_norm_ (all parameters, torch semantics) + Adam on one flat buffer by one CTA: the part of adam_kernel after the
// data-parallel gather, shared with pop_adam_kernel
__device__ __forceinline__ void adam_clip_step(int64_t P, float* __restrict__ params, const float* __restrict__ g_in,
                                               float* __restrict__ m1, float* __restrict__ m2, float lr_over_bc1, float beta1,
                                               float beta2, float eps, float sqrt_bc2, float max_norm, float inv_m, float ent_c,
                                               float vf_c, float* __restrict__ stats_out) {
  __shared__ double sh[32];
  __shared__ float coef_s, norm_s;
  double ss = 0.0;
  for (int64_t i = threadIdx.x; i < P; i += blockDim.x) { const double g = g_in[i]; ss += g * g; }
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 32; ++w) t += sh[w];
    const float total = (float)sqrt(t);
    float coef = max_norm / (total + 1e-6f);
    coef = coef > 1.0f ? 1.0f : coef;
    coef_s = coef; norm_s = total;
  }
  __syncthreads();
  const float coef = coef_s;
  for (int64_t i = threadIdx.x; i < P; i += blockDim.x) {
    const float g = g_in[i] * coef;
    float m = m1[i], v = m2[i];
    m = m + (g - m) * (1.0f - beta1);                        // exp_avg.lerp_(grad, 1 - beta1)
    v = v * beta2 + (1.0f - beta2) * g * g;                  // exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2)
    const float denom = sqrtf(v) / sqrt_bc2 + eps;
    params[i] = params[i] - lr_over_bc1 * (m / denom);       // param.addcdiv_(exp_avg, denom, value=-step_size)
    m1[i] = m; m2[i] = v;
  }
  if (stats_out && threadIdx.x < AUR_NUM_STATS) {
    const float* st = g_in + P;
    float v = 0.0f;
    if (threadIdx.x <= AUR_STAT_CLIPFRAC) v = st[threadIdx.x] * inv_m;
    if (threadIdx.x == AUR_STAT_GRAD_NORM) v = norm_s;
    if (threadIdx.x == AUR_STAT_LOSS)
      v = st[AUR_STAT_POLICY_LOSS] * inv_m - ent_c * (st[AUR_STAT_ENTROPY] * inv_m) + (st[AUR_STAT_VALUE_LOSS] * inv_m) * vf_c;
    stats_out[threadIdx.x] = v;
  }
}

// clip_grad_norm_ (all parameters, torch semantics) + Adam, one CTA (P ~ 9e3).
__global__ void __launch_bounds__(1024) adam_kernel(int64_t P, float* __restrict__ params, float* __restrict__ g_in,
                                                   float* __restrict__ m1, float* __restrict__ m2, float lr_over_bc1,
                                                   float beta1, float beta2, float eps, float sqrt_bc2, float max_norm,
                                                   float inv_m, float ent_c, float vf_c, float* __restrict__ stats_out, DpDev dp) {
  if (dp.world > 1) {
    // data-parallel: the all-reduce happens HERE.  Every rank pushed its [grads | stats] sums into our exchange
    // area (grad_reduce_kernel); wait for the flags, add the G vectors in rank order (bit-identical on every
    // rank), keep the global sums in g_in, then clip + Adam as usual on replicated parameters.
    unsigned char* me = dp.peer[dp.rank];
    const uint64_t t_in = global_timer_ns();
    if ((int)threadIdx.x < dp.world) dp_wait_flag(reinterpret_cast<const uint32_t*>(me + DP_OFF_FLAG_GRAD) + threadIdx.x, dp.seq, me);
    __syncthreads();
    if (threadIdx.x == 0) {                              // wall time this rank stood still waiting for the slowest peer
      unsigned long long* w = reinterpret_cast<unsigned long long*>(me + DP_OFF_WAIT) + 4;
      w[0] += (unsigned long long)(global_timer_ns() - t_in);
      w[1] += 1ull;
    }
    // a wait gave up (a peer is gone): the sums are incomplete - do NOT step the parameters on them; the status word stays set
    // and the host raises on every rank (ppo.train checks it once per update)
    if (*reinterpret_cast<volatile uint32_t*>(me + DP_OFF_STATUS) != 0u) return;
    const int gs = dp_grad_stride(P);
    const float* rg = reinterpret_cast<const float*>(me + DP_OFF_GRAD) + (size_t)(dp.seq & 1u) * DP_MAX * gs;
    for (int64_t i = threadIdx.x; i < P + AUR_NUM_STATS; i += blockDim.x) {
      float g = 0.0f;
      for (int r = 0; r < dp.world; ++r) g += __ldcg(rg + (size_t)r * gs + i);
      g_in[i] = g;
    }
    __syncthreads();
  }
  adam_clip_step(P, params, g_in, m1, m2, lr_over_bc1, beta1, beta2, eps, sqrt_bc2, max_norm, inv_m, ent_c, vf_c, stats_out);
}

// Population clip + Adam (aur_pop_update_apply): one CTA per member with the member's learning rate, step count, bias
// corrections (host table) and coefficients; at the end of an epoch a member over its target_kl leaves `active`.
struct PopAdam {
  int64_t P;
  float* params;
  const float* grads;
  float *m1, *m2;
  int64_t* steps;
  int32_t* active;
  const aur_pop_hparams* hp;
  const double* bc;
  int64_t bc_len;
  double frac;
  float beta1, beta2, eps, inv_m;
  float* stats;
  int stats_rows, stats_row, epoch_end;
};
__global__ void __launch_bounds__(1024) pop_adam_kernel(PopAdam a) {
  const int k = blockIdx.x;
  if (!a.active[k]) return;
  const int64_t step = a.steps[k] + 1;
  if (step >= a.bc_len) return;                        // the host sizes the table for every step of the run
  const aur_pop_hparams h = a.hp[k];
  const double lr = h.learning_rate * a.frac;          // ppo.run_update: frac * learning_rate (1.0 without the anneal)
  const double bc1 = a.bc[2 * step], bc2 = a.bc[2 * step + 1];
  const float* g = a.grads + (size_t)k * (a.P + AUR_NUM_STATS);
  float* st = a.stats ? a.stats + ((size_t)k * a.stats_rows + a.stats_row) * AUR_NUM_STATS : nullptr;
  adam_clip_step(a.P, a.params + (size_t)k * a.P, g, a.m1 + (size_t)k * a.P, a.m2 + (size_t)k * a.P, (float)(lr / bc1), a.beta1,
                 a.beta2, a.eps, (float)sqrt(bc2), (float)h.max_grad_norm, a.inv_m, (float)h.entropy_coeff, (float)h.value_coeff, st);
  if (threadIdx.x == 0) {
    a.steps[k] = step;
    // ppo.py:271-273 on the value the stats row holds (fp32, compared in double as `stats_rows[n - 1, 4].item() > target_kl`)
    if (a.epoch_end && (double)(g[a.P + AUR_STAT_APPROX_KL] * a.inv_m) > h.target_kl) a.active[k] = 0;
  }
}

// 0 = SIMT fp32 (ppo_grad_kernel, kept as an independent cross-check), 1 = tcgen05 bf16x2-split with two threads per
// sample, 2 = the same with four threads per sample (ppo_grad_tc_kernel<2|4>).  AUR_UPDATE_IMPL=simt|tc|tc4 or
// aur_ppo_update_set_impl() select it.
#ifndef AUR_UPDATE_DEFAULT_IMPL
#define AUR_UPDATE_DEFAULT_IMPL 1
#endif
static int g_update_impl = -1;
static int update_impl() {
  if (g_update_impl < 0) {
    const char* e = getenv("AUR_UPDATE_IMPL");
    if (!e) g_update_impl = AUR_UPDATE_DEFAULT_IMPL;
    else if (e[0] == 's' || e[0] == '0') g_update_impl = 0;
    else if (e[0] == '2' || (e[0] == 't' && e[1] == 'c' && e[2] == '4')) g_update_impl = 2;
    else if (e[0] == '3' || e[0] == 'g') g_update_impl = 3;
    else g_update_impl = 1;
  }
  return g_update_impl;
}
static int upd_grid_x() {
  int g = sm_count() / 2;
  return g < 1 ? 1 : g;
}
// workspace: [2][grid_x][PSTRIDE] partials | moments partials (fp64) | ticket
static size_t ws_partials_floats() { return (size_t)2 * sm_count() * UPD_PSTRIDE; }
static size_t ws_bytes() { return ws_partials_floats() * sizeof(float) + (2 * MOM_CTAS) * sizeof(double) + 64; }

// update_generic.cu: the kernel for every shape other than 64 x 2 / widths <= 4 (and, with impl 3, a cross-check there)
int check_generic_policy(const aur_policy_desc& p, const char* who);
size_t gen_workspace_floats(const aur_policy_desc& p);
int gen_pstride(const aur_policy_desc& p);
int launch_ppo_grad_generic(const UpdDev& d, const aur_policy_desc& p, float* ws, int* gx_out, float** part_out, cudaStream_t s);
// update_wide.cu: hidden 128 / 256 layer by layer on tensor cores
bool wide_eligible(const aur_policy_desc& p);
size_t wide_workspace_bytes(const aur_policy_desc& p);
int update_wide_enabled();
void set_update_wide(int on);
int launch_ppo_grad_wide(const UpdDev& d, const aur_policy_desc& p, float* ws, int* gx_out, float** part_out, cudaStream_t s);

static bool is_headline_shape(const aur_policy_desc& p) {
  return p.hidden_dim == 64 && p.num_layers == 2 && p.obs_dim >= 1 && p.obs_dim <= POL_IN_PAD && p.act_dim >= 1 &&
         p.act_dim <= POL_OUT_MAX;
}
static int check_update_policy(const aur_policy_desc& p, const char* who) {
  if (is_headline_shape(p)) return 0;
  return check_generic_policy(p, who);
}

}  // namespace aur

extern "C" int64_t aur_ppo_update_workspace_bytes(const aur_policy_desc* desc) {
  if (!desc) return AUR_ERR_ARG;
  int rc = aur::check_update_policy(*desc, "aur_ppo_update_workspace_bytes");
  if (rc) return rc;
  // [specialised kernels' partials | moments partials | tickets] then the generic kernel's staged parameters + slabs
  return (int64_t)(aur::ws_bytes() + aur::gen_workspace_floats(*desc) * sizeof(float) + aur::wide_workspace_bytes(*desc));
}

namespace aur {
static int make_dp(const aur_dp_ctx* c, uint32_t seq, DpDev& d, const char* who) {
  d.world = 1; d.rank = 0; d.seq = seq;
  d.mom_seq = 0; d.mom_index = 0;
  for (int r = 0; r < DP_MAX; ++r) d.peer[r] = nullptr;
  if (!c || c->world <= 1) return 0;
  if (c->world > DP_MAX || c->rank < 0 || c->rank >= c->world || seq == 0) {
    set_error("%s: bad data-parallel context (world %d, rank %d, seq %u)", who, c->world, c->rank, seq); return AUR_ERR_ARG;
  }
  for (int r = 0; r < c->world; ++r) {
    if (!c->peer[r]) { set_error("%s: exchange area of rank %d is not mapped", who, r); return AUR_ERR_ARG; }
    d.peer[r] = static_cast<unsigned char*>(c->peer[r]);
  }
  d.world = c->world; d.rank = c->rank;
  return 0;
}
}  // namespace aur

extern "C" int aur_ppo_adv_moments(int64_t m, const int32_t* idx, int64_t idx_offset, const float* advantages,
                                   double* moments_out, float* workspace, void* stream) {
  return aur_ppo_adv_moments_dp(m, idx, idx_offset, advantages, moments_out, workspace, nullptr, 0, stream);
}

extern "C" int aur_ppo_adv_moments_dp(int64_t m, const int32_t* idx, int64_t idx_offset, const float* advantages,
                                      double* moments_out, float* workspace, const aur_dp_ctx* dp, uint32_t seq, void* stream) {
  using namespace aur;
  DpDev dpd;
  { int rc = make_dp(dp, seq, dpd, "aur_ppo_adv_moments_dp"); if (rc) return rc; }
  if (m <= 0 || !advantages || !moments_out || !workspace) { set_error("aur_ppo_adv_moments: bad arguments"); return AUR_ERR_ARG; }
  double* partial = reinterpret_cast<double*>(workspace + ws_partials_floats());
  unsigned int* ticket = stream_tickets((cudaStream_t)stream);      // library-owned: the workspace need not be zeroed
  if (!ticket) return AUR_ERR_ARG;
  long long grid = (m + 255) / 256;
  if (grid > MOM_CTAS) grid = MOM_CTAS;
  adv_moments_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((long long)m, idx, (long long)idx_offset, advantages,
                                                                      partial, ticket, moments_out, dpd);
  AUR_LAUNCH_OK("adv_moments_kernel");
  return 0;
}

extern "C" int aur_ppo_adv_moments_multi(int32_t n_mb, int64_t m, const int32_t* idx, int64_t idx_stride, const float* advantages,
                                         double* moments_out, float* workspace, const aur_dp_ctx* dp, uint32_t mom_seq, void* stream) {
  using namespace aur;
  if (n_mb <= 0 || n_mb > DP_MAXMB || m <= 0 || idx_stride < m || !advantages || !moments_out || !workspace) {
    set_error("aur_ppo_adv_moments_multi: bad arguments (1 <= n_mb <= %d, idx_stride >= m)", DP_MAXMB); return AUR_ERR_ARG;
  }
  DpDev dpd;
  { int rc = make_dp(dp, mom_seq ? mom_seq : 1u, dpd, "aur_ppo_adv_moments_multi"); if (rc) return rc; }
  if (dpd.world > 1 && mom_seq == 0) { set_error("aur_ppo_adv_moments_multi: data-parallel needs mom_seq >= 1"); return AUR_ERR_ARG; }
  dpd.mom_seq = mom_seq;
  // all n_mb x cpm CTAs share the moment-partial region of the workspace (2 x MOM_CTAS doubles)
  int cpm = MOM_CTAS / n_mb;
  if (cpm < 1) cpm = 1;
  const long long need = (m + 255) / 256;
  if (cpm > need) cpm = (int)need;
  double* partial = reinterpret_cast<double*>(workspace + ws_partials_floats());
  unsigned int* tickets = stream_tickets((cudaStream_t)stream);
  if (!tickets) return AUR_ERR_ARG;
  adv_moments_multi_kernel<<<dim3((unsigned)cpm, (unsigned)n_mb), 256, 0, (cudaStream_t)stream>>>(
      (long long)m, idx, (long long)idx_stride, advantages, partial, tickets + 16, moments_out, dpd);
  AUR_LAUNCH_OK("adv_moments_multi_kernel");
  return 0;
}

extern "C" int aur_ppo_update_set_impl(int impl) {
  if (impl < 0 || impl > 3) { aur::set_error("aur_ppo_update_set_impl: impl must be 0 (simt), 1 (tensor core), 2 (tensor core, 4 threads per sample) or 3 (shape-generic)"); return AUR_ERR_ARG; }
  aur::g_update_impl = impl;
  return 0;
}
extern "C" int aur_ppo_update_get_impl(void) { return aur::update_impl(); }
extern "C" int aur_ppo_update_set_wide(int on) {
  if (on != 0 && on != 1) { aur::set_error("aur_ppo_update_set_wide: 0 (shape-generic SIMT kernel) or 1 (layer-wise tensor-core path)"); return AUR_ERR_ARG; }
  aur::set_update_wide(on);
  return 0;
}
extern "C" int aur_ppo_update_get_wide(void) { return aur::update_wide_enabled(); }

extern "C" int aur_ppo_update_grad(const aur_update_args* args, void* stream) {
  using namespace aur;
  if (!args) { set_error("aur_ppo_update_grad: null args"); return AUR_ERR_ARG; }
  const aur_update_args& u = *args;
  int rc = check_update_policy(u.policy, "aur_ppo_update_grad");
  if (rc) return rc;
  if (u.m_local < 0 || u.m_total <= 0 || !u.obs || !u.actions || !u.logprobs || !u.advantages || !u.returns || !u.values ||
      !u.params || !u.workspace || !u.grads_out || (u.norm_adv && !u.adv_moments)) {
    set_error("aur_ppo_update_grad: bad arguments"); return AUR_ERR_ARG;
  }
  UpdDev d;
  d.m_local = u.m_local; d.idx = u.idx; d.idx_offset = u.idx_offset;
  d.obs = u.obs; d.actions = u.actions; d.logprobs = u.logprobs; d.advantages = u.advantages; d.returns = u.returns;
  d.values = u.values; d.params = u.params;
  d.obs_dim = u.policy.obs_dim; d.act_dim = u.policy.act_dim; d.continuous = u.policy.continuous;
  d.norm_adv = u.norm_adv; d.clip_vloss = u.clip_vloss;
  d.clip = u.clip_coeff;
  d.clip_lo = (float)(1.0 - (double)u.clip_coeff); d.clip_hi = (float)(1.0 + (double)u.clip_coeff);
  d.ent_c = u.entropy_coeff; d.vf_c = u.value_coeff; d.inv_m = (float)(1.0 / (double)u.m_total);
  d.moments = u.adv_moments; d.partials = u.workspace;
  { int rc2 = make_dp(u.dp, u.dp_seq, d.dp, "aur_ppo_update_grad"); if (rc2) return rc2; }
  if (u.mom_seq) {
    if (u.mom_index < 0 || u.mom_index >= DP_MAXMB) { set_error("aur_ppo_update_grad: mom_index %d outside 0..%d", u.mom_index, DP_MAXMB - 1); return AUR_ERR_ARG; }
    d.dp.mom_seq = u.mom_seq; d.dp.mom_index = u.mom_index;
  }
  if ((u.rec_actor != nullptr) != (u.rec_critic != nullptr)) { set_error("aur_ppo_update_grad: give both record arrays or neither"); return AUR_ERR_ARG; }
  if (u.rec_actor && u.policy.continuous && u.policy.act_dim > 2) { set_error("aur_ppo_update_grad: records hold at most 2 action dims"); return AUR_ERR_ARG; }
  d.rec_actor = reinterpret_cast<const float4*>(u.rec_actor); d.rec_critic = reinterpret_cast<const float4*>(u.rec_critic);
  static DeviceOnce attr_set;
  if (attr_set.first()) {
    AUR_CUDA_OK(cudaFuncSetAttribute(ppo_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UPD_SMEM));
    attr_set.done();
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int impl = is_headline_shape(u.policy) ? update_impl() : 3;
  int gx, pstride = UPD_PSTRIDE;
  const float* partials = u.workspace;
  if (impl == 3 && wide_eligible(u.policy) && update_wide_enabled()) {
    float* part = nullptr;
    int rc2 = launch_ppo_grad_wide(d, u.policy, u.workspace + ws_bytes() / sizeof(float) + gen_workspace_floats(u.policy), &gx, &part, s);
    if (rc2) return rc2;
    partials = part; pstride = gen_pstride(u.policy);
  } else if (impl == 3) {
    float* part = nullptr;
    int rc2 = launch_ppo_grad_generic(d, u.policy, u.workspace + ws_bytes() / sizeof(float), &gx, &part, s);
    if (rc2) return rc2;
    partials = part; pstride = gen_pstride(u.policy);
  } else if (impl >= 1) {
    gx = sm_count();
    int rc2 = launch_ppo_grad_tc(d, gx, impl == 2 ? 4 : 2, s);
    if (rc2) return rc2;
  } else {
    gx = upd_grid_x();
    ppo_grad_kernel<<<dim3(gx, 2), UPD_THREADS, UPD_SMEM, s>>>(d);
    AUR_LAUNCH_OK("ppo_grad_kernel");
  }
  const int64_t P = policy_param_count(u.policy);
  const int total = (int)(P + AUR_NUM_STATS);
  unsigned int* ticket2 = stream_tickets(s);
  if (!ticket2) return AUR_ERR_ARG;
  ticket2 += 1;
  grad_reduce_kernel<<<(4 * total + 255) / 256, 256, 0, s>>>(partials, gx, u.policy.obs_dim, u.policy.act_dim, u.policy.continuous,
                                                        u.policy.hidden_dim, u.policy.num_layers, pstride, u.grads_out, d.dp,
                                                        ticket2, PopRed{});
  AUR_LAUNCH_OK("grad_reduce_kernel");
  return 0;
}

extern "C" int aur_ppo_update_apply(const aur_policy_desc* desc, float* params, float* grads_packed, float* adam_m,
                                    float* adam_v, double lr, double beta1, double beta2, double eps, int64_t step,
                                    double max_grad_norm, int64_t m_total, double entropy_coeff, double value_coeff,
                                    float* stats_out, void* stream) {
  return aur_ppo_update_apply_dp(desc, params, grads_packed, adam_m, adam_v, lr, beta1, beta2, eps, step, max_grad_norm, m_total,
                                 entropy_coeff, value_coeff, stats_out, nullptr, 0, stream);
}

extern "C" int aur_ppo_update_apply_dp(const aur_policy_desc* desc, float* params, float* grads_packed, float* adam_m,
                                       float* adam_v, double lr, double beta1, double beta2, double eps, int64_t step,
                                       double max_grad_norm, int64_t m_total, double entropy_coeff, double value_coeff,
                                       float* stats_out, const aur_dp_ctx* dp, uint32_t seq, void* stream) {
  using namespace aur;
  DpDev dpd;
  { int rc = make_dp(dp, seq, dpd, "aur_ppo_update_apply_dp"); if (rc) return rc; }
  if (!desc || !params || !grads_packed || !adam_m || !adam_v || step < 1 || m_total <= 0) {
    set_error("aur_ppo_update_apply: bad arguments"); return AUR_ERR_ARG;
  }
  const int64_t P = policy_param_count(*desc);
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
  adam_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(P, params, grads_packed, adam_m, adam_v, (float)(lr / bc1), (float)beta1,
                                                   (float)beta2, (float)eps, (float)sqrt(bc2), (float)max_grad_norm,
                                                   (float)(1.0 / (double)m_total), (float)entropy_coeff, (float)value_coeff,
                                                   stats_out, dpd);
  AUR_LAUNCH_OK("adam_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------------------ populations
namespace aur {
int check_pop(const aur_pop_desc* pop, const char* who) {
  if (!pop || pop->K < 1 || pop->K > 65535 || pop->n_member < 1 || !pop->seeds) {
    set_error("%s: bad population (need 1 <= K <= 65535, n_member >= 1, a device seed array)", who); return AUR_ERR_ARG;
  }
  return 0;
}
int check_pop_policy(const aur_policy_desc& p, const char* who) {
  if (!is_headline_shape(p) || (p.continuous && p.act_dim > 2)) {
    set_error("%s: populations run the 64 x 2 tensor-core kernels (hidden 64, 2 layers, obs_dim <= 4, act_dim <= 4, <= 2 continuous "
              "dims); got hidden %d, %d layers, obs %d, act %d - no fallback", who, p.hidden_dim, p.num_layers, p.obs_dim, p.act_dim);
    return AUR_ERR_UNSUPPORTED;
  }
  return 0;
}
// CTAs per net and member: a single run's count (#SM), or fewer when the member's minibatch has fewer tiles of 128 samples
static int pop_grad_ctas(int64_t m) {
  const int64_t tiles = (m + 127) / 128;
  return (int)(tiles < sm_count() ? tiles : sm_count());
}
// CTAs per minibatch of the advantage moments: as aur_ppo_adv_moments_multi computes it
static int pop_moment_ctas(int32_t n_mb, int64_t m) {
  int cpm = MOM_CTAS / n_mb;
  if (cpm < 1) cpm = 1;
  const long long need = (m + 255) / 256;
  if (cpm > need) cpm = (int)need;
  return cpm;
}
static size_t pop_grad_ws_floats(int K, int64_t m) { return (size_t)K * 2 * pop_grad_ctas(m) * UPD_PSTRIDE; }
}  // namespace aur

extern "C" int64_t aur_pop_update_workspace_bytes(const aur_pop_desc* pop, const aur_policy_desc* desc, int32_t n_mb, int64_t m) {
  using namespace aur;
  int rc = check_pop(pop, "aur_pop_update_workspace_bytes");
  if (rc) return rc;
  if (!desc) { set_error("aur_pop_update_workspace_bytes: null policy"); return AUR_ERR_ARG; }
  if ((rc = check_pop_policy(*desc, "aur_pop_update_workspace_bytes"))) return rc;
  if (n_mb < 1 || n_mb > DP_MAXMB || m < 1) { set_error("aur_pop_update_workspace_bytes: need 1 <= n_mb <= %d, m >= 1", DP_MAXMB); return AUR_ERR_ARG; }
  // [K][2][c][PSTRIDE] gradient partials | [K][n_mb][cpm][2] fp64 moment partials
  return (int64_t)(pop_grad_ws_floats(pop->K, m) * sizeof(float) + (size_t)pop->K * n_mb * pop_moment_ctas(n_mb, m) * 2 * sizeof(double));
}

extern "C" int aur_pop_adv_moments_multi(const aur_pop_desc* pop, int32_t n_mb, int64_t m, const int32_t* idx, const float* advantages,
                                         double* moments_out, float* workspace, void* stream) {
  using namespace aur;
  int rc = check_pop(pop, "aur_pop_adv_moments_multi");
  if (rc) return rc;
  if (n_mb <= 0 || n_mb > DP_MAXMB || m <= 0 || !idx || !advantages || !moments_out || !workspace) {
    set_error("aur_pop_adv_moments_multi: bad arguments (1 <= n_mb <= %d, m >= 1, non-null arrays)", DP_MAXMB); return AUR_ERR_ARG;
  }
  const int cpm = pop_moment_ctas(n_mb, m);
  double* partial = reinterpret_cast<double*>(workspace + pop_grad_ws_floats(pop->K, m));
  DpDev dpd;
  make_dp(nullptr, 1u, dpd, "aur_pop_adv_moments_multi");
  cudaStream_t s = (cudaStream_t)stream;
  adv_moments_multi_kernel<true><<<dim3((unsigned)cpm, (unsigned)n_mb, (unsigned)pop->K), 256, 0, s>>>(
      (long long)m, idx, (long long)m, advantages, partial, nullptr, moments_out, dpd);
  AUR_LAUNCH_OK("adv_moments_multi_kernel (population)");
  const int entries = pop->K * n_mb;
  pop_moments_final_kernel<<<(entries + 127) / 128, 128, 0, s>>>(entries, cpm, (long long)m, partial, moments_out);
  AUR_LAUNCH_OK("pop_moments_final_kernel");
  return 0;
}

extern "C" int aur_pop_update_grad(const aur_pop_desc* pop, const aur_pop_update_args* args, void* stream) {
  using namespace aur;
  int rc = check_pop(pop, "aur_pop_update_grad");
  if (rc) return rc;
  if (!args) { set_error("aur_pop_update_grad: null args"); return AUR_ERR_ARG; }
  const aur_pop_update_args& u = *args;
  if ((rc = check_pop_policy(u.policy, "aur_pop_update_grad"))) return rc;
  if (u.m < 1 || u.n_mb < 1 || u.n_mb > DP_MAXMB || u.mb_index < 0 || u.mb_index >= u.n_mb || !u.idx || !u.rec_actor || !u.rec_critic ||
      !u.params || !u.hparams || !u.active || !u.workspace || !u.grads_out || (u.norm_adv && !u.adv_moments) ||
      ((uintptr_t)u.rec_actor & 31) || ((uintptr_t)u.rec_critic & 31)) {
    set_error("aur_pop_update_grad: bad arguments"); return AUR_ERR_ARG;
  }
  const int64_t P = policy_param_count(u.policy);
  UpdDev d{};
  d.m_local = u.m; d.idx = u.idx + (size_t)u.mb_index * u.m; d.idx_offset = 0;
  d.params = u.params;
  d.obs_dim = u.policy.obs_dim; d.act_dim = u.policy.act_dim; d.continuous = u.policy.continuous;
  d.norm_adv = u.norm_adv; d.clip_vloss = u.clip_vloss;
  d.inv_m = (float)(1.0 / (double)u.m);
  d.moments = u.norm_adv ? u.adv_moments + 3 * (size_t)u.mb_index : nullptr;
  d.partials = u.workspace;
  make_dp(nullptr, 0u, d.dp, "aur_pop_update_grad");
  d.rec_actor = reinterpret_cast<const float4*>(u.rec_actor); d.rec_critic = reinterpret_cast<const float4*>(u.rec_critic);
  const int gx = pop_grad_ctas(u.m);
  PopUpd pu;
  pu.hp = u.hparams; pu.active = u.active; pu.P = P;
  pu.idx_stride = (long long)u.n_mb * u.m; pu.mom_stride = 3LL * u.n_mb; pu.part_stride = 2LL * gx * UPD_PSTRIDE;
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = launch_ppo_grad_tc_pop(d, pu, gx, pop->K, s))) return rc;
  PopRed pr;
  pr.chunk_ncta = sm_count(); pr.part_stride = pu.part_stride; pr.grads_stride = P + AUR_NUM_STATS; pr.active = u.active;
  const int total = (int)(P + AUR_NUM_STATS);
  grad_reduce_kernel<true><<<dim3((4 * total + 255) / 256, pop->K), 256, 0, s>>>(
      u.workspace, gx, u.policy.obs_dim, u.policy.act_dim, u.policy.continuous, u.policy.hidden_dim, u.policy.num_layers, UPD_PSTRIDE,
      u.grads_out, d.dp, nullptr, pr);
  AUR_LAUNCH_OK("grad_reduce_kernel (population)");
  return 0;
}

extern "C" int aur_pop_update_apply(const aur_pop_desc* pop, const aur_policy_desc* desc, const aur_pop_hparams* hparams, float* params,
                                    const float* grads, float* adam_m, float* adam_v, int64_t* steps, int32_t* active, const double* bc,
                                    int64_t bc_len, double frac, double beta1, double beta2, double eps, int64_t m_total,
                                    float* stats_out, int32_t stats_rows, int32_t stats_row, int32_t epoch_end, void* stream) {
  using namespace aur;
  int rc = check_pop(pop, "aur_pop_update_apply");
  if (rc) return rc;
  if (!desc || !hparams || !params || !grads || !adam_m || !adam_v || !steps || !active || !bc || bc_len < 2 || m_total <= 0 ||
      (stats_out && (stats_rows < 1 || stats_row < 0 || stats_row >= stats_rows))) {
    set_error("aur_pop_update_apply: bad arguments"); return AUR_ERR_ARG;
  }
  if ((rc = check_pop_policy(*desc, "aur_pop_update_apply"))) return rc;
  PopAdam a;
  a.P = policy_param_count(*desc);
  a.params = params; a.grads = grads; a.m1 = adam_m; a.m2 = adam_v; a.steps = steps; a.active = active; a.hp = hparams;
  a.bc = bc; a.bc_len = bc_len; a.frac = frac;
  a.beta1 = (float)beta1; a.beta2 = (float)beta2; a.eps = (float)eps; a.inv_m = (float)(1.0 / (double)m_total);
  a.stats = stats_out; a.stats_rows = stats_rows; a.stats_row = stats_row; a.epoch_end = epoch_end ? 1 : 0;
  pop_adam_kernel<<<pop->K, 1024, 0, (cudaStream_t)stream>>>(a);
  AUR_LAUNCH_OK("pop_adam_kernel");
  return 0;
}
