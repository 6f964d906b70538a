// Declarations shared by the SIMT (update.cu) and tensor-core (update_tc.cu) minibatch-update kernels.
#pragma once
#include "policy.cuh"

namespace aur {

constexpr int UPD_THREADS = 256;
constexpr int UPD_S = 256;             // samples per tile (one per thread in the per-sample phases)
constexpr int UPD_LD = UPD_S + 4;      // feature-major row stride: 16-B aligned, 4 banks per row
constexpr int UPD_H = 64;
constexpr int UPD_PSTRIDE = 4800;      // floats per CTA partial: net gradients + AUR_NUM_STATS
constexpr int UPD_STAT_OFF = UPD_PSTRIDE - AUR_NUM_STATS;
constexpr int UPD_SW = 4800;           // smem floats reserved for one net (padded layout)
constexpr int UPD_WD = 2 * UPD_H * UPD_H;   // a 64x64 matrix with every entry duplicated: [k][n][2]
constexpr int UPD_SMEM_FLOATS = UPD_SW + 2 * UPD_WD + UPD_H + 2 * UPD_H * UPD_LD + 2 * 4 * UPD_LD + 4 * UPD_H;
constexpr size_t UPD_SMEM = sizeof(float) * UPD_SMEM_FLOATS;
constexpr int MOM_CTAS = 148 * 8;      // advantage-moment CTAs: the gather is latency-bound, eight CTAs per SM keep ~64 loads in flight per SM x 8

// ---- data-parallel exchange over peer memory (dp.cu): every rank owns one exchange area that all ranks of the
// node map (CUDA IPC).  Producers PUSH their values into every peer's area over NVLink and then release a
// sequence-numbered flag there; consumers only ever poll and read their OWN area.  Two slots (seq & 1) because a
// rank can run at most one minibatch ahead of a peer that is still reading.
constexpr int DP_MAX = 16;
constexpr int DP_OFF_FLAG_MOM = 0;         // u32 [DP_MAX]
constexpr int DP_OFF_FLAG_GRAD = 64;       // u32 [DP_MAX]
constexpr int DP_OFF_STATUS = 128;         // u32: 1 = a wait timed out
constexpr int DP_OFF_WAIT = 136;           // u64 [6]: spin ns on peers' gradient flags summed over the spinning threads, number of spins;
                                           // the same for moment flags; then WALL ns the Adam kernel stood still until every peer's
                                           // gradients had arrived (entry -> all flags seen), number of Adam launches
constexpr int DP_OFF_FLAG_MOMX = 192;      // u32 [DP_MAX]: iteration counter of the moments exchanged ahead (aur_ppo_adv_moments_multi)
constexpr int DP_OFF_MOM = 256;            // f64 [2][DP_MAX][4]
constexpr int DP_MAXMB = AUR_DP_MAX_MINIBATCHES;
constexpr int DP_OFF_MOMX = DP_OFF_MOM + 2 * DP_MAX * 4 * 8;             // f64 [2][DP_MAX][DP_MAXMB][4]: moments of a whole iteration
constexpr int DP_OFF_GRAD = DP_OFF_MOMX + 2 * DP_MAX * DP_MAXMB * 4 * 8; // f32 [2][DP_MAX][dp_grad_stride]
__host__ __device__ inline int dp_grad_stride(int64_t P) { return (int)((P + AUR_NUM_STATS + 63) / 64 * 64); }
__host__ __device__ inline int64_t dp_area_bytes(int64_t P) { return DP_OFF_GRAD + (int64_t)2 * DP_MAX * dp_grad_stride(P) * 4; }
struct DpDev {
  int world, rank;                         // world <= 1: not data-parallel
  uint32_t seq;                            // minibatch sequence number (same on every rank), starts at 1
  unsigned char* peer[DP_MAX];             // exchange area of every rank as mapped here; peer[rank] is local
  // advantage moments exchanged ahead for the whole iteration (aur_ppo_adv_moments_multi): mom_seq != 0 selects them
  uint32_t mom_seq;
  int mom_index;
};

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// wait until the peer's flag in OUR area reaches seq; gives up after 20 s (status word) instead of hanging the GPU
// (which: 0 = gradient flags, 1 = moment flags - the time spent spinning is accumulated per kind in the exchange area, so the
// skew between ranks is measured, not inferred: aur_dp_wait_stats)
__device__ __forceinline__ void dp_wait_flag(const uint32_t* flag, uint32_t seq, unsigned char* my_area, int which = 0) {
  if ((int32_t)(ld_acquire_sys(flag) - seq) >= 0) return;
  const uint64_t t0 = global_timer_ns();
  while ((int32_t)(ld_acquire_sys(flag) - seq) < 0) {
    __nanosleep(64);
    if (global_timer_ns() - t0 > 20000000000ull) { *reinterpret_cast<volatile uint32_t*>(my_area + DP_OFF_STATUS) = 1u; break; }
  }
  unsigned long long* w = reinterpret_cast<unsigned long long*>(my_area + DP_OFF_WAIT) + 2 * which;
  atomicAdd(w, (unsigned long long)(global_timer_ns() - t0));
  atomicAdd(w + 1, 1ull);
}
#endif

struct UpdDev {
  long long m_local;
  const int32_t* idx;
  long long idx_offset;
  const float *obs, *actions, *logprobs, *advantages, *returns, *values, *params;
  int obs_dim, act_dim, continuous, norm_adv, clip_vloss;
  float clip, clip_lo, clip_hi, ent_c, vf_c, inv_m;
  const double* moments;
  float* partials;      // [2][gridDim.x][UPD_PSTRIDE]
  const float4 *rec_actor, *rec_critic;   // optional packed records (aur_ppo_pack_records): 2 x float4 per sample, else NULL
  DpDev dp;
};

#ifdef __CUDACC__
// sum, sum of squares and count of the advantages of the WHOLE minibatch: local (a.moments) or, data-parallel, the
// per-rank moments every rank pushed into our exchange area, added in rank order (identical on every rank)
__device__ __forceinline__ void load_adv_moments(const UpdDev& a, double& s, double& ss, double& n) {
  if (a.dp.world > 1) {
    unsigned char* me = a.dp.peer[a.dp.rank];
    s = 0.0; ss = 0.0; n = 0.0;
    if (a.dp.mom_seq) {                      // exchanged once for the whole iteration: normally no wait at all here
      const uint32_t* flags = reinterpret_cast<const uint32_t*>(me + DP_OFF_FLAG_MOMX);
      const double* rm = reinterpret_cast<const double*>(me + DP_OFF_MOMX) + (size_t)(a.dp.mom_seq & 1u) * DP_MAX * DP_MAXMB * 4 +
                         (size_t)a.dp.mom_index * 4;
      for (int r = 0; r < a.dp.world; ++r) {
        dp_wait_flag(flags + r, a.dp.mom_seq, me, 1);
        const double* q = rm + (size_t)r * DP_MAXMB * 4;
        s += __ldcg(q); ss += __ldcg(q + 1); n += __ldcg(q + 2);
      }
      return;
    }
    const uint32_t* flags = reinterpret_cast<const uint32_t*>(me + DP_OFF_FLAG_MOM);
    const double* rm = reinterpret_cast<const double*>(me + DP_OFF_MOM) + (a.dp.seq & 1u) * DP_MAX * 4;
    for (int r = 0; r < a.dp.world; ++r) {
      dp_wait_flag(flags + r, a.dp.seq, me, 1);
      s += __ldcg(rm + r * 4); ss += __ldcg(rm + r * 4 + 1); n += __ldcg(rm + r * 4 + 2);
    }
  } else {
    s = a.moments[0]; ss = a.moments[1]; n = a.moments[2];
  }
}
__device__ __forceinline__ void adv_norm_from_moments(double s, double ss, double n, float& mean_out, float& den_out) {
  const double mean = s / n;
  double var = (ss - s * mean) / (n - 1.0);          // unbiased (torch .std())
  if (var < 0.0) var = 0.0;
  mean_out = (float)mean;
  den_out = (float)sqrt(var) + 1e-8f;
}
__device__ __forceinline__ void adv_norm_consts(const UpdDev& a, float& mean_out, float& den_out) {
  double s, ss, n;
  load_adv_moments(a, s, ss, n);
  adv_norm_from_moments(s, ss, n, mean_out, den_out);
}
#endif



// population form of the tensor-core update (aur_pop_update_grad): member k = blockIdx.y reads params + k * P, idx + k * idx_stride,
// moments + k * mom_stride and writes partials + k * part_stride; members with active[k] == 0 are skipped
struct PopUpd {
  const aur_pop_hparams* hp;
  const int32_t* active;
  long long P, idx_stride, mom_stride, part_stride;
};

// tensor-core implementation (update_tc.cu): both nets per CTA, grid = gx CTAs; same partial layout
int launch_ppo_grad_tc(const UpdDev& d, int gx, int threads_per_sample, cudaStream_t s);
int launch_ppo_grad_tc_pop(const UpdDev& d, const PopUpd& pop, int gx, int K, cudaStream_t s);
size_t ppo_grad_tc_smem_bytes();

}  // namespace aur
