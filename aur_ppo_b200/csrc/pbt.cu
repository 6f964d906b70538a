// Population-based training (Jaderberg et al., 2017) between population iterations: a ranking of the members' fitness and
// the exploit / explore copies, all inside the population's own stacked [K][...] buffers -- no host round trip, no
// checkpoint files.  The decision rule is stated once, in include/aur_ppo.h ("population-based training"); oracle/pbt_ref.py
// restates it in NumPy (tests/test_pbt_gpu.py compares with np.array_equal).
//
//   pop_episode_fitness_kernel   fitness[k] = mean return of member k's episodes since the last snapshot (NaN if none)
//   pbt_rank_kernel              rank[K] / order[K] / n_valid by counting: O(K^2) compares over shared-memory tiles, no sort
//   pbt_exploit_kernel           grid (chunks, K): a recipient's blocks copy their chunk of the donor's rows and columns
#include <math.h>

#include "common.cuh"
#include "policy.cuh"

namespace aur {

int check_pop(const aur_pop_desc* pop, const char* who);                    // update.cu
int check_pop_policy(const aur_policy_desc& p, const char* who);

constexpr int PBT_RANK_THREADS = 256;
constexpr int PBT_COPY_THREADS = 256;
constexpr int PBT_COPY_FLOATS = 2048;     // floats of each [P] row one block copies (two float4 per thread)

__global__ void __launch_bounds__(256) pop_episode_fitness_kernel(int K, const double* __restrict__ totals,
                                                                  double* __restrict__ snapshot, double* __restrict__ fitness) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const double c = totals[3 * k + 0], r = totals[3 * k + 1], l = totals[3 * k + 2];
  const double dc = c - snapshot[3 * k + 0];
  fitness[k] = dc > 0.0 ? (r - snapshot[3 * k + 1]) / dc : __longlong_as_double(0x7FF8000000000000LL);
  snapshot[3 * k + 0] = c;
  snapshot[3 * k + 1] = r;
  snapshot[3 * k + 2] = l;
}

// Member k is ranked when fitness[k] is not NaN; rank[k] = #{ranked j : f_j > f_k, or f_j == f_k and j < k} (IEEE compares,
// so -0.0 == +0.0 and +-inf order as numbers), order[rank[k]] = k, order[K] = n_valid.  Every thread scans the whole vector.
__global__ void __launch_bounds__(PBT_RANK_THREADS) pbt_rank_kernel(int K, const double* __restrict__ fitness,
                                                                    int32_t* __restrict__ rank, int32_t* __restrict__ order) {
  __shared__ double tile[PBT_RANK_THREADS];
  const int k = blockIdx.x * PBT_RANK_THREADS + threadIdx.x;
  const double f = k < K ? fitness[k] : 0.0;
  int above = 0, valid = 0;
  for (int base = 0; base < K; base += PBT_RANK_THREADS) {
    __syncthreads();
    if (base + (int)threadIdx.x < K) tile[threadIdx.x] = fitness[base + threadIdx.x];
    __syncthreads();
    const int n = K - base < PBT_RANK_THREADS ? K - base : PBT_RANK_THREADS;
    for (int i = 0; i < n; ++i) {
      const double g = tile[i];
      const int j = base + i;
      valid += !isnan(g);
      above += (g > f) || (g == f && j < k);      // false for NaN g
    }
  }
  if (k >= K) return;
  if (isnan(f)) {
    rank[k] = -1;
  } else {
    rank[k] = above;
    order[above] = k;
  }
  if (k == 0) order[K] = valid;
}

struct PbtCopy {
  int K;
  int64_t P;
  const int32_t* rank;
  const int32_t* order;          // [K + 1], order[K] = n_valid
  double q, down, up;
  uint32_t mask;
  uint32_t r_lo, r_hi, key_lo, key_hi;
  float* rows[3];                // params, adam_m, adam_v [K][P]
  int64_t* steps;
  aur_pop_hparams* hp;
  double* norm;                  // [>= 2D + 4][norm_ld] or nullptr
  int64_t norm_ld, n_member;
  int norm_rows;                 // 2D + 4: observation and return statistics (the return accumulator row 2D + 4 is kept)
  int32_t* donor_out;
};

__device__ __forceinline__ void copy_row_chunk(float* __restrict__ dst, const float* __restrict__ src, int64_t lo, int64_t hi) {
  // 16-byte copies when source and destination share their alignment; scalar head and tail
  if ((((uintptr_t)(dst + lo)) & 15) == (((uintptr_t)(src + lo)) & 15)) {
    int64_t a = lo;
    while (a < hi && (((uintptr_t)(dst + a)) & 15)) ++a;                 // <= 3 elements
    const int64_t nv = (hi - a) >> 2;
    for (int64_t i = lo + threadIdx.x; i < a; i += blockDim.x) dst[i] = src[i];
    const float4* s4 = reinterpret_cast<const float4*>(src + a);
    float4* d4 = reinterpret_cast<float4*>(dst + a);
    for (int64_t i = threadIdx.x; i < nv; i += blockDim.x) d4[i] = s4[i];
    for (int64_t i = a + 4 * nv + threadIdx.x; i < hi; i += blockDim.x) dst[i] = src[i];
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) dst[i] = src[i];
  }
}

__global__ void __launch_bounds__(PBT_COPY_THREADS) pbt_exploit_kernel(PbtCopy c) {
  const int k = blockIdx.y;
  const int rk = c.rank[k];
  const int n_valid = c.order[c.K];
  const int n_sel = (int)floor(c.q * (double)n_valid);
  if (n_sel == 0 || rk < n_valid - n_sel) {                  // also rk == -1: not ranked
    if (blockIdx.x == 0 && threadIdx.x == 0) c.donor_out[k] = -1;
    return;
  }
  const Philox w = philox4x32_10((uint32_t)k, c.r_lo, c.r_hi, AUR_PBT_PHILOX_C3, c.key_lo, c.key_hi);
  const int d = c.order[((uint64_t)w.c[0] * (uint64_t)n_sel) >> 32];
  // [P] rows: chunk blockIdx.x of PBT_COPY_FLOATS elements
  const int64_t lo = (int64_t)blockIdx.x * PBT_COPY_FLOATS;
  const int64_t hi = lo + PBT_COPY_FLOATS < c.P ? lo + PBT_COPY_FLOATS : c.P;
  if (lo < hi) {
#pragma unroll
    for (int a = 0; a < 3; ++a) copy_row_chunk(c.rows[a] + (size_t)k * c.P, c.rows[a] + (size_t)d * c.P, lo, hi);
  }
  // wrapper statistics: columns d * n + j -> k * n + j of rows 0 .. 2D + 3, j split evenly over the blocks
  if (c.norm) {
    const int64_t per = (c.n_member + gridDim.x - 1) / gridDim.x;
    const int64_t j0 = (int64_t)blockIdx.x * per;
    const int64_t j1 = j0 + per < c.n_member ? j0 + per : c.n_member;
    const int64_t w_cols = j1 > j0 ? j1 - j0 : 0;
    for (int64_t i = threadIdx.x; i < w_cols * c.norm_rows; i += blockDim.x) {
      const int64_t row = i / w_cols, j = j0 + i % w_cols;
      c.norm[row * c.norm_ld + (int64_t)k * c.n_member + j] = c.norm[row * c.norm_ld + (int64_t)d * c.n_member + j];
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const double* src = reinterpret_cast<const double*>(c.hp + d);      // the six fields, in declaration order
    double* dst = reinterpret_cast<double*>(c.hp + k);
    for (int j = 0; j < 6; ++j) {
      double v = src[j];
      if ((c.mask >> j) & 1u) v = v * (((w.c[1] >> j) & 1u) ? c.up : c.down);
      dst[j] = v;
    }
    c.steps[k] = c.steps[d];
    c.donor_out[k] = d;
  }
}

}  // namespace aur

extern "C" int aur_pop_episode_fitness(const aur_pop_desc* pop, const double* totals, double* snapshot, double* fitness_out,
                                       void* stream) {
  using namespace aur;
  int rc = check_pop(pop, "aur_pop_episode_fitness");
  if (rc) return rc;
  if (!totals || !snapshot || !fitness_out) { set_error("aur_pop_episode_fitness: null pointer"); return AUR_ERR_ARG; }
  pop_episode_fitness_kernel<<<(pop->K + 255) / 256, 256, 0, (cudaStream_t)stream>>>(pop->K, totals, snapshot, fitness_out);
  AUR_LAUNCH_OK("pop_episode_fitness_kernel");
  return 0;
}

extern "C" int aur_pop_pbt_step(const aur_pop_desc* pop, const aur_policy_desc* desc, const aur_pop_pbt_args* args,
                                void* stream) {
  using namespace aur;
  int rc = check_pop(pop, "aur_pop_pbt_step");
  if (rc) return rc;
  if (!desc || !args) { set_error("aur_pop_pbt_step: null desc or args"); return AUR_ERR_ARG; }
  if ((rc = check_pop_policy(*desc, "aur_pop_pbt_step"))) return rc;
  const aur_pop_pbt_args& a = *args;
  if (!(a.q > 0.0 && a.q <= 0.5)) { set_error("aur_pop_pbt_step: q must be in (0, 0.5] (got %g)", a.q); return AUR_ERR_ARG; }
  if (!(a.down > 0.0 && isfinite(a.down) && a.up > 0.0 && isfinite(a.up))) {
    set_error("aur_pop_pbt_step: the factors must be finite and > 0 (got down %g, up %g)", a.down, a.up); return AUR_ERR_ARG;
  }
  if (a.mask >> 6) { set_error("aur_pop_pbt_step: mask 0x%x has bits above 5 (aur_pop_hparams has six fields)", a.mask); return AUR_ERR_ARG; }
  if (!a.fitness || !a.params || !a.adam_m || !a.adam_v || !a.steps || !a.hparams || !a.rank_out || !a.donor_out || !a.order) {
    set_error("aur_pop_pbt_step: null pointer"); return AUR_ERR_ARG;
  }
  if (a.norm && a.norm_ld < (int64_t)pop->K * pop->n_member) {
    set_error("aur_pop_pbt_step: norm_ld %lld < K * n_member", (long long)a.norm_ld); return AUR_ERR_ARG;
  }
  PbtCopy c;
  c.K = pop->K;
  c.P = policy_param_count(*desc);
  c.rank = a.rank_out; c.order = a.order;
  c.q = a.q; c.down = a.down; c.up = a.up; c.mask = a.mask;
  c.r_lo = (uint32_t)a.round; c.r_hi = (uint32_t)(a.round >> 32);
  c.key_lo = (uint32_t)a.seed; c.key_hi = (uint32_t)(a.seed >> 32);
  c.rows[0] = a.params; c.rows[1] = a.adam_m; c.rows[2] = a.adam_v;
  c.steps = a.steps; c.hp = a.hparams;
  c.norm = a.norm; c.norm_ld = a.norm_ld; c.n_member = pop->n_member; c.norm_rows = 2 * desc->obs_dim + 4;
  c.donor_out = a.donor_out;
  cudaStream_t s = (cudaStream_t)stream;
  pbt_rank_kernel<<<(pop->K + PBT_RANK_THREADS - 1) / PBT_RANK_THREADS, PBT_RANK_THREADS, 0, s>>>(pop->K, a.fitness, a.rank_out,
                                                                                                  a.order);
  AUR_LAUNCH_OK("pbt_rank_kernel");
  const unsigned chunks = (unsigned)((c.P + PBT_COPY_FLOATS - 1) / PBT_COPY_FLOATS);
  pbt_exploit_kernel<<<dim3(chunks, (unsigned)pop->K), PBT_COPY_THREADS, 0, s>>>(c);
  AUR_LAUNCH_OK("pbt_exploit_kernel");
  return 0;
}
