// Minibatch shuffle (row U, src/ppo.py:214-215 `np.random.shuffle(b_inds)`): a keyed bijection of [0, n) written
// straight to the int32 index array the update kernels gather through -- no sort, no host round trip.
// The permutation is an (unbalanced, alternating) Feistel network over exactly bits = ceil(log2 n) bits, halves of
// ceil(bits/2) and floor(bits/2) bits that swap every round (round function: a 32-bit multiply-xorshift mix of
// the right half and a Philox4x32-10-derived round key), with cycle-walking: indices that land outside [0, n)
// are encrypted again until they fall inside, which keeps it a bijection on [0, n).  The domain is < 2n, so a
// thread walks < 2 times on average and not at all when n is a power of two.
// The numpy restatement in oracle/ppo_ref.py (feistel_shuffle) is bit-identical (tests/test_shuffle_gpu.py).
#include "common.cuh"

namespace aur {

constexpr int SHUF_ROUNDS = 8;
struct ShufKeys { uint32_t k[SHUF_ROUNDS]; };

__host__ __device__ __forceinline__ uint32_t shuf_mix(uint32_t v) {
  v *= 0x9E3779B1u; v ^= v >> 15;
  v *= 0x85EBCA77u; v ^= v >> 13;
  v *= 0xC2B2AE3Du; v ^= v >> 16;
  return v;
}
__host__ __device__ __forceinline__ uint32_t shuf_encrypt(uint32_t x, int wa, int wb, const ShufKeys& keys) {
  const uint32_t ma = (1u << wa) - 1u, mb = (1u << wb) - 1u;
  uint32_t L = x >> wb, R = x & mb;                 // L: wa bits, R: wb bits
#pragma unroll
  for (int r = 0; r < SHUF_ROUNDS; r += 2) {
    uint32_t t = L ^ (shuf_mix(R + keys.k[r]) & ma);       // (L: wa, R: wb) -> (R: wb, t: wa)
    L = R; R = t;
    t = L ^ (shuf_mix(R + keys.k[r + 1]) & mb);            // (L: wb, R: wa) -> (R: wa, t: wb)
    L = R; R = t;
  }
  return (L << wb) | R;
}

__global__ void __launch_bounds__(256) shuffle_kernel(long long n, int wa, int wb, ShufKeys keys, int32_t* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t x = (uint32_t)i;
  do { x = shuf_encrypt(x, wa, wb, keys); } while ((long long)x >= n);
  out[i] = (int32_t)x;
}

// Population form (aur_pop_shuffle_indices): grid (ceil(n / 256), K, epochs); member k's epoch e is the permutation of
// aur_shuffle_indices(n, seeds[k], stream_id0 + e), its round keys derived here (one Philox call per round, as the host does
// for a single run), each local index j written as the population's global row.
__global__ void __launch_bounds__(256) pop_shuffle_kernel(long long n, int wa, int wb, const uint64_t* __restrict__ seeds,
                                                        uint64_t stream_id0, long long n_member, long long NK,
                                                        int32_t* __restrict__ out) {
  __shared__ ShufKeys keys;
  const int k = blockIdx.y, e = blockIdx.z;
  if (threadIdx.x < SHUF_ROUNDS) {
    const uint64_t seed = seeds[k], stream_id = stream_id0 + (uint64_t)e;
    keys.k[threadIdx.x] = philox4x32_10((uint32_t)threadIdx.x, (uint32_t)stream_id, (uint32_t)(stream_id >> 32), 0x5AFE5EEDu,
                                        (uint32_t)seed, (uint32_t)(seed >> 32)).c[0];
  }
  __syncthreads();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const ShufKeys kk = keys;
  uint32_t x = (uint32_t)i;
  do { x = shuf_encrypt(x, wa, wb, kk); } while ((long long)x >= n);
  const long long t = (long long)x / n_member;
  out[((long long)k * gridDim.z + e) * n + i] = (int32_t)(t * NK + (long long)k * n_member + ((long long)x - t * n_member));
}

// Packed per-sample records for the minibatch gather: the update reads ONE 32-byte sector per sample and net instead
// of one sector per gathered array (4-byte elements at random rows cost 32 B of DRAM traffic each).
//   actor  record: obs[0..3] (zero padded) | action[0], old logprob, advantage, action[1]
//   critic record: obs[0..3] (zero padded) | return, old value, 0, 0
__global__ void __launch_bounds__(256) pack_records_kernel(long long B, int obs_dim, int act_w, const float* __restrict__ obs,
                                                         const float* __restrict__ act, const float* __restrict__ logp,
                                                         const float* __restrict__ adv, const float* __restrict__ ret,
                                                         const float* __restrict__ val, float4* __restrict__ rec_a,
                                                         float4* __restrict__ rec_c) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  float x[4] = {0.f, 0.f, 0.f, 0.f};
  for (int c = 0; c < obs_dim; ++c) x[c] = obs[i * obs_dim + c];
  const float4 o = make_float4(x[0], x[1], x[2], x[3]);
  rec_a[2 * i] = o;
  rec_a[2 * i + 1] = make_float4(act[i * act_w], logp[i], adv[i], act_w > 1 ? act[i * act_w + 1] : 0.0f);
  rec_c[2 * i] = o;
  rec_c[2 * i + 1] = make_float4(ret[i], val[i], 0.0f, 0.0f);
}

}  // namespace aur

extern "C" int aur_ppo_pack_records(int64_t B, int32_t obs_dim, int32_t action_width, const float* obs, const float* actions,
                                    const float* logprobs, const float* advantages, const float* returns, const float* values,
                                    float* rec_actor, float* rec_critic, void* stream) {
  using namespace aur;
  if (B < 0 || obs_dim < 1 || obs_dim > 4 || action_width < 1 || action_width > 2) {
    set_error("aur_ppo_pack_records: obs_dim 1..4 and action width 1..2 fit a record (got %d, %d); use the unpacked arrays otherwise",
              obs_dim, action_width);
    return AUR_ERR_UNSUPPORTED;
  }
  if (B == 0) return 0;
  if (!obs || !actions || !logprobs || !advantages || !returns || !values || !rec_actor || !rec_critic ||
      ((uintptr_t)rec_actor & 31) || ((uintptr_t)rec_critic & 31)) {
    set_error("aur_ppo_pack_records: null or not 32-byte aligned buffer"); return AUR_ERR_ARG;
  }
  pack_records_kernel<<<(unsigned)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>((long long)B, obs_dim, action_width, obs, actions,
                                                                                  logprobs, advantages, returns, values,
                                                                                  (float4*)rec_actor, (float4*)rec_critic);
  AUR_LAUNCH_OK("pack_records_kernel");
  return 0;
}

extern "C" int aur_shuffle_indices(int64_t n, uint64_t seed, uint64_t stream_id, int32_t* out, void* stream) {
  using namespace aur;
  if (n < 0 || n > 0x7FFFFFFFLL || (n > 0 && !out)) { set_error("aur_shuffle_indices: n must be in [0, 2^31) and out non-null"); return AUR_ERR_ARG; }
  if (n == 0) return 0;
  int bits = 1;
  while ((1LL << bits) < n) ++bits;
  const int wa = (bits + 1) / 2, wb = bits - wa > 0 ? bits - wa : 0;
  ShufKeys keys;
  for (int r = 0; r < SHUF_ROUNDS; ++r)
    keys.k[r] = philox4x32_10((uint32_t)r, (uint32_t)stream_id, (uint32_t)(stream_id >> 32), 0x5AFE5EEDu, (uint32_t)seed,
                              (uint32_t)(seed >> 32)).c[0];
  shuffle_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((long long)n, wa, wb, keys, out);
  AUR_LAUNCH_OK("shuffle_kernel");
  return 0;
}

extern "C" int aur_pop_shuffle_indices(const aur_pop_desc* pop, int32_t T, int32_t epochs, uint64_t stream_id0, int32_t* out,
                                       void* stream) {
  using namespace aur;
  if (!pop || pop->K < 1 || pop->n_member < 1 || !pop->seeds || T < 1 || epochs < 1 || !out) {
    set_error("aur_pop_shuffle_indices: bad arguments"); return AUR_ERR_ARG;
  }
  const long long n = (long long)T * pop->n_member, NK = (long long)pop->K * pop->n_member;
  if ((long long)T * NK > 0x7FFFFFFFLL || pop->K > 65535 || epochs > 65535) {
    set_error("aur_pop_shuffle_indices: K * T * n_member must be < 2^31 (got K %d, T %d, n_member %lld)", pop->K, T,
              (long long)pop->n_member);
    return AUR_ERR_ARG;
  }
  int bits = 1;
  while ((1LL << bits) < n) ++bits;
  const int wa = (bits + 1) / 2, wb = bits - wa > 0 ? bits - wa : 0;
  pop_shuffle_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)pop->K, (unsigned)epochs), 256, 0, (cudaStream_t)stream>>>(
      n, wa, wb, pop->seeds, stream_id0, (long long)pop->n_member, NK, out);
  AUR_LAUNCH_OK("pop_shuffle_kernel");
  return 0;
}
