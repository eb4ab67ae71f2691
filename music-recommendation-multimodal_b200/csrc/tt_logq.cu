// logQ correction of in-batch negatives (Yi et al., RecSys 2019): every negative of a batch is another row's positive,
// so an item is sampled as a negative in proportion to its popularity q. The loss kernels subtract log q_j from every
// logit of column j (tt_infonce_rows_off / tt_infonce_grad_off); the kernels here produce those offsets on the device,
// inside the captured step:
//   tt_logq_table_gather  : off[i] = table[ids[i]] (a fixed log q per id), floor for ids outside [0, N);
//   tt_logq_stream_update : the streaming frequency estimator (Algorithm 2 of the paper), made order-free so the state
//                           is bit-identical from run to run and on every data-parallel replica.
// Estimator state: h arrays of H = 2^log2H slots, A (int64, the last step a slot was seen) and Bv (fp32, the
// estimated interval between sightings). Per step t (= ++*step_dev): every slot hit by at least one id of the step is
// updated ONCE, Bv <- (1-alpha) Bv + alpha (t - A), A <- t, however many ids hit it; then off[i] = -log(max_k Bv_k).
// The update runs in ONE CTA: the slot's first atomicExch(&A[s], t) that returns a value other than t owns it (A only
// ever holds earlier steps before this one), so which thread updates a slot changes from run to run but the value it
// writes does not. One CTA also orders "all updates" before "all reads" with a __syncthreads.
#include "../../include/tt_b200.h"
#include "tt_common.cuh"

namespace tt {

constexpr int kLogqThreads = 1024;
constexpr int kLogqMaxHashes = 4;

// Low log2H bits of the splitmix64 finaliser of id + (k + 1) * golden ratio: array k's slot of `id`.
__device__ __forceinline__ uint32_t logq_slot(int64_t id, int k, int log2H) {
  uint64_t z = static_cast<uint64_t>(id) + static_cast<uint64_t>(k + 1) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return static_cast<uint32_t>(z & ((1ull << log2H) - 1));
}

__global__ void __launch_bounds__(kLogqThreads) logq_stream_update_kernel(const int64_t* __restrict__ ids, int n,
                                                                          int64_t* __restrict__ A, float* __restrict__ Bv,
                                                                          int h, int log2H, int64_t* __restrict__ step_dev,
                                                                          float alpha, float one_minus_alpha,
                                                                          float* __restrict__ off) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ long long s_t;
  if (threadIdx.x == 0) {
    s_t = static_cast<long long>(*step_dev) + 1;
    *step_dev = s_t;
  }
  __syncthreads();
  const long long t = s_t;
  const size_t H = size_t(1) << log2H;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t id = ids[i];
    for (int k = 0; k < h; ++k) {
      const size_t s = k * H + logq_slot(id, k, log2H);
      const long long prev = atomicExch(reinterpret_cast<unsigned long long*>(A + s), static_cast<unsigned long long>(t));
      if (prev != t) {
        const float gap = __ll2float_rn(t - prev);
        Bv[s] = __fadd_rn(__fmul_rn(one_minus_alpha, Bv[s]), __fmul_rn(alpha, gap));
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t id = ids[i];
    float b = 0.f;
    for (int k = 0; k < h; ++k) b = fmaxf(b, __ldcg(Bv + k * H + logq_slot(id, k, log2H)));
    off[i] = -logf(b);
  }
}

__global__ void __launch_bounds__(256) logq_table_gather_kernel(const int64_t* __restrict__ ids, int n,
                                                                const float* __restrict__ table, int64_t N, float floor_,
                                                                float* __restrict__ off) {
  pdl_launch_dependents();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t id = ids[i];
  off[i] = (id >= 0 && id < N) ? table[id] : floor_;
}

}  // namespace tt

using namespace tt;

extern "C" int tt_logq_stream_update(const int64_t* ids, int n, int64_t* A, float* Bv, int h, int log2H,
                                     int64_t* step_dev, float alpha, float one_minus_alpha, float* off_out,
                                     void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(ids && A && Bv && step_dev && off_out && n > 0, "tt_logq_stream_update: bad arguments");
  TT_REQUIRE(h >= 1 && h <= kLogqMaxHashes, "tt_logq_stream_update: %d hash arrays outside [1, %d]", h, kLogqMaxHashes);
  TT_REQUIRE(log2H >= 0 && log2H <= 28, "tt_logq_stream_update: 2^%d slots outside [1, 2^28]", log2H);
  TT_REQUIRE(alpha > 0.f && alpha <= 1.f && one_minus_alpha >= 0.f && one_minus_alpha < 1.f,
             "tt_logq_stream_update: alpha %g / 1 - alpha %g outside (0, 1] / [0, 1)", alpha, one_minus_alpha);
  TT_CHECK_CUDA(launch_k(logq_stream_update_kernel, dim3(1), dim3(kLogqThreads), 0, stream, ids, n, A, Bv, h, log2H,
                         step_dev, alpha, one_minus_alpha, off_out));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_logq_table_gather(const int64_t* ids, int n, const float* table, int64_t N, float floor_,
                                    float* off_out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(ids && table && off_out && n > 0 && N > 0, "tt_logq_table_gather: bad arguments");
  TT_CHECK_CUDA(launch_k(logq_table_gather_kernel, dim3((n + 255) / 256), dim3(256), 0, stream, ids, n, table, N,
                         floor_, off_out));
  TT_LAUNCH_CHECK();
  return TT_OK;
}
