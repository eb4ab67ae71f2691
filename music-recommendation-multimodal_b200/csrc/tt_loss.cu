// Symmetric InfoNCE with same-user collision masking (src/models/two_tower.py:106-140),
// organised as ROW problems so the same kernels serve one GPU and data-parallel training
// with all-gathered negatives:
//   S  = U_loc I_all^T / tau   rows = local users,  positives at column pos0 + i
//   S' = I_loc U_all^T / tau   rows = local items,  positives at column pos0 + i
// loss = 1/2 (mean_i CE(S_i) + mean_i CE(S'_i)). The column softmax term of dS needs the
// log-sum-exp of each COLUMN over all rows of all ranks, which is exactly the row LSE of the
// other matrix at the owning rank: two tiny all-gathers, no reduce-scatter.
//
// Kernels: (1) mask in place + row log-sum-exp (warp per row, online max/sum, shuffles),
// (2) dS = c * (exp(S - lse_row) + exp(S - lse_col) - 2*onehot) as bf16, (3) scalar loss.
#include "../../include/tt_b200.h"
#include "tt_common.cuh"

namespace tt {

// kOffset: every logit of column j enters the row's log-sum-exp and positive as x - col_off[j] (logQ correction of
// sampled negatives, tt_infonce_rows_off); masked entries are -1e4 before the offset. The offsets come last in the
// parameter list so that the kOffset = false instantiation keeps the parameter layout (and code) of the plain kernel.
template <bool kOffset>
__global__ void __launch_bounds__(256) infonce_rows_kernel(float* __restrict__ S, int R, int C, int ld,
                                                           const int64_t* __restrict__ uid_rows,
                                                           const int64_t* __restrict__ uid_cols, int pos0,
                                                           float* __restrict__ row_lse, float* __restrict__ pos_logit,
                                                           const float* __restrict__ col_off) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= R) return;
  float* s = S + static_cast<size_t>(row) * ld;
  const int pos = pos0 + row;
  const bool masked = uid_rows != nullptr;
  const int64_t uid = masked ? uid_rows[row] : 0;
  float m = -INFINITY, l = 0.f;
  for (int j = lane; j < C; j += 32) {
    float x = s[j];
    if (masked && j != pos && uid_cols[j] == uid) {
      x = -1e4f;  // the reference's fill value (fp16-safe), two_tower.py:124
      s[j] = x;
    }
    if (kOffset) x -= col_off[j];
    const float nm = fmaxf(m, x);
    l = l * __expf(m - nm) + __expf(x - nm);
    m = nm;
  }
  // combine the 32 (m, l) pairs
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
    const float l2 = __shfl_xor_sync(0xffffffffu, l, o);
    const float nm = fmaxf(m, m2);
    const float a = (m == -INFINITY) ? 0.f : l * __expf(m - nm);
    const float b = (m2 == -INFINITY) ? 0.f : l2 * __expf(m2 - nm);
    l = a + b;
    m = nm;
  }
  if (lane == 0) {
    row_lse[row] = m + __logf(l);
    pos_logit[row] = kOffset ? s[pos] - col_off[pos] : s[pos];
  }
}

// kOffset: dS = coef * (exp(S - col_off[j] - row_lse[i]) + exp(S - row_off[pos0 + i] - col_lse[j]) - 2*onehot): the
// row direction subtracts its columns' offsets, the column direction the offset of this row's own entity.
template <bool kOffset>
__global__ void __launch_bounds__(256) infonce_grad_kernel(const float* __restrict__ S, int R, int C, int ld,
                                                           const float* __restrict__ row_lse,
                                                           const float* __restrict__ col_lse, int pos0, float coef,
                                                           __nv_bfloat16* __restrict__ dS, int ld_d,
                                                           const float* __restrict__ col_off,
                                                           const float* __restrict__ row_off) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.y;
  const int j = (blockIdx.x * blockDim.x + threadIdx.x) * 2;
  if (j >= C) return;
  const float lr = row_lse[row];
  const float ro = kOffset ? row_off[pos0 + row] : 0.f;
  const float* s = S + static_cast<size_t>(row) * ld;
  float g[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int c = j + k;
    float v = 0.f;
    if (c < C) {
      const float x = s[c];
      if (kOffset) {
        v = __expf(x - col_off[c] - lr) + __expf(x - ro - col_lse[c]);
      } else {
        v = __expf(x - lr) + __expf(x - col_lse[c]);
      }
      if (c == pos0 + row) v -= 2.f;
      v *= coef;
    }
    g[k] = v;
  }
  if (j + 1 < C || (ld_d & 1) == 0) {
    *reinterpret_cast<uint32_t*>(dS + static_cast<size_t>(row) * ld_d + j) = pack_bf16(g[0], g[1]);
  } else {
    dS[static_cast<size_t>(row) * ld_d + j] = __float2bfloat16_rn(g[0]);
  }
}

// loss = coef * ( sum_i (lse_a[i] - pos_a[i]) + sum_i (lse_b[i] - pos_b[i]) ); single block, deterministic.
__global__ void __launch_bounds__(256) infonce_loss_kernel(const float* lse_a, const float* pos_a, const float* lse_b,
                                                           const float* pos_b, int R, float coef, float* loss) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s[256];
  float acc = 0.f;
  for (int i = threadIdx.x; i < R; i += 256) acc += (lse_a[i] - pos_a[i]) + (lse_b[i] - pos_b[i]);
  s[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *loss = s[0] * coef;
}

// In-batch Recall@k of `evaluate` (src/train.py:95-103): row i hits when its positive column is among the k
// best logits of the row. One warp per row counts the entries that precede the positive in the canonical order
// (logit descending, column ascending) — the rank of the positive — so no top-k list is ever formed.
// acc[0] += hits, acc[1] += rows (integers held in fp32: exact below 2^24, summation order irrelevant).
__global__ void __launch_bounds__(256) inbatch_recall_kernel(const float* __restrict__ S, int R, int C, int ld, int pos0,
                                                             int k, float* __restrict__ acc) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ int s_hits;
  if (threadIdx.x == 0) s_hits = 0;
  __syncthreads();
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row < R) {
    const float* s = S + static_cast<size_t>(row) * ld;
    const int pos = pos0 + row;
    const float d = s[pos];
    int better = 0;
    for (int j = lane; j < C; j += 32) {
      const float x = s[j];
      better += (x > d) || (x == d && j < pos);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) better += __shfl_xor_sync(0xffffffffu, better, o);
    if (lane == 0 && better < k) atomicAdd(&s_hits, 1);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_hits) atomicAdd(acc, static_cast<float>(s_hits));
    const int first = (blockIdx.x * blockDim.x) >> 5;
    const int rows_here = min(R - first, static_cast<int>(blockDim.x >> 5));
    if (rows_here > 0) atomicAdd(acc + 1, static_cast<float>(rows_here));
  }
}

}  // namespace tt

using namespace tt;

extern "C" int tt_inbatch_recall(const float* S, int R, int C, int ld, int pos0, int k, float* acc, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(S && acc && R > 0 && C > 0 && ld >= C && k > 0, "tt_inbatch_recall: bad arguments");
  TT_REQUIRE(pos0 >= 0 && pos0 + R <= C, "tt_inbatch_recall: positives [%d, %d) outside %d columns", pos0, pos0 + R, C);
  TT_CHECK_CUDA(launch_k(inbatch_recall_kernel, dim3((R * 32 + 255) / 256), dim3(256), 0, stream, S, R, C, ld, pos0, k, acc));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_infonce_rows(float* S, int R, int C, int ld, const int64_t* uid_rows, const int64_t* uid_cols,
                               int pos0, float* row_lse, float* pos_logit, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(S && row_lse && pos_logit && R > 0 && C > 0 && ld >= C, "tt_infonce_rows: bad arguments");
  TT_REQUIRE((uid_rows == nullptr) == (uid_cols == nullptr), "tt_infonce_rows: uid_rows/uid_cols come together");
  TT_REQUIRE(pos0 >= 0 && pos0 + R <= C, "tt_infonce_rows: positives [%d, %d) outside %d columns", pos0, pos0 + R, C);
  TT_CHECK_CUDA(launch_k(infonce_rows_kernel<false>, dim3((R * 32 + 255) / 256), dim3(256), 0, stream, S, R, C, ld, uid_rows, uid_cols, pos0, row_lse, pos_logit, nullptr));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_infonce_rows_off(float* S, int R, int C, int ld, const int64_t* uid_rows, const int64_t* uid_cols,
                                   int pos0, const float* col_off, float* row_lse, float* pos_logit, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(S && col_off && row_lse && pos_logit && R > 0 && C > 0 && ld >= C, "tt_infonce_rows_off: bad arguments");
  TT_REQUIRE((uid_rows == nullptr) == (uid_cols == nullptr), "tt_infonce_rows_off: uid_rows/uid_cols come together");
  TT_REQUIRE(pos0 >= 0 && pos0 + R <= C, "tt_infonce_rows_off: positives [%d, %d) outside %d columns", pos0, pos0 + R, C);
  TT_CHECK_CUDA(launch_k(infonce_rows_kernel<true>, dim3((R * 32 + 255) / 256), dim3(256), 0, stream, S, R, C, ld, uid_rows, uid_cols, pos0, row_lse, pos_logit, col_off));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

static dim3 infonce_grad_grid(int R, int C) {
  dim3 grid((C / 2 + 255) / 256 + ((C / 2) % 256 == 0 && C % 2 ? 1 : 0), R);
  if (grid.x == 0) grid.x = 1;
  return grid;
}

extern "C" int tt_infonce_grad(const float* S, int R, int C, int ld, const float* row_lse, const float* col_lse,
                               int pos0, float coef, void* dS_bf16, int ld_d, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(S && row_lse && col_lse && dS_bf16 && R > 0 && C > 0, "tt_infonce_grad: bad arguments");
  TT_REQUIRE(ld_d % 2 == 0, "tt_infonce_grad: ld_d must be even");
  TT_CHECK_CUDA(launch_k(infonce_grad_kernel<false>, infonce_grad_grid(R, C), dim3(256), 0, stream, S, R, C, ld, row_lse, col_lse, pos0, coef, static_cast<__nv_bfloat16*>(dS_bf16), ld_d, nullptr, nullptr));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_infonce_grad_off(const float* S, int R, int C, int ld, const float* row_lse, const float* col_lse,
                                   int pos0, float coef, const float* col_off, const float* row_off, void* dS_bf16,
                                   int ld_d, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(S && row_lse && col_lse && col_off && row_off && dS_bf16 && R > 0 && C > 0 && ld >= C,
             "tt_infonce_grad_off: bad arguments");
  TT_REQUIRE(ld_d % 2 == 0 && ld_d >= C, "tt_infonce_grad_off: ld_d must be even and at least C");
  TT_REQUIRE(pos0 >= 0 && pos0 + R <= C, "tt_infonce_grad_off: positives [%d, %d) outside %d columns", pos0, pos0 + R, C);
  TT_CHECK_CUDA(launch_k(infonce_grad_kernel<true>, infonce_grad_grid(R, C), dim3(256), 0, stream, S, R, C, ld, row_lse, col_lse, pos0, coef, static_cast<__nv_bfloat16*>(dS_bf16), ld_d, col_off, row_off));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_infonce_loss(const float* lse_a, const float* pos_a, const float* lse_b, const float* pos_b, int R,
                               float coef, float* loss, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(lse_a && pos_a && lse_b && pos_b && loss && R > 0, "tt_infonce_loss: bad arguments");
  TT_CHECK_CUDA(launch_k(infonce_loss_kernel, dim3(1), dim3(256), 0, stream, lse_a, pos_a, lse_b, pos_b, R, coef, loss));
  TT_LAUNCH_CHECK();
  return TT_OK;
}
