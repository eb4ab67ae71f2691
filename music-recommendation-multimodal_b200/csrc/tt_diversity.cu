// Diversified recommendations: exact maximal-marginal-relevance (MMR) selection of k items from each user's
// candidate pool (the exact top P of the retrieval path, canonical order).
//
//   lambda = 1 - diversity, mu = 1 - lambda (fp64, from the host). m_j = max sim(c_j, s) over the picks s so far
//   (0 before the first pick); sim = fp32 rows, fp64 accumulate, one rounding to fp32 (the finalize re-score's
//   arithmetic). Step t picks the unpicked position j with c_j >= 0 and the largest
//   obj_j = lambda * r_j - mu * m_j, evaluated as two correctly rounded fp64 products and one subtraction (no FMA);
//   a tie goes to the smaller j.
//
//   grid: one cluster of two CTAs per user. CTA c holds pool positions [c*H, min((c+1)*H, P)), H = ceil(P/2), as fp32
//   rows in dynamic shared memory (H KB, loaded by 1 KB bulk async copies), so every row is read from HBM once per
//   user and P = 256 fits in two 128 KB halves. Per step each CTA finds its best position, the pair exchanges the two
//   candidates through distributed shared memory and both take the same winner; then each CTA copies the winner's
//   row (from its own or its peer's shared memory) and updates m_j of its unpicked positions with one dot product
//   each: at most (k-1) * P dot products per user, never the P x P Gram matrix. Every sum has a fixed order, so the
//   result is bit-identical from run to run and on every rank.
#include <cooperative_groups.h>

#include "../../include/tt_b200.h"
#include "tt_common.cuh"

namespace cg = cooperative_groups;

namespace tt {
namespace {

constexpr int kD = 256;
constexpr int kMaxPool = 256;
constexpr int kHalf = kMaxPool / 2;     // pool positions per CTA
constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

struct MmrParams {
  const int32_t* pool_idx;  // [U, P] global ids, -1 = no candidate
  const float* pool_score;  // [U, P] exact relevances
  const float* rows;        // source table (mode 0) or gathered rows [U, P, 256] (mode 1)
  int U, P, k, half, source, item_base, num_rows;
  double lam, mu;
  int32_t* out_idx;         // [U, k]
  float* out_score;         // [U, k]
};

// one step's best candidate of a CTA: objective and pool position (-1 = none)
struct Best {
  double obj;
  int pos;
};

__device__ __forceinline__ bool better(double a, int ia, double b, int ib) {
  if (ib < 0) return ia >= 0;
  if (ia < 0) return false;
  return a > b || (a == b && ia < ib);
}

__device__ __forceinline__ void bulk_load_1k(void* dst, const void* src, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], 1024, [%2];" ::"r"(smem_u32(dst)),
      "l"(src), "r"(smem_u32(bar))
      : "memory");
}

__global__ void __launch_bounds__(kThreads) mmr_select_kernel(const MmrParams p) {
  pdl_launch_dependents();
  extern __shared__ __align__(128) uint8_t smem_raw[];
  float* s_rows = reinterpret_cast<float*>(smem_raw);       // [half][256]
  __shared__ float s_rel[kHalf], s_m[kHalf];
  __shared__ __align__(16) float s_pick[kD];
  __shared__ int s_id[kHalf];
  __shared__ int s_picked[kHalf];
  __shared__ Best s_warp[kWarps];
  __shared__ Best s_best[2];                                // this CTA's candidate, double-buffered by step parity
  __shared__ __align__(8) uint64_t s_bar;

  cg::cluster_group cluster = cg::this_cluster();
  const int rank = static_cast<int>(cluster.block_rank());
  const int u = blockIdx.x >> 1;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int base = rank * p.half;                          // pool position of this CTA's local row 0
  const int nloc = max(0, min(p.half, p.P - base));
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    fence_barrier_init();
  }
  pdl_wait();
  __syncthreads();

  // candidates and their rows
  const size_t urow = static_cast<size_t>(u) * p.P;
  if (tid < kHalf) {
    int id = -1;
    float r = -INFINITY;
    if (tid < nloc) {
      id = p.pool_idx[urow + base + tid];
      r = p.pool_score[urow + base + tid];
      if (p.source == 0 && (id < p.item_base || id - p.item_base >= p.num_rows)) id = -1;
    }
    s_id[tid] = id;
    s_rel[tid] = r;
    s_m[tid] = 0.f;
    s_picked[tid] = 0;
  }
  __syncthreads();
  if (warp == 0) {
    int bytes = 0;
    // k = 1 takes the first pick only, which needs no row
    for (int i = lane; p.k > 1 && i < nloc; i += 32) {
      const int id = s_id[i];
      if (id < 0) continue;
      const float* src = p.source == 0 ? p.rows + static_cast<size_t>(id - p.item_base) * kD
                                       : p.rows + (urow + base + i) * kD;
      bulk_load_1k(s_rows + i * kD, src, &s_bar);
      bytes += 1024;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bytes += __shfl_xor_sync(0xffffffffu, bytes, o);
    if (lane == 0) mbar_arrive_expect_tx(&s_bar, static_cast<uint32_t>(bytes));
  }

  int n_out = 0;
  bool rows_ready = false;
  for (int t = 0; t < p.k; ++t) {
    // this CTA's best unpicked admissible position: one position per thread, warp then CTA argmax
    Best b{0.0, -1};
    if (tid < nloc && s_id[tid] >= 0 && !s_picked[tid]) {
      const double o = __dsub_rn(__dmul_rn(p.lam, static_cast<double>(s_rel[tid])),
                                 __dmul_rn(p.mu, static_cast<double>(s_m[tid])));
      b = Best{o, base + tid};
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, b.obj, o);
      const int ib = __shfl_xor_sync(0xffffffffu, b.pos, o);
      if (better(ob, ib, b.obj, b.pos)) b = Best{ob, ib};
    }
    if (lane == 0) s_warp[warp] = b;
    __syncthreads();
    if (tid == 0) {
      Best c = s_warp[0];
      for (int w = 1; w < kWarps; ++w)
        if (better(s_warp[w].obj, s_warp[w].pos, c.obj, c.pos)) c = s_warp[w];
      s_best[t & 1] = c;
    }
    cluster.sync();
    // both CTAs combine the pair's candidates in the same way and reach the same winner
    const Best b0 = *cluster.map_shared_rank(&s_best[t & 1], 0);
    const Best b1 = *cluster.map_shared_rank(&s_best[t & 1], 1);
    const Best w = better(b1.obj, b1.pos, b0.obj, b0.pos) ? b1 : b0;
    if (w.pos < 0) break;                                   // no admissible candidate left
    const int owner = w.pos / p.half, wl = w.pos - owner * p.half;
    if (owner == rank && tid == 0) {
      s_picked[wl] = 1;
      p.out_idx[static_cast<size_t>(u) * p.k + t] = s_id[wl];
      p.out_score[static_cast<size_t>(u) * p.k + t] = s_rel[wl];
    }
    n_out = t + 1;
    if (t + 1 == p.k) break;
    if (t == 0) {                                           // rows are first needed here: ours and the peer's
      mbar_wait(&s_bar, 0);
      rows_ready = true;
      cluster.sync();
    }
    // the winner's row, from our shared memory or the peer's (rows are never written after the load)
    {
      const float* src = cluster.map_shared_rank(s_rows + static_cast<size_t>(wl) * kD, owner);
      s_pick[tid] = src[tid];
    }
    __syncthreads();
    float pk[8];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float4 x = reinterpret_cast<const float4*>(s_pick)[h * 32 + lane];
      pk[4 * h] = x.x; pk[4 * h + 1] = x.y; pk[4 * h + 2] = x.z; pk[4 * h + 3] = x.w;
    }
    // m_j of the unpicked admissible positions: one warp per row, fp64 accumulate in a fixed order
    for (int i = warp; i < nloc; i += kWarps) {
      if (s_id[i] < 0 || s_picked[i]) continue;             // warp-uniform
      const float* row = s_rows + static_cast<size_t>(i) * kD;
      double acc = 0.0;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 x = reinterpret_cast<const float4*>(row)[h * 32 + lane];
        acc += static_cast<double>(pk[4 * h]) * x.x + static_cast<double>(pk[4 * h + 1]) * x.y +
               static_cast<double>(pk[4 * h + 2]) * x.z + static_cast<double>(pk[4 * h + 3]) * x.w;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      const float sim = static_cast<float>(acc);
      if (lane == 0) s_m[i] = t == 0 ? sim : fmaxf(s_m[i], sim);   // m_j: 0 only before the first pick
    }
    __syncthreads();
  }
  // fewer admissible candidates than k: -1 / -inf tail (written by rank 0 only)
  if (rank == 0) {
    for (int t = n_out + tid; t < p.k; t += kThreads) {
      p.out_idx[static_cast<size_t>(u) * p.k + t] = -1;
      p.out_score[static_cast<size_t>(u) * p.k + t] = -INFINITY;
    }
  }
  if (!rows_ready) mbar_wait(&s_bar, 0);                   // no bulk copy may outlive the CTA
  cluster.sync();                                           // the peer may still read our rows / candidate
}

// Sharded catalogs: out[u, j] = row of pool id c_uj when this shard owns it (item_base <= id < item_base + num_rows),
// zeros otherwise. One warp per (u, j).
__global__ void __launch_bounds__(256) mmr_gather_kernel(const int32_t* __restrict__ pool_idx, int n, const float* table,
                                                         int item_base, int num_rows, float* out) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t r = static_cast<size_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= static_cast<size_t>(n)) return;
  const int id = pool_idx[r];
  const bool mine = id >= item_base && id - item_base < num_rows;
  float4* dst = reinterpret_cast<float4*>(out + r * kD);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (mine) x = __ldg(reinterpret_cast<const float4*>(table + static_cast<size_t>(id - item_base) * kD) + h * 32 + lane);
    dst[h * 32 + lane] = x;
  }
}

}  // namespace
}  // namespace tt

using namespace tt;

extern "C" int tt_mmr_select(const int32_t* pool_idx, const float* pool_score, int U, int P, int k, double lam,
                             double mu, int source, const float* rows, int item_base, int num_rows, int32_t* out_idx,
                             float* out_score, void* stream) {
  TT_REQUIRE(U >= 0, "tt_mmr_select: U=%d < 0", U);
  TT_REQUIRE(1 <= k && k <= P && P <= kMaxPool, "tt_mmr_select: need 1 <= k=%d <= P=%d <= %d", k, P, kMaxPool);
  TT_REQUIRE(lam >= 0.0 && lam <= 1.0 && mu >= 0.0 && mu <= 1.0, "tt_mmr_select: lambda / mu outside [0, 1]");
  TT_REQUIRE(source == TT_MMR_ROWS_TABLE || source == TT_MMR_ROWS_GATHERED, "tt_mmr_select: unknown row source %d",
             source);
  if (U == 0) return TT_OK;   // an empty batch: its tensors may have no storage (null data pointers)
  TT_REQUIRE(pool_idx && pool_score && rows && out_idx && out_score, "tt_mmr_select: null pointer");
  TT_REQUIRE(source != TT_MMR_ROWS_TABLE || num_rows > 0, "tt_mmr_select: empty table");
  TT_REQUIRE((reinterpret_cast<uintptr_t>(rows) & 15) == 0, "tt_mmr_select: rows must be 16-byte aligned");
  TT_REQUIRE(U <= (1 << 30) - 1, "tt_mmr_select: U=%d is too many for one launch", U);
  MmrParams p;
  p.pool_idx = pool_idx; p.pool_score = pool_score; p.rows = rows;
  p.U = U; p.P = P; p.k = k; p.half = (P + 1) / 2; p.source = source;
  p.item_base = item_base; p.num_rows = num_rows;
  p.lam = lam; p.mu = mu;
  p.out_idx = out_idx; p.out_score = out_score;
  const size_t smem = static_cast<size_t>(p.half) * kD * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    TT_CHECK_CUDA(cudaFuncSetAttribute(mmr_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       kHalf * kD * static_cast<int>(sizeof(float))));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(2 * U));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  TT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, mmr_select_kernel, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_mmr_gather_rows(const int32_t* pool_idx, int n, const float* table, int item_base, int num_rows,
                                  float* out, void* stream) {
  TT_REQUIRE(n >= 0, "tt_mmr_gather_rows: n=%d < 0", n);
  if (n == 0) return TT_OK;
  TT_REQUIRE(pool_idx && table && out && num_rows > 0, "tt_mmr_gather_rows: bad arguments");
  const unsigned blocks = static_cast<unsigned>((static_cast<size_t>(n) + 7) / 8);
  TT_CHECK_CUDA(launch_k(mmr_gather_kernel, dim3(blocks), dim3(256), 0, static_cast<cudaStream_t>(stream), pool_idx, n,
                         table, item_base, num_rows, out));
  TT_LAUNCH_CHECK();
  return TT_OK;
}
