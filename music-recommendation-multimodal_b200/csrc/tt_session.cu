// Incremental user tower for listening sessions: one new query row per user attends over that user's cached keys
// and values.
//
// The encoder is causal and a history is a right-padded prefix, so appending item p to a history of length p leaves
// every earlier position's output unchanged in every layer. Per layer only the new row's Q/K/V are computed (a GEMM
// of n rows); this kernel stores the new K/V row in the cache and runs the single-query attention of that row over
// positions 0..p of its slot.
//
//   cache layout: one K and one V plane per layer, bf16 [capacity, H, L, 64]. A (slot, head) is one contiguous stretch
//   of L x 128 bytes, so the keys a CTA reads are one sequential stream.
//   grid: one cluster of S CTAs per (row, head). CTA s takes keys [s*chunk, min((s+1)*chunk, p+1)), so a single user
//   at L = 2048 spreads over 4 x 8 CTAs. Each warp keeps an online softmax over its keys (8 keys x 4 dim quarters per
//   warp instruction, 16-byte loads); the 4 warps are combined in shared memory, then CTA rank 0 combines the S CTAs
//   through distributed shared memory, always in rank order: results are bit-identical from run to run.
//   The new key/value of row p is read from qkv, never from the cache the same kernel writes.
#include <cooperative_groups.h>

#include "../../include/tt_b200.h"
#include "tt_common.cuh"

namespace cg = cooperative_groups;

namespace tt {
namespace {

constexpr int kDh = 64;
constexpr int kThreads = 128;
constexpr int kMaxL = 4096;
constexpr int kMaxSplits = 8;      // portable cluster size
constexpr int kKeysPerSplit = 256; // below this many keys per CTA the split count stops growing
constexpr float kLog2e = 1.4426950408889634f;

struct SessionAttnParams {
  const __nv_bfloat16* qkv;  // [n, 3*H*64]: Q | K | V of the new rows
  __nv_bfloat16* kc;         // [capacity, H, L, 64]
  __nv_bfloat16* vc;         // [capacity, H, L, 64]
  const int32_t* slots;      // [n]
  const int32_t* pos;        // [n]
  int n, H, L, capacity, splits, chunk;
  __nv_bfloat16* ctx;        // [n, H*64]
};

__device__ __forceinline__ void load16(const __nv_bfloat16* p, float (&v)[16]) {
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const uint4 x = __ldg(reinterpret_cast<const uint4*>(p) + u);
    const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const float2 f = unpack_bf16(w[h]);
      v[u * 8 + h * 2] = f.x;
      v[u * 8 + h * 2 + 1] = f.y;
    }
  }
}

// partial softmax state of a set of keys: running max m (log2 domain), sum l, unnormalised output acc[64]
struct Partial {
  float m, l, acc[kDh];
};

__global__ void __launch_bounds__(kThreads) session_attn_kernel(const SessionAttnParams p) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ Partial s_warp[kThreads / 32];
  __shared__ Partial s_cta;
  cg::cluster_group cluster = cg::this_cluster();
  const int split = static_cast<int>(cluster.block_rank());
  const int rh = blockIdx.x / p.splits;
  const int r = rh / p.H, h = rh % p.H;
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ks = lane >> 2, dq = lane & 3;
  const int D = p.H * kDh;
  const int slot = p.slots[r], pos = p.pos[r];
  const bool valid = slot >= 0 && slot < p.capacity && pos >= 0 && pos < p.L;
  const __nv_bfloat16* qrow = p.qkv + static_cast<size_t>(r) * 3 * D + h * kDh;
  const __nv_bfloat16* knew = qrow + D;
  const __nv_bfloat16* vnew = qrow + 2 * D;
  const size_t plane = valid ? (static_cast<size_t>(slot) * p.H + h) * p.L * kDh : 0;
  const int k0 = split * p.chunk;
  const int k1 = valid ? min(k0 + p.chunk, pos + 1) : 0;
  if (valid && pos >= k0 && pos < k0 + p.chunk && threadIdx.x < 16) {   // the new row's K | V into the cache
    const int t = threadIdx.x & 7;
    const __nv_bfloat16* src = threadIdx.x < 8 ? knew : vnew;
    __nv_bfloat16* dst = (threadIdx.x < 8 ? p.kc : p.vc) + plane + static_cast<size_t>(pos) * kDh;
    reinterpret_cast<uint4*>(dst)[t] = __ldg(reinterpret_cast<const uint4*>(src) + t);
  }
  float q[16];
  load16(qrow + dq * 16, q);
  const float c1 = 0.125f * kLog2e;
  float m = -INFINITY, l = 0.f, acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  // warp w takes keys j0 + ks, j0 = k0 + 8w, k0 + 8w + 32, ...; the ks = 0 key of every iteration is live, so the
  // running max is finite from the first iteration on
#pragma unroll 2
  for (int j0 = k0 + wib * 8; j0 < k1; j0 += 32) {
    const int j = j0 + ks;
    float s = -INFINITY, v[16];
    if (j < k1) {
      const __nv_bfloat16* kr = j == pos ? knew : p.kc + plane + static_cast<size_t>(j) * kDh;
      const __nv_bfloat16* vr = j == pos ? vnew : p.vc + plane + static_cast<size_t>(j) * kDh;
      float k[16];
      load16(kr + dq * 16, k);
      load16(vr + dq * 16, v);
      float d = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) d += k[i] * q[i];
      s = d;
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = 0.f;
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s *= c1;
    float gm = fmaxf(s, __shfl_xor_sync(0xffffffffu, s, 4));
    gm = fmaxf(gm, __shfl_xor_sync(0xffffffffu, gm, 8));
    gm = fmaxf(gm, __shfl_xor_sync(0xffffffffu, gm, 16));
    const float mn = fmaxf(m, gm);
    const float alpha = exp2f(m - mn);
    const float pj = exp2f(s - mn);
    l = l * alpha + pj;
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = acc[i] * alpha + pj * v[i];
    m = mn;
  }
  // sum over the 8 key slots of the warp (the 4 lanes of a key carry the same l)
#pragma unroll
  for (int o = 4; o < 32; o <<= 1) {
    l += __shfl_xor_sync(0xffffffffu, l, o);
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
  }
  if (ks == 0) {
#pragma unroll
    for (int i = 0; i < 16; ++i) s_warp[wib].acc[dq * 16 + i] = acc[i];
    if (dq == 0) { s_warp[wib].m = m; s_warp[wib].l = l; }
  }
  __syncthreads();
  // the CTA's keys: combine the 4 warps in warp order (a warp without keys has m = -inf and weight 0)
  if (threadIdx.x < kDh) {
    const int d = threadIdx.x;
    float M = -INFINITY;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) M = fmaxf(M, s_warp[w].m);
    float L = 0.f, a = 0.f;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) {
      const float f = s_warp[w].m == -INFINITY ? 0.f : exp2f(s_warp[w].m - M);
      L += s_warp[w].l * f;
      a += s_warp[w].acc[d] * f;
    }
    s_cta.acc[d] = a;
    if (d == 0) { s_cta.m = M; s_cta.l = L; }
  }
  cluster.sync();
  // rank 0 combines the S CTAs of the row in rank order
  if (split == 0 && threadIdx.x < kDh) {
    const int d = threadIdx.x;
    float M = -INFINITY;
    for (int c = 0; c < p.splits; ++c) M = fmaxf(M, cluster.map_shared_rank(&s_cta, c)->m);
    float L = 0.f, a = 0.f;
    for (int c = 0; c < p.splits; ++c) {
      const Partial* o = cluster.map_shared_rank(&s_cta, c);
      const float mc = o->m;
      const float f = mc == -INFINITY ? 0.f : exp2f(mc - M);
      L += o->l * f;
      a += o->acc[d] * f;
    }
    p.ctx[static_cast<size_t>(r) * D + h * kDh + d] = __float2bfloat16_rn(valid ? a / L : 0.f);
  }
  cluster.sync();   // the other CTAs' shared memory stays alive until rank 0 has read it
}

}  // namespace
}  // namespace tt

using namespace tt;

extern "C" int tt_session_attn(const void* qkv, void* k_cache, void* v_cache, const int32_t* slots, const int32_t* pos,
                               int n, int H, int L, int capacity, void* ctx, void* stream_) {
  TT_REQUIRE(qkv && k_cache && v_cache && slots && pos && ctx, "tt_session_attn: null pointer");
  TT_REQUIRE(n > 0 && H > 0 && capacity > 0, "tt_session_attn: bad arguments");
  TT_REQUIRE(L >= 1 && L <= kMaxL, "tt_session_attn: L=%d outside [1, %d]", L, kMaxL);
  SessionAttnParams p;
  p.qkv = static_cast<const __nv_bfloat16*>(qkv);
  p.kc = static_cast<__nv_bfloat16*>(k_cache);
  p.vc = static_cast<__nv_bfloat16*>(v_cache);
  p.slots = slots; p.pos = pos;
  p.n = n; p.H = H; p.L = L; p.capacity = capacity;
  p.splits = min(kMaxSplits, (L + kKeysPerSplit - 1) / kKeysPerSplit);
  p.chunk = ((L + p.splits - 1) / p.splits + 31) / 32 * 32;
  p.ctx = static_cast<__nv_bfloat16*>(ctx);
  const size_t blocks = static_cast<size_t>(n) * H * p.splits;
  TT_REQUIRE(blocks < (1ull << 31), "tt_session_attn: %d rows is too many for one launch", n);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(blocks));
  cfg.blockDim = dim3(kThreads);
  cfg.stream = static_cast<cudaStream_t>(stream_);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = p.splits;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  TT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, session_attn_kernel, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}
