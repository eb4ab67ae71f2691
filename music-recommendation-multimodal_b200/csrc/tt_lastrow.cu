// Last-layer specialisation of the SASRec user tower (SURVEY.md §8 a5).
//
// The reference gathers out[b, len_b - 1] after the LAST encoder layer (src/models/user_tower.py:
// 122-132); nothing else of that layer's output is ever read, and its pad/other rows carry zero
// gradient. So in the last layer only K and V are needed for every position; the query, the
// attention output, out_proj, both residual adds, norm2 and the FFN are needed for ONE row per
// sequence. These kernels implement that exactly: without dropout, the same results as the full
// computation. With dropout the masks differ: the out_proj / linear1 / linear2 GEMMs of the pruned
// layer run on the compact [B, .] rows, so their epilogues hash the compact row b where the full
// schedule hashes the token row b*L + last_b (tt_attn_lastq_* keep the full-sequence index). Both
// are valid draws of the same dropout, not the same draw.
//   tt_gather_rows        : rows[b] = x[b*L + last_idx[b]]  (fp32 and/or bf16 copies)
//   tt_scatter_rows_add   : x[b*L + last_idx[b]] (+)= rows[b]
//   tt_attn_lastq_fwd/bwd : causal attention for the single query row len-1 of every
//                           (sequence, head): one warp per (b, h), lane-per-key dot products,
//                           warp-shuffle softmax, lane-per-dim-pair P*V. HBM/L2-bound gathers of
//                           128-byte K/V rows; no tensor cores (2*L*64 MACs per problem).
#include "../../include/tt_b200.h"
#include "tt_common.cuh"

namespace tt {

static constexpr int kDh = 64;
static constexpr int kMaxL = 512;
static constexpr float kLog2e = 1.4426950408889634f;

__global__ void gather_rows_kernel(const float* __restrict__ x32, const __nv_bfloat16* __restrict__ x16,
                                   const int32_t* __restrict__ last_idx, int B, int L, int W,
                                   float* __restrict__ out32, __nv_bfloat16* __restrict__ out16) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= B) return;
  const size_t row = static_cast<size_t>(b) * L + last_idx[b];
  for (int c = lane * 4; c < W; c += 128) {
    if (x32 && out32)
      *reinterpret_cast<float4*>(out32 + static_cast<size_t>(b) * W + c) =
          __ldg(reinterpret_cast<const float4*>(x32 + row * W + c));
    if (x16 && out16)
      *reinterpret_cast<uint2*>(out16 + static_cast<size_t>(b) * W + c) =
          __ldg(reinterpret_cast<const uint2*>(x16 + row * W + c));
  }
}

__global__ void scatter_rows_add_kernel(const float* __restrict__ rows, const int32_t* __restrict__ last_idx, int B,
                                        int L, int W, float* __restrict__ x, int accumulate) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= B) return;
  const size_t row = static_cast<size_t>(b) * L + last_idx[b];
  for (int c = lane * 4; c < W; c += 128) {
    float4 v = __ldg(reinterpret_cast<const float4*>(rows + static_cast<size_t>(b) * W + c));
    float4* dst = reinterpret_cast<float4*>(x + row * W + c);
    if (accumulate) {
      const float4 o = *dst;
      v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
    }
    *dst = v;
  }
}

struct LastQParams {
  const __nv_bfloat16* q;     // [B, H*64]
  const __nv_bfloat16* qkv;   // [B*L, 3*H*64] (K, V thirds used)
  const int32_t* last_idx;    // [B]
  int B, L, H;
  float scale;
  uint32_t drop_thresh; float drop_scale; uint64_t seed; const uint64_t* seed_dev; uint32_t site;
  __nv_bfloat16* ctx;         // [B, H*64]
  float* lse;                 // [B, H]
  // backward
  const __nv_bfloat16* dctx;  // [B, H*64]
  __nv_bfloat16* dq;          // [B, H*64]
  __nv_bfloat16* dqkv;        // [B*L, 3*H*64]: K and V thirds written for every position (zeros beyond len)
};

// Lane layout inside a warp: 8 key slots x 4 dim quarters. Lane (ks, dq) = (lane >> 2, lane & 3)
// handles key j = 8*it + ks and dims [16*dq, 16*dq + 16) (two 16-byte loads), so a warp instruction
// reads 8 keys x 128 contiguous bytes; the 4 partial dot products meet with two shuffles.
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
__device__ __forceinline__ float dot16(const float (&a)[16], const float (&b)[16]) {
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) acc += a[i] * b[i];
  return acc;
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}
// 16 scaled values -> 16 bf16 = one 32-byte store: a whole sector per lane (two 16-byte stores left every sector
// half-written until the second instruction; the four lanes of a key row cover its 128 bytes)
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t (&w)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]),
               "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}
__device__ __forceinline__ void store16_scaled(__nv_bfloat16* p, const float (&v)[16], float s) {
  uint32_t w[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) w[e] = pack_bf16(v[2 * e] * s, v[2 * e + 1] * s);
  st_global_v8(p, w);
}

// One block (4 warps) per (b, h). The 32 key slots of an iteration are spread over the block:
// warp w, lane (ks, dq) handles key j = 32*it + 8*w + ks, dims [16*dq, 16*dq+16). Row max / sum and
// the per-dim outputs are combined across the 4 warps through shared memory.
__device__ __forceinline__ float block4_max(float v, float* s4, int wib, int lane) {
  v = warp_max(v);
  if (lane == 0) s4[wib] = v;
  __syncthreads();
  const float r = fmaxf(fmaxf(s4[0], s4[1]), fmaxf(s4[2], s4[3]));
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block4_sum(float v, float* s4, int wib, int lane) {
  v = warp_sum(v);
  if (lane == 0) s4[wib] = v;
  __syncthreads();
  const float r = (s4[0] + s4[1]) + (s4[2] + s4[3]);
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(128) attn_lastq_fwd_kernel(const LastQParams p) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s_p[kMaxL];
  __shared__ float s_acc[4][64];
  __shared__ float s4[4];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ks = lane >> 2, dq = lane & 3;
  const int bh = blockIdx.x;
  const int b = bh / p.H, h = bh % p.H;
  const int D = p.H * kDh;
  const int last = p.last_idx[b];
  const int len = last + 1;
  float q[16];
  load16(p.q + static_cast<size_t>(b) * D + h * kDh + dq * 16, q);
  const __nv_bfloat16* kbase = p.qkv + static_cast<size_t>(b) * p.L * 3 * D + D + h * kDh;
  const __nv_bfloat16* vbase = kbase + D;
  const float c1 = p.scale * kLog2e;
  float m = -INFINITY;
  for (int j0 = 0; j0 < len; j0 += 32) {
    const int j = j0 + wib * 8 + ks;
    float s = -INFINITY;
    if (j < len) {
      float k[16];
      load16(kbase + static_cast<size_t>(j) * 3 * D + dq * 16, k);
      s = dot16(k, q);
    }
    s = quad_sum(s) * c1;          // (-inf stays -inf for keys beyond len)
    if (dq == 0 && j < len) s_p[j] = s;
    m = fmaxf(m, s);
  }
  m = block4_max(m, s4, wib, lane);   // (also orders the s_p writes before the reads below)
  const uint64_t seed = p.seed + ((p.drop_thresh && p.seed_dev) ? *p.seed_dev : 0ull);
  const uint32_t dkey = drop_key(seed, p.site);
  const uint64_t didx0 = (static_cast<uint64_t>(bh) * p.L + last) * p.L;
  float l = 0.f;
  for (int j = threadIdx.x; j < len; j += 128) {
    float e = exp2f(s_p[j] - m);
    l += e;
    if (p.drop_thresh) e = drop_keep_k(dkey, didx0 + j, p.drop_thresh) ? e * p.drop_scale : 0.f;
    s_p[j] = e;
  }
  l = block4_sum(l, s4, wib, lane);
  // ctx[d] = sum_j p_j V[j][d]: warp w takes keys j = w, w+4, ...; lane owns dims (2*lane, 2*lane+1)
  float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
  int j = wib;
  for (; j + 4 < len; j += 8) {
    const float p0 = s_p[j], p1 = s_p[j + 4];
    const float2 v0 = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(vbase + static_cast<size_t>(j) * 3 * D) + lane));
    const float2 v1 = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(vbase + static_cast<size_t>(j + 4) * 3 * D) + lane));
    a0 += p0 * v0.x; a1 += p0 * v0.y;
    b0 += p1 * v1.x; b1 += p1 * v1.y;
  }
  for (; j < len; j += 4) {
    const float p0 = s_p[j];
    const float2 v0 = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(vbase + static_cast<size_t>(j) * 3 * D) + lane));
    a0 += p0 * v0.x; a1 += p0 * v0.y;
  }
  s_acc[wib][2 * lane] = a0 + b0;
  s_acc[wib][2 * lane + 1] = a1 + b1;
  __syncthreads();
  if (wib == 0) {
    const float inv = 1.f / l;
    const float o0 = (s_acc[0][2 * lane] + s_acc[1][2 * lane]) + (s_acc[2][2 * lane] + s_acc[3][2 * lane]);
    const float o1 = (s_acc[0][2 * lane + 1] + s_acc[1][2 * lane + 1]) + (s_acc[2][2 * lane + 1] + s_acc[3][2 * lane + 1]);
    reinterpret_cast<uint32_t*>(p.ctx + static_cast<size_t>(b) * D + h * kDh)[lane] = pack_bf16(o0 * inv, o1 * inv);
    if (lane == 0 && p.lse) p.lse[bh] = (m + log2f(l)) / kLog2e;   // natural-log sum-exp of the scaled scores
  }
}

__global__ void __launch_bounds__(128) attn_lastq_bwd_kernel(const LastQParams p) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s_ds[kMaxL];
  __shared__ float s_acc[4][64];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ks = lane >> 2, dq = lane & 3;
  const int bh = blockIdx.x;
  const int b = bh / p.H, h = bh % p.H;
  const int D = p.H * kDh;
  const int last = p.last_idx[b];
  const int len = last + 1;
  float q[16], g[16];
  load16(p.q + static_cast<size_t>(b) * D + h * kDh + dq * 16, q);
  load16(p.dctx + static_cast<size_t>(b) * D + h * kDh + dq * 16, g);
  float delta;   // dctx . ctx
  {
    const float2 o = unpack_bf16(reinterpret_cast<const uint32_t*>(p.ctx + static_cast<size_t>(b) * D + h * kDh)[lane]);
    const float2 d = unpack_bf16(reinterpret_cast<const uint32_t*>(p.dctx + static_cast<size_t>(b) * D + h * kDh)[lane]);
    delta = warp_sum(o.x * d.x + o.y * d.y);
  }
  const size_t seq0 = static_cast<size_t>(b) * p.L;
  const __nv_bfloat16* kbase = p.qkv + seq0 * 3 * D + D + h * kDh;
  const __nv_bfloat16* vbase = kbase + D;
  __nv_bfloat16* dkbase = p.dqkv + seq0 * 3 * D + D + h * kDh;
  __nv_bfloat16* dvbase = dkbase + D;
  const float c1 = p.scale * kLog2e;
  const float lse2 = p.lse[bh] * kLog2e;
  const uint64_t seed = p.seed + ((p.drop_thresh && p.seed_dev) ? *p.seed_dev : 0ull);
  const uint32_t dkey = drop_key(seed, p.site);
  const uint64_t didx0 = (static_cast<uint64_t>(bh) * p.L + last) * p.L;
  for (int j0 = 0; j0 < p.L; j0 += 32) {
    const int j = j0 + wib * 8 + ks;
    const bool inrange = j < p.L;      // every lane stays in the loop: the quad shuffles use the full mask
    __nv_bfloat16* dk = dkbase + static_cast<size_t>(j) * 3 * D + dq * 16;
    __nv_bfloat16* dv = dvbase + static_cast<size_t>(j) * 3 * D + dq * 16;
    float sdot = 0.f, vdot = 0.f;
    const bool live = j < len;
    if (live) {
      float k[16], v[16];
      load16(kbase + static_cast<size_t>(j) * 3 * D + dq * 16, k);
      load16(vbase + static_cast<size_t>(j) * 3 * D + dq * 16, v);
      sdot = dot16(k, q);
      vdot = dot16(v, g);
    }
    sdot = quad_sum(sdot);
    vdot = quad_sum(vdot);
    if (live) {
      const float pr = exp2f(sdot * c1 - lse2);
      float dp = vdot, pd = pr;
      if (p.drop_thresh) {
        const bool keep = drop_keep_k(dkey, didx0 + j, p.drop_thresh);
        pd = keep ? pr * p.drop_scale : 0.f;
        dp = keep ? dp * p.drop_scale : 0.f;
      }
      const float ds = pr * (dp - delta) * p.scale;
      if (dq == 0) s_ds[j] = ds;
      store16_scaled(dk, q, ds);    // dK_j = dS_j * q
      store16_scaled(dv, g, pd);    // dV_j = Pd_j * dO
    } else if (inrange) {
      const uint32_t z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      st_global_v8(dk, z);
      st_global_v8(dv, z);
    }
  }
  __syncthreads();
  // dq[d] = sum_j dS_j K[j][d]: warp w takes keys j = w, w+4, ...
  float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
  int j = wib;
  for (; j + 4 < len; j += 8) {
    const float d0 = s_ds[j], d1 = s_ds[j + 4];
    const float2 k0 = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(kbase + static_cast<size_t>(j) * 3 * D) + lane));
    const float2 k1 = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(kbase + static_cast<size_t>(j + 4) * 3 * D) + lane));
    a0 += d0 * k0.x; a1 += d0 * k0.y;
    b0 += d1 * k1.x; b1 += d1 * k1.y;
  }
  for (; j < len; j += 4) {
    const float d0 = s_ds[j];
    const float2 k0 = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(kbase + static_cast<size_t>(j) * 3 * D) + lane));
    a0 += d0 * k0.x; a1 += d0 * k0.y;
  }
  s_acc[wib][2 * lane] = a0 + b0;
  s_acc[wib][2 * lane + 1] = a1 + b1;
  __syncthreads();
  if (wib == 0) {
    const float o0 = (s_acc[0][2 * lane] + s_acc[1][2 * lane]) + (s_acc[2][2 * lane] + s_acc[3][2 * lane]);
    const float o1 = (s_acc[0][2 * lane + 1] + s_acc[1][2 * lane + 1]) + (s_acc[2][2 * lane + 1] + s_acc[3][2 * lane + 1]);
    reinterpret_cast<uint32_t*>(p.dq + static_cast<size_t>(b) * D + h * kDh)[lane] = pack_bf16(o0, o1);
  }
}

static uint32_t drop_threshold(float p) {
  if (p <= 0.f) return 0;
  double t = static_cast<double>(p) * 4294967296.0;
  uint32_t v = t >= 4294967295.0 ? 4294967295u : static_cast<uint32_t>(t);
  return v == 0 ? 1 : v;
}

}  // namespace tt

using namespace tt;

extern "C" int tt_gather_rows(const float* x_f32, const void* x_bf16, const int32_t* last_idx, int B, int L, int W,
                              float* out_f32, void* out_bf16, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(last_idx && B > 0 && L > 0 && W > 0 && W % 4 == 0, "tt_gather_rows: bad arguments");
  TT_REQUIRE((x_f32 && out_f32) || (x_bf16 && out_bf16), "tt_gather_rows: nothing to gather");
  TT_CHECK_CUDA(launch_k(gather_rows_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, stream, x_f32, static_cast<const __nv_bfloat16*>(x_bf16), last_idx, B, L, W, out_f32, static_cast<__nv_bfloat16*>(out_bf16)));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_scatter_rows_add(const float* rows, const int32_t* last_idx, int B, int L, int W, float* x,
                                   int accumulate, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(rows && last_idx && x && B > 0 && L > 0 && W > 0 && W % 4 == 0, "tt_scatter_rows_add: bad arguments");
  TT_CHECK_CUDA(launch_k(scatter_rows_add_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, stream, rows, last_idx, B, L, W, x, accumulate));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

static int fill_lastq(LastQParams& p, const void* q, const void* qkv, const int32_t* last_idx, int B, int L, int H,
                      float drop_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site, const char* who) {
  TT_REQUIRE(q && qkv && last_idx && B > 0 && L > 0 && H > 0, "%s: bad arguments", who);
  TT_REQUIRE(L <= kMaxL, "%s: L=%d > %d unsupported", who, L, kMaxL);
  TT_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "%s: drop_p out of range", who);
  p.q = static_cast<const __nv_bfloat16*>(q);
  p.qkv = static_cast<const __nv_bfloat16*>(qkv);
  p.last_idx = last_idx;
  p.B = B; p.L = L; p.H = H;
  p.scale = 0.125f;
  p.drop_thresh = drop_threshold(drop_p);
  p.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  p.seed = seed; p.seed_dev = seed_dev; p.site = site;
  p.ctx = nullptr; p.lse = nullptr; p.dctx = nullptr; p.dq = nullptr; p.dqkv = nullptr;
  return TT_OK;
}

extern "C" int tt_attn_lastq_fwd(const void* q, const void* qkv, const int32_t* last_idx, void* ctx, float* lse, int B,
                                 int L, int H, float drop_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site,
                                 void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  LastQParams p;
  int rc = fill_lastq(p, q, qkv, last_idx, B, L, H, drop_p, seed, seed_dev, site, "tt_attn_lastq_fwd");
  if (rc) return rc;
  TT_REQUIRE(ctx, "tt_attn_lastq_fwd: null ctx");
  p.ctx = static_cast<__nv_bfloat16*>(ctx);
  p.lse = lse;
  TT_CHECK_CUDA(launch_k(attn_lastq_fwd_kernel, dim3(B * H), dim3(128), 0, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_attn_lastq_bwd(const void* q, const void* qkv, const int32_t* last_idx, const void* ctx,
                                 const void* dctx, const float* lse, void* dq, void* dqkv, int B, int L, int H,
                                 float drop_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  LastQParams p;
  int rc = fill_lastq(p, q, qkv, last_idx, B, L, H, drop_p, seed, seed_dev, site, "tt_attn_lastq_bwd");
  if (rc) return rc;
  TT_REQUIRE(ctx && dctx && lse && dq && dqkv, "tt_attn_lastq_bwd: null pointer");
  p.ctx = const_cast<__nv_bfloat16*>(static_cast<const __nv_bfloat16*>(ctx));
  p.dctx = static_cast<const __nv_bfloat16*>(dctx);
  p.lse = const_cast<float*>(lse);
  p.dq = static_cast<__nv_bfloat16*>(dq);
  p.dqkv = static_cast<__nv_bfloat16*>(dqkv);
  TT_CHECK_CUDA(launch_k(attn_lastq_bwd_kernel, dim3(B * H), dim3(128), 0, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}
