// Bandwidth-bound row-wise kernels of the two-tower path: embedding gather + positional add +
// LayerNorm, LayerNorm / ReLU / dropout / L2-normalise chains and their backward passes,
// last-valid-step gather + demographic concat, BatchNorm1d (batch or running statistics),
// scatter-add of ID-embedding gradients.
//
// Layout rule: one warp per row, each lane owns NV float4 columns strided by 32 lanes
// (col = (k*32 + lane)*4 + c), so every load/store instruction of a warp covers 512
// contiguous bytes. Reductions are warp shuffles; no shared memory except for the
// cross-warp parameter-gradient combine.
#include "../../include/tt_b200.h"
#include "tt_common.cuh"
#include <vector>

namespace tt {

static constexpr int kRowThreads = 256;  // 8 warps per block

template <int NV>
__device__ __forceinline__ void load_row(const float* __restrict__ p, int lane, float (&v)[4 * NV]) {
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(p) + k * 32 + lane);
    v[4 * k] = x.x; v[4 * k + 1] = x.y; v[4 * k + 2] = x.z; v[4 * k + 3] = x.w;
  }
}
template <int NV>
__device__ __forceinline__ void store_row(float* __restrict__ p, int lane, const float (&v)[4 * NV]) {
#pragma unroll
  for (int k = 0; k < NV; ++k)
    reinterpret_cast<float4*>(p)[k * 32 + lane] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
}
template <int NV>
__device__ __forceinline__ void store_row_bf16(__nv_bfloat16* __restrict__ p, int lane, const float (&v)[4 * NV]) {
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    uint2 u;
    u.x = pack_bf16(v[4 * k], v[4 * k + 1]);
    u.y = pack_bf16(v[4 * k + 2], v[4 * k + 3]);
    reinterpret_cast<uint2*>(p)[k * 32 + lane] = u;
  }
}
template <int NV>
__device__ __forceinline__ void load_row_bf16(const __nv_bfloat16* __restrict__ p, int lane, float (&v)[4 * NV]) {
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p) + k * 32 + lane);
    const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y);
    v[4 * k] = a.x; v[4 * k + 1] = a.y; v[4 * k + 2] = b.x; v[4 * k + 3] = b.y;
  }
}
// column index of element e (0..4*NV) owned by `lane`
template <int NV>
__device__ __forceinline__ int col_of(int lane, int e) { return ((e >> 2) * 32 + lane) * 4 + (e & 3); }

template <int NV>
__device__ __forceinline__ void ln_stats(const float (&v)[4 * NV], float eps, float& mean, float& rstd) {
  constexpr int W = 128 * NV;
  float s = 0.f;
#pragma unroll
  for (int e = 0; e < 4 * NV; ++e) s += v[e];
  mean = warp_sum(s) * (1.f / W);
  float q = 0.f;
#pragma unroll
  for (int e = 0; e < 4 * NV; ++e) { const float d = v[e] - mean; q += d * d; }
  rstd = rsqrtf(warp_sum(q) * (1.f / W) + eps);
}

__device__ __forceinline__ uint64_t read_seed(uint64_t seed, const uint64_t* seed_dev) {
  return seed_dev ? seed + *seed_dev : seed;
}
// Dropout over a lane's row slice: elements come in float4 groups with 4-aligned column indices,
// so (e, e+1) pairs share one hash. keep[] (optional) receives the decisions.
template <int NV>
__device__ __forceinline__ void row_dropout(float (&v)[4 * NV], uint32_t key, uint64_t row, int width, int lane,
                                            uint32_t thresh, float scale, bool* keep) {
#pragma unroll
  for (int e = 0; e < 4 * NV; e += 2) {
    const uint64_t idx = row * static_cast<uint64_t>(width) + static_cast<uint64_t>(col_of<NV>(lane, e));
    bool k0, k1;
    if (idx < 0xFFFFFFFEull) drop_keep_pair(key, static_cast<uint32_t>(idx), thresh, k0, k1);
    else { k0 = drop_keep_k(key, idx, thresh); k1 = drop_keep_k(key, idx + 1, thresh); }
    v[e] = k0 ? v[e] * scale : 0.f;
    v[e + 1] = k1 ? v[e + 1] * scale : 0.f;
    if (keep) { keep[e] = k0; keep[e + 1] = k1; }
  }
}

static uint32_t drop_threshold(float p) {
  if (p <= 0.f) return 0;
  double t = static_cast<double>(p) * 4294967296.0;
  uint32_t v = t >= 4294967295.0 ? 4294967295u : static_cast<uint32_t>(t);
  return v == 0 ? 1 : v;
}

// --------------------------------------------------------------------------------------------
// fp32 -> bf16 cast (dense weight shadow copies), grid-stride, 16 B in / 8 B out per thread-step
// --------------------------------------------------------------------------------------------
__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, size_t n4) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(src) + i);
    uint2 u;
    u.x = pack_bf16(x.x, x.y);
    u.y = pack_bf16(x.z, x.w);
    reinterpret_cast<uint2*>(dst)[i] = u;
  }
}

// --------------------------------------------------------------------------------------------
// last valid index per history: len-1 clamped at 0 (user_tower.py:122-128)
// --------------------------------------------------------------------------------------------
__global__ void last_index_kernel(const int64_t* __restrict__ ids, const int64_t* __restrict__ mask, int B, int L,
                                  int32_t* __restrict__ last_idx) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B) return;
  int cnt = 0;
  for (int i = lane; i < L; i += 32) {
    const int64_t m = mask ? mask[static_cast<size_t>(warp) * L + i] : ids[static_cast<size_t>(warp) * L + i];
    cnt += (m != 0);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) last_idx[warp] = max(cnt - 1, 0);
}

// --------------------------------------------------------------------------------------------
// x0 = dropout(LN_emb(E[id] + P[pos]));  h = LN_next(x0) as bf16       (user_tower.py:86-93 and
// the first norm1 of the encoder). D = 256.
// --------------------------------------------------------------------------------------------
struct EmbedParams {
  const int64_t* ids;
  const float* E;
  const float* P;
  const float* ln_w; const float* ln_b;
  const float* nw; const float* nb;
  int T, L;
  uint32_t drop_thresh; float drop_scale; uint64_t seed; const uint64_t* seed_dev; uint32_t site;
  float* x0;
  __nv_bfloat16* h;
};

// One token row of embed_ln_fwd (one warp): table row E[id] and position row P[pos] -> x0, h at output row `row`.
// Shared by the [B, L] kernel (pos = row % L, dropout) and the explicit-position one (sessions: no dropout).
__device__ __forceinline__ void embed_ln_row(const EmbedParams& p, int64_t id, int pos, int row, int lane,
                                             const float (&w)[8], const float (&b)[8], const float (&nw)[8],
                                             const float (&nb)[8], uint64_t seed) {
  constexpr int NV = 2;
  float e[8], q[8];
  load_row<NV>(p.E + static_cast<size_t>(id) * 256, lane, e);
  load_row<NV>(p.P + static_cast<size_t>(pos) * 256, lane, q);
#pragma unroll
  for (int i = 0; i < 8; ++i) e[i] += q[i];
  float mean, rstd;
  ln_stats<NV>(e, 1e-5f, mean, rstd);
#pragma unroll
  for (int i = 0; i < 8; ++i) e[i] = (e[i] - mean) * rstd * w[i] + b[i];
  if (p.drop_thresh) row_dropout<NV>(e, drop_key(seed, p.site), row, 256, lane, p.drop_thresh, p.drop_scale, nullptr);
  store_row<NV>(p.x0 + static_cast<size_t>(row) * 256, lane, e);
  ln_stats<NV>(e, 1e-5f, mean, rstd);
#pragma unroll
  for (int i = 0; i < 8; ++i) e[i] = (e[i] - mean) * rstd * nw[i] + nb[i];
  store_row_bf16<NV>(p.h + static_cast<size_t>(row) * 256, lane, e);
}

__global__ void __launch_bounds__(kRowThreads) embed_ln_fwd_kernel(const EmbedParams p) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int NV = 2;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  float w[8], b[8], nw[8], nb[8];
  load_row<NV>(p.ln_w, lane, w);
  load_row<NV>(p.ln_b, lane, b);
  load_row<NV>(p.nw, lane, nw);
  load_row<NV>(p.nb, lane, nb);
  const uint64_t seed = p.drop_thresh ? read_seed(p.seed, p.seed_dev) : 0;
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < p.T; row += warps_total)
    embed_ln_row(p, p.ids[row], row % p.L, row, lane, w, b, nw, nb, seed);
}

// Rows at explicit positions: row r is item ids[r] at position pos[r] (p.T = n rows; no dropout).
__global__ void __launch_bounds__(kRowThreads) embed_ln_fwd_pos_kernel(const EmbedParams p,
                                                                        const int32_t* __restrict__ pos) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int NV = 2;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  float w[8], b[8], nw[8], nb[8];
  load_row<NV>(p.ln_w, lane, w);
  load_row<NV>(p.ln_b, lane, b);
  load_row<NV>(p.nw, lane, nw);
  load_row<NV>(p.nb, lane, nb);
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < p.T; row += warps_total)
    embed_ln_row(p, p.ids[row], pos[row], row, lane, w, b, nw, nb, 0);
}

// --------------------------------------------------------------------------------------------
// Generic row chain:  [LN] -> [ReLU] -> [dropout] -> [L2 normalise] on fp32 rows of width 128*NV.
// --------------------------------------------------------------------------------------------
struct ChainParams {
  const float* x;      // [R, W]
  int R;
  const float* ln_w; const float* ln_b;  // nullptr => no LayerNorm
  float ln_eps;
  int relu;
  uint32_t drop_thresh; float drop_scale; uint64_t seed; const uint64_t* seed_dev; uint32_t site;
  int l2norm; float l2_eps;
  float* out_f32;          // nullable
  __nv_bfloat16* out_bf16; // nullable
  // backward only
  const float* dout;       // [R, W] gradient w.r.t. the chain output
  const __nv_bfloat16* dout_bf16;   // the same as bf16 (exclusive with dout): what a dgrad GEMM hands back under autocast
  const float* resid;      // nullable [R, W]: added to dx
  const float* resid_rows; // nullable [R / resid_L, W]: added to row b*resid_L + resid_idx[b] of sequence b only
  const int32_t* resid_idx;
  int resid_L;
  float* dx_f32;           // nullable
  __nv_bfloat16* dx_bf16;  // nullable; receives dropout2(dx) when drop2_thresh != 0
  uint32_t drop2_thresh; float drop2_scale; uint32_t site2;
  float* dgamma; float* dbeta;  // accumulated (atomicAdd) when LN is on
  float* dx_colsum;             // nullable [W]: column sums of what is written to dx_bf16
};

template <int NV>
__global__ void __launch_bounds__(kRowThreads) chain_fwd_kernel(const ChainParams p) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int W = 128 * NV, E = 4 * NV;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  float w[E], b[E];
  if (p.ln_w) { load_row<NV>(p.ln_w, lane, w); load_row<NV>(p.ln_b, lane, b); }
  const uint64_t seed = p.drop_thresh ? read_seed(p.seed, p.seed_dev) : 0;
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < p.R; row += warps_total) {
    float v[E];
    load_row<NV>(p.x + static_cast<size_t>(row) * W, lane, v);
    if (p.ln_w) {
      float mean, rstd;
      ln_stats<NV>(v, p.ln_eps, mean, rstd);
#pragma unroll
      for (int i = 0; i < E; ++i) v[i] = (v[i] - mean) * rstd * w[i] + b[i];
    }
    if (p.relu) {
#pragma unroll
      for (int i = 0; i < E; ++i) v[i] = v[i] < 0.f ? 0.f : v[i];   // NaN-propagating like torch.relu
    }
    if (p.drop_thresh) row_dropout<NV>(v, drop_key(seed, p.site), row, W, lane, p.drop_thresh, p.drop_scale, nullptr);
    if (p.l2norm) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < E; ++i) s += v[i] * v[i];
      const float inv = 1.f / fmaxf(sqrtf(warp_sum(s)), p.l2_eps);
#pragma unroll
      for (int i = 0; i < E; ++i) v[i] *= inv;
    }
    if (p.out_f32) store_row<NV>(p.out_f32 + static_cast<size_t>(row) * W, lane, v);
    if (p.out_bf16) store_row_bf16<NV>(p.out_bf16 + static_cast<size_t>(row) * W, lane, v);
  }
}

// Backward of the chain: the forward is recomputed from x, then
// dout -> [L2 bwd] -> [dropout] -> [ReLU] -> [LN bwd] -> (+resid) -> dx.
template <int NV>
__global__ void __launch_bounds__(kRowThreads, 2) chain_bwd_kernel(const ChainParams p) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int W = 128 * NV, E = 4 * NV;
  __shared__ float s_red[3][kRowThreads / 32][W];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  float w[E], b[E], dg[E], db[E], cs[E];
#pragma unroll
  for (int i = 0; i < E; ++i) { dg[i] = 0.f; db[i] = 0.f; cs[i] = 0.f; w[i] = 1.f; b[i] = 0.f; }
  if (p.ln_w) { load_row<NV>(p.ln_w, lane, w); load_row<NV>(p.ln_b, lane, b); }
  const uint64_t seed = (p.drop_thresh || p.drop2_thresh) ? read_seed(p.seed, p.seed_dev) : 0;
  // Software pipeline: the three input rows of the NEXT iteration are requested before this row's
  // arithmetic (two warp reductions deep), so each warp keeps two rows of loads in flight.
  int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  float xn[E], gn[E], rn[E];
  if (row < p.R) {
    load_row<NV>(p.x + static_cast<size_t>(row) * W, lane, xn);
    if (p.dout_bf16) load_row_bf16<NV>(p.dout_bf16 + static_cast<size_t>(row) * W, lane, gn);
    else load_row<NV>(p.dout + static_cast<size_t>(row) * W, lane, gn);
    if (p.resid) load_row<NV>(p.resid + static_cast<size_t>(row) * W, lane, rn);
  }
  for (; row < p.R; row += warps_total) {
    float x[E], g[E], r[E], xhat[E], y[E];
#pragma unroll
    for (int i = 0; i < E; ++i) { x[i] = xn[i]; g[i] = gn[i]; r[i] = rn[i]; }
    const int nrow = row + warps_total;
    if (nrow < p.R) {
      load_row<NV>(p.x + static_cast<size_t>(nrow) * W, lane, xn);
      if (p.dout_bf16) load_row_bf16<NV>(p.dout_bf16 + static_cast<size_t>(nrow) * W, lane, gn);
      else load_row<NV>(p.dout + static_cast<size_t>(nrow) * W, lane, gn);
      if (p.resid) load_row<NV>(p.resid + static_cast<size_t>(nrow) * W, lane, rn);
    }
    float mean = 0.f, rstd = 1.f;
    if (p.ln_w) {
      ln_stats<NV>(x, p.ln_eps, mean, rstd);
#pragma unroll
      for (int i = 0; i < E; ++i) { xhat[i] = (x[i] - mean) * rstd; y[i] = xhat[i] * w[i] + b[i]; }
    } else {
#pragma unroll
      for (int i = 0; i < E; ++i) { xhat[i] = x[i]; y[i] = x[i]; }
    }
    // forward tail (ReLU, dropout) recomputed to obtain the L2 input z and the masks
    float z[E];
    bool keep[E];
#pragma unroll
    for (int i = 0; i < E; ++i) {
      z[i] = (p.relu && y[i] < 0.f) ? 0.f : y[i];
      keep[i] = true;
    }
    if (p.drop_thresh) row_dropout<NV>(z, drop_key(seed, p.site), row, W, lane, p.drop_thresh, p.drop_scale, keep);
    if (p.l2norm) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < E; ++i) s += z[i] * z[i];
      const float nrm = sqrtf(warp_sum(s));
      const float inv = 1.f / fmaxf(nrm, p.l2_eps);
      float dot = 0.f;
#pragma unroll
      for (int i = 0; i < E; ++i) dot += g[i] * z[i];
      dot = warp_sum(dot) * inv * inv;  // (g . zn) / n  with zn = z*inv
      const bool clamped = nrm < p.l2_eps;
#pragma unroll
      for (int i = 0; i < E; ++i) g[i] = clamped ? g[i] * inv : (g[i] - z[i] * dot) * inv;
    }
#pragma unroll
    for (int i = 0; i < E; ++i) {
      if (p.drop_thresh) g[i] = keep[i] ? g[i] * p.drop_scale : 0.f;
      if (p.relu && y[i] <= 0.f) g[i] = 0.f;
    }
    if (p.ln_w) {
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int i = 0; i < E; ++i) {
        dg[i] += g[i] * xhat[i];
        db[i] += g[i];
        g[i] *= w[i];
        s1 += g[i];
        s2 += g[i] * xhat[i];
      }
      s1 = warp_sum(s1) * (1.f / W);
      s2 = warp_sum(s2) * (1.f / W);
#pragma unroll
      for (int i = 0; i < E; ++i) g[i] = rstd * (g[i] - s1 - xhat[i] * s2);
    }
    if (p.resid) {
#pragma unroll
      for (int i = 0; i < E; ++i) g[i] += r[i];
    } else if (p.resid_rows) {
      const int b = row / p.resid_L;
      if (row - b * p.resid_L == __ldg(p.resid_idx + b)) {     // warp-uniform: one row per sequence
        float rr[E];
        load_row<NV>(p.resid_rows + static_cast<size_t>(b) * W, lane, rr);
#pragma unroll
        for (int i = 0; i < E; ++i) g[i] += rr[i];
      }
    }
    if (p.dx_f32) store_row<NV>(p.dx_f32 + static_cast<size_t>(row) * W, lane, g);
    if (p.dx_bf16) {
      if (p.drop2_thresh)
        row_dropout<NV>(g, drop_key(seed, p.site2), row, W, lane, p.drop2_thresh, p.drop2_scale, nullptr);
      store_row_bf16<NV>(p.dx_bf16 + static_cast<size_t>(row) * W, lane, g);
      if (p.dx_colsum) {
#pragma unroll
        for (int i = 0; i < E; ++i) cs[i] += __bfloat162float(__float2bfloat16_rn(g[i]));
      }
    }
  }
  // cross-warp combine of the per-column accumulators, one atomicAdd per column per block
  const bool need_ln = p.ln_w != nullptr, need_cs = p.dx_colsum != nullptr;
  if (!need_ln && !need_cs) return;
#pragma unroll
  for (int i = 0; i < E; ++i) {
    const int c = col_of<NV>(lane, i);
    s_red[0][wib][c] = dg[i];
    s_red[1][wib][c] = db[i];
    s_red[2][wib][c] = cs[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < W; c += blockDim.x) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
    for (int k = 0; k < kRowThreads / 32; ++k) { a0 += s_red[0][k][c]; a1 += s_red[1][k][c]; a2 += s_red[2][k][c]; }
    if (need_ln) { atomicAdd(p.dgamma + c, a0); atomicAdd(p.dbeta + c, a1); }
    if (need_cs) atomicAdd(p.dx_colsum + c, a2);
  }
}

// --------------------------------------------------------------------------------------------
// cat[b] = [x[b*L + last_idx[b]] | G[gender[b]] | C[country[b]]]  as bf16 [B, 304]
// (user_tower.py:132-139). One warp per sequence.
// --------------------------------------------------------------------------------------------
__global__ void gather_cat_kernel(const float* __restrict__ x, const int32_t* __restrict__ last_idx,
                                  const int64_t* __restrict__ gender, const int64_t* __restrict__ country,
                                  const float* __restrict__ G, const float* __restrict__ C, int B, int L,
                                  __nv_bfloat16* __restrict__ cat) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* row = x + (static_cast<size_t>(b) * L + last_idx[b]) * 256;
  __nv_bfloat16* o = cat + static_cast<size_t>(b) * 304;
  float v[8];
  load_row<2>(row, lane, v);
  store_row_bf16<2>(o, lane, v);
  const int64_t gi = gender ? gender[b] : 0, ci = country ? country[b] : 0;
  if (lane < 16) o[256 + lane] = __float2bfloat16_rn(G[gi * 16 + lane]);
  o[272 + lane] = __float2bfloat16_rn(C[ci * 32 + lane]);
}

// Backward of the above: dcat fp32 [B, 304] -> dx_top (zero-initialised by the caller) rows,
// atomics into dG / dC.
__global__ void gather_cat_bwd_kernel(const float* __restrict__ dcat, const int32_t* __restrict__ last_idx,
                                      const int64_t* __restrict__ gender, const int64_t* __restrict__ country,
                                      int B, int L, float* __restrict__ dx, __nv_bfloat16* __restrict__ dx_bf16,
                                      float* __restrict__ dG, float* __restrict__ dC) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* g = dcat + static_cast<size_t>(b) * 304;
  const size_t row = static_cast<size_t>(b) * L + last_idx[b];
  float v[8];
  load_row<2>(g, lane, v);
  if (dx) store_row<2>(dx + row * 256, lane, v);
  if (dx_bf16) store_row_bf16<2>(dx_bf16 + row * 256, lane, v);
  const int64_t gi = gender ? gender[b] : 0, ci = country ? country[b] : 0;
  if (lane < 16) atomicAdd(dG + gi * 16 + lane, g[256 + lane]);
  atomicAdd(dC + ci * 32 + lane, g[272 + lane]);
}

// --------------------------------------------------------------------------------------------
// concat of the four modality embeddings -> bf16 [B, 4*m]   (item_tower.py:147)
// --------------------------------------------------------------------------------------------
__global__ void concat4_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c,
                               const float* __restrict__ d, int B, int m, __nv_bfloat16* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t n = static_cast<size_t>(B) * 4 * m;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int row = static_cast<int>(i / (4 * m)), col = static_cast<int>(i % (4 * m));
    const int which = col / m, k = col % m;
    const float* src = which == 0 ? a : (which == 1 ? b : (which == 2 ? c : d));
    out[i] = __float2bfloat16_rn(__ldg(src + static_cast<size_t>(row) * m + k));
  }
}

// --------------------------------------------------------------------------------------------
// BatchNorm1d + ReLU + dropout over [B, C] fp32 -> bf16 (item_tower.py:124-126).
// training: batch mean / biased variance (two passes), running stats updated with the unbiased
// variance and momentum; eval: running stats. Block = 32 columns x 8 row-lanes.
// --------------------------------------------------------------------------------------------
struct BnParams {
  const float* y; int B, C;
  const float* w; const float* b;
  float* running_mean; float* running_var; int64_t* num_batches;
  int training; float momentum, eps;
  uint32_t drop_thresh; float drop_scale; uint64_t seed; const uint64_t* seed_dev; uint32_t site;
  float* save_mean; float* save_rstd;
  __nv_bfloat16* out;
  // backward
  const float* dout;      // fp32 [B, C] grad w.r.t. the bf16 output
  __nv_bfloat16* dy;      // bf16 [B, C] grad w.r.t. y
  float* dgamma; float* dbeta; float* dy_colsum;
};

__device__ __forceinline__ float block_col_reduce(float v, float (*s)[33]) {
  // blockDim = (32, 8): sum over threadIdx.y for each threadIdx.x
  s[threadIdx.y][threadIdx.x] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) t += s[k][threadIdx.x];
  __syncthreads();
  return t;
}

__global__ void __launch_bounds__(256) bn_fwd_kernel(const BnParams p) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool active = c < p.C;
  float mean, rstd;
  if (p.training) {
    float a = 0.f;
    if (active) for (int r = threadIdx.y; r < p.B; r += 8) a += p.y[static_cast<size_t>(r) * p.C + c];
    mean = block_col_reduce(a, s) / p.B;
    float q = 0.f;
    if (active) for (int r = threadIdx.y; r < p.B; r += 8) { const float d = p.y[static_cast<size_t>(r) * p.C + c] - mean; q += d * d; }
    const float var = block_col_reduce(q, s) / p.B;
    rstd = rsqrtf(var + p.eps);
    if (active && threadIdx.y == 0) {
      p.save_mean[c] = mean;
      p.save_rstd[c] = rstd;
      const float unbiased = p.B > 1 ? var * p.B / (p.B - 1) : var;
      p.running_mean[c] = (1.f - p.momentum) * p.running_mean[c] + p.momentum * mean;
      p.running_var[c] = (1.f - p.momentum) * p.running_var[c] + p.momentum * unbiased;
      if (c == 0 && p.num_batches) *p.num_batches += 1;
    }
  } else {
    mean = active ? p.running_mean[c] : 0.f;
    rstd = active ? rsqrtf(p.running_var[c] + p.eps) : 0.f;
  }
  if (!active) return;
  const float g = p.w[c], be = p.b[c];
  const uint64_t seed = p.drop_thresh ? read_seed(p.seed, p.seed_dev) : 0;
  for (int r = threadIdx.y; r < p.B; r += 8) {
    const size_t i = static_cast<size_t>(r) * p.C + c;
    float v = (p.y[i] - mean) * rstd * g + be;
    v = v < 0.f ? 0.f : v;   // NaN-propagating like torch.relu
    if (p.drop_thresh) v = drop_keep(seed, p.site, i, p.drop_thresh) ? v * p.drop_scale : 0.f;
    p.out[i] = __float2bfloat16_rn(v);
  }
}

__global__ void __launch_bounds__(256) bn_bwd_kernel(const BnParams p) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool active = c < p.C;
  const float mean = active ? p.save_mean[c] : 0.f, rstd = active ? p.save_rstd[c] : 0.f;
  const float g = active ? p.w[c] : 0.f, be = active ? p.b[c] : 0.f;
  const uint64_t seed = p.drop_thresh ? read_seed(p.seed, p.seed_dev) : 0;
  float s1 = 0.f, s2 = 0.f;
  if (active) {
    for (int r = threadIdx.y; r < p.B; r += 8) {
      const size_t i = static_cast<size_t>(r) * p.C + c;
      const float xh = (p.y[i] - mean) * rstd;
      float d = p.dout[i];
      if (p.drop_thresh) d = drop_keep(seed, p.site, i, p.drop_thresh) ? d * p.drop_scale : 0.f;
      if (xh * g + be <= 0.f) d = 0.f;
      s1 += d;
      s2 += d * xh;
    }
  }
  s1 = block_col_reduce(s1, s);
  s2 = block_col_reduce(s2, s);
  if (!active) return;
  if (threadIdx.y == 0) { atomicAdd(p.dbeta + c, s1); atomicAdd(p.dgamma + c, s2); }
  const float m1 = s1 / p.B, m2 = s2 / p.B;
  float cs = 0.f;
  for (int r = threadIdx.y; r < p.B; r += 8) {
    const size_t i = static_cast<size_t>(r) * p.C + c;
    const float xh = (p.y[i] - mean) * rstd;
    float d = p.dout[i];
    if (p.drop_thresh) d = drop_keep(seed, p.site, i, p.drop_thresh) ? d * p.drop_scale : 0.f;
    if (xh * g + be <= 0.f) d = 0.f;
    const __nv_bfloat16 o = __float2bfloat16_rn(g * rstd * (d - m1 - xh * m2));
    p.dy[i] = o;
    cs += __bfloat162float(o);
  }
  if (p.dy_colsum) {
    // reuse the reduction buffer: all threads of the column group reach this point together
    __shared__ float s3[8][33];
    s3[threadIdx.y][threadIdx.x] = cs;
    __syncthreads();
    if (threadIdx.y == 0) {
      float t = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) t += s3[k][threadIdx.x];
      atomicAdd(p.dy_colsum + c, t);
    }
  }
}

// --------------------------------------------------------------------------------------------
// Backward of embed_ln_fwd w.r.t. its first LayerNorm: dx0 [T,256] -> dE (scatter-add, id 0
// skipped: padding_idx), dP (per position), d(ln_w), d(ln_b). The pre-LN sum E[id]+P[pos] is
// re-gathered instead of being stored.
// Grid (L, S): block (pos, s) handles position `pos` for every S-th group of 8 sequences, so dP takes
// S atomics per element; S is chosen for ~6 blocks per SM (see embed_bwd_impl).
// --------------------------------------------------------------------------------------------
// Fixed-point scale of the deterministic table-gradient accumulation: 2^40 (resolution 9.1e-13, |sum| < 8.3e6).
static constexpr float kGradFixScale = 1099511627776.f;

struct EmbedBwdParams {
  const int64_t* ids; const float* E; const float* P; const float* ln_w; const float* ln_b;
  const float* dx0; int B, L;
  uint32_t drop_thresh; float drop_scale; uint64_t seed; const uint64_t* seed_dev; uint32_t site;
  float* dE; float* dP; float* dgamma; float* dbeta;
  // deterministic mode (both set): token `row` adds its gradient row into acc64[acc_slot[row]] in 64-bit fixed
  // point instead of dE (slot 0 = padding: skipped); tt_rows_scatter_add_i64 then rounds each sum once
  unsigned long long* acc64; const int64_t* acc_slot;
};

__global__ void __launch_bounds__(kRowThreads, 2) embed_ln_bwd_kernel(const EmbedBwdParams p) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int NV = 2, E_ = 8, W = 256;
  __shared__ float s_red[3][kRowThreads / 32][W];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int pos = blockIdx.x;
  float w[E_], dg[E_], db[E_], dp[E_], q[E_];
  load_row<NV>(p.ln_w, lane, w);
  load_row<NV>(p.P + static_cast<size_t>(pos) * W, lane, q);
#pragma unroll
  for (int i = 0; i < E_; ++i) { dg[i] = 0.f; db[i] = 0.f; dp[i] = 0.f; }
  const uint64_t seed = p.drop_thresh ? read_seed(p.seed, p.seed_dev) : 0;
  // The id -> table row -> arithmetic chain is two dependent memory latencies per row; the ids run two
  // rows ahead and the (table row, gradient row) pair one row ahead of the arithmetic.
  const int stride = (kRowThreads / 32) * gridDim.y;
  int b = wib * gridDim.y + blockIdx.y;
  int64_t id_n = 0, id_nn = 0;
  float e_n[E_], g_n[E_];
  if (b < p.B) {
    id_n = p.ids[static_cast<size_t>(b) * p.L + pos];
    load_row<NV>(p.E + static_cast<size_t>(id_n) * W, lane, e_n);
    load_row<NV>(p.dx0 + (static_cast<size_t>(b) * p.L + pos) * W, lane, g_n);
  }
  if (b + stride < p.B) id_nn = p.ids[static_cast<size_t>(b + stride) * p.L + pos];
  for (; b < p.B; b += stride) {
    const size_t row = static_cast<size_t>(b) * p.L + pos;
    const int64_t id = id_n;
    float e[E_], g[E_], xhat[E_];
#pragma unroll
    for (int i = 0; i < E_; ++i) { e[i] = e_n[i]; g[i] = g_n[i]; }
    id_n = id_nn;
    if (b + stride < p.B) {
      load_row<NV>(p.E + static_cast<size_t>(id_n) * W, lane, e_n);
      load_row<NV>(p.dx0 + (static_cast<size_t>(b + stride) * p.L + pos) * W, lane, g_n);
    }
    if (b + 2 * stride < p.B) id_nn = p.ids[static_cast<size_t>(b + 2 * stride) * p.L + pos];
#pragma unroll
    for (int i = 0; i < E_; ++i) e[i] += q[i];
    float mean, rstd;
    ln_stats<NV>(e, 1e-5f, mean, rstd);
#pragma unroll
    for (int i = 0; i < E_; ++i) xhat[i] = (e[i] - mean) * rstd;
    if (p.drop_thresh) row_dropout<NV>(g, drop_key(seed, p.site), row, W, lane, p.drop_thresh, p.drop_scale, nullptr);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < E_; ++i) {
      dg[i] += g[i] * xhat[i];
      db[i] += g[i];
      g[i] *= w[i];
      s1 += g[i];
      s2 += g[i] * xhat[i];
    }
    s1 = warp_sum(s1) * (1.f / W);
    s2 = warp_sum(s2) * (1.f / W);
#pragma unroll
    for (int i = 0; i < E_; ++i) {
      g[i] = rstd * (g[i] - s1 - xhat[i] * s2);
      dp[i] += g[i];
    }
    if (p.acc64) {
      // Integer addition is associative: whatever order the tokens of an id arrive in, the 64-bit sum is the
      // same, so the table gradient is bit-identical from run to run (floating-point atomics are not).
      const int64_t slot = p.acc_slot[row];
      if (slot != 0) {
        unsigned long long* dst = p.acc64 + static_cast<size_t>(slot) * W;
#pragma unroll
        for (int k = 0; k < NV; ++k)
#pragma unroll
          for (int e = 0; e < 4; ++e)
            atomicAdd(dst + (k * 32 + lane) * 4 + e,
                      static_cast<unsigned long long>(__float2ll_rn(g[4 * k + e] * kGradFixScale)));
      }
    } else if (id != 0) {
      float* dst = p.dE + static_cast<size_t>(id) * W;
#pragma unroll
      for (int k = 0; k < NV; ++k)
        red_add_f32x4(dst + (k * 32 + lane) * 4, g[4 * k + 0], g[4 * k + 1], g[4 * k + 2], g[4 * k + 3]);
    }
  }
#pragma unroll
  for (int i = 0; i < E_; ++i) {
    const int c = col_of<NV>(lane, i);
    s_red[0][wib][c] = dg[i];
    s_red[1][wib][c] = db[i];
    s_red[2][wib][c] = dp[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < W; c += blockDim.x) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
    for (int k = 0; k < kRowThreads / 32; ++k) {
      a0 += s_red[0][k][c]; a1 += s_red[1][k][c]; a2 += s_red[2][k][c];
    }
    atomicAdd(p.dgamma + c, a0);
    atomicAdd(p.dbeta + c, a1);
    atomicAdd(p.dP + static_cast<size_t>(pos) * W + c, a2);  // gridDim.y blocks per position
  }
}

// --------------------------------------------------------------------------------------------
// Fused AdamW over a flat fp32 parameter buffer (torch.optim.AdamW semantics, train.py:302),
// dense and decoupled: every element decays every step. Optionally refreshes a bf16 shadow of
// a sub-range and zeroes the gradient in the same pass. `step_dev` holds the 1-based step
// count as a device scalar so the launch is CUDA-graph replayable.
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                                    float* __restrict__ v, size_t n4, float lr, float beta1,
                                                    float beta2, float eps, float wd, float grad_scale,
                                                    const int64_t* step_dev,
                                                    __nv_bfloat16* __restrict__ shadow, size_t shadow_begin4,
                                                    size_t shadow_end4, int zero_grad) {
  pdl_launch_dependents();
  pdl_wait();
  const float step = static_cast<float>(*step_dev);
  const float bc1 = 1.f - powf(beta1, step);
  const float bc2_sqrt = sqrtf(1.f - powf(beta2, step));
  const float step_size = lr / bc1;
  const float decay = 1.f - lr * wd;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = reinterpret_cast<const float4*>(g)[i];
    const float4 gs = make_float4(gg.x * grad_scale, gg.y * grad_scale, gg.z * grad_scale, gg.w * grad_scale);
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    float* pa = reinterpret_cast<float*>(&pp);
    const float* ga = reinterpret_cast<const float*>(&gs);
    float* ma = reinterpret_cast<float*>(&mm);
    float* va = reinterpret_cast<float*>(&vv);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float x = pa[k] * decay;
      ma[k] = beta1 * ma[k] + (1.f - beta1) * ga[k];
      va[k] = beta2 * va[k] + (1.f - beta2) * ga[k] * ga[k];
      const float denom = sqrtf(va[k]) / bc2_sqrt + eps;
      pa[k] = x - step_size * ma[k] / denom;
    }
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
    // ID-table rows no token of the batch touched (60 % of them at c2) already hold a zero gradient: skip
    // the 16-byte store (bit patterns compared, so a -0.0 is rewritten as +0.0 like before)
    if (zero_grad && ((__float_as_uint(gg.x) | __float_as_uint(gg.y) | __float_as_uint(gg.z) | __float_as_uint(gg.w)) != 0u))
      reinterpret_cast<float4*>(g)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (shadow && i >= shadow_begin4 && i < shadow_end4) {
      uint2 u;
      u.x = pack_bf16(pp.x, pp.y);
      u.y = pack_bf16(pp.z, pp.w);
      reinterpret_cast<uint2*>(shadow)[i - shadow_begin4] = u;
    }
  }
}

// --------------------------------------------------------------------------------------------
// Catalog indexing tail (src/evaluate_metrics.py:70-102 after the item tower's last Linear): LayerNorm
// (item_tower.py:128) -> F.normalize eps 1e-12 (two_tower.py:168) -> NaN -> 0 (:79-81) -> F.normalize eps 1e-8
// (:85) -> row `ids[r]` of the dense (V, 256) cache table, fp32 and the bf16 copy retrieval scores with.
// The reference applies nan_to_num to a whole batch when any element is NaN; on finite elements that is the
// identity, and +-inf cannot survive the first normalisation (inf / inf = NaN), so the per-element rule here
// is the same function. One warp per item: 1 KB in, 1 KB + 512 B out.
// --------------------------------------------------------------------------------------------
// The row arithmetic of both indexing kernels: y row (one lane's 8 values) -> the cache row's values.
__device__ __forceinline__ void index_row_values(const float* __restrict__ yrow, int lane, const float (&w)[8],
                                                 const float (&b)[8], float (&v)[8]) {
  constexpr int NV = 2, E = 8;
  load_row<NV>(yrow, lane, v);
  float mean, rstd;
  ln_stats<NV>(v, 1e-5f, mean, rstd);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < E; ++i) { v[i] = (v[i] - mean) * rstd * w[i] + b[i]; s += v[i] * v[i]; }
  float inv = 1.f / fmaxf(sqrtf(warp_sum(s)), 1e-12f);
  s = 0.f;
#pragma unroll
  for (int i = 0; i < E; ++i) {
    v[i] *= inv;
    if (v[i] != v[i]) v[i] = 0.f;
    s += v[i] * v[i];
  }
  inv = 1.f / fmaxf(sqrtf(warp_sum(s)), 1e-8f);
#pragma unroll
  for (int i = 0; i < E; ++i) v[i] *= inv;
}

__global__ void __launch_bounds__(kRowThreads) index_rows_kernel(const float* __restrict__ y, int R,
                                                                 const float* __restrict__ ln_w,
                                                                 const float* __restrict__ ln_b,
                                                                 const int64_t* __restrict__ ids, int64_t V,
                                                                 float* __restrict__ table,
                                                                 __nv_bfloat16* __restrict__ table_bf16) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int NV = 2, E = 8, W = 256;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  float w[E], b[E];
  load_row<NV>(ln_w, lane, w);
  load_row<NV>(ln_b, lane, b);
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < R; row += warps_total) {
    const int64_t id = ids[row];
    if (id < 0 || id >= V) continue;             // out-of-table ids are dropped (the reference would raise)
    float v[E];
    index_row_values(y + static_cast<size_t>(row) * W, lane, w, b, v);
    store_row<NV>(table + static_cast<size_t>(id) * W, lane, v);
    if (table_bf16) store_row_bf16<NV>(table_bf16 + static_cast<size_t>(id) * W, lane, v);
  }
}

// Live update of a built index (rows [item_base, item_base + N) of the catalog): the rows of index_rows_kernel for
// the ids this index owns, their retired bits cleared, and the item-side terms of the retrieval certificate
// (max ||bf16(e) - e||, max ||bf16(e)||) raised to cover them.
__global__ void __launch_bounds__(kRowThreads) index_rows_live_kernel(const float* __restrict__ y, int R,
                                                                      const float* __restrict__ ln_w,
                                                                      const float* __restrict__ ln_b,
                                                                      const int64_t* __restrict__ ids,
                                                                      int64_t item_base, int N,
                                                                      float* __restrict__ table,
                                                                      __nv_bfloat16* __restrict__ table_bf16,
                                                                      uint32_t* __restrict__ retired,
                                                                      float* __restrict__ stats) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int NV = 2, E = 8, W = 256;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  float w[E], b[E];
  load_row<NV>(ln_w, lane, w);
  load_row<NV>(ln_b, lane, b);
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < R; row += warps_total) {
    const int64_t local = ids[row] - item_base;
    if (local < 0 || local >= N) continue;       // another shard's row
    float v[E];
    index_row_values(y + static_cast<size_t>(row) * W, lane, w, b, v);
    store_row<NV>(table + static_cast<size_t>(local) * W, lane, v);
    store_row_bf16<NV>(table_bf16 + static_cast<size_t>(local) * W, lane, v);
    float d2 = 0.f, n2 = 0.f;
#pragma unroll
    for (int i = 0; i < E; i += 2) {
      const float2 r = unpack_bf16(pack_bf16(v[i], v[i + 1]));
      const float e0 = r.x - v[i], e1 = r.y - v[i + 1];
      d2 += e0 * e0 + e1 * e1;
      n2 += r.x * r.x + r.y * r.y;
    }
    d2 = warp_sum(d2);
    n2 = warp_sum(n2);
    if (lane == 0) {
      if (retired) atomicAnd(retired + (local >> 5), ~(1u << (local & 31)));   // rows share words
      // rounded up by a few ulps: these feed an upper bound
      atomicMax(reinterpret_cast<int*>(stats), __float_as_int(sqrtf(d2) * 1.00001f));
      atomicMax(reinterpret_cast<int*>(stats) + 1, __float_as_int(sqrtf(n2) * 1.00001f));
    }
  }
}

// Retire ids of this index: zero their fp32 and bf16 rows, set their retired bits. One warp per id.
__global__ void __launch_bounds__(kRowThreads) catalog_retire_kernel(const int64_t* __restrict__ ids, int n,
                                                                     int64_t item_base, int N,
                                                                     float* __restrict__ table,
                                                                     __nv_bfloat16* __restrict__ table_bf16,
                                                                     uint32_t* __restrict__ retired) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int NV = 2, E = 8, W = 256;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  float z[E];
#pragma unroll
  for (int i = 0; i < E; ++i) z[i] = 0.f;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps_total) {
    const int64_t local = ids[r] - item_base;
    if (local < 0 || local >= N) continue;
    store_row<NV>(table + static_cast<size_t>(local) * W, lane, z);
    store_row_bf16<NV>(table_bf16 + static_cast<size_t>(local) * W, lane, z);
    if (lane == 0) atomicOr(retired + (local >> 5), 1u << (local & 31));
  }
}

__global__ void increment_kernel(int64_t* a, uint64_t* b) {
  pdl_launch_dependents();
  pdl_wait();
  if (a) *a += 1;
  if (b) *b += 0x9E3779B97F4A7C15ULL;
}

static int row_grid(int rows) {
  const int blocks = (rows + (kRowThreads / 32) - 1) / (kRowThreads / 32);
  const int cap = num_sms() * 8;
  return blocks < cap ? (blocks > 0 ? blocks : 1) : cap;
}

}  // namespace tt

using namespace tt;

extern "C" int tt_cast_bf16(const float* src, void* dst, int64_t n, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(src && dst && n > 0 && n % 4 == 0, "tt_cast_bf16: n must be a positive multiple of 4");
  const size_t n4 = static_cast<size_t>(n / 4);
  int grid = static_cast<int>((n4 + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  TT_CHECK_CUDA(launch_k(cast_bf16_kernel, dim3(grid), dim3(256), 0, stream, src, static_cast<__nv_bfloat16*>(dst), n4));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_last_index(const int64_t* ids, const int64_t* mask, int B, int L, int32_t* last_idx, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE((ids || mask) && last_idx && B > 0 && L > 0, "tt_last_index: bad arguments");
  TT_CHECK_CUDA(launch_k(last_index_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, stream, ids, mask, B, L, last_idx));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

static int embed_fwd_impl(const int64_t* ids, const float* E, const float* P, const float* ln_w, const float* ln_b,
                          const float* next_w, const float* next_b, int B, int L, float drop_p, uint64_t seed,
                          const uint64_t* seed_dev, uint32_t site, float* x0, void* h_bf16, cudaStream_t stream) {
  TT_REQUIRE(ids && P && ln_w && ln_b && next_w && next_b && x0 && h_bf16, "tt_embed_ln_fwd: null pointer");
  TT_REQUIRE(B > 0 && L > 0, "tt_embed_ln_fwd: empty batch");
  EmbedParams p;
  p.ids = ids; p.E = E; p.P = P; p.ln_w = ln_w; p.ln_b = ln_b; p.nw = next_w; p.nb = next_b;
  p.T = B * L; p.L = L;
  p.drop_thresh = drop_threshold(drop_p);
  p.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  p.seed = seed; p.seed_dev = seed_dev; p.site = site;
  p.x0 = x0; p.h = static_cast<__nv_bfloat16*>(h_bf16);
  TT_CHECK_CUDA(launch_k(embed_ln_fwd_kernel, dim3(row_grid(p.T)), dim3(kRowThreads), 0, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

static int embed_bwd_impl(const int64_t* ids, const float* E, const float* P, const float* ln_w, const float* ln_b,
                          const float* dx0, int B, int L, float drop_p, uint64_t seed, const uint64_t* seed_dev,
                          uint32_t site, float* dE, float* dP, float* dgamma, float* dbeta, cudaStream_t stream,
                          unsigned long long* acc64 = nullptr, const int64_t* acc_slot = nullptr) {
  TT_REQUIRE(ids && P && ln_w && ln_b && dx0 && dP && dgamma && dbeta, "tt_embed_ln_bwd: null pointer");
  EmbedBwdParams p;
  p.ids = ids; p.E = E; p.P = P; p.ln_w = ln_w; p.ln_b = ln_b; p.dx0 = dx0; p.B = B; p.L = L;
  p.drop_thresh = drop_threshold(drop_p);
  p.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  p.seed = seed; p.seed_dev = seed_dev; p.site = site;
  p.dE = dE; p.dP = dP; p.dgamma = dgamma; p.dbeta = dbeta;
  p.acc64 = acc64; p.acc_slot = acc_slot;
  // ~6 blocks per SM in total (three waves at two resident blocks per SM): measured on the c2 step (L = 200), 1 / 2 /
  // 3 / 4 / 6 / 8 blocks per position -> 1.172 / 1.169 / 1.160 / 1.158 / 1.161 / 1.161 ms per step; one block per
  // position left every warp with a 32-row serial id -> row -> atomics chain and the SMs two thirds empty
  int splits = (6 * num_sms() + L / 2) / L;
  if (splits < 1) splits = 1;
  if (splits > (B + 7) / 8) splits = (B + 7) / 8;
  TT_CHECK_CUDA(launch_k(embed_ln_bwd_kernel, dim3(L, splits), dim3(kRowThreads), 0, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_embed_ln_fwd(const int64_t* ids, const float* E, const float* P, const float* ln_w,
                               const float* ln_b, const float* next_w, const float* next_b, int B, int L,
                               float drop_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site, float* x0,
                               void* h_bf16, void* stream_) {
  TT_REQUIRE(E, "tt_embed_ln_fwd: null table");
  return embed_fwd_impl(ids, E, P, ln_w, ln_b, next_w, next_b, B, L, drop_p, seed, seed_dev, site, x0, h_bf16,
                        static_cast<cudaStream_t>(stream_));
}

extern "C" int tt_embed_ln_fwd_pos(const int64_t* ids, const int32_t* pos, const float* E, const float* P,
                                   const float* ln_w, const float* ln_b, const float* next_w, const float* next_b,
                                   int n, float* x0, void* h_bf16, void* stream_) {
  TT_REQUIRE(ids && pos && E && P && ln_w && ln_b && next_w && next_b && x0 && h_bf16,
             "tt_embed_ln_fwd_pos: null pointer");
  TT_REQUIRE(n > 0, "tt_embed_ln_fwd_pos: empty batch");
  EmbedParams p;
  p.ids = ids; p.E = E; p.P = P; p.ln_w = ln_w; p.ln_b = ln_b;
  p.nw = next_w; p.nb = next_b;
  p.T = n; p.L = 0;
  p.drop_thresh = 0; p.drop_scale = 1.f; p.seed = 0; p.seed_dev = nullptr; p.site = 0;
  p.x0 = x0; p.h = static_cast<__nv_bfloat16*>(h_bf16);
  TT_CHECK_CUDA(launch_k(embed_ln_fwd_pos_kernel, dim3(row_grid(n)), dim3(kRowThreads), 0,
                         static_cast<cudaStream_t>(stream_), p, pos));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_embed_ln_bwd(const int64_t* ids, const float* E, const float* P, const float* ln_w,
                               const float* ln_b, const float* dx0, int B, int L, float drop_p, uint64_t seed,
                               const uint64_t* seed_dev, uint32_t site, float* dE, float* dP, float* dgamma,
                               float* dbeta, void* stream_) {
  TT_REQUIRE(E && dE, "tt_embed_ln_bwd: null table");
  return embed_bwd_impl(ids, E, P, ln_w, ln_b, dx0, B, L, drop_p, seed, seed_dev, site, dE, dP, dgamma, dbeta,
                        static_cast<cudaStream_t>(stream_));
}

extern "C" int tt_embed_ln_bwd_det(const int64_t* ids, const float* E, const float* P, const float* ln_w,
                                   const float* ln_b, const float* dx0, int B, int L, float drop_p, uint64_t seed,
                                   const uint64_t* seed_dev, uint32_t site, const int64_t* slot_of_token, int64_t* acc64,
                                   float* dP, float* dgamma, float* dbeta, void* stream_) {
  TT_REQUIRE(E && slot_of_token && acc64, "tt_embed_ln_bwd_det: null pointer");
  return embed_bwd_impl(ids, E, P, ln_w, ln_b, dx0, B, L, drop_p, seed, seed_dev, site, nullptr, dP, dgamma, dbeta,
                        static_cast<cudaStream_t>(stream_), reinterpret_cast<unsigned long long*>(acc64),
                        slot_of_token);
}

static int fill_chain(ChainParams& p, const tt_chain_args* a, const char* who) {
  TT_REQUIRE(a && a->x && a->rows > 0, "%s: bad arguments", who);
  TT_REQUIRE(a->width == 256 || a->width == 512, "%s: width %d unsupported (256 or 512)", who, a->width);
  TT_REQUIRE((a->ln_w == nullptr) == (a->ln_b == nullptr), "%s: ln_w/ln_b must come together", who);
  p.x = a->x; p.R = a->rows;
  p.ln_w = a->ln_w; p.ln_b = a->ln_b; p.ln_eps = a->ln_eps > 0.f ? a->ln_eps : 1e-5f;
  p.relu = a->relu;
  p.drop_thresh = drop_threshold(a->drop_p);
  p.drop_scale = a->drop_p > 0.f ? 1.f / (1.f - a->drop_p) : 1.f;
  p.seed = a->drop_seed; p.seed_dev = a->drop_seed_dev; p.site = a->drop_site;
  p.l2norm = a->l2norm; p.l2_eps = a->l2_eps > 0.f ? a->l2_eps : 1e-12f;
  p.out_f32 = a->out_f32; p.out_bf16 = static_cast<__nv_bfloat16*>(a->out_bf16);
  p.dout = a->dout; p.dout_bf16 = static_cast<const __nv_bfloat16*>(a->dout_bf16); p.resid = a->resid; p.dx_f32 = a->dx_f32;
  p.resid_rows = a->resid_rows; p.resid_idx = a->resid_last_idx; p.resid_L = a->resid_seq_len;
  TT_REQUIRE(!(a->resid && a->resid_rows), "%s: resid and resid_rows are exclusive", who);
  TT_REQUIRE(!a->resid_rows || (a->resid_last_idx && a->resid_seq_len > 0 && a->rows % a->resid_seq_len == 0),
             "%s: resid_rows needs resid_last_idx and a seq_len dividing rows", who);
  p.dx_bf16 = static_cast<__nv_bfloat16*>(a->dx_bf16);
  p.drop2_thresh = drop_threshold(a->drop2_p);
  p.drop2_scale = a->drop2_p > 0.f ? 1.f / (1.f - a->drop2_p) : 1.f;
  p.site2 = a->drop2_site;
  p.dgamma = a->dgamma; p.dbeta = a->dbeta; p.dx_colsum = a->dx_colsum;
  return TT_OK;
}

extern "C" int tt_chain_fwd(const tt_chain_args* a, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ChainParams p;
  int rc = fill_chain(p, a, "tt_chain_fwd");
  if (rc) return rc;
  TT_REQUIRE(p.out_f32 || p.out_bf16, "tt_chain_fwd: no output");
  if (a->width == 256) TT_CHECK_CUDA(launch_k(chain_fwd_kernel<2>, dim3(row_grid(p.R)), dim3(kRowThreads), 0, stream, p));
  else TT_CHECK_CUDA(launch_k(chain_fwd_kernel<4>, dim3(row_grid(p.R)), dim3(kRowThreads), 0, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_chain_bwd(const tt_chain_args* a, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ChainParams p;
  int rc = fill_chain(p, a, "tt_chain_bwd");
  if (rc) return rc;
  TT_REQUIRE((p.dout != nullptr) != (p.dout_bf16 != nullptr) && (p.dx_f32 || p.dx_bf16),
             "tt_chain_bwd: exactly one of dout / dout_bf16 and a dx output are required");
  TT_REQUIRE(!p.ln_w || (p.dgamma && p.dbeta), "tt_chain_bwd: LayerNorm needs dgamma/dbeta");
  TT_REQUIRE(a->width == 256, "tt_chain_bwd: width %d unsupported (256)", a->width);
  int grid = row_grid(p.R);
  if (grid > num_sms() * 2) grid = num_sms() * 2;  // bounds the per-block atomic combine
  TT_CHECK_CUDA(launch_k(chain_bwd_kernel<2>, dim3(grid), dim3(kRowThreads), 0, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_gather_cat_fwd(const float* x, const int32_t* last_idx, const int64_t* gender,
                                 const int64_t* country, const float* G, const float* C, int B, int L, void* cat,
                                 void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(x && last_idx && G && C && cat && B > 0, "tt_gather_cat_fwd: bad arguments");
  TT_CHECK_CUDA(launch_k(gather_cat_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, stream, x, last_idx, gender, country, G, C, B, L, static_cast<__nv_bfloat16*>(cat)));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_gather_cat_bwd(const float* dcat, const int32_t* last_idx, const int64_t* gender,
                                 const int64_t* country, int B, int L, float* dx, void* dx_bf16, float* dG, float* dC,
                                 void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(dcat && last_idx && dG && dC && (dx || dx_bf16) && B > 0, "tt_gather_cat_bwd: bad arguments");
  TT_CHECK_CUDA(launch_k(gather_cat_bwd_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, stream, dcat, last_idx, gender, country, B, L, dx, static_cast<__nv_bfloat16*>(dx_bf16), dG, dC));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_concat4_bf16(const float* a, const float* b, const float* c, const float* d, int B, int m,
                               void* out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(a && b && c && d && out && B > 0 && m > 0, "tt_concat4_bf16: bad arguments");
  const size_t n = static_cast<size_t>(B) * 4 * m;
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  TT_CHECK_CUDA(launch_k(concat4_kernel, dim3(grid), dim3(256), 0, stream, a, b, c, d, B, m, static_cast<__nv_bfloat16*>(out)));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

static int fill_bn(BnParams& p, const tt_bn_args* a, const char* who) {
  TT_REQUIRE(a && a->y && a->w && a->b && a->B > 0 && a->C > 0, "%s: bad arguments", who);
  TT_REQUIRE(a->C % 32 == 0, "%s: C must be a multiple of 32", who);
  p.y = a->y; p.B = a->B; p.C = a->C; p.w = a->w; p.b = a->b;
  p.running_mean = a->running_mean; p.running_var = a->running_var; p.num_batches = a->num_batches_tracked;
  p.training = a->training; p.momentum = a->momentum; p.eps = a->eps > 0.f ? a->eps : 1e-5f;
  p.drop_thresh = drop_threshold(a->drop_p);
  p.drop_scale = a->drop_p > 0.f ? 1.f / (1.f - a->drop_p) : 1.f;
  p.seed = a->drop_seed; p.seed_dev = a->drop_seed_dev; p.site = a->drop_site;
  p.save_mean = a->save_mean; p.save_rstd = a->save_rstd;
  p.out = static_cast<__nv_bfloat16*>(a->out_bf16);
  p.dout = a->dout; p.dy = static_cast<__nv_bfloat16*>(a->dy_bf16);
  p.dgamma = a->dgamma; p.dbeta = a->dbeta; p.dy_colsum = a->dy_colsum;
  return TT_OK;
}

extern "C" int tt_bn_relu_fwd(const tt_bn_args* a, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  BnParams p;
  int rc = fill_bn(p, a, "tt_bn_relu_fwd");
  if (rc) return rc;
  TT_REQUIRE(p.out && p.running_mean && p.running_var, "tt_bn_relu_fwd: missing output or running stats");
  TT_REQUIRE(!p.training || (p.save_mean && p.save_rstd), "tt_bn_relu_fwd: training needs save_mean/save_rstd");
  TT_CHECK_CUDA(launch_k(bn_fwd_kernel, dim3((p.C + 31) / 32), dim3(dim3(32, 8)), 0, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_bn_relu_bwd(const tt_bn_args* a, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  BnParams p;
  int rc = fill_bn(p, a, "tt_bn_relu_bwd");
  if (rc) return rc;
  TT_REQUIRE(p.dout && p.dy && p.dgamma && p.dbeta && p.save_mean && p.save_rstd, "tt_bn_relu_bwd: missing buffers");
  TT_CHECK_CUDA(launch_k(bn_bwd_kernel, dim3((p.C + 31) / 32), dim3(dim3(32, 8)), 0, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_adamw_step(float* p, float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                             float eps, float weight_decay, float grad_scale, const int64_t* step_dev,
                             void* shadow_bf16, int64_t shadow_begin, int64_t shadow_end, int zero_grad, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(p && g && m && v && step_dev && n > 0 && n % 4 == 0, "tt_adamw_step: bad arguments");
  TT_REQUIRE(shadow_begin % 4 == 0 && shadow_end % 4 == 0 && shadow_begin <= shadow_end && shadow_end <= n,
             "tt_adamw_step: shadow range must be 4-aligned and inside [0, n]");
  const size_t n4 = static_cast<size_t>(n / 4);
  int grid = static_cast<int>((n4 + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  TT_CHECK_CUDA(launch_k(adamw_kernel, dim3(grid), dim3(256), 0, stream, p, g, m, v, n4, lr, beta1, beta2, eps, weight_decay, grad_scale, step_dev, static_cast<__nv_bfloat16*>(shadow_bf16), static_cast<size_t>(shadow_begin / 4), static_cast<size_t>(shadow_end / 4), zero_grad));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_index_rows(const float* y, int R, const float* ln_w, const float* ln_b, const int64_t* ids,
                             int64_t V, float* table, void* table_bf16, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(y && ln_w && ln_b && ids && table && R > 0 && V > 0, "tt_index_rows: bad arguments");
  TT_CHECK_CUDA(launch_k(index_rows_kernel, dim3(row_grid(R)), dim3(kRowThreads), 0, stream, y, R, ln_w, ln_b, ids, V, table, static_cast<__nv_bfloat16*>(table_bf16)));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

// The update id list on the host: every id in [1, vocab_size) and none twice, checked before any launch.
static int check_update_ids(const int64_t* ids, int n, int64_t vocab_size, cudaStream_t stream, const char* what) {
  std::vector<int64_t> h(static_cast<size_t>(n));
  TT_CHECK_CUDA(cudaMemcpyAsync(h.data(), ids, static_cast<size_t>(n) * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  TT_CHECK_CUDA(cudaStreamSynchronize(stream));
  std::vector<uint64_t> seen(static_cast<size_t>((vocab_size + 63) / 64), 0ull);
  for (int i = 0; i < n; ++i) {
    const int64_t id = h[i];
    TT_REQUIRE(id >= 1 && id < vocab_size, "%s: id %lld outside [1, %lld)", what, static_cast<long long>(id),
               static_cast<long long>(vocab_size));
    uint64_t& word = seen[static_cast<size_t>(id >> 6)];
    TT_REQUIRE(!((word >> (id & 63)) & 1ull), "%s: id %lld appears twice", what, static_cast<long long>(id));
    word |= 1ull << (id & 63);
  }
  return TT_OK;
}

extern "C" int tt_index_rows_live(const float* y, int R, const float* ln_w, const float* ln_b, const int64_t* ids,
                                  int64_t vocab_size, int64_t item_base, int N, float* table, void* table_bf16,
                                  uint32_t* retired_bits, float* stats, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(y && ln_w && ln_b && ids && table && table_bf16 && stats && R > 0 && N > 0,
             "tt_index_rows_live: bad arguments");
  TT_REQUIRE(item_base >= 0 && item_base + N <= vocab_size, "tt_index_rows_live: rows [%lld, %lld) outside the catalog of %lld",
             static_cast<long long>(item_base), static_cast<long long>(item_base + N), static_cast<long long>(vocab_size));
  const int rc = check_update_ids(ids, R, vocab_size, stream, "tt_index_rows_live");
  if (rc) return rc;
  TT_CHECK_CUDA(launch_k(index_rows_live_kernel, dim3(row_grid(R)), dim3(kRowThreads), 0, stream, y, R, ln_w, ln_b, ids, item_base, N, table, static_cast<__nv_bfloat16*>(table_bf16), retired_bits, stats));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_catalog_retire(const int64_t* ids, int n, int64_t vocab_size, int64_t item_base, int N, float* table,
                                 void* table_bf16, uint32_t* retired_bits, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(ids && table && table_bf16 && retired_bits && n > 0 && N > 0, "tt_catalog_retire: bad arguments");
  TT_REQUIRE(item_base >= 0 && item_base + N <= vocab_size, "tt_catalog_retire: rows [%lld, %lld) outside the catalog of %lld",
             static_cast<long long>(item_base), static_cast<long long>(item_base + N), static_cast<long long>(vocab_size));
  const int rc = check_update_ids(ids, n, vocab_size, stream, "tt_catalog_retire");
  if (rc) return rc;
  TT_CHECK_CUDA(launch_k(catalog_retire_kernel, dim3(row_grid(n)), dim3(kRowThreads), 0, stream, ids, n, item_base, N, table, static_cast<__nv_bfloat16*>(table_bf16), retired_bits));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_step_counters_advance(int64_t* step_dev, uint64_t* seed_dev, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_CHECK_CUDA(launch_k(increment_kernel, dim3(1), dim3(1), 0, stream, step_dev, seed_dev));
  TT_LAUNCH_CHECK();
  return TT_OK;
}
