// Causal self-attention for the SASRec user tower on tcgen05 (sm_100a), d_head = 64.
//
// Replaces the scaled_dot_product_attention call the reference reaches through
// nn.TransformerEncoderLayer (src/models/user_tower.py:37-45,111-116). The reference feeds a
// dense additive (causal + key-padding) float mask; here the histories are right-padded, so
// for every VALID query row the causal predicate alone is the full mask (keys <= query <
// length) and no mask tensor exists. Pad-query rows produce finite values nobody reads.
//
// Forward: one CTA (128 threads = 128 query rows = 128 TMEM lanes) per (sequence, head,
// 128-row query tile). All S_j = Q K_j^T tiles (j <= query tile) are issued up front into
// TMEM (128 columns each, L <= 512), the row max is taken from TMEM, then per key tile
// P_j = exp2(.) is written as bf16 into a 128B-swizzled K-major smem tile (double-buffered)
// and O += P_j V_j accumulates in TMEM (V consumed MN-major straight from the QKV buffer's
// layout). O reuses the first 64 columns of S_0 once S_0 has been drained.
//
// Backward: one CTA per (sequence, head) walks key tiles j and query tiles i >= j with the
// five products of the standard attention backward, all on tcgen05 (see attn_bwd_kernel).
#include "../../include/tt_b200.h"
#include "tt_common.cuh"

namespace tt {

static constexpr int kDh = 64;
static constexpr int kTile = 128;
static constexpr uint32_t kTileBytes = kTile * kDh * 2;  // 16 KB: 128 rows x 64 bf16
static constexpr float kLog2e = 1.4426950408889634f;

struct AttnParams {
  int B, L, H;
  int nq;            // query tiles per sequence
  float scale;       // 1/sqrt(d_head)
  uint32_t drop_thresh;
  float drop_scale;
  uint64_t drop_seed;
  const uint64_t* drop_seed_dev;
  uint32_t drop_site;
  __nv_bfloat16* ctx;  // [T, H*64]
  float* lse;          // [B, H, L]
};

// Write 8 consecutive bf16 (one 16-byte unit) of row r, unit u (0..7) into a K-major
// 128B-swizzled [128][64] bf16 tile.
__device__ __forceinline__ void st_swizzled_unit(uint8_t* tile, int r, int u, uint4 v) {
  *reinterpret_cast<uint4*>(tile + r * 128 + ((u ^ (r & 7)) << 4)) = v;
}

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// 32 fp32 accumulator columns -> 32 bf16 = 64 bytes of one row, as two 32-byte stores: every store fills a whole
// sector (the rows of a warp are 1.5 KB apart, so nothing coalesces across lanes; 16-byte stores left half-written
// sectors for the L2 to merge). dst is 64-byte aligned (row pitch, head offset and column half all are).
__device__ __forceinline__ void store_row32_bf16(__nv_bfloat16* dst, const uint32_t (&r)[32]) {
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    uint32_t w[8];
#pragma unroll
    for (int e = 0; e < 8; ++e)
      w[e] = pack_bf16(__uint_as_float(r[u * 16 + 2 * e]), __uint_as_float(r[u * 16 + 2 * e + 1]));
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + u * 16), "r"(w[0]), "r"(w[1]),
                 "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
                 : "memory");
  }
}

// Forward. 256 threads: warp w -> TMEM lane quarter (w & 3), column half (w >> 2). Thread
// (row, hf) owns query row `row` of the tile and the 64-column half `hf` of every 128-key tile.
// Shared memory per CTA (nq = 2): Q 16 KB + K slots 32 KB (reused for V_1.. once the S MMAs have retired) + V_0
// 16 KB + P 32 KB = 96 KB -> two CTAs per SM (TMEM: 128 or 256 columns each).
__global__ void __launch_bounds__(256, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hf = warp >> 2;
  const int row = q * 32 + lane;
  const int bh_count = p.B * p.H;
  const int qt = p.nq - 1 - static_cast<int>(blockIdx.x) / bh_count;  // heavy tiles first
  const int bh = static_cast<int>(blockIdx.x) % bh_count;
  const int b = bh / p.H, h = bh % p.H;
  const int n_kv = qt + 1;
  const int D = p.H * kDh;

  uint8_t* sQ = smem;
  uint8_t* sKV = sQ + kTileBytes;
  uint8_t* sV0 = sKV + static_cast<size_t>(p.nq) * kTileBytes;   // V_0 has its own slot: loaded with Q / K, not after S
  uint8_t* sP = sV0 + kTileBytes;                                 // 2 chunks x 16 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * kTileBytes);
  uint64_t* bar_qk = bars + 0;
  uint64_t* bar_v = bars + 1;
  uint64_t* bar_s = bars + 2;
  uint64_t* bar_pv = bars + 3;
  uint64_t* bar_v0 = bars + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
  float* s_red = reinterpret_cast<float*>(bars + 7);  // [2][128]

  uint32_t tmem_cols = 128;
  while (tmem_cols < static_cast<uint32_t>(n_kv * kTile)) tmem_cols <<= 1;

  if (tid == 0) {
    tma_prefetch_desc(&tmQKV);
    mbar_init(bar_qk, 1);
    mbar_init(bar_v, 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_pv, 1);
    mbar_init(bar_v0, 1);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) {
    tmem_alloc(tmem_slot, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // The trigger comes AFTER this CTA owns its TMEM columns: a dependent CTA scheduled early on the same
  // SM could otherwise take them first and wait forever for this grid to finish.
  pdl_launch_dependents();
  pdl_wait();   // prologue (barriers, TMEM, tensor-map prefetch) overlapped the previous kernel's tail

  const int seq_row0 = b * p.L;
  const int q_row0 = seq_row0 + qt * kTile;

  if (tid == 0) {
    mbar_arrive_expect_tx(bar_qk, (1 + n_kv) * kTileBytes);
    tma_load_2d(sQ, &tmQKV, bar_qk, h * kDh, q_row0);
    for (int j = 0; j < n_kv; ++j)
      tma_load_2d(sKV + static_cast<size_t>(j) * kTileBytes, &tmQKV, bar_qk, D + h * kDh, seq_row0 + j * kTile);
    mbar_arrive_expect_tx(bar_v0, kTileBytes);
    tma_load_2d(sV0, &tmQKV, bar_v0, 2 * D + h * kDh, seq_row0);
    mbar_wait(bar_qk, 0);
    tc_fence_after();
    const uint32_t idesc_s = umma_idesc_bf16(kTile, kTile, false, false);
    // descriptors once per tile, a k-step adds its byte offset >> 4 to the address field (addresses < 256 KB)
    const uint64_t q_desc = umma_desc_kmajor(smem_u32(sQ));
    for (int j = 0; j < n_kv; ++j) {
      const uint64_t k_desc = umma_desc_kmajor(smem_u32(sKV + static_cast<size_t>(j) * kTileBytes));
#pragma unroll
      for (int k = 0; k < kDh / 16; ++k)
        umma_bf16(tmem_base + j * kTile, q_desc + (k * 32 >> 4), k_desc + (k * 32 >> 4), idesc_s, k > 0 ? 1u : 0u);
    }
    umma_commit(bar_s);
    // the K slots are free once the S MMAs retired: V_1.. take their place (needed one P tile later than V_0)
    if (n_kv > 1) {
      mbar_wait(bar_s, 0);
      mbar_arrive_expect_tx(bar_v, (n_kv - 1) * kTileBytes);
      for (int j = 1; j < n_kv; ++j)
        tma_load_2d(sKV + static_cast<size_t>(j - 1) * kTileBytes, &tmQKV, bar_v, 2 * D + h * kDh, seq_row0 + j * kTile);
    }
  }

  // ---- pass A: row maximum over the causal prefix (each thread: its column half) ----------
  mbar_wait(bar_s, 0);
  __syncwarp();
  tc_fence_after();
  const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  const int q_pos = qt * kTile + row;  // position of this thread's query inside the sequence
  const bool dead_rows = qt * kTile + q * 32 >= p.L;
  float m = -INFINITY;
  for (int j = 0; j < n_kv; ++j) {
    const bool diag = (j == qt);
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      const int cg = 2 * hf + cc;       // 32-column chunk index inside the key tile
      // nothing to do (warp-uniform): above the diagonal for every row of this warp, or the warp's 32 query rows /
      // the chunk's 32 keys lie wholly beyond the sequence (L = 200: a quarter of the second tile's warps)
      if ((diag && cg > q) || dead_rows || j * kTile + cg * 32 >= p.L) continue;
      uint32_t r[32];
      tmem_ld32(lane_base + j * kTile + cg * 32, r);
      tmem_ld_wait();
      const int kv0 = j * kTile + cg * 32;
#pragma unroll
      for (int t = 0; t < 32; ++t) {
        const float s = __uint_as_float(r[t]);
        if (!diag || kv0 + t <= q_pos) m = fmaxf(m, s);
      }
    }
  }
  s_red[hf * 128 + row] = m;
  __syncthreads();
  m = fmaxf(s_red[row], s_red[128 + row]);
  __syncthreads();
  const float c1 = p.scale * kLog2e;
  const float mc = m * c1;
  const uint64_t seed = p.drop_seed + ((p.drop_thresh && p.drop_seed_dev) ? *p.drop_seed_dev : 0ull);
  const uint32_t dkey = drop_key(seed, p.drop_site);

  // ---- pass B: P_j -> smem (bf16, swizzled), O += P_j V_j ------------------------------
  float l = 0.f;
  const uint32_t idesc_pv = umma_idesc_bf16(kTile, kDh, false, true);
  uint8_t* chunk = sP + static_cast<size_t>(hf) * kTileBytes;  // this thread's 64 key columns
  for (int j = 0; j < n_kv; ++j) {
    if (j >= 1) mbar_wait(bar_pv, (j - 1) & 1);  // previous P tile consumed
    __syncwarp();
    const bool diag = (j == qt);
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      const int cg = 2 * hf + cc;
      const int u0 = cc * 4;
      if (!((diag && cg > q) || dead_rows || j * kTile + cg * 32 >= p.L)) {
        uint32_t r[32];
        tmem_ld32(lane_base + j * kTile + cg * 32, r);
        tmem_ld_wait();
        const int kv0 = j * kTile + cg * 32;
        const uint32_t didx0 = (static_cast<uint32_t>(bh) * p.L + q_pos) * p.L + kv0;
        float pv[32];
#pragma unroll
        for (int t = 0; t < 32; ++t) {
          float e = fast_exp2(__uint_as_float(r[t]) * c1 - mc);
          if (diag && kv0 + t > q_pos) e = 0.f;
          l += e;
          pv[t] = e;
        }
        if (p.drop_thresh) {
          if ((didx0 & 3u) == 0u) {          // L % 4 == 0: four keys per hash word
#pragma unroll
            for (int t = 0; t < 32; t += 4) {
              bool k[4];
              drop_keep_quad(dkey, didx0 + t, p.drop_thresh, k);
#pragma unroll
              for (int e = 0; e < 4; ++e) pv[t + e] = k[e] ? pv[t + e] * p.drop_scale : 0.f;
            }
          } else if ((didx0 & 1u) == 0u) {
#pragma unroll
            for (int t = 0; t < 32; t += 2) {
              bool k0, k1;
              drop_keep_pair(dkey, didx0 + t, p.drop_thresh, k0, k1);
              pv[t] = k0 ? pv[t] * p.drop_scale : 0.f;
              pv[t + 1] = k1 ? pv[t + 1] * p.drop_scale : 0.f;
            }
          } else {
#pragma unroll
            for (int t = 0; t < 32; ++t)
              pv[t] = drop_keep_k(dkey, didx0 + t, p.drop_thresh) ? pv[t] * p.drop_scale : 0.f;
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint4 v;
          v.x = pack_bf16(pv[u * 8 + 0], pv[u * 8 + 1]);
          v.y = pack_bf16(pv[u * 8 + 2], pv[u * 8 + 3]);
          v.z = pack_bf16(pv[u * 8 + 4], pv[u * 8 + 5]);
          v.w = pack_bf16(pv[u * 8 + 6], pv[u * 8 + 7]);
          st_swizzled_unit(chunk, row, u0 + u, v);
        }
      } else {
#pragma unroll
        for (int u = 0; u < 4; ++u) st_swizzled_unit(chunk, row, u0 + u, make_uint4(0, 0, 0, 0));
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      if (j == 0) mbar_wait(bar_v0, 0);
      else if (j == 1) mbar_wait(bar_v, 0);
      const uint64_t p_desc = umma_desc_kmajor(smem_u32(sP));
      const uint64_t v_desc = umma_desc_mnmajor(smem_u32(j == 0 ? sV0 : sKV + static_cast<size_t>(j - 1) * kTileBytes), kTileBytes);
#pragma unroll
      for (int k = 0; k < kTile / 16; ++k) {
        // A = P: chunk (k/4), 32 B per 16 kv columns; B = V rows (MN-major): 16 kv rows = 2048 B
        umma_bf16(tmem_base, p_desc + (((k >> 2) * kTileBytes + (k & 3) * 32) >> 4), v_desc + (k * 2048 >> 4), idesc_pv,
                  (j > 0 || k > 0) ? 1u : 0u);
      }
      umma_commit(bar_pv);
    }
  }

  // ---- epilogue: O / l -> ctx, log-sum-exp -> lse ---------------------------------------
  s_red[hf * 128 + row] = l;
  mbar_wait(bar_pv, (n_kv - 1) & 1);
  __syncthreads();
  tc_fence_after();
  l = s_red[row] + s_red[128 + row];
  {
    const float inv_l = 1.f / l;
    const bool valid = q_pos < p.L;
    __nv_bfloat16* orow = p.ctx + static_cast<size_t>(seq_row0 + q_pos) * D + h * kDh + hf * 32;
    uint32_t r[32];
    tmem_ld32(lane_base + hf * 32, r);
    tmem_ld_wait();
    if (valid) {
#pragma unroll
      for (int t = 0; t < 32; ++t) r[t] = __float_as_uint(__uint_as_float(r[t]) * inv_l);
      store_row32_bf16(orow, r);   // two 32-byte stores: whole sectors (rows are 512 B apart, nothing coalesces)
      if (hf == 0 && p.lse) p.lse[static_cast<size_t>(bh) * p.L + q_pos] = m * p.scale + __logf(l);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

// --------------------------------------------------------------------------------------------
// Forward, persistent and pipelined (L <= 256). The kernel above is a chain of dependent latencies per CTA
// (TMEM allocation -> TMA -> S MMAs -> row max -> P -> PV MMA -> epilogue) with two CTAs per SM to hide them.
// Here a CTA per SM walks (sequence, head) items; per item the (query tile u, key tile j <= u) pairs are
// (0,0), (1,0), (1,1), S tile t = pair index at TMEM columns 128 t, O_u at 384 + 64 u:
//   * warps 0-15: thread (row, 32-column chunk). Per query tile: row max over its S tiles (combined across the
//     four chunk groups through shared memory), then per pair P = dropout(exp2(.)) -> bf16 -> one of two
//     32 KB P tiles. O_u is divided by the row sum and stored one pair AFTER its last PV MMA was issued, so
//     that MMA is never waited for;
//   * warp 16 (control flow by the whole warp, issue by one elected lane): TMA loads and MMAs. The S tile t
//     of the NEXT item is issued as soon as every thread has read tile t of this one for the last time, so
//     it is ready long before it is needed; Q / K of the next item are requested when this item's S MMAs
//     have retired, V (two sets of slots) one item ahead.
// --------------------------------------------------------------------------------------------
static constexpr int kFwdComputeThreads = 512;
static constexpr int kFwdThreads = kFwdComputeThreads + 128;

__global__ void __launch_bounds__(kFwdThreads, 1)
attn_fwd_persist_kernel(const __grid_constant__ CUtensorMap tmQKV, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int D = p.H * kDh;
  const int nq = p.nq;                         // 1 or 2
  const int np = nq == 2 ? 3 : 1;              // (query tile, key tile) pairs per item
  const int n_items = p.B * p.H;

  uint8_t* sQ = smem;                          // [2]
  uint8_t* sK = sQ + 2 * kTileBytes;           // [2]
  uint8_t* sV = sK + 2 * kTileBytes;           // [2 sets][2]
  uint8_t* sP = sV + 4 * kTileBytes;           // [2 slots] x (2 chunks of 64 key columns)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 4 * kTileBytes);
  uint64_t* bar_q = bars + 0;       // [2] Q_u landed (a phase per item)
  uint64_t* bar_k = bars + 2;       // [2] K_j landed (a phase per item)
  uint64_t* bar_v = bars + 4;       // [2 sets][2] V_j landed (a phase per two items)
  uint64_t* bar_s = bars + 8;       // [3] S tile t ready (a phase per item)
  uint64_t* bar_sfree = bars + 11;  // [3] every thread has read S tile t for the last time (a phase per item)
  uint64_t* bar_pfull = bars + 14;  // [2] P slot staged (a phase per use)
  uint64_t* bar_pv = bars + 16;     // [2] the PV MMAs reading P slot s retired (a phase per use)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);
  float* s_sum = reinterpret_cast<float*>(bars + 20);   // [3 buffers][4 chunk groups][128 rows]

  if (tid == 0) {
    tma_prefetch_desc(&tmQKV);
    for (int i = 0; i < 8; ++i) mbar_init(bars + i, 1);
    for (int i = 0; i < 3; ++i) mbar_init(bar_s + i, 1);
    for (int i = 0; i < 3; ++i) mbar_init(bar_sfree + i, kFwdComputeThreads);
    for (int i = 0; i < 2; ++i) mbar_init(bar_pfull + i, kFwdComputeThreads);
    for (int i = 0; i < 2; ++i) mbar_init(bar_pv + i, 1);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 16) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();
  constexpr uint32_t T_O = 384;

  if (warp >= 16) {
    if (warp == 16) {
      // ======================= issuer =========================================================
      const uint32_t idesc_s = umma_idesc_bf16(kTile, kTile, false, false);
      const uint32_t idesc_pv = umma_idesc_bf16(kTile, kDh, false, true);
      auto load_qk = [&](int item) {          // Q_u -> slot u, K_j -> slot j
        const int b = item / p.H, h = item % p.H;
        if (elect_one()) {
          for (int u = 0; u < nq; ++u) {
            mbar_arrive_expect_tx(bar_q + u, kTileBytes);
            tma_load_2d(sQ + static_cast<size_t>(u) * kTileBytes, &tmQKV, bar_q + u, h * kDh, b * p.L + u * kTile);
            mbar_arrive_expect_tx(bar_k + u, kTileBytes);
            tma_load_2d(sK + static_cast<size_t>(u) * kTileBytes, &tmQKV, bar_k + u, D + h * kDh, b * p.L + u * kTile);
          }
        }
        __syncwarp();
      };
      auto load_v = [&](int item, int set) {
        const int b = item / p.H, h = item % p.H;
        if (elect_one()) {
          for (int j = 0; j < nq; ++j) {
            mbar_arrive_expect_tx(bar_v + set * 2 + j, kTileBytes);
            tma_load_2d(sV + static_cast<size_t>(set * 2 + j) * kTileBytes, &tmQKV, bar_v + set * 2 + j, 2 * D + h * kDh,
                        b * p.L + j * kTile);
          }
        }
        __syncwarp();
      };
      auto issue_s = [&](int t) {              // S tile t = Q_u K_j^T, (u, j) = (0,0), (1,0), (1,1)
        const int u = t == 0 ? 0 : 1, j = t == 2 ? 1 : 0;
        const uint64_t dq = umma_desc_kmajor(smem_u32(sQ + static_cast<size_t>(u) * kTileBytes));
        const uint64_t dk = umma_desc_kmajor(smem_u32(sK + static_cast<size_t>(j) * kTileBytes));
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k)
            umma_bf16(tmem_base + t * kTile, dq + (k * 32 >> 4), dk + (k * 32 >> 4), idesc_s, k > 0 ? 1u : 0u);
          umma_commit(bar_s + t);
        }
        __syncwarp();
      };
      auto issue_pv = [&](int t, int slot, int set) {   // O_u (+)= P[slot] V_j
        const int u = t == 0 ? 0 : 1, j = t == 2 ? 1 : 0;
        const uint64_t dp = umma_desc_kmajor(smem_u32(sP + static_cast<size_t>(slot) * 2 * kTileBytes));
        const uint64_t dv = umma_desc_mnmajor(smem_u32(sV + static_cast<size_t>(set * 2 + j) * kTileBytes), kTileBytes);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < kTile / 16; ++k)
            umma_bf16(tmem_base + T_O + u * kDh, dp + (((k >> 2) * kTileBytes + (k & 3) * 32) >> 4), dv + (k * 2048 >> 4),
                      idesc_pv, (j > 0 || k > 0) ? 1u : 0u);
          umma_commit(bar_pv + slot);
        }
        __syncwarp();
      };

      int item = blockIdx.x;
      load_qk(item);
      load_v(item, 0);
      for (int t = 0; t < np; ++t) {
        const int u = t == 0 ? 0 : 1, j = t == 2 ? 1 : 0;
        mbar_wait(bar_q + u, 0);
        mbar_wait(bar_k + j, 0);
        tc_fence_after();
        issue_s(t);
      }
      uint32_t gk = 0;
      for (uint32_t n = 0; item < n_items; ++n, item += gridDim.x) {
        const int next = item + static_cast<int>(gridDim.x);
        const bool has_next = next < n_items;
        const uint32_t par = n & 1u, npar = (n + 1u) & 1u;
        const int set = static_cast<int>(n & 1u);
        mbar_wait(bar_s + (np - 1), par);        // this item's S MMAs retired: the Q / K slots are free
        if (has_next) load_qk(next);
        for (int t = 0; t < np; ++t, ++gk) {
          const int u = t == 0 ? 0 : 1, j = t == 2 ? 1 : 0;
          const int slot = static_cast<int>(gk & 1u);
          mbar_wait(bar_pfull + slot, (gk >> 1) & 1u);
          if (t == 0 || t == 2) mbar_wait(bar_v + set * 2 + j, (n >> 1) & 1u);   // first use of V_j in this item
          tc_fence_after();
          issue_pv(t, slot, set);
          if (has_next) {
            if (t == 0) {
              // the other V set was last read by the previous item's last PV MMAs
              if (gk >= 1) mbar_wait(bar_pv + ((gk - 1u) & 1u), ((gk - 1u) >> 1) & 1u);
              load_v(next, set ^ 1);
            }
            mbar_wait(bar_sfree + t, par);        // S tile t fully consumed: the next item's tile takes its columns
            mbar_wait(bar_q + u, npar);
            mbar_wait(bar_k + j, npar);
            tc_fence_after();
            issue_s(t);
          }
        }
      }
    }
  } else {
    // ======================= compute warps ====================================================
    const int q = warp & 3, cg = warp >> 2;     // TMEM lane quarter, 32-column chunk of a key tile
    const int row = q * 32 + lane;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float c1 = p.scale * kLog2e;
    const uint64_t seed = p.drop_seed + ((p.drop_thresh && p.drop_seed_dev) ? *p.drop_seed_dev : 0ull);
    const uint32_t dkey = drop_key(seed, p.drop_site);
    const int u0 = (cg & 1) * 4;
    // state of the query tile whose O is still to be stored (one pair after its last PV MMA was issued)
    int d_item = -1, d_u = 0, d_buf = 0;
    float d_m = 0.f;
    uint32_t d_gk = 0;
    auto drain = [&]() {
      // O_u / l -> ctx, log-sum-exp -> lse: thread (row, chunk group) takes 16 of the 64 columns
      mbar_wait(bar_pv + (d_gk & 1u), (d_gk >> 1) & 1u);
      __syncwarp();
      tc_fence_after();
      const float* ls = s_sum + d_buf * 4 * kTile;
      const float l = (ls[row] + ls[kTile + row]) + (ls[2 * kTile + row] + ls[3 * kTile + row]);
      const int q_pos = d_u * kTile + row;
      uint32_t r[16];
      tmem_ld16(lane_base + T_O + d_u * kDh + cg * 16, r);
      tmem_ld_wait();
      tc_fence_before();
      if (q_pos < p.L) {
        const int b = d_item / p.H, h = d_item % p.H;
        const float inv_l = 1.f / l;
        uint32_t w[8];
#pragma unroll
        for (int e = 0; e < 8; ++e)
          w[e] = pack_bf16(__uint_as_float(r[2 * e]) * inv_l, __uint_as_float(r[2 * e + 1]) * inv_l);
        __nv_bfloat16* dst = p.ctx + static_cast<size_t>(b * p.L + q_pos) * D + h * kDh + cg * 16;
        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(w[0]), "r"(w[1]),
                     "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
                     : "memory");
        if (cg == 0 && p.lse) p.lse[static_cast<size_t>(d_item) * p.L + q_pos] = d_m * p.scale + __logf(l);
      }
      d_item = -1;
    };

    uint32_t gk = 0, gu = 0;     // global pair / query-tile counters of this CTA
    int item = blockIdx.x;
    for (uint32_t n = 0; item < n_items; ++n, item += gridDim.x) {
      for (int u = 0; u < nq; ++u, ++gu) {
        const int q_pos = u * kTile + row;
        const bool dead_rows = u * kTile + q * 32 >= p.L;
        const int buf = static_cast<int>(gu % 3u);
        // ---- row maximum over the causal prefix: S tiles (u, 0..u). Every thread scans its WHOLE row (the four
        // threads of a row repeat each other's 128 comparisons per tile): combining four partial maxima needed a
        // 512-thread barrier per query tile, and the warps' skew made that wait a fifth of the kernel.
        float m = -INFINITY;
        for (int j = 0; j <= u; ++j) {
          const int t = u + j;
          const bool diag = (j == u);
          mbar_wait(bar_s + t, n & 1u);
          __syncwarp();
          tc_fence_after();
          if (dead_rows) continue;
          for (int c = 0; c < 4; ++c) {
            if ((diag && c > q) || j * kTile + c * 32 >= p.L) break;     // nothing further right is visible to these rows
            uint32_t r[32];
            tmem_ld32(lane_base + t * kTile + c * 32, r);
            tmem_ld_wait();
            if (diag && c == q) {
              const int kv0 = j * kTile + c * 32;
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (kv0 + e <= q_pos) m = fmaxf(m, __uint_as_float(r[e]));
            } else {
#pragma unroll
              for (int e = 0; e < 32; ++e) m = fmaxf(m, __uint_as_float(r[e]));
            }
          }
        }
        const float mc = m * c1;
        // ---- per pair: P -> shared memory, then the PV MMAs are the issuer's business ---------------
        float l = 0.f;
        for (int j = 0; j <= u; ++j, ++gk) {
          const int t = u + j;
          const bool diag = (j == u);
          const bool active = !((diag && cg > q) || dead_rows || j * kTile + cg * 32 >= p.L);
          const int slot = static_cast<int>(gk & 1u);
          uint8_t* chunk = sP + static_cast<size_t>(slot) * 2 * kTileBytes + static_cast<size_t>(cg >> 1) * kTileBytes;
          uint4 v[4];
#pragma unroll
          for (int x = 0; x < 4; ++x) v[x] = make_uint4(0, 0, 0, 0);
          if (active) {
            uint32_t r[32];
            tmem_ld32(lane_base + t * kTile + cg * 32, r);
            tmem_ld_wait();
            tc_fence_before();
            mbar_arrive(bar_sfree + t);
            const int kv0 = j * kTile + cg * 32;
            const uint32_t didx0 = (static_cast<uint32_t>(item) * p.L + q_pos) * p.L + kv0;
            float pv[32];
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              float x = fast_exp2(__uint_as_float(r[e]) * c1 - mc);
              if (diag && kv0 + e > q_pos) x = 0.f;
              l += x;
              pv[e] = x;
            }
            if (p.drop_thresh) {
              if ((didx0 & 3u) == 0u) {          // L % 4 == 0: four keys per hash word
#pragma unroll
                for (int e = 0; e < 32; e += 4) {
                  bool k[4];
                  drop_keep_quad(dkey, didx0 + e, p.drop_thresh, k);
#pragma unroll
                  for (int x = 0; x < 4; ++x) pv[e + x] = k[x] ? pv[e + x] * p.drop_scale : 0.f;
                }
              } else if ((didx0 & 1u) == 0u) {
#pragma unroll
                for (int e = 0; e < 32; e += 2) {
                  bool k0, k1;
                  drop_keep_pair(dkey, didx0 + e, p.drop_thresh, k0, k1);
                  pv[e] = k0 ? pv[e] * p.drop_scale : 0.f;
                  pv[e + 1] = k1 ? pv[e + 1] * p.drop_scale : 0.f;
                }
              } else {
#pragma unroll
                for (int e = 0; e < 32; ++e)
                  pv[e] = drop_keep_k(dkey, didx0 + e, p.drop_thresh) ? pv[e] * p.drop_scale : 0.f;
              }
            }
#pragma unroll
            for (int x = 0; x < 4; ++x) {
              v[x].x = pack_bf16(pv[x * 8 + 0], pv[x * 8 + 1]);
              v[x].y = pack_bf16(pv[x * 8 + 2], pv[x * 8 + 3]);
              v[x].z = pack_bf16(pv[x * 8 + 4], pv[x * 8 + 5]);
              v[x].w = pack_bf16(pv[x * 8 + 6], pv[x * 8 + 7]);
            }
          } else {
            tc_fence_before();
            mbar_arrive(bar_sfree + t);
          }
          // the PV MMAs that read this P slot two pairs ago have retired
          if (gk >= 2) mbar_wait(bar_pv + slot, ((gk >> 1) - 1u) & 1u);
#pragma unroll
          for (int x = 0; x < 4; ++x) st_swizzled_unit(chunk, row, u0 + x, v[x]);
          // Row-sum partials of the four chunk groups meet through shared memory without a barrier of their own:
          // written before this pair's arrive, read (drain) after the wait for the PV MMAs that the issuer started
          // once all 512 arrives were in. Three buffers: a thread can only be staging a pair if every thread has
          // arrived for the pair two before, i.e. has finished the drain that preceded that arrive.
          if (j == u) s_sum[(buf * 4 + cg) * kTile + row] = l;
          // the query tile whose last PV MMAs were issued one pair ago: its O is complete by now
          if (d_item >= 0) drain();
          fence_proxy_async_smem();
          mbar_arrive(bar_pfull + slot);
          if (j == u) { d_item = item; d_u = u; d_buf = buf; d_m = m; d_gk = gk; }
        }
      }
    }
    if (d_item >= 0) {
      asm volatile("bar.sync 1, %0;" ::"n"(kFwdComputeThreads) : "memory");   // the last tile's row sums are all written
      drain();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_dealloc(tmem_base, 512);
}

// --------------------------------------------------------------------------------------------
// Backward. One CTA (256 threads) per (sequence, head). For key tile j and query tile i >= j:
//   S   = Q_i K_j^T                    (TMEM cols [0,128))
//   dP  = dO_i V_j^T                   (TMEM cols [128,256))
//   P   = exp2(scale*log2e*S - lse_i*log2e) under the causal mask; Pd = dropout(P)
//   dS  = P * (dropout(dP) - delta_i) * scale,  delta_i = rowsum(dO_i * O_i)
//   dV_j += Pd^T dO_i   (A = Pd stored [q][kv] read MN-major, B = dO_i read MN-major)
//   dK_j += dS^T Q_i    (A = dS read MN-major,               B = Q_i  read MN-major)
//   dQ_i += dS K_j      (A = dS K-major,                     B = K_j  read MN-major)
// dV_j, dK_j live in TMEM (cols [256,320), [320,384)) across the inner loop; dQ_i
// (cols [384 + 64*i ...)) is kept for every query tile: two tiles (L <= 256) in the fast layout,
// four (L <= 512) in the LONG layout described at the kernel.
// Pd and dS are staged as bf16 in 128B-swizzled smem tiles. Thread (row, hf) owns query row
// `row` and the 64-column half `hf` of the 128-key tile (warp & 3 = TMEM lane quarter).
// --------------------------------------------------------------------------------------------
// Keep decisions of 32 consecutive elements starting at didx0 as a bit mask: one hash per 4 (2, 1) elements
// depending on the alignment of didx0 — the same decisions drop_keep_k gives element by element.
__device__ __forceinline__ uint32_t drop_keepmask32(uint32_t dkey, uint32_t didx0, uint32_t thresh) {
  uint32_t keepmask = 0u;
  if ((didx0 & 3u) == 0u) {
#pragma unroll
    for (int t = 0; t < 32; t += 4) {
      bool k[4];
      drop_keep_quad(dkey, didx0 + t, thresh, k);
#pragma unroll
      for (int e = 0; e < 4; ++e) keepmask |= (k[e] ? 1u : 0u) << (t + e);
    }
  } else if ((didx0 & 1u) == 0u) {
#pragma unroll
    for (int t = 0; t < 32; t += 2) {
      bool k0, k1;
      drop_keep_pair(dkey, didx0 + t, thresh, k0, k1);
      keepmask |= (k0 ? 1u : 0u) << t;
      keepmask |= (k1 ? 1u : 0u) << (t + 1);
    }
  } else {
#pragma unroll
    for (int t = 0; t < 32; ++t) keepmask |= (drop_keep_k(dkey, didx0 + t, thresh) ? 1u : 0u) << t;
  }
  return keepmask;
}

struct AttnBwdParams {
  int B, L, H, nq;
  float scale;
  uint32_t drop_thresh;
  float drop_scale;
  uint64_t drop_seed;
  const uint64_t* drop_seed_dev;
  uint32_t drop_site;
  const __nv_bfloat16* ctx;   // O  [T, H*64]
  const __nv_bfloat16* dctx;  // dO [T, H*64]
  const float* lse;           // [B,H,L]
  __nv_bfloat16* dqkv;        // [T, 3*H*64]
};

// LONG = false: L <= 256 (two query tiles): S and dP have their own TMEM columns and are issued
//   together. LONG = true: L <= 512 (four query tiles): the four dQ accumulators need 256 columns,
//   so S and dP SHARE one 128-column region — P is formed from S first (un-dropped P parked as bf16
//   in the dS tile), then dP = dO V^T overwrites S and dS replaces the parked P.
// CG = column groups: 128*CG threads, thread (row, g) owns 4/CG of the four 32-column chunks of every
// 128-key tile. The per-iteration element-wise phase between the two MMA groups is latency-bound, so the
// fast layout runs it with 16 warps (CG = 4); LONG keeps 8 (its register tiles are larger).
template <bool LONG, int CG>
__global__ void __launch_bounds__(128 * CG, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, grp = warp >> 2;
  constexpr int CPT = 4 / CG;   // 32-column chunks per thread per key tile
  const int row = q * 32 + lane;
  const int bh = blockIdx.x;
  const int b = bh / p.H, h = bh % p.H;
  const int D = p.H * kDh;
  const int nq = p.nq;
  const int seq_row0 = b * p.L;

  // smem: Q[slots], dO[slots], K_j, V_j, Pd (2 chunks), dS (2 chunks). The fast layout keeps every
  // query tile resident; LONG re-loads Q_i / dO_i per (j, i) iteration into a single slot.
  const int slots = LONG ? 1 : nq;
  uint8_t* sQ = smem;
  uint8_t* sDO = sQ + static_cast<size_t>(slots) * kTileBytes;
  uint8_t* sK = sDO + static_cast<size_t>(slots) * kTileBytes;
  uint8_t* sV = sK + kTileBytes;
  uint8_t* sPd = sV + kTileBytes;
  uint8_t* sDS = sPd + 2 * kTileBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDS + 2 * kTileBytes);
  uint64_t* bar_q = bars + 0;    // Q/dO tiles loaded
  uint64_t* bar_kv = bars + 1;   // K_j/V_j loaded (phase per j)
  uint64_t* bar_mm1 = bars + 2;  // S and dP ready (phase per (j,i))
  uint64_t* bar_mm2 = bars + 3;  // dV/dK/dQ MMAs of this (j,i) retired
  uint64_t* bar_mm1b = bars + 4; // LONG: dP ready (after S has been consumed)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
  float* sDelta = reinterpret_cast<float*>(bars + 8);  // [nq*128]
  float* sLse = sDelta + nq * kTile;                   // [nq*128], pre-multiplied by log2e

  const uint32_t tmem_cols = 512;
  if (tid == 0) {
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmDO);
    mbar_init(bar_q, 1);
    mbar_init(bar_kv, 1);
    mbar_init(bar_mm1, 1);
    mbar_init(bar_mm2, 1);
    mbar_init(bar_mm1b, 1);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) {
    tmem_alloc(tmem_slot, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // The trigger comes AFTER this CTA owns its TMEM columns: a dependent CTA scheduled early on the same
  // SM could otherwise take them first and wait forever for this grid to finish.
  pdl_launch_dependents();
  pdl_wait();   // prologue (barriers, TMEM, tensor-map prefetch) overlapped the previous kernel's tail
  const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  constexpr uint32_t T_S = 0, T_DP = LONG ? 0 : 128, T_DV = LONG ? 128 : 256, T_DK = LONG ? 192 : 320,
                     T_DQ = LONG ? 256 : 384;

  if (!LONG && tid == 0) {
    mbar_arrive_expect_tx(bar_q, 2 * nq * kTileBytes);
    for (int i = 0; i < nq; ++i) {
      tma_load_2d(sQ + static_cast<size_t>(i) * kTileBytes, &tmQKV, bar_q, h * kDh, seq_row0 + i * kTile);
      tma_load_2d(sDO + static_cast<size_t>(i) * kTileBytes, &tmDO, bar_q, h * kDh, seq_row0 + i * kTile);
    }
  }
  // delta_i = rowsum(dO * O), lse -> smem (generic loads; rows beyond L are treated as zero)
  for (int pos = tid; pos < nq * kTile; pos += 128 * CG) {
    float delta = 0.f, lse2 = 0.f;
    if (pos < p.L) {
      const uint4* o = reinterpret_cast<const uint4*>(p.ctx + static_cast<size_t>(seq_row0 + pos) * D + h * kDh);
      const uint4* g = reinterpret_cast<const uint4*>(p.dctx + static_cast<size_t>(seq_row0 + pos) * D + h * kDh);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const uint4 a = __ldg(o + u), c = __ldg(g + u);
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, cw[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const float2 x = unpack_bf16(aw[w]), y = unpack_bf16(cw[w]);
          delta += x.x * y.x + x.y * y.y;
        }
      }
      lse2 = p.lse[static_cast<size_t>(bh) * p.L + pos] * kLog2e;
    }
    sDelta[pos] = delta;
    sLse[pos] = lse2;
  }
  __syncthreads();

  const float c1 = p.scale * kLog2e;
  const uint64_t seed = p.drop_seed + ((p.drop_thresh && p.drop_seed_dev) ? *p.drop_seed_dev : 0ull);
  const uint32_t dkey = drop_key(seed, p.drop_site);
  const uint32_t idesc_s = umma_idesc_bf16(kTile, kTile, false, false);    // Q K^T, dO V^T
  const uint32_t idesc_t = umma_idesc_bf16(kTile, kDh, true, true);        // X^T Y (dV, dK)
  const uint32_t idesc_q = umma_idesc_bf16(kTile, kDh, false, true);       // dS K
  uint32_t it = 0;  // (j,i) iteration counter -> mbarrier phase
  uint32_t dq_started = 0;  // bit i set once dQ_i has received its first MMA

  for (int j = 0; j < nq; ++j) {
    if (tid == 0) {
      // previous key tile's MMAs (which read sK/sV) have retired: bar_mm2 waited in-loop
      mbar_arrive_expect_tx(bar_kv, 2 * kTileBytes);
      tma_load_2d(sK, &tmQKV, bar_kv, D + h * kDh, seq_row0 + j * kTile);
      tma_load_2d(sV, &tmQKV, bar_kv, 2 * D + h * kDh, seq_row0 + j * kTile);
    }
    for (int i = j; i < nq; ++i, ++it) {
      const int slot = LONG ? 0 : i;
      if (tid == 0) {
        if constexpr (LONG) {   // the previous iteration's MMAs retired (bar_mm2): the slot is free
          mbar_arrive_expect_tx(bar_q, 2 * kTileBytes);
          tma_load_2d(sQ, &tmQKV, bar_q, h * kDh, seq_row0 + i * kTile);
          tma_load_2d(sDO, &tmDO, bar_q, h * kDh, seq_row0 + i * kTile);
          mbar_wait(bar_q, it & 1);
        } else {
          if (it == 0) mbar_wait(bar_q, 0);
        }
        if (i == j) mbar_wait(bar_kv, j & 1);
        tc_fence_after();
        const uint32_t q_base = smem_u32(sQ + static_cast<size_t>(slot) * kTileBytes);
        const uint32_t do_base = smem_u32(sDO + static_cast<size_t>(slot) * kTileBytes);
        const uint32_t k_base = smem_u32(sK), v_base = smem_u32(sV);
#pragma unroll
        for (int k = 0; k < kDh / 16; ++k)
          umma_bf16(tmem_base + T_S, umma_desc_kmajor(q_base + k * 32), umma_desc_kmajor(k_base + k * 32),
                    idesc_s, k > 0 ? 1u : 0u);
        if constexpr (!LONG) {
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k)
            umma_bf16(tmem_base + T_DP, umma_desc_kmajor(do_base + k * 32), umma_desc_kmajor(v_base + k * 32),
                      idesc_s, k > 0 ? 1u : 0u);
        }
        umma_commit(bar_mm1);
      }
      mbar_wait(bar_mm1, it & 1);
      __syncwarp();
      tc_fence_after();

      const int q_pos = i * kTile + row;
      const float lse2 = sLse[q_pos];
      const float delta = sDelta[q_pos];
      const bool diag = (i == j);
      const bool row_ok = q_pos < p.L;
      if constexpr (LONG) {
        // ---- part A: P from S. Pd -> sPd, un-dropped P parked (bf16) in the dS tile ---------------
        uint32_t km[CPT];   // dropout keep bits of this thread's chunks, formed once and reused by part B
#pragma unroll
        for (int cc = 0; cc < CPT; ++cc) {
          const int cg = CPT * grp + cc;
          const int u0 = (cg & 1) * 4;
          uint8_t* pchunk = sPd + static_cast<size_t>(cg >> 1) * kTileBytes;
          uint8_t* dchunk = sDS + static_cast<size_t>(cg >> 1) * kTileBytes;
          if (!(diag && cg > q)) {
            uint32_t rs[32];
            tmem_ld32(lane_base + T_S + cg * 32, rs);
            tmem_ld_wait();
            const int kv0 = j * kTile + cg * 32;
            const uint32_t didx0 = (static_cast<uint32_t>(bh) * p.L + q_pos) * p.L + kv0;
            km[cc] = p.drop_thresh ? drop_keepmask32(dkey, didx0, p.drop_thresh) : 0xFFFFFFFFu;
            float pr[32], pd[32];
#pragma unroll
            for (int t = 0; t < 32; ++t) {
              float x = fast_exp2(__uint_as_float(rs[t]) * c1 - lse2);
              if ((diag && kv0 + t > q_pos) || !row_ok) x = 0.f;
              pr[t] = x;
              pd[t] = ((km[cc] >> t) & 1u) ? x * p.drop_scale : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              uint4 v, w;
              v.x = pack_bf16(pd[u * 8 + 0], pd[u * 8 + 1]);
              v.y = pack_bf16(pd[u * 8 + 2], pd[u * 8 + 3]);
              v.z = pack_bf16(pd[u * 8 + 4], pd[u * 8 + 5]);
              v.w = pack_bf16(pd[u * 8 + 6], pd[u * 8 + 7]);
              w.x = pack_bf16(pr[u * 8 + 0], pr[u * 8 + 1]);
              w.y = pack_bf16(pr[u * 8 + 2], pr[u * 8 + 3]);
              w.z = pack_bf16(pr[u * 8 + 4], pr[u * 8 + 5]);
              w.w = pack_bf16(pr[u * 8 + 6], pr[u * 8 + 7]);
              st_swizzled_unit(pchunk, row, u0 + u, v);
              st_swizzled_unit(dchunk, row, u0 + u, w);
            }
          } else {
            km[cc] = 0u;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              st_swizzled_unit(pchunk, row, u0 + u, make_uint4(0, 0, 0, 0));
              st_swizzled_unit(dchunk, row, u0 + u, make_uint4(0, 0, 0, 0));
            }
          }
        }
        // ---- dP = dO V^T overwrites S once every thread has drained it --------------------------
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
          tc_fence_after();
          const uint32_t do_base = smem_u32(sDO + static_cast<size_t>(slot) * kTileBytes);
          const uint32_t v_base = smem_u32(sV);
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k)
            umma_bf16(tmem_base + T_DP, umma_desc_kmajor(do_base + k * 32), umma_desc_kmajor(v_base + k * 32),
                      idesc_s, k > 0 ? 1u : 0u);
          umma_commit(bar_mm1b);
        }
        mbar_wait(bar_mm1b, it & 1);
        __syncwarp();
        tc_fence_after();
        // ---- part B: dS = P * (dropout(dP) - delta) * scale replaces the parked P ------------------
#pragma unroll
        for (int cc = 0; cc < CPT; ++cc) {
          const int cg = CPT * grp + cc;
          const int u0 = (cg & 1) * 4;
          uint8_t* pchunk = sPd + static_cast<size_t>(cg >> 1) * kTileBytes;
          uint8_t* dchunk = sDS + static_cast<size_t>(cg >> 1) * kTileBytes;
          if (!(diag && cg > q)) {
            uint32_t rp[32];
            tmem_ld32(lane_base + T_DP + cg * 32, rp);
            tmem_ld_wait();
            const int kv0 = j * kTile + cg * 32;
            const uint32_t didx0 = (static_cast<uint32_t>(bh) * p.L + q_pos) * p.L + kv0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              uint4* slot = reinterpret_cast<uint4*>(dchunk + row * 128 + (((u0 + u) ^ (row & 7)) << 4));
              const uint4 pw = *slot;
              const uint32_t w[4] = {pw.x, pw.y, pw.z, pw.w};
              float ds[8];
#pragma unroll
              for (int h2 = 0; h2 < 4; ++h2) {
                const float2 pr2 = unpack_bf16(w[h2]);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const int t = u * 8 + h2 * 2 + e;
                  const float prv = e ? pr2.y : pr2.x;
                  const bool keep = (km[cc] >> t) & 1u;
                  const float dp = keep ? __uint_as_float(rp[t]) * p.drop_scale : 0.f;
                  ds[h2 * 2 + e] = prv * (dp - delta) * p.scale;
                }
              }
              uint4 o;
              o.x = pack_bf16(ds[0], ds[1]);
              o.y = pack_bf16(ds[2], ds[3]);
              o.z = pack_bf16(ds[4], ds[5]);
              o.w = pack_bf16(ds[6], ds[7]);
              *slot = o;
            }
          }
        }
      } else {
#pragma unroll
      for (int cc = 0; cc < CPT; ++cc) {
        const int cg = CPT * grp + cc;
        const int u0 = (cg & 1) * 4;
        uint8_t* pchunk = sPd + static_cast<size_t>(cg >> 1) * kTileBytes;
        uint8_t* dchunk = sDS + static_cast<size_t>(cg >> 1) * kTileBytes;
        if (!(diag && cg > q)) {
          uint32_t rs[32], rp[32];
          tmem_ld32(lane_base + T_S + cg * 32, rs);
          tmem_ld32(lane_base + T_DP + cg * 32, rp);
          tmem_ld_wait();
          const int kv0 = j * kTile + cg * 32;
          const uint32_t didx0 = (static_cast<uint32_t>(bh) * p.L + q_pos) * p.L + kv0;
          const uint32_t keepmask = p.drop_thresh ? drop_keepmask32(dkey, didx0, p.drop_thresh) : 0xFFFFFFFFu;
          float pd[32], ds[32];
#pragma unroll
          for (int t = 0; t < 32; ++t) {
            float pr = fast_exp2(__uint_as_float(rs[t]) * c1 - lse2);
            if ((diag && kv0 + t > q_pos) || !row_ok) pr = 0.f;
            const bool keep = (keepmask >> t) & 1u;
            const float dp = keep ? __uint_as_float(rp[t]) * p.drop_scale : 0.f;
            pd[t] = keep ? pr * p.drop_scale : 0.f;
            ds[t] = pr * (dp - delta) * p.scale;
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            uint4 v, w;
            v.x = pack_bf16(pd[u * 8 + 0], pd[u * 8 + 1]);
            v.y = pack_bf16(pd[u * 8 + 2], pd[u * 8 + 3]);
            v.z = pack_bf16(pd[u * 8 + 4], pd[u * 8 + 5]);
            v.w = pack_bf16(pd[u * 8 + 6], pd[u * 8 + 7]);
            w.x = pack_bf16(ds[u * 8 + 0], ds[u * 8 + 1]);
            w.y = pack_bf16(ds[u * 8 + 2], ds[u * 8 + 3]);
            w.z = pack_bf16(ds[u * 8 + 4], ds[u * 8 + 5]);
            w.w = pack_bf16(ds[u * 8 + 6], ds[u * 8 + 7]);
            st_swizzled_unit(pchunk, row, u0 + u, v);
            st_swizzled_unit(dchunk, row, u0 + u, w);
          }
        } else {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            st_swizzled_unit(pchunk, row, u0 + u, make_uint4(0, 0, 0, 0));
            st_swizzled_unit(dchunk, row, u0 + u, make_uint4(0, 0, 0, 0));
          }
        }
      }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncthreads();
      if (tid == 0) {
        tc_fence_after();
        const uint32_t pd_base = smem_u32(sPd), ds_base = smem_u32(sDS);
        const uint32_t q_base = smem_u32(sQ + static_cast<size_t>(slot) * kTileBytes);
        const uint32_t do_base = smem_u32(sDO + static_cast<size_t>(slot) * kTileBytes);
        const uint32_t k_base = smem_u32(sK);
        // Pd / dS are stored [q row][kv col] in two 64-column chunks. Read as the TRANSPOSED
        // operand (M = kv, contraction = q) they are MN-major: 16 q rows = 2048 B per K step,
        // 64-wide kv chunks are kTileBytes apart.
#pragma unroll
        for (int k = 0; k < kTile / 16; ++k)   // dV_j += Pd^T dO_i
          umma_bf16(tmem_base + T_DV, umma_desc_mnmajor(pd_base + k * 2048, kTileBytes),
                    umma_desc_mnmajor(do_base + k * 2048, kTileBytes), idesc_t, (i > j || k > 0) ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < kTile / 16; ++k)   // dK_j += dS^T Q_i
          umma_bf16(tmem_base + T_DK, umma_desc_mnmajor(ds_base + k * 2048, kTileBytes),
                    umma_desc_mnmajor(q_base + k * 2048, kTileBytes), idesc_t, (i > j || k > 0) ? 1u : 0u);
        const uint32_t first = ((dq_started >> i) & 1u) ? 0u : 1u;
#pragma unroll
        for (int k = 0; k < kTile / 16; ++k)   // dQ_i += dS K_j (A K-major, B = K_j rows MN-major)
          umma_bf16(tmem_base + T_DQ + i * kDh,
                    umma_desc_kmajor(ds_base + (k >> 2) * kTileBytes + (k & 3) * 32),
                    umma_desc_mnmajor(k_base + k * 2048, kTileBytes), idesc_q, (first && k == 0) ? 0u : 1u);
        dq_started |= (1u << i);
        umma_commit(bar_mm2);
      }
      // Pd/dS (and, on the last i, K_j/V_j) may only be overwritten once these MMAs retire.
      mbar_wait(bar_mm2, it & 1);
      __syncwarp();
      tc_fence_after();
    }
    // ---- dK_j, dV_j complete: TMEM -> dqkv (each thread: 32 of the 64 columns) -------------
    if (CG == 2 || grp < 2) {
      // 64 output columns = two 32-column halves: warps of groups 0/1 (CG = 4: groups 0,1 take dK, 2,3 dV)
      const int hf = grp & 1;
      const int pos = j * kTile + row;
      __nv_bfloat16* grow = p.dqkv + static_cast<size_t>(seq_row0 + pos) * (3 * D) + h * kDh + hf * 32;
      uint32_t rk[32];
      tmem_ld32(lane_base + T_DK + hf * 32, rk);
      tmem_ld_wait();
      if (pos < p.L) store_row32_bf16(grow + D, rk);
    }
    if (CG == 2 || grp >= 2) {
      const int hf = grp & 1;
      const int pos = j * kTile + row;
      __nv_bfloat16* grow = p.dqkv + static_cast<size_t>(seq_row0 + pos) * (3 * D) + h * kDh + hf * 32;
      uint32_t rv[32];
      tmem_ld32(lane_base + T_DV + hf * 32, rv);
      tmem_ld_wait();
      if (pos < p.L) store_row32_bf16(grow + 2 * D, rv);
    }
    tc_fence_before();
    __syncthreads();  // everyone has drained dK/dV before the next j overwrites them
    tc_fence_after();
  }

  // ---- dQ_i -> dqkv ---------------------------------------------------------------------
  for (int i = (CG == 2 ? 0 : (grp >> 1)); i < nq; i += (CG == 2 ? 1 : 2)) {   // CG = 4: groups (0,1) / (2,3) alternate tiles
    const int hf = grp & 1;
    const int pos = i * kTile + row;
    uint32_t r[32];
    tmem_ld32(lane_base + T_DQ + i * kDh + hf * 32, r);
    tmem_ld_wait();
    if (pos < p.L)
      store_row32_bf16(p.dqkv + static_cast<size_t>(seq_row0 + pos) * (3 * D) + h * kDh + hf * 32, r);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

// --------------------------------------------------------------------------------------------
// Backward, persistent and pipelined (L <= 256: one or two 128-row tiles). The kernel above spends most
// of a CTA's life in chains of dependent latencies (TMEM allocation -> TMA -> MMA -> element-wise -> MMA,
// one CTA per SM, nothing to overlap them with). Here a CTA per SM walks (sequence, head) items:
//   * warps 0-15 (512 threads): the element-wise phase, thread (row, 32-column chunk) as above; they
//     never issue anything, they only wait on / arrive at mbarriers;
//   * warp 16, one lane: every TMA load and every MMA. S/dP of iteration g+1 are issued as soon as all
//     512 threads hold S/dP of iteration g in registers (bar_drain), so those MMAs run under the
//     element-wise phase of g; operand tiles of the NEXT item are loaded into each shared-memory slot
//     as soon as the last MMA reading the slot has retired (Q0/dO0 after iteration 0, K0/V0 after
//     iteration 1, the rest after iteration 2), so no load latency is exposed between items;
//   * warp 17: delta = rowsum(dO * O) and the log-sum-exps of the next item, double-buffered.
// Iterations of an item (key tile j, query tile i): (0,0), (0,1), (1,1); TMEM columns as in the fast
// layout above. One __syncthreads at each end of the kernel, none inside.
// --------------------------------------------------------------------------------------------
static constexpr int kBwdComputeThreads = 512;
static constexpr int kBwdCtrlRegs = 56, kBwdComputeRegs = 104;   // 512 * 104 + 128 * 56 <= 640 * 96
static constexpr int kBwdThreads = kBwdComputeThreads + 128;   // + one warpgroup: issuer warp, delta warp, two idle

__global__ void __launch_bounds__(kBwdThreads, 1)
attn_bwd_persist_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                        const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int D = p.H * kDh;
  const int nq = p.nq;                       // 1 or 2
  const int niter = nq == 2 ? 3 : 1;
  const int n_items = p.B * p.H;

  uint8_t* sQ = smem;                        // [2] tiles
  uint8_t* sDO = sQ + 2 * kTileBytes;        // [2]
  uint8_t* sK = sDO + 2 * kTileBytes;        // [2]
  uint8_t* sV = sK + 2 * kTileBytes;         // [2]
  uint8_t* sPd = sV + 2 * kTileBytes;        // 2 chunks
  uint8_t* sDS = sPd + 2 * kTileBytes;       // 2 chunks
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDS + 2 * kTileBytes);
  uint64_t* bar_q = bars + 0;      // [2] Q_i + dO_i landed (one phase per item)
  uint64_t* bar_kv = bars + 2;     // [2] K_j + V_j landed (one phase per item)
  uint64_t* bar_mm1 = bars + 4;    // S and dP of iteration g ready
  uint64_t* bar_drain = bars + 5;  // all compute threads hold S/dP of iteration g in registers
  uint64_t* bar_stage = bars + 6;  // Pd / dS of iteration g are in shared memory
  uint64_t* bar_mm2 = bars + 7;    // dV/dK/dQ MMAs of iteration g retired
  uint64_t* bar_dfull = bars + 8;  // [2] delta / lse buffer filled
  uint64_t* bar_dfree = bars + 10; // [2] delta / lse buffer no longer read
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
  float* sDelta = reinterpret_cast<float*>(bars + 14);  // [2][256]
  float* sLse = sDelta + 2 * 2 * kTile;                 // [2][256], pre-multiplied by log2e

  if (tid == 0) {
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmDO);
    mbar_init(bar_q + 0, 1);
    mbar_init(bar_q + 1, 1);
    mbar_init(bar_kv + 0, 1);
    mbar_init(bar_kv + 1, 1);
    mbar_init(bar_mm1, 1);
    mbar_init(bar_drain, kBwdComputeThreads);
    mbar_init(bar_stage, kBwdComputeThreads);
    mbar_init(bar_mm2, 1);
    mbar_init(bar_dfull + 0, 96);
    mbar_init(bar_dfull + 1, 96);
    mbar_init(bar_dfree + 0, kBwdComputeThreads);
    mbar_init(bar_dfree + 1, kBwdComputeThreads);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 16) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();
  constexpr uint32_t T_S = 0, T_DP = 128, T_DV = 256, T_DK = 320, T_DQ = 384;

  // 640 threads start with 96 registers each (the 20-warp allocation granule). The element-wise phase wants
  // 64 raw values + ~40 of state per thread: the control warpgroup hands registers over to the compute warpgroups.
  if (warp >= 16) {
  reg_dealloc<kBwdCtrlRegs>();
  if (warp == 16) {
    // ======================= issuer: TMA loads and MMAs, one lane ==============================
    if (lane == 0) {
      const uint32_t idesc_s = umma_idesc_bf16(kTile, kTile, false, false);    // Q K^T, dO V^T
      const uint32_t idesc_t = umma_idesc_bf16(kTile, kDh, true, true);        // X^T Y (dV, dK)
      const uint32_t idesc_q = umma_idesc_bf16(kTile, kDh, false, true);       // dS K
      auto load_q = [&](int item, int i) {      // Q_i, dO_i of `item` -> slot i
        const int b = item / p.H, h = item % p.H;
        mbar_arrive_expect_tx(bar_q + i, 2 * kTileBytes);
        tma_load_2d(sQ + static_cast<size_t>(i) * kTileBytes, &tmQKV, bar_q + i, h * kDh, b * p.L + i * kTile);
        tma_load_2d(sDO + static_cast<size_t>(i) * kTileBytes, &tmDO, bar_q + i, h * kDh, b * p.L + i * kTile);
      };
      auto load_kv = [&](int item, int j) {     // K_j, V_j of `item` -> slot j
        const int b = item / p.H, h = item % p.H;
        mbar_arrive_expect_tx(bar_kv + j, 2 * kTileBytes);
        tma_load_2d(sK + static_cast<size_t>(j) * kTileBytes, &tmQKV, bar_kv + j, D + h * kDh, b * p.L + j * kTile);
        tma_load_2d(sV + static_cast<size_t>(j) * kTileBytes, &tmQKV, bar_kv + j, 2 * D + h * kDh, b * p.L + j * kTile);
      };
      // Descriptors are formed once per tile; a k-step only adds its byte offset (>> 4) to the start-address
      // field (shared-memory addresses < 256 KB: the 14-bit field cannot carry). The issue loop of the 24
      // accumulator MMAs is on the critical path of every iteration: ~8 instead of ~14 instructions per MMA.
      auto issue_mm1 = [&](int j, int i) {      // S = Q_i K_j^T, dP = dO_i V_j^T
        const uint64_t dq = umma_desc_kmajor(smem_u32(sQ + static_cast<size_t>(i) * kTileBytes));
        const uint64_t dd = umma_desc_kmajor(smem_u32(sDO + static_cast<size_t>(i) * kTileBytes));
        const uint64_t dk = umma_desc_kmajor(smem_u32(sK + static_cast<size_t>(j) * kTileBytes));
        const uint64_t dv = umma_desc_kmajor(smem_u32(sV + static_cast<size_t>(j) * kTileBytes));
#pragma unroll
        for (int k = 0; k < kDh / 16; ++k)
          umma_bf16(tmem_base + T_S, dq + (k * 32 >> 4), dk + (k * 32 >> 4), idesc_s, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < kDh / 16; ++k)
          umma_bf16(tmem_base + T_DP, dd + (k * 32 >> 4), dv + (k * 32 >> 4), idesc_s, k > 0 ? 1u : 0u);
        umma_commit(bar_mm1);
      };
      auto issue_mm2 = [&](int j, int i) {
        const uint64_t dpd = umma_desc_mnmajor(smem_u32(sPd), kTileBytes);
        const uint64_t dds = umma_desc_mnmajor(smem_u32(sDS), kTileBytes);
        const uint64_t ddsk = umma_desc_kmajor(smem_u32(sDS));
        const uint64_t dq = umma_desc_mnmajor(smem_u32(sQ + static_cast<size_t>(i) * kTileBytes), kTileBytes);
        const uint64_t dd = umma_desc_mnmajor(smem_u32(sDO + static_cast<size_t>(i) * kTileBytes), kTileBytes);
        const uint64_t dk = umma_desc_mnmajor(smem_u32(sK + static_cast<size_t>(j) * kTileBytes), kTileBytes);
        const uint32_t acc_kv = i > j ? 1u : 0u;   // first query tile of a key tile starts dV_j / dK_j
        const uint32_t acc_q = j > 0 ? 1u : 0u;    // key tile 0 starts dQ_i
#pragma unroll
        for (int k = 0; k < kTile / 16; ++k)   // dV_j += Pd^T dO_i
          umma_bf16(tmem_base + T_DV, dpd + (k * 2048 >> 4), dd + (k * 2048 >> 4), idesc_t, (acc_kv || k > 0) ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < kTile / 16; ++k)   // dK_j += dS^T Q_i
          umma_bf16(tmem_base + T_DK, dds + (k * 2048 >> 4), dq + (k * 2048 >> 4), idesc_t, (acc_kv || k > 0) ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < kTile / 16; ++k)   // dQ_i += dS K_j (A K-major: 64-column chunk k/4, 32 B per k-step inside)
          umma_bf16(tmem_base + T_DQ + i * kDh, ddsk + (((k >> 2) * kTileBytes + (k & 3) * 32) >> 4),
                    dk + (k * 2048 >> 4), idesc_q, (acc_q || k > 0) ? 1u : 0u);
        umma_commit(bar_mm2);
      };

      int item = blockIdx.x;
      if (item < n_items) {
        load_q(item, 0);
        load_kv(item, 0);
        if (nq == 2) {
          load_q(item, 1);
          load_kv(item, 1);
        }
        mbar_wait(bar_q + 0, 0);
        mbar_wait(bar_kv + 0, 0);
        tc_fence_after();
        issue_mm1(0, 0);
      }
      uint32_t g = 0;
      for (uint32_t n = 0; item < n_items; ++n, item += gridDim.x) {
        const int next = item + static_cast<int>(gridDim.x);
        const bool has_next = next < n_items;
        const uint32_t par = n & 1u, npar = (n + 1u) & 1u;
        for (int it = 0; it < niter; ++it, ++g) {
          const int j = it == 2 ? 1 : 0, i = it == 0 ? 0 : 1;
          mbar_wait(bar_drain, g & 1u);          // S/dP(g) sit in registers: their columns are free
          tc_fence_after();
          if (it + 1 < niter) {                   // next iteration of this item: (0,1) or (1,1)
            if (it == 0) mbar_wait(bar_q + 1, par); else mbar_wait(bar_kv + 1, par);
            tc_fence_after();
            issue_mm1(it == 0 ? 0 : 1, 1);
          }
          if (niter == 3 && it == 2 && has_next) {   // first iteration of the next item; its tiles were requested
            mbar_wait(bar_q + 0, npar);              // after iterations 0 and 1 of this item (K0/V0 about one
            mbar_wait(bar_kv + 0, npar);             // element-wise phase ago: the stage barrier below is later still)
            tc_fence_after();
            issue_mm1(0, 0);
          }
          mbar_wait(bar_stage, g & 1u);          // Pd / dS of g staged (and every earlier TMEM drain done)
          tc_fence_after();
          issue_mm2(j, i);
          if (niter == 3) {
            mbar_wait(bar_mm2, g & 1u);          // the slots this iteration read last are free now
            if (has_next) {
              if (it == 0) load_q(next, 0);
              else if (it == 1) load_kv(next, 0);
              else { load_q(next, 1); load_kv(next, 1); }
            }
          } else {
            mbar_wait(bar_mm2, g & 1u);
            if (has_next) {
              load_q(next, 0);
              load_kv(next, 0);
              mbar_wait(bar_q + 0, npar);
              mbar_wait(bar_kv + 0, npar);
              tc_fence_after();
              issue_mm1(0, 0);
            }
          }
        }
      }
    }
  } else {
    // ======================= warps 17-19: delta / lse of the item after the one being processed ====
    // (the first item's values are formed by the compute threads themselves, one position each: nothing else
    // for them to do at kernel start, and it takes one load round trip instead of three)
    int item = blockIdx.x + gridDim.x;
    for (uint32_t n = 1; item < n_items; ++n, item += gridDim.x) {
      const uint32_t bsel = n & 1u;
      if (n >= 2) mbar_wait(bar_dfree + bsel, ((n >> 1) - 1u) & 1u);
      const int b = item / p.H, h = item % p.H;
      const int seq_row0 = b * p.L;
      for (int pos = (warp - 17) * 32 + lane; pos < nq * kTile; pos += 96) {
        float delta = 0.f, lse2 = 0.f;
        if (pos < p.L) {
          const uint4* o = reinterpret_cast<const uint4*>(p.ctx + static_cast<size_t>(seq_row0 + pos) * D + h * kDh);
          const uint4* gq = reinterpret_cast<const uint4*>(p.dctx + static_cast<size_t>(seq_row0 + pos) * D + h * kDh);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const uint4 a = __ldg(o + u), c = __ldg(gq + u);
            const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, cw[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              const float2 x = unpack_bf16(aw[w]), y = unpack_bf16(cw[w]);
              delta += x.x * y.x + x.y * y.y;
            }
          }
          lse2 = p.lse[static_cast<size_t>(item) * p.L + pos] * kLog2e;
        }
        sDelta[bsel * 2 * kTile + pos] = delta;
        sLse[bsel * 2 * kTile + pos] = lse2;
      }
      mbar_arrive(bar_dfull + bsel);
    }
  }
  } else {
    reg_alloc<kBwdComputeRegs>();
    // ======================= compute warps ====================================================
    const int q = warp & 3, grp = warp >> 2;   // TMEM lane quarter, 32-column chunk of the key tile
    const int row = q * 32 + lane;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float c1 = p.scale * kLog2e;
    const uint64_t seed = p.drop_seed + ((p.drop_thresh && p.drop_seed_dev) ? *p.drop_seed_dev : 0ull);
    const uint32_t dkey = drop_key(seed, p.drop_site);
    const int cg = grp;
    const int u0 = (cg & 1) * 4;
    uint8_t* pchunk = sPd + static_cast<size_t>(cg >> 1) * kTileBytes;
    uint8_t* dchunk = sDS + static_cast<size_t>(cg >> 1) * kTileBytes;
    // Key tile j of `ditem` complete: dK_j, dV_j TMEM -> dqkv (warp groups 0,1: the two 32-column halves of dK;
    // 2,3: of dV); with_dq: the item is complete, dQ_i -> dqkv (groups (0,1) take tile 0, (2,3) tile 1).
    // Called one iteration AFTER the MMAs were issued, so their completion barrier has long flipped.
    auto drain = [&](int ditem, int j, bool with_dq) {
      __syncwarp();
      tc_fence_after();
      const int b = ditem / p.H, h = ditem % p.H;
      const int hf = grp & 1;
      const int pos = j * kTile + row;
      __nv_bfloat16* base = p.dqkv + static_cast<size_t>(b * p.L) * (3 * D) + h * kDh + hf * 32;
      uint32_t r[32];
      tmem_ld32(lane_base + (grp < 2 ? T_DK : T_DV) + hf * 32, r);
      tmem_ld_wait();
      if (pos < p.L) store_row32_bf16(base + static_cast<size_t>(pos) * (3 * D) + (grp < 2 ? D : 2 * D), r);
      const int qi = grp >> 1;
      if (with_dq && qi < nq) {
        const int qpos = qi * kTile + row;
        tmem_ld32(lane_base + T_DQ + qi * kDh + hf * 32, r);
        tmem_ld_wait();
        if (qpos < p.L) store_row32_bf16(base + static_cast<size_t>(qpos) * (3 * D), r);
      }
      tc_fence_before();
    };
    uint32_t g = 0;
    int item = blockIdx.x;
    if (tid < nq * kTile) {   // delta / lse of this CTA's first item
      const int b = item / p.H, h = item % p.H;
      float delta = 0.f, lse2 = 0.f;
      if (tid < p.L) {
        const uint4* o = reinterpret_cast<const uint4*>(p.ctx + static_cast<size_t>(b * p.L + tid) * D + h * kDh);
        const uint4* gq = reinterpret_cast<const uint4*>(p.dctx + static_cast<size_t>(b * p.L + tid) * D + h * kDh);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const uint4 a = __ldg(o + u), c = __ldg(gq + u);
          const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, cw[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const float2 x = unpack_bf16(aw[w]), y = unpack_bf16(cw[w]);
            delta += x.x * y.x + x.y * y.y;
          }
        }
        lse2 = p.lse[static_cast<size_t>(item) * p.L + tid] * kLog2e;
      }
      sDelta[tid] = delta;
      sLse[tid] = lse2;
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kBwdComputeThreads) : "memory");
    for (uint32_t n = 0; item < n_items; ++n, item += gridDim.x) {
      const uint32_t bsel = n & 1u;
      // buffer 1 is filled for items 1, 3, ... (completion n >> 1), buffer 0 for items 2, 4, ... ((n >> 1) - 1)
      if (n > 0) mbar_wait(bar_dfull + bsel, ((n >> 1) - (bsel ? 0u : 1u)) & 1u);
      for (int it = 0; it < niter; ++it, ++g) {
        const int j = it == 2 ? 1 : 0, i = it == 0 ? 0 : 1;
        const int q_pos = i * kTile + row;
        const float lse2 = sLse[bsel * 2 * kTile + q_pos];
        const float delta = sDelta[bsel * 2 * kTile + q_pos];
        if (it == niter - 1) mbar_arrive(bar_dfree + bsel);   // last read of this buffer
        const bool diag = (i == j);
        const bool row_ok = q_pos < p.L;
        // inactive (warp-uniform): above the diagonal, or all 32 query rows / all 32 key columns beyond the sequence
        const bool active = !(diag && cg > q) && (i * kTile + q * 32 < p.L) && (j * kTile + cg * 32 < p.L);
        // the dropout decisions of this thread's 32 elements do not depend on S / dP: formed while the MMAs run
        const int kv0 = j * kTile + cg * 32;
        uint32_t keepmask = 0xFFFFFFFFu;
        if (active && p.drop_thresh) {
          const uint32_t didx0 = (static_cast<uint32_t>(item) * p.L + q_pos) * p.L + kv0;
          keepmask = 0u;
          if ((didx0 & 3u) == 0u) {
#pragma unroll
            for (int t = 0; t < 32; t += 4) {
              bool k[4];
              drop_keep_quad(dkey, didx0 + t, p.drop_thresh, k);
#pragma unroll
              for (int e = 0; e < 4; ++e) keepmask |= (k[e] ? 1u : 0u) << (t + e);
            }
          } else if ((didx0 & 1u) == 0u) {
#pragma unroll
            for (int t = 0; t < 32; t += 2) {
              bool k0, k1;
              drop_keep_pair(dkey, didx0 + t, p.drop_thresh, k0, k1);
              keepmask |= (k0 ? 1u : 0u) << t;
              keepmask |= (k1 ? 1u : 0u) << (t + 1);
            }
          } else {
#pragma unroll
            for (int t = 0; t < 32; ++t)
              keepmask |= (drop_keep_k(dkey, didx0 + t, p.drop_thresh) ? 1u : 0u) << t;
          }
        }
        mbar_wait(bar_mm1, g & 1u);
        __syncwarp();
        tc_fence_after();
        // Two halves of 16 columns: 32 raw registers live instead of 64 (the element-wise phase also carries the
        // 32 packed results and ~30 registers of state; 64 raw ones spilled). S / dP are released to the MMAs of
        // the next iteration once the second half sits in registers, i.e. after half of the arithmetic.
        uint4 vp[4], vd[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) vp[u] = vd[u] = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          uint32_t rs[16], rp[16];
          if (active) {
            tmem_ld16(lane_base + T_S + cg * 32 + half * 16, rs);
            tmem_ld16(lane_base + T_DP + cg * 32 + half * 16, rp);
            tmem_ld_wait();
          }
          if (half == 1) {
            tc_fence_before();
            mbar_arrive(bar_drain);
          }
          if (active) {
#pragma unroll
            for (int uu = 0; uu < 2; ++uu) {
              const int u = half * 2 + uu;
              float pd[8], ds[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int t = u * 8 + e;
                float pr = fast_exp2(__uint_as_float(rs[uu * 8 + e]) * c1 - lse2);
                if ((diag && kv0 + t > q_pos) || !row_ok) pr = 0.f;
                const bool keep = (keepmask >> t) & 1u;
                const float dp = keep ? __uint_as_float(rp[uu * 8 + e]) * p.drop_scale : 0.f;
                pd[e] = keep ? pr * p.drop_scale : 0.f;
                ds[e] = pr * (dp - delta) * p.scale;
              }
              vp[u].x = pack_bf16(pd[0], pd[1]);
              vp[u].y = pack_bf16(pd[2], pd[3]);
              vp[u].z = pack_bf16(pd[4], pd[5]);
              vp[u].w = pack_bf16(pd[6], pd[7]);
              vd[u].x = pack_bf16(ds[0], ds[1]);
              vd[u].y = pack_bf16(ds[2], ds[3]);
              vd[u].z = pack_bf16(ds[4], ds[5]);
              vd[u].w = pack_bf16(ds[6], ds[7]);
            }
          }
        }
        // The previous iteration's MMAs no longer read Pd / dS; this wait is also what the deferred drain of
        // their dK/dV/dQ accumulators needs. It was issued a whole element-wise phase ago: no stall.
        if (g > 0) {
          mbar_wait(bar_mm2, (g - 1u) & 1u);
          if (it != 1) drain(it == 0 ? item - static_cast<int>(gridDim.x) : item, (niter == 3 && it == 0) ? 1 : 0, it == 0);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          st_swizzled_unit(pchunk, row, u0 + u, vp[u]);
          st_swizzled_unit(dchunk, row, u0 + u, vd[u]);
        }
        fence_proxy_async_smem();
        mbar_arrive(bar_stage);
      }
    }
    if (g > 0) {   // the last item's key tile nq-1 and its dQ
      mbar_wait(bar_mm2, (g - 1u) & 1u);
      drain(item - static_cast<int>(gridDim.x), nq - 1, true);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_dealloc(tmem_base, 512);
}

// ============================================================================================
// Long histories, 512 < L <= 4096. The kernels above keep every S tile (forward) or every dQ accumulator (backward)
// of a sequence in TMEM, which caps L at 512. The kernels below walk the key / query tiles of one 128-row tile with
// TMEM and shared memory that do not depend on L. Dropout hashes the 64-bit element index ((b*H + h)*L + q)*L + k
// (B*H*L^2 passes 2^32 from B = 65 at L = 4096), exactly as drop_keep_k and the single-query kernels do.
// ============================================================================================
static constexpr int kLongMaxL = 4096;

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}

// drop_keepmask32 for a 64-bit element index
__device__ __forceinline__ uint32_t drop_keepmask32_64(uint32_t dkey, uint64_t didx0, uint32_t thresh) {
  uint32_t keepmask = 0u;
  if ((didx0 & 3u) == 0u) {
#pragma unroll
    for (int t = 0; t < 32; t += 4) {
      bool k[4];
      drop_keep_quad64(dkey, didx0 + t, thresh, k);
#pragma unroll
      for (int e = 0; e < 4; ++e) keepmask |= (k[e] ? 1u : 0u) << (t + e);
    }
  } else if ((didx0 & 1u) == 0u) {
#pragma unroll
    for (int t = 0; t < 32; t += 2) {
      bool k0, k1;
      drop_keep_pair64(dkey, didx0 + t, thresh, k0, k1);
      keepmask |= (k0 ? 1u : 0u) << t;
      keepmask |= (k1 ? 1u : 0u) << (t + 1);
    }
  } else {
#pragma unroll
    for (int t = 0; t < 32; ++t) keepmask |= (drop_keep_k(dkey, didx0 + t, thresh) ? 1u : 0u) << t;
  }
  return keepmask;
}

// Forward, L > 512. One CTA (256 threads) per (sequence, head, 128-row query tile), heavy tiles first; thread (row,
// hf) as in attn_fwd_kernel. Online softmax over the key tiles j = 0..qt:
//   S_j = Q K_j^T -> TMEM columns [0, 128); the row max of S_j raises the running max m;
//   P_j = dropout(exp2((S_j - m) * scale * log2e)) -> bf16, 128B-swizzled smem tile; O_j = P_j V_j -> TMEM columns
//   [128, 192), a fresh accumulator per tile;
//   O_{j-1} is folded into the thread's 32 output columns in registers (O = O * exp2((m_old - m_new) * c) + O_{j-1})
//   while S_{j+1} and P_j V_j are under way.
// TMEM: 256 columns. Shared memory: Q, K, V[2], P (two 64-column chunks) = 96 KB. Two CTAs per SM. K_{j+1} is
// requested once S_j has retired, V_{j+1} once P_{j-1} V_{j-1} has.
__global__ void __launch_bounds__(256, 2)
attn_fwd_long_kernel(const __grid_constant__ CUtensorMap tmQKV, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hf = warp >> 2;
  const int row = q * 32 + lane;
  const int bh_count = p.B * p.H;
  const int qt = p.nq - 1 - static_cast<int>(blockIdx.x) / bh_count;  // heavy tiles first
  const int bh = static_cast<int>(blockIdx.x) % bh_count;
  const int b = bh / p.H, h = bh % p.H;
  const int n_kv = qt + 1;
  const int D = p.H * kDh;
  constexpr uint32_t kCols = 256, T_O = 128;

  uint8_t* sQ = smem;
  uint8_t* sK = sQ + kTileBytes;
  uint8_t* sV = sK + kTileBytes;          // [2]
  uint8_t* sP = sV + 2 * kTileBytes;      // 2 chunks
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * kTileBytes);
  uint64_t* bar_k = bars + 0;    // Q + K_0, then K_j: phase j
  uint64_t* bar_v = bars + 1;    // [2] V slot j & 1: phase j >> 1
  uint64_t* bar_s = bars + 3;    // S_j retired: phase j
  uint64_t* bar_pv = bars + 4;   // P_j V_j retired: phase j
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
  float* s_red = reinterpret_cast<float*>(bars + 6);  // [2][128]

  if (tid == 0) {
    tma_prefetch_desc(&tmQKV);
    for (int i = 0; i < 5; ++i) mbar_init(bars + i, 1);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) {
    tmem_alloc(tmem_slot, kCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  const int seq_row0 = b * p.L;
  const uint32_t idesc_s = umma_idesc_bf16(kTile, kTile, false, false);
  const uint32_t idesc_pv = umma_idesc_bf16(kTile, kDh, false, true);
  const uint64_t q_desc = umma_desc_kmajor(smem_u32(sQ));
  const uint64_t k_desc = umma_desc_kmajor(smem_u32(sK));
  auto issue_s = [&]() {
#pragma unroll
    for (int k = 0; k < kDh / 16; ++k)
      umma_bf16(tmem_base, q_desc + (k * 32 >> 4), k_desc + (k * 32 >> 4), idesc_s, k > 0 ? 1u : 0u);
    umma_commit(bar_s);
  };
  auto load_v = [&](int j) {
    mbar_arrive_expect_tx(bar_v + (j & 1), kTileBytes);
    tma_load_2d(sV + static_cast<size_t>(j & 1) * kTileBytes, &tmQKV, bar_v + (j & 1), 2 * D + h * kDh,
                seq_row0 + j * kTile);
  };
  if (tid == 0) {
    mbar_arrive_expect_tx(bar_k, 2 * kTileBytes);
    tma_load_2d(sQ, &tmQKV, bar_k, h * kDh, seq_row0 + qt * kTile);
    tma_load_2d(sK, &tmQKV, bar_k, D + h * kDh, seq_row0);
    load_v(0);
    if (n_kv > 1) load_v(1);
    mbar_wait(bar_k, 0);
    tc_fence_after();
    issue_s();
  }

  const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  const int q_pos = qt * kTile + row;
  const bool dead_rows = qt * kTile + q * 32 >= p.L;   // warp-uniform: all 32 rows beyond the sequence
  const float c1 = p.scale * kLog2e;
  const uint64_t seed = p.drop_seed + ((p.drop_thresh && p.drop_seed_dev) ? *p.drop_seed_dev : 0ull);
  const uint32_t dkey = drop_key(seed, p.drop_site);
  const uint64_t didx_row = (static_cast<uint64_t>(bh) * p.L + q_pos) * p.L;
  uint8_t* chunk = sP + static_cast<size_t>(hf) * kTileBytes;
  float m = -INFINITY;      // running row max of the raw scores
  float l = 0.f;            // this thread's half of the row sum, relative to m
  float m_o = -INFINITY;    // the max that o[] is relative to
  float o[32];
#pragma unroll
  for (int t = 0; t < 32; ++t) o[t] = 0.f;
  // o = o * exp2((m_o - m_new) * c1) + (the thread's 32 columns of P_{j} V_{j}, relative to m_new)
  auto fold = [&](float m_new) {
    uint32_t r[32];
    tmem_ld32(lane_base + T_O + hf * 32, r);
    tmem_ld_wait();
    const float a = fast_exp2((m_o - m_new) * c1);
#pragma unroll
    for (int t = 0; t < 32; ++t) o[t] = fmaf(o[t], a, __uint_as_float(r[t]));
    m_o = m_new;
  };

  for (int j = 0; j < n_kv; ++j) {
    const bool diag = (j == qt);
    mbar_wait(bar_s, j & 1);
    __syncwarp();
    tc_fence_after();
    if (tid == 0 && j + 1 < n_kv) {   // S_j retired: the K slot is free
      mbar_arrive_expect_tx(bar_k, kTileBytes);
      tma_load_2d(sK, &tmQKV, bar_k, D + h * kDh, seq_row0 + (j + 1) * kTile);
    }
    // ---- row max of S_j (each thread: its column half) ----
    float mt = -INFINITY;
    if (!dead_rows) {
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int cg = 2 * hf + cc;
        const int kv0 = j * kTile + cg * 32;
        if ((diag && cg > q) || kv0 >= p.L) continue;
        uint32_t r[32];
        tmem_ld32(lane_base + cg * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int t = 0; t < 32; ++t)
          if (!diag || kv0 + t <= q_pos) mt = fmaxf(mt, __uint_as_float(r[t]));
      }
    }
    s_red[hf * 128 + row] = mt;
    __syncthreads();
    const float m_prev = m;
    m = fmaxf(m, fmaxf(s_red[row], s_red[128 + row]));
    // ---- P_{j-1} V_{j-1} retired: fold it in; the P tile and its V slot are free ----
    if (j >= 1) {
      mbar_wait(bar_pv, (j - 1) & 1);
      __syncwarp();
      tc_fence_after();
      if (!dead_rows) fold(m_prev);
    }
    const float mc = m * c1;
    if (!dead_rows) l *= fast_exp2((m_prev - m) * c1);
    // ---- P_j -> shared memory ----
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      const int cg = 2 * hf + cc;
      const int u0 = cc * 4;
      const int kv0 = j * kTile + cg * 32;
      if (!((diag && cg > q) || dead_rows || kv0 >= p.L)) {
        uint32_t r[32];
        tmem_ld32(lane_base + cg * 32, r);
        tmem_ld_wait();
        const uint32_t keep = p.drop_thresh ? drop_keepmask32_64(dkey, didx_row + kv0, p.drop_thresh) : 0xFFFFFFFFu;
        float pv[32];
#pragma unroll
        for (int t = 0; t < 32; ++t) {
          float e = fast_exp2(__uint_as_float(r[t]) * c1 - mc);
          if (diag && kv0 + t > q_pos) e = 0.f;
          l += e;
          pv[t] = ((keep >> t) & 1u) ? e * p.drop_scale : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint4 v;
          v.x = pack_bf16(pv[u * 8 + 0], pv[u * 8 + 1]);
          v.y = pack_bf16(pv[u * 8 + 2], pv[u * 8 + 3]);
          v.z = pack_bf16(pv[u * 8 + 4], pv[u * 8 + 5]);
          v.w = pack_bf16(pv[u * 8 + 6], pv[u * 8 + 7]);
          st_swizzled_unit(chunk, row, u0 + u, v);
        }
      } else {
#pragma unroll
        for (int u = 0; u < 4; ++u) st_swizzled_unit(chunk, row, u0 + u, make_uint4(0, 0, 0, 0));
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      if (j + 1 < n_kv) {
        mbar_wait(bar_k, (j + 1) & 1);
        tc_fence_after();
        issue_s();
        if (j >= 1) load_v(j + 1);   // P_{j-1} V_{j-1} retired: slot (j + 1) & 1 is free
      }
      mbar_wait(bar_v + (j & 1), (j >> 1) & 1);
      tc_fence_after();
      const uint64_t p_desc = umma_desc_kmajor(smem_u32(sP));
      const uint64_t v_desc = umma_desc_mnmajor(smem_u32(sV + static_cast<size_t>(j & 1) * kTileBytes), kTileBytes);
#pragma unroll
      for (int k = 0; k < kTile / 16; ++k)
        umma_bf16(tmem_base + T_O, p_desc + (((k >> 2) * kTileBytes + (k & 3) * 32) >> 4), v_desc + (k * 2048 >> 4),
                  idesc_pv, k > 0 ? 1u : 0u);
      umma_commit(bar_pv);
    }
  }

  // ---- epilogue: O / l -> ctx, log-sum-exp -> lse ----
  mbar_wait(bar_pv, (n_kv - 1) & 1);
  __syncwarp();
  tc_fence_after();
  if (!dead_rows) fold(m);
  s_red[hf * 128 + row] = l;
  __syncthreads();
  l = s_red[row] + s_red[128 + row];
  if (q_pos < p.L) {
    const float inv_l = 1.f / l;
    uint32_t r[32];
#pragma unroll
    for (int t = 0; t < 32; ++t) r[t] = __float_as_uint(o[t] * inv_l);
    store_row32_bf16(p.ctx + static_cast<size_t>(seq_row0 + q_pos) * D + h * kDh + hf * 32, r);
    if (hf == 0 && p.lse) p.lse[static_cast<size_t>(bh) * p.L + q_pos] = m * p.scale + __logf(l);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, kCols);
}

// Backward, L > 512: two kernels, no atomics, so dqkv is the same bit for bit from run to run.
//   DQ = false: one CTA per (sequence, head, key tile j) walks the query tiles i = j..nq-1 and accumulates dV_j, dK_j;
//   DQ = true:  one CTA per (sequence, head, query tile i) walks the key tiles j = 0..i and accumulates dQ_i.
// Both recompute S = Q_i K_j^T and dP = dO_i V_j^T and form P, Pd and dS exactly as attn_bwd_kernel does, so the two
// halves of the gradient see the same dS. The tile of the CTA (K_j / V_j, or Q_i / dO_i) stays in shared memory, the
// walked tiles stream through two slots. Warp roles as in attn_bwd_persist_kernel:
//   * warps 0-15: the element-wise phase, thread (row, 32-column chunk); they arrive at bar_drain once S / dP of the
//     iteration sit in registers, so the next iteration's S / dP MMAs run under the element-wise phase;
//   * warp 16, one lane: TMA loads and MMAs;
//   * warp 17: delta_i = rowsum(dO_i * O_i) and the log-sum-exps of the coming query tile, double-buffered (DQ: once,
//     the query tile is fixed). O_i arrives by TMA with the walked dO_i (DQ: with the CTA's own tiles), so delta is
//     formed from shared memory.
// TMEM: S [0,128), dP [128,256), accumulators [256,384); 512 allocated, one CTA per SM.
static constexpr int kLongBwdThreads = kBwdComputeThreads + 64;

template <bool DQ>
__global__ void __launch_bounds__(kLongBwdThreads, 1)
attn_bwd_long_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                     const __grid_constant__ CUtensorMap tmO, const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int D = p.H * kDh;
  const int bh_count = p.B * p.H;
  const int tile = DQ ? p.nq - 1 - static_cast<int>(blockIdx.x) / bh_count   // heavy tiles first
                      : static_cast<int>(blockIdx.x) / bh_count;
  const int bh = static_cast<int>(blockIdx.x) % bh_count;
  const int b = bh / p.H, h = bh % p.H;
  const int n_it = DQ ? tile + 1 : p.nq - tile;
  const int seq_row0 = b * p.L;
  // iteration it: query tile i, key tile j
  auto qtile = [&](int it) { return DQ ? tile : tile + it; };
  auto ktile = [&](int it) { return DQ ? it : tile; };

  uint8_t* sF = smem;                        // [2] the CTA's own tiles: K_j, V_j (DQ: Q_i, dO_i)
  uint8_t* sX = sF + 2 * kTileBytes;         // [2 slots] walked Q_i (DQ: K_j)
  uint8_t* sY = sX + 2 * kTileBytes;         // [2 slots] walked dO_i (DQ: V_j)
  uint8_t* sDS = sY + 2 * kTileBytes;        // 2 chunks
  uint8_t* sPd = sDS + 2 * kTileBytes;       // 2 chunks (not DQ)
  uint8_t* sO = sPd + (DQ ? 0 : 2) * kTileBytes;   // [2 slots] O_i of the walked query tiles (DQ: [1], the own one)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sO + (DQ ? 1 : 2) * kTileBytes);
  uint64_t* bar_fix = bars + 0;    // own tiles landed
  uint64_t* bar_ld = bars + 1;     // [2] slot it & 1 landed: phase it >> 1
  uint64_t* bar_mm1 = bars + 3;    // S / dP of iteration it ready
  uint64_t* bar_drain = bars + 4;  // every compute thread holds S / dP of iteration it
  uint64_t* bar_stage = bars + 5;  // Pd / dS of iteration it staged
  uint64_t* bar_mm2 = bars + 6;    // accumulator MMAs of iteration it retired
  uint64_t* bar_dfull = bars + 7;  // [2] delta / lse buffer filled
  uint64_t* bar_dfree = bars + 9;  // [2] delta / lse buffer read
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 11);
  float* sDelta = reinterpret_cast<float*>(bars + 12);  // [2][128]
  float* sLse = sDelta + 2 * kTile;                     // [2][128], times log2e

  if (tid == 0) {
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 4; ++i) mbar_init(bars + i, 1);
    mbar_init(bar_drain, kBwdComputeThreads);
    mbar_init(bar_stage, kBwdComputeThreads);
    mbar_init(bar_mm2, 1);
    mbar_init(bar_dfull + 0, 32);
    mbar_init(bar_dfull + 1, 32);
    mbar_init(bar_dfree + 0, kBwdComputeThreads);
    mbar_init(bar_dfree + 1, kBwdComputeThreads);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 16) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();
  constexpr uint32_t T_S = 0, T_DP = 128, T_ACC = 256;   // dV_j | dK_j, or dQ_i

  if (warp >= 16) {
    if (warp == 16) {
      // ======================= issuer: TMA loads and MMAs, one lane ==============================
      if (lane == 0) {
        const uint32_t idesc_s = umma_idesc_bf16(kTile, kTile, false, false);    // Q K^T, dO V^T
        const uint32_t idesc_t = umma_idesc_bf16(kTile, kDh, true, true);        // X^T Y (dV, dK)
        const uint32_t idesc_q = umma_idesc_bf16(kTile, kDh, false, true);       // dS K
        auto load_walk = [&](int it) {
          const int s = it & 1;
          mbar_arrive_expect_tx(bar_ld + s, (DQ ? 2 : 3) * kTileBytes);
          if (DQ) {
            const int j = ktile(it);
            tma_load_2d(sX + static_cast<size_t>(s) * kTileBytes, &tmQKV, bar_ld + s, D + h * kDh, seq_row0 + j * kTile);
            tma_load_2d(sY + static_cast<size_t>(s) * kTileBytes, &tmQKV, bar_ld + s, 2 * D + h * kDh, seq_row0 + j * kTile);
          } else {
            const int i = qtile(it);
            tma_load_2d(sX + static_cast<size_t>(s) * kTileBytes, &tmQKV, bar_ld + s, h * kDh, seq_row0 + i * kTile);
            tma_load_2d(sY + static_cast<size_t>(s) * kTileBytes, &tmDO, bar_ld + s, h * kDh, seq_row0 + i * kTile);
            tma_load_2d(sO + static_cast<size_t>(s) * kTileBytes, &tmO, bar_ld + s, h * kDh, seq_row0 + i * kTile);
          }
        };
        mbar_arrive_expect_tx(bar_fix, (DQ ? 3 : 2) * kTileBytes);
        if (DQ) {
          tma_load_2d(sF, &tmQKV, bar_fix, h * kDh, seq_row0 + tile * kTile);
          tma_load_2d(sF + kTileBytes, &tmDO, bar_fix, h * kDh, seq_row0 + tile * kTile);
          tma_load_2d(sO, &tmO, bar_fix, h * kDh, seq_row0 + tile * kTile);
        } else {
          tma_load_2d(sF, &tmQKV, bar_fix, D + h * kDh, seq_row0 + tile * kTile);
          tma_load_2d(sF + kTileBytes, &tmQKV, bar_fix, 2 * D + h * kDh, seq_row0 + tile * kTile);
        }
        load_walk(0);
        if (n_it > 1) load_walk(1);
        // Q, dO, K, V of iteration it (slot it & 1)
        auto tq = [&](int it) { return smem_u32(DQ ? sF : sX + static_cast<size_t>(it & 1) * kTileBytes); };
        auto tdo = [&](int it) { return smem_u32(DQ ? sF + kTileBytes : sY + static_cast<size_t>(it & 1) * kTileBytes); };
        auto tk = [&](int it) { return smem_u32(DQ ? sX + static_cast<size_t>(it & 1) * kTileBytes : sF); };
        auto tv = [&](int it) { return smem_u32(DQ ? sY + static_cast<size_t>(it & 1) * kTileBytes : sF + kTileBytes); };
        auto issue_mm1 = [&](int it) {
          const uint64_t dq = umma_desc_kmajor(tq(it)), dd = umma_desc_kmajor(tdo(it));
          const uint64_t dk = umma_desc_kmajor(tk(it)), dv = umma_desc_kmajor(tv(it));
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k)
            umma_bf16(tmem_base + T_S, dq + (k * 32 >> 4), dk + (k * 32 >> 4), idesc_s, k > 0 ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k)
            umma_bf16(tmem_base + T_DP, dd + (k * 32 >> 4), dv + (k * 32 >> 4), idesc_s, k > 0 ? 1u : 0u);
          umma_commit(bar_mm1);
        };
        auto issue_mm2 = [&](int it) {
          const uint32_t acc = it > 0 ? 1u : 0u;
          if (DQ) {
            const uint64_t ddsk = umma_desc_kmajor(smem_u32(sDS));
            const uint64_t dk = umma_desc_mnmajor(tk(it), kTileBytes);
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)   // dQ_i += dS K_j
              umma_bf16(tmem_base + T_ACC, ddsk + (((k >> 2) * kTileBytes + (k & 3) * 32) >> 4), dk + (k * 2048 >> 4),
                        idesc_q, (acc || k > 0) ? 1u : 0u);
          } else {
            const uint64_t dpd = umma_desc_mnmajor(smem_u32(sPd), kTileBytes);
            const uint64_t dds = umma_desc_mnmajor(smem_u32(sDS), kTileBytes);
            const uint64_t dq = umma_desc_mnmajor(tq(it), kTileBytes);
            const uint64_t dd = umma_desc_mnmajor(tdo(it), kTileBytes);
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)   // dV_j += Pd^T dO_i
              umma_bf16(tmem_base + T_ACC, dpd + (k * 2048 >> 4), dd + (k * 2048 >> 4), idesc_t, (acc || k > 0) ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)   // dK_j += dS^T Q_i
              umma_bf16(tmem_base + T_ACC + kDh, dds + (k * 2048 >> 4), dq + (k * 2048 >> 4), idesc_t,
                        (acc || k > 0) ? 1u : 0u);
          }
          umma_commit(bar_mm2);
        };
        mbar_wait(bar_fix, 0);
        mbar_wait(bar_ld + 0, 0);
        tc_fence_after();
        issue_mm1(0);
        for (int it = 0; it < n_it; ++it) {
          mbar_wait(bar_drain, it & 1);          // S / dP(it) sit in registers: their columns are free
          tc_fence_after();
          if (it + 1 < n_it) {
            mbar_wait(bar_ld + ((it + 1) & 1), ((it + 1) >> 1) & 1);
            tc_fence_after();
            issue_mm1(it + 1);
          }
          mbar_wait(bar_stage, it & 1);
          tc_fence_after();
          issue_mm2(it);
          mbar_wait(bar_mm2, it & 1);            // slot it & 1 is read for the last time
          if (it + 2 < n_it) load_walk(it + 2);
        }
      }
    } else {
      // ======================= warp 17: delta / lse of the coming query tiles ====================
      const int n_fill = DQ ? 1 : n_it;
      for (int it = 0; it < n_fill; ++it) {
        const int s = it & 1;
        if (it >= 2) mbar_wait(bar_dfree + s, ((it >> 1) - 1) & 1);
        if (DQ) mbar_wait(bar_fix, 0);
        else mbar_wait(bar_ld + s, (it >> 1) & 1);
        const uint8_t* to = sO + static_cast<size_t>(DQ ? 0 : s) * kTileBytes;
        const uint8_t* tg = DQ ? sF + kTileBytes : sY + static_cast<size_t>(s) * kTileBytes;
        const int i = qtile(it);
        float lse[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int pos = i * kTile + lane + 32 * k;
          lse[k] = pos < p.L ? p.lse[static_cast<size_t>(bh) * p.L + pos] : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int r = lane + 32 * k;
          float delta = 0.f;
          if (i * kTile + r < p.L) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const int off = r * 128 + ((u ^ (r & 7)) << 4);
              const uint4 a = *reinterpret_cast<const uint4*>(to + off), c = *reinterpret_cast<const uint4*>(tg + off);
              const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, cw[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                const float2 x = unpack_bf16(aw[w]), y = unpack_bf16(cw[w]);
                delta += x.x * y.x + x.y * y.y;
              }
            }
          }
          sDelta[s * kTile + r] = delta;
          sLse[s * kTile + r] = lse[k] * kLog2e;
        }
        mbar_arrive(bar_dfull + s);
      }
    }
  } else {
    // ======================= compute warps ====================================================
    const int q = warp & 3, cg = warp >> 2;   // TMEM lane quarter, 32-column chunk of the key tile
    const int row = q * 32 + lane;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float c1 = p.scale * kLog2e;
    const uint64_t seed = p.drop_seed + ((p.drop_thresh && p.drop_seed_dev) ? *p.drop_seed_dev : 0ull);
    const uint32_t dkey = drop_key(seed, p.drop_site);
    const int u0 = (cg & 1) * 4;
    for (int it = 0; it < n_it; ++it) {
      const int i = qtile(it), j = ktile(it);
      const int s = DQ ? 0 : (it & 1);
      const int q_pos = i * kTile + row;
      const int kv0 = j * kTile + cg * 32;
      const bool diag = (i == j);
      const bool row_ok = q_pos < p.L;
      // inactive (warp-uniform): above the diagonal, or all 32 query rows / all 32 key columns beyond the sequence
      const bool active = !(diag && cg > q) && (i * kTile + q * 32 < p.L) && (kv0 < p.L);
      const uint32_t keepmask = (active && p.drop_thresh)
          ? drop_keepmask32_64(dkey, (static_cast<uint64_t>(bh) * p.L + q_pos) * p.L + kv0, p.drop_thresh)
          : 0xFFFFFFFFu;
      mbar_wait(bar_dfull + s, DQ ? 0u : static_cast<uint32_t>((it >> 1) & 1));
      const float lse2 = sLse[s * kTile + row];
      const float delta = sDelta[s * kTile + row];
      if (!DQ) mbar_arrive(bar_dfree + s);
      mbar_wait(bar_mm1, it & 1);
      __syncwarp();
      tc_fence_after();
      uint4 vp[4], vd[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) vp[u] = vd[u] = make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int u = 0; u < 4; ++u) {     // four 8-column quarters: 16 raw registers live
        uint32_t rs[8], rp[8];
        if (active) {
          tmem_ld8(lane_base + T_S + cg * 32 + u * 8, rs);
          tmem_ld8(lane_base + T_DP + cg * 32 + u * 8, rp);
          tmem_ld_wait();
        }
        if (u == 3) {
          tc_fence_before();
          mbar_arrive(bar_drain);
        }
        if (active) {
          {
            float pd[8], ds[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int t = u * 8 + e;
              float pr = fast_exp2(__uint_as_float(rs[e]) * c1 - lse2);
              if ((diag && kv0 + t > q_pos) || !row_ok) pr = 0.f;
              const bool keep = (keepmask >> t) & 1u;
              const float dp = keep ? __uint_as_float(rp[e]) * p.drop_scale : 0.f;
              pd[e] = keep ? pr * p.drop_scale : 0.f;
              ds[e] = pr * (dp - delta) * p.scale;
            }
            vp[u].x = pack_bf16(pd[0], pd[1]);
            vp[u].y = pack_bf16(pd[2], pd[3]);
            vp[u].z = pack_bf16(pd[4], pd[5]);
            vp[u].w = pack_bf16(pd[6], pd[7]);
            vd[u].x = pack_bf16(ds[0], ds[1]);
            vd[u].y = pack_bf16(ds[2], ds[3]);
            vd[u].z = pack_bf16(ds[4], ds[5]);
            vd[u].w = pack_bf16(ds[6], ds[7]);
          }
        }
      }
      if (it > 0) mbar_wait(bar_mm2, (it - 1) & 1);   // the previous MMAs no longer read Pd / dS
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (!DQ) st_swizzled_unit(sPd + (cg >> 1) * kTileBytes, row, u0 + u, vp[u]);
        st_swizzled_unit(sDS + (cg >> 1) * kTileBytes, row, u0 + u, vd[u]);
      }
      fence_proxy_async_smem();
      mbar_arrive(bar_stage);
    }
    // ---- accumulators complete: TMEM -> dqkv (groups 0,1: the two 32-column halves of dV_j / dQ_i; 2,3: of dK_j) ----
    mbar_wait(bar_mm2, (n_it - 1) & 1);
    __syncwarp();
    tc_fence_after();
    if (!DQ || cg < 2) {
      const int hf = cg & 1;
      const int pos = tile * kTile + row;
      uint32_t r[32];
      tmem_ld32(lane_base + T_ACC + (cg >> 1) * kDh + hf * 32, r);
      tmem_ld_wait();
      // dQ -> the Q third; dV_j (cg < 2) -> the V third, dK_j -> the K third
      const int third = DQ ? 0 : (cg < 2 ? 2 : 1);
      if (pos < p.L)
        store_row32_bf16(p.dqkv + static_cast<size_t>(seq_row0 + pos) * (3 * D) + third * D + h * kDh + hf * 32, r);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_dealloc(tmem_base, 512);
}

static int make_rows_map(CUtensorMap* m, const void* base, int rows, int cols) {
  uint64_t dims[2] = {static_cast<uint64_t>(cols), static_cast<uint64_t>(rows)};
  uint64_t str[1] = {static_cast<uint64_t>(cols) * 2};
  uint32_t box[2] = {kDh, kTile};
  return make_tmap_bf16(m, base, 2, dims, str, box);
}

static uint32_t drop_threshold(float p) {
  if (p <= 0.f) return 0;
  double t = static_cast<double>(p) * 4294967296.0;
  uint32_t v = t >= 4294967295.0 ? 4294967295u : static_cast<uint32_t>(t);
  return v == 0 ? 1 : v;
}

}  // namespace tt

extern "C" int tt_attn_causal_fwd(const void* qkv, void* ctx, float* lse, int B, int L, int H, float drop_p,
                                  uint64_t drop_seed, const uint64_t* drop_seed_dev, uint32_t drop_site,
                                  void* stream_) {
  using namespace tt;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(qkv && ctx, "tt_attn_causal_fwd: null pointer");
  TT_REQUIRE(B > 0 && L > 0 && H > 0, "tt_attn_causal_fwd: empty problem");
  TT_REQUIRE(L <= kLongMaxL, "tt_attn_causal_fwd: L=%d > %d unsupported", L, kLongMaxL);
  TT_REQUIRE(static_cast<int64_t>(B) * L <= INT32_MAX, "tt_attn_causal_fwd: B*L=%lld rows too many",
             static_cast<long long>(B) * L);
  TT_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "tt_attn_causal_fwd: drop_p out of range");
  const int D = H * kDh;
  AttnParams p;
  p.B = B; p.L = L; p.H = H;
  p.nq = (L + kTile - 1) / kTile;
  p.scale = 0.125f;
  p.drop_thresh = drop_threshold(drop_p);
  p.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  p.drop_seed = drop_seed;
  p.drop_seed_dev = drop_seed_dev;
  p.drop_site = drop_site;
  p.ctx = static_cast<__nv_bfloat16*>(ctx);
  p.lse = lse;
  CUtensorMap tm;
  int rc = make_rows_map(&tm, qkv, B * L, 3 * D);
  if (rc) return rc;
  if (L > 512) {
    const size_t lsmem = 1024 + 6 * static_cast<size_t>(kTileBytes) + 48 + 2 * 128 * sizeof(float);
    static bool lconfigured = false;
    if (!lconfigured) {
      TT_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lsmem));
      lconfigured = true;
    }
    TT_CHECK_CUDA(launch_k(attn_fwd_long_kernel, dim3(B * H * p.nq), dim3(256), lsmem, stream, tm, p));
    TT_LAUNCH_CHECK();
    return TT_OK;
  }
  const size_t smem = 1024 + static_cast<size_t>(1 + p.nq + 1 + 2) * kTileBytes + 64 + 2 * 128 * sizeof(float);
  static bool configured = false;
  if (!configured) {
    TT_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    configured = true;
  }
  TT_REQUIRE(smem <= 232448, "tt_attn_causal_fwd: shared memory %zu too large", smem);
  // TT_ATTN_FWD=legacy keeps the one-CTA-per-(sequence, head, query tile) kernel for L <= 256
  const char* mode = getenv("TT_ATTN_FWD");
  const bool legacy = mode && mode[0] == 'l';
  if (p.nq <= 2 && !legacy) {
    const size_t psmem = 1024 + 12 * static_cast<size_t>(kTileBytes) + 256 + 3 * 4 * kTile * sizeof(float);
    static bool pconfigured = false;
    if (!pconfigured) {
      TT_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
      pconfigured = true;
    }
    const int grid = B * H < num_sms() ? B * H : num_sms();
    TT_CHECK_CUDA(launch_k(attn_fwd_persist_kernel, dim3(grid), dim3(kFwdThreads), psmem, stream, tm, p));
    TT_LAUNCH_CHECK();
    return TT_OK;
  }
  TT_CHECK_CUDA(launch_k(attn_fwd_kernel, dim3(B * H * p.nq), dim3(256), smem, stream, tm, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_attn_causal_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse, void* dqkv,
                                  int B, int L, int H, float drop_p, uint64_t drop_seed,
                                  const uint64_t* drop_seed_dev, uint32_t drop_site, void* stream_) {
  using namespace tt;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(qkv && ctx && dctx && lse && dqkv, "tt_attn_causal_bwd: null pointer");
  TT_REQUIRE(B > 0 && L > 0 && H > 0, "tt_attn_causal_bwd: empty problem");
  TT_REQUIRE(L <= kLongMaxL, "tt_attn_causal_bwd: L=%d > %d unsupported", L, kLongMaxL);
  TT_REQUIRE(static_cast<int64_t>(B) * L <= INT32_MAX, "tt_attn_causal_bwd: B*L=%lld rows too many",
             static_cast<long long>(B) * L);
  const int D = H * kDh;
  AttnBwdParams p;
  p.B = B; p.L = L; p.H = H;
  p.nq = (L + kTile - 1) / kTile;
  p.scale = 0.125f;
  p.drop_thresh = drop_threshold(drop_p);
  p.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  p.drop_seed = drop_seed;
  p.drop_seed_dev = drop_seed_dev;
  p.drop_site = drop_site;
  p.ctx = static_cast<const __nv_bfloat16*>(ctx);
  p.dctx = static_cast<const __nv_bfloat16*>(dctx);
  p.lse = lse;
  p.dqkv = static_cast<__nv_bfloat16*>(dqkv);
  CUtensorMap tmQ, tmDO;
  int rc = make_rows_map(&tmQ, qkv, B * L, 3 * D);
  if (rc) return rc;
  rc = make_rows_map(&tmDO, dctx, B * L, D);
  if (rc) return rc;
  if (L > 512) {
    // dK / dV (a CTA per key tile) and dQ (a CTA per query tile): 12 and 9 tiles of shared memory
    const size_t ksmem = 1024 + 12 * static_cast<size_t>(kTileBytes) + 96 + 2 * 2 * kTile * sizeof(float);
    const size_t qsmem = ksmem - 3 * static_cast<size_t>(kTileBytes);
    CUtensorMap tmO;
    rc = make_rows_map(&tmO, ctx, B * L, D);
    if (rc) return rc;
    static bool lconfigured = false;
    if (!lconfigured) {
      TT_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_long_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ksmem));
      TT_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_long_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, qsmem));
      lconfigured = true;
    }
    const dim3 grid(B * H * p.nq);
    TT_CHECK_CUDA(launch_k(attn_bwd_long_kernel<false>, grid, dim3(kLongBwdThreads), ksmem, stream, tmQ, tmDO, tmO, p));
    TT_LAUNCH_CHECK();
    TT_CHECK_CUDA(launch_k(attn_bwd_long_kernel<true>, grid, dim3(kLongBwdThreads), qsmem, stream, tmQ, tmDO, tmO, p));
    TT_LAUNCH_CHECK();
    return TT_OK;
  }
  const int slots = p.nq <= 2 ? p.nq : 1;
  const size_t smem = 1024 + static_cast<size_t>(2 * slots + 2 + 4) * kTileBytes + 128 +
                      static_cast<size_t>(2 * p.nq * kTile) * sizeof(float);
  static bool configured = false;
  if (!configured) {
    TT_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<false, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    TT_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    TT_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<true, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    configured = true;
  }
  TT_REQUIRE(smem <= 232448, "tt_attn_causal_bwd: shared memory %zu too large", smem);
  // TT_ATTN_BWD=legacy keeps the one-CTA-per-(sequence, head) kernel for L <= 256 (A/B runs, bit-equality test)
  const char* mode = getenv("TT_ATTN_BWD");
  const bool legacy = mode && mode[0] == 'l';
  if (p.nq <= 2 && !legacy) {
    const size_t psmem = 1024 + 12 * static_cast<size_t>(kTileBytes) + 128 + 2 * 2 * 2 * kTile * sizeof(float);
    static bool pconfigured = false;
    if (!pconfigured) {
      TT_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
      pconfigured = true;
    }
    const int grid = B * H < num_sms() ? B * H : num_sms();
    TT_CHECK_CUDA(launch_k(attn_bwd_persist_kernel, dim3(grid), dim3(kBwdThreads), psmem, stream, tmQ, tmDO, p));
  } else if (p.nq <= 2) {
    TT_CHECK_CUDA(launch_k(attn_bwd_kernel<false, 4>, dim3(B * H), dim3(512), smem, stream, tmQ, tmDO, p));
  } else {
    // L <= 512: 16 warps in the element-wise phase (CG = 4) like the fast layout; TT_ATTN_BWD_LONG_CG=2 keeps 8
    static int long_cg = -1;
    if (long_cg < 0) { const char* e = getenv("TT_ATTN_BWD_LONG_CG"); long_cg = e ? atoi(e) : 4; }
    if (long_cg == 4) TT_CHECK_CUDA(launch_k(attn_bwd_kernel<true, 4>, dim3(B * H), dim3(512), smem, stream, tmQ, tmDO, p));
    else TT_CHECK_CUDA(launch_k(attn_bwd_kernel<true, 2>, dim3(B * H), dim3(256), smem, stream, tmQ, tmDO, p));
  }
  TT_LAUNCH_CHECK();
  return TT_OK;
}
