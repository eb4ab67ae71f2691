// Persistent warp-specialised tcgen05 GEMM for sm_100a.
//
//   C[M,N] = epilogue(alpha * A[M,K] * B[N,K]^T), bf16 operands, fp32 accumulate in TMEM.
//
// One CTA per SM, 640 threads:
//   warp 0      : TMA producer (one elected lane) — A/B tiles, 128B swizzle, N-stage ring
//   warp 1      : MMA issuer (one elected lane)  — tcgen05.mma M=128, N=block_n, K=16
//   warp 2      : TMEM allocator (2 accumulator buffers of block_n columns)
//   warps 2, 3  : optional column sums of the A operand (the bias gradient that belongs to a dgrad GEMM's
//                 dY operand), read from the staged A tiles while the MMAs run
//   warps 4..19 : epilogue — tcgen05.ld (warp % 4 = TMEM lane quarter, the four warps of a quarter
//                 take every 4th 32-column chunk), fused bias / ReLU / dropout / gate / residual;
//                 all global traffic goes through a swizzled per-warp smem tile so loads/stores
//                 are coalesced, split-K via red.v4
// Three pipelines: smem full/empty (TMA<->MMA), TMEM full/empty (MMA<->epilogue) and the
// static persistent tile loop. Operands may be K-major or MN-major (the transposed
// layouts dgrad/wgrad need), selected by template flags and the UMMA descriptors.
#include "../../include/tt_b200.h"
#include "tt_common.cuh"

namespace tt {

struct GemmParams {
  int M, N, K;
  int block_n, stages, k_splits;
  float alpha;
  const float* bias;
  int relu;
  uint32_t drop_thresh;
  float drop_scale;
  uint64_t drop_seed;
  const uint64_t* drop_seed_dev;
  uint32_t drop_site;
  const __nv_bfloat16* gate;
  int ld_gate;
  float gate_scale;
  const float* residual;
  int ld_res;
  float* out_f32;
  int ld_f32;
  __nv_bfloat16* out_bf16;
  int ld_bf16;
  int accumulate;
  int pair;         // 1 = CTA pairs (cluster of 2, tcgen05 cta_group::2): a pair computes a 256-row x block_n tile;
                    // each CTA stages its 128 rows of A and HALF of the B tile, the leader issues M=256 MMAs
  int stg_bytes;    // per-epilogue-warp staging tile bytes (the 256 B bias slices follow the 16 tiles)
  int tma_store;    // 1: finished 32 x 32 output blocks leave through TMA tensor stores straight from the (swizzled)
                    // staging tile instead of a transposed LDS + STG pass by the warp
  float* a_colsum;  // optional [K]: += column sums of the (K-major) A operand, taken from the staged tiles by warps 2 and 3
};

static constexpr int kBlockM = 128;
static constexpr int kBlockK = 64;
static constexpr uint32_t kABytes = kBlockM * kBlockK * 2;  // 16 KB
static constexpr int kEpiWarps = 16;
static constexpr int kGemmThreads = 128 + 32 * kEpiWarps;   // 4 control warps + 16 epilogue warps
static constexpr uint32_t kStageBytesF32 = 32 * 128;    // 32 rows x 128 B staging tile (fp32 output / residual)
static constexpr uint32_t kStageBytesBf16 = 32 * 64;    // 32 rows x 64 B (bf16 output / gate only)
static constexpr uint32_t kBiasBytesPerWarp = 256;      // 2 chunks x 32 floats

// Per-warp staging tile: 32 rows x 128 B, 16-byte units XOR-swizzled by (row & 7) so that both
// the row-per-lane accesses (thread = accumulator row) and the transposed, coalesced accesses
// (8 lanes = one 128 B row segment) are bank-conflict free.
__device__ __forceinline__ uint4* stg_unit(uint8_t* stg, int row, int unit) {
  return reinterpret_cast<uint4*>(stg + row * 128 + ((unit ^ (row & 7)) << 4));
}
// bf16 variant: 32 rows x 64 B. Two rows share a 128 B bank line, so the 4 units are swizzled by
// (row >> 1) & 3: eight consecutive rows (one row-per-lane wavefront) and 2 rows x 4 units (one
// transposed wavefront) both cover all 32 banks exactly once.
__device__ __forceinline__ uint4* stg_unit_bf(uint8_t* stg, int row, int unit) {
  return reinterpret_cast<uint4*>(stg + row * 64 + ((unit ^ ((row >> 1) & 3)) << 4));
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Asynchronously fetch the residual (fp32, 32 rows x 128 B) or gate (bf16, 32 rows x 64 B) block of
// one 32-column chunk into the warp's "in" tile: global -> shared without registers, coalesced
// (4 rows x 128 B resp. 8 rows x 64 B per warp instruction), one chunk ahead of its use.
__device__ __forceinline__ void epi_prefetch(const GemmParams& p, uint8_t* in, int lane, int row0, int col0) {
  if (p.residual) {
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int rr = it * 4 + (lane >> 3), u = lane & 7;
      const int gr = row0 + rr, gc = col0 + u * 4;
      if (gr < p.M && gc + 4 <= p.N) cp_async16(stg_unit(in, rr, u), p.residual + static_cast<size_t>(gr) * p.ld_res + gc);
    }
  } else if (p.gate) {
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int rr = it * 8 + (lane >> 2), u = lane & 3;
      const int gr = row0 + rr, gc = col0 + u * 8;
      if (gr < p.M && gc + 8 <= p.N) cp_async16(stg_unit_bf(in, rr, u), p.gate + static_cast<size_t>(gr) * p.ld_gate + gc);
    }
  }
  cp_async_commit();
}

// L2 prefetch of the residual / gate lines of one (tile, warp): lane = row, one 128-byte (fp32) or
// 64-byte (bf16) segment per 32-column chunk. Issued a whole tile ahead, so the later cp.async only
// pays L2 latency.
__device__ __forceinline__ void epi_prefetch_l2(const GemmParams& p, int lane, int row0, int colbase, int sub,
                                                int nchunks) {
  const int gr = row0 + lane;
  if (gr >= p.M) return;
  for (int c = sub; c < nchunks; c += kEpiWarps / 4) {
    const int gc = colbase + c * 32;
    if (gc >= p.N) break;
    const void* ptr = p.residual ? static_cast<const void*>(p.residual + static_cast<size_t>(gr) * p.ld_res + gc)
                                 : static_cast<const void*>(p.gate + static_cast<size_t>(gr) * p.ld_gate + gc);
    asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr));
  }
}

// One 32-column chunk of one accumulator row per lane. `next_col0` >= 0 asks for the prefetch of
// the warp's next chunk once the staging tile (`in` and `out` may be the same tile) is free again.
// The staging tile may still be read by a TMA store issued from it: wait (lane 0 issued it) before it is rewritten.
__device__ __forceinline__ void stg_acquire(const GemmParams& p, int lane) {
  if (p.tma_store) {
    if (lane == 0) tma_store_wait_read();
    __syncwarp();
  }
}

__device__ __forceinline__ void gemm_epilogue_chunk(const GemmParams& p, const uint32_t (&r)[32], uint8_t* out,
                                                    uint8_t* in, const float* sbias, int lane, int row0, int col0,
                                                    int next_col0, uint32_t dkey, const CUtensorMap* tmO32,
                                                    const CUtensorMap* tmO16) {
  const int row = row0 + lane;
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  // alpha and bias in one packed FFMA2 per column pair; alpha == 1 without bias costs nothing
  if (p.bias) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 b = *reinterpret_cast<const float4*>(sbias + j);   // same address in every lane: broadcast
      ffma2(v[j], v[j + 1], p.alpha, p.alpha, b.x, b.y);
      ffma2(v[j + 2], v[j + 3], p.alpha, p.alpha, b.z, b.w);
    }
  } else if (p.alpha != 1.f) {
#pragma unroll
    for (int j = 0; j < 32; j += 2) fmul2(v[j], v[j + 1], p.alpha, p.alpha);
  }
  if (p.relu) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = v[j] < 0.f ? 0.f : v[j];   // torch.relu keeps NaN (fmaxf would drop it)
  }
  if (p.drop_thresh) {
    // N % 4 == 0 and col0 % 32 == 0: the four columns j..j+3 share one hash word
    const uint32_t base = static_cast<uint32_t>(row) * static_cast<uint32_t>(p.N) + static_cast<uint32_t>(col0);
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      bool k[4];
      drop_keep_quad(dkey, base + j, p.drop_thresh, k);
      fmul2(v[j], v[j + 1], k[0] ? p.drop_scale : 0.f, k[1] ? p.drop_scale : 0.f);
      fmul2(v[j + 2], v[j + 3], k[2] ? p.drop_scale : 0.f, k[3] ? p.drop_scale : 0.f);
    }
  }
  if (p.residual || p.gate) {
    cp_async_wait_all();
    __syncwarp();
    if (p.residual) {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float4 x = *reinterpret_cast<const float4*>(stg_unit(in, lane, u));
        fadd2(v[4 * u], v[4 * u + 1], x.x, x.y);
        fadd2(v[4 * u + 2], v[4 * u + 3], x.z, x.w);
      }
    } else {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint4 x = *stg_unit_bf(in, lane, u);
        const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          // gate > 0 on the packed bf16 pair without unpacking: a positive bf16 is a positive int16
          const bool g0 = static_cast<int32_t>(w[h] << 16) > 0;
          const bool g1 = static_cast<int32_t>(w[h]) > 0xFFFF;
          const int j = u * 8 + h * 2;
          fmul2(v[j], v[j + 1], g0 ? p.gate_scale : 0.f, g1 ? p.gate_scale : 0.f);
        }
      }
    }
    __syncwarp();
  }
  if (p.out_f32) {
    stg_acquire(p, lane);
#pragma unroll
    for (int u = 0; u < 8; ++u)
      *reinterpret_cast<float4*>(stg_unit(out, lane, u)) = make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
    if (p.tma_store) {
      // the tile is laid out exactly as the 128-byte TMA swizzle expects (unit ^ (row & 7)); rows / columns beyond
      // M / N are clipped by the tensor map
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) { tma_store_2d(tmO32, out, col0, row0); tma_store_commit(); }
    } else {
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int rr = it * 4 + (lane >> 3), u = lane & 7;
      const int gr = row0 + rr, gc = col0 + u * 4;
      if (gr < p.M && gc + 4 <= p.N) {
        const float4 x = *reinterpret_cast<const float4*>(stg_unit(out, rr, u));
        float* o = p.out_f32 + static_cast<size_t>(gr) * p.ld_f32 + gc;
        if (p.accumulate) red_add_f32x4(o, x.x, x.y, x.z, x.w);
        else *reinterpret_cast<float4*>(o) = x;
      }
    }
    __syncwarp();
    }
  }
  if (p.out_bf16) {
    stg_acquire(p, lane);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      uint4 x;
      x.x = pack_bf16(v[u * 8 + 0], v[u * 8 + 1]);
      x.y = pack_bf16(v[u * 8 + 2], v[u * 8 + 3]);
      x.z = pack_bf16(v[u * 8 + 4], v[u * 8 + 5]);
      x.w = pack_bf16(v[u * 8 + 6], v[u * 8 + 7]);
      *stg_unit_bf(out, lane, u) = x;
    }
    if (p.tma_store) {   // 64-byte TMA swizzle == unit ^ ((row >> 1) & 3)
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) { tma_store_2d(tmO16, out, col0, row0); tma_store_commit(); }
    } else {
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int rr = it * 8 + (lane >> 2), u = lane & 3;
      const int gr = row0 + rr, gc = col0 + u * 8;
      if (gr < p.M && gc + 8 <= p.N)
        *reinterpret_cast<uint4*>(p.out_bf16 + static_cast<size_t>(gr) * p.ld_bf16 + gc) = *stg_unit_bf(out, rr, u);
    }
    __syncwarp();
    }
  }
  // the staging tile is free again: fetch the residual / gate block of this warp's next chunk
  if ((p.residual || p.gate) && next_col0 >= 0) {
    stg_acquire(p, lane);
    epi_prefetch(p, in, lane, row0, next_col0);
  }
}

template <bool A_MN, bool B_MN, bool PAIR>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmO32, const __grid_constant__ CUtensorMap tmO16,
                 const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int stages = p.stages;
  const int block_n = p.block_n;
  // CTA-pair mode (p.pair): the two CTAs of a cluster take row blocks 2i and 2i+1 of the same column block
  // and k range. Each stages its own A rows and HALF of the B tile (rows / 64-wide chunks [rank * half, +half));
  // the leader's single MMA thread issues cta_group::2 MMAs (M = 256) that read both CTAs' shared memory and
  // write 128 TMEM lanes in each. Per SM that is a third fewer operand bytes through TMA and the tensor
  // pipe reads 8 KB instead of 12 KB of shared memory per 256-wide MMA. Barrier protocol as in score_topk:
  // TMA bytes of both CTAs complete on the LEADER's full barrier, tcgen05.commit is multicast to the empty /
  // accumulator-full barriers of both CTAs, epilogue warps of both release the accumulator on the leader.
  constexpr bool pair = PAIR;   // a kernel that contains cta_group::2 instructions can only be launched as a cluster of 2
  uint32_t rank = 0;
  if constexpr (pair) rank = cluster_ctarank();
  const int worker = pair ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int n_workers = pair ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  const uint32_t b_bytes = (static_cast<uint32_t>(block_n) * kBlockK * 2) >> (pair ? 1 : 0);   // per CTA

  const int kblocks = (p.K + kBlockK - 1) / kBlockK;
  uint8_t* sA = smem;
  uint8_t* sB = smem + static_cast<size_t>(stages) * kABytes;
  uint8_t* sStage = sB + static_cast<size_t>(stages) * b_bytes;  // kEpiWarps staging tiles
  uint8_t* sBias = sStage + static_cast<size_t>(kEpiWarps) * p.stg_bytes;     // kEpiWarps x 256 B when p.bias
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sBias + (p.bias ? kEpiWarps * kBiasBytesPerWarp : 0u));
  uint64_t* empty_bar = full_bar + stages;
  uint64_t* tfull_bar = empty_bar + stages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* cs_bar = tempty_bar + 2;            // pair mode + column sums: "MMAs of this stage retired" in both CTAs
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(cs_bar + stages);
  float* csum = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 15) & ~static_cast<uintptr_t>(15));   // [2 warps][kblocks * 64] when p.a_colsum
  const bool colsum = p.a_colsum != nullptr;

  const uint32_t tmem_cols = static_cast<uint32_t>(2 * block_n);  // 128 / 256 / 512

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && elect_one()) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], colsum ? 3 : 1);   // MMA commit (+ the two column-sum warps)
      mbar_init(&cs_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], pair ? 2 * kEpiWarps : kEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (pair) { tmem_alloc_pair(tmem_slot, tmem_cols); tmem_relinquish_pair(); }
    else      { tmem_alloc(tmem_slot, tmem_cols); tmem_relinquish(); }
  }
  tc_fence_before();
  __syncwarp();                   // elected lanes rejoin their warps: barrier.cluster is .aligned
  if constexpr (pair) cluster_sync_all();   // both CTAs' barriers and TMEM exist before anything is signalled across
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // The trigger comes AFTER this CTA owns its TMEM columns: a dependent CTA scheduled early on the same
  // SM could otherwise take them first and wait forever for this grid to finish.
  pdl_launch_dependents();
  pdl_wait();   // prologue (barriers, TMEM, tensor-map prefetch) overlapped the previous kernel's tail

  const int tiles_m = (p.M + kBlockM - 1) / kBlockM;
  const int tiles_n = (p.N + block_n - 1) / block_n;
  const int tiles_mw = pair ? (tiles_m + 1) / 2 : tiles_m;      // row blocks (pairs of them) a worker walks
  const int num_tiles = tiles_mw * tiles_n * p.k_splits;
  // row block of work item mn: in pair mode the odd CTA may get one past the end (odd tiles_m): it still
  // loads (zero-filled) in lockstep and stores nothing.
  auto m_block = [&](int mn) { return pair ? 2 * (mn / tiles_n) + static_cast<int>(rank) : mn / tiles_n; };
  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = worker; t < num_tiles; t += n_workers) {
        const int split = t % p.k_splits;
        const int mn = t / p.k_splits;
        const int m_blk = m_block(mn), n_blk = mn % tiles_n;
        const int kb0 = static_cast<int>(static_cast<long long>(split) * kblocks / p.k_splits);
        const int kb1 = static_cast<int>(static_cast<long long>(split + 1) * kblocks / p.k_splits);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          uint8_t* a_dst = sA + static_cast<size_t>(stage) * kABytes;
          uint8_t* b_dst = sB + static_cast<size_t>(stage) * b_bytes;
          if constexpr (pair) {
            if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * (kABytes + b_bytes));
            if (A_MN) tma_load_3d_pair(a_dst, &tmA, &full_bar[stage], 0, kb * kBlockK, m_blk * (kBlockM / 64));
            else      tma_load_2d_pair(a_dst, &tmA, &full_bar[stage], kb * kBlockK, m_blk * kBlockM);
            if (B_MN) tma_load_3d_pair(b_dst, &tmB, &full_bar[stage], 0, kb * kBlockK,
                                       n_blk * (block_n / 64) + static_cast<int>(rank) * (block_n / 128));
            else      tma_load_2d_pair(b_dst, &tmB, &full_bar[stage], kb * kBlockK,
                                       n_blk * block_n + static_cast<int>(rank) * (block_n / 2));
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], kABytes + b_bytes);
            if (A_MN) tma_load_3d(a_dst, &tmA, &full_bar[stage], 0, kb * kBlockK, m_blk * (kBlockM / 64));
            else      tma_load_2d(a_dst, &tmA, &full_bar[stage], kb * kBlockK, m_blk * kBlockM);
            if (B_MN) tma_load_3d(b_dst, &tmB, &full_bar[stage], 0, kb * kBlockK, n_blk * (block_n / 64));
            else      tma_load_2d(b_dst, &tmB, &full_bar[stage], kb * kBlockK, n_blk * block_n);
          }
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0 && elect_one()) {
      const uint32_t idesc = umma_idesc_bf16(pair ? 2 * kBlockM : kBlockM, block_n, A_MN, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int t = worker; t < num_tiles; t += n_workers) {
        const int split = t % p.k_splits;
        const int kb0 = static_cast<int>(static_cast<long long>(split) * kblocks / p.k_splits);
        const int kb1 = static_cast<int>(static_cast<long long>(split + 1) * kblocks / p.k_splits);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * block_n);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_base = smem_u32(sA + static_cast<size_t>(stage) * kABytes);
          const uint32_t b_base = smem_u32(sB + static_cast<size_t>(stage) * b_bytes);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            // K-major: +32 B per 16 K-elements inside the 128 B swizzled row.
            // MN-major: +16 K-rows of 128 B; 64-wide MN chunks are kBlockK*128 B apart.
            const uint64_t adesc = A_MN ? umma_desc_mnmajor(a_base + k * 2048, kBlockK * 128)
                                        : umma_desc_kmajor(a_base + k * 32);
            const uint64_t bdesc = B_MN ? umma_desc_mnmajor(b_base + k * 2048, kBlockK * 128)
                                        : umma_desc_kmajor(b_base + k * 32);
            if constexpr (pair) umma_bf16_pair(d_tmem, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            else      umma_bf16(d_tmem, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          if constexpr (pair) {
            umma_commit_pair(&empty_bar[stage]);   // both CTAs' smem slots reusable once these MMAs retire
            // the follower's full barrier is never signalled (all TMA bytes land on the leader's): its column-sum
            // warps take "the MMAs that read this stage have retired" as "the tile is there"
            if (colsum) umma_commit_pair(&cs_bar[stage]);
          } else {
            umma_commit(&empty_bar[stage]);
          }
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
        if constexpr (pair) umma_commit_pair(&tfull_bar[acc]);       // accumulator complete -> both CTAs' epilogues
        else      umma_commit(&tfull_bar[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else if (warp < 4 && colsum) {
    // warps 2 and 3: column sums of this CTA's A tiles (K-major: row r = 128 B, 16-byte unit u stored at
    // u ^ (r & 7)). Lane = (row group rg, logical unit u): 4 rows per instruction, no bank conflicts; warp 2
    // takes rows 0..63, warp 3 rows 64..127. Every (row block, k-block) tile is staged exactly once per
    // column block, so only the tiles of column block 0 are summed. Rows beyond M arrive zero-filled.
    const int w2 = warp - 2;
    float* my = csum + w2 * (kblocks * kBlockK);
    for (int i = lane; i < kblocks * kBlockK; i += 32) my[i] = 0.f;
    __syncwarp();
    const int u = lane & 7, rg = lane >> 3;
    int stage = 0;
    uint32_t phase = 0;
    for (int t = worker; t < num_tiles; t += n_workers) {
      const int split = t % p.k_splits;
      const int mn = t / p.k_splits;
      const bool take = (mn % tiles_n) == 0;
      const int kb0 = static_cast<int>(static_cast<long long>(split) * kblocks / p.k_splits);
      const int kb1 = static_cast<int>(static_cast<long long>(split + 1) * kblocks / p.k_splits);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(pair ? &cs_bar[stage] : &full_bar[stage], phase);
        if (take) {
          const uint8_t* a = sA + static_cast<size_t>(stage) * kABytes + static_cast<size_t>(w2) * 64 * 128;
          float acc[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll 8
          for (int i = 0; i < 16; ++i) {
            const int r = i * 4 + rg;
            const uint4 x = *reinterpret_cast<const uint4*>(a + r * 128 + ((u ^ (r & 7)) << 4));
            const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int h = 0; h < 4; ++h)
              fadd2(acc[2 * h], acc[2 * h + 1], __uint_as_float(w[h] << 16), __uint_as_float(w[h] & 0xFFFF0000u));
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 8);
            acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 16);
          }
          if (rg == 0) {
            float4* dst = reinterpret_cast<float4*>(my + kb * kBlockK + u * 8);
            float4 lo = dst[0], hi = dst[1];
            lo.x += acc[0]; lo.y += acc[1]; lo.z += acc[2]; lo.w += acc[3];
            hi.x += acc[4]; hi.y += acc[5]; hi.z += acc[6]; hi.w += acc[7];
            dst[0] = lo; dst[1] = hi;
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);   // this warp is done with the slot
        if (++stage == stages) { stage = 0; phase ^= 1u; }
      }
    }
    __syncwarp();
    for (int i = lane; i < p.K; i += 32) {
      const float v = my[i];
      if (v != 0.f) atomicAdd(p.a_colsum + i, v);
    }
  }
  if (warp >= 4) {
    // 16 epilogue warps (4 per scheduler: the chunk pipeline is a chain of TMEM / shared / global
    // latencies, hidden by switching warps rather than by unrolling). warp % 4 selects the TMEM lane
    // quarter (hardware rule); the four warps sharing a quarter take every 4th 32-column chunk.
    const int ew = warp - 4;
    const int q = ew & 3, sub = ew >> 2;
    uint8_t* stg = sStage + static_cast<size_t>(ew) * p.stg_bytes;
    float* sbias = reinterpret_cast<float*>(sBias + static_cast<size_t>(ew) * kBiasBytesPerWarp);   // [2 chunks][32]
    const uint64_t seed = p.drop_seed + ((p.drop_thresh && p.drop_seed_dev) ? *p.drop_seed_dev : 0ull);
    const uint32_t dkey = drop_key(seed, p.drop_site);
    const int nchunks = block_n / 32;
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool has_in = p.residual || p.gate;
    if (has_in && worker < num_tiles) {
      const int mn = worker / p.k_splits;
      epi_prefetch_l2(p, lane, m_block(mn) * kBlockM + q * 32, (mn % tiles_n) * block_n, sub, nchunks);
    }
    for (int t = worker; t < num_tiles; t += n_workers) {
      const int mn = t / p.k_splits;
      const int m_blk = m_block(mn), n_blk = mn % tiles_n;
      const int row0 = m_blk * kBlockM + q * 32;
      const int colbase = n_blk * block_n;
      if (has_in && t + n_workers < num_tiles) {   // next tile's lines -> L2 while this one computes
        const int mn2 = (t + n_workers) / p.k_splits;
        epi_prefetch_l2(p, lane, m_block(mn2) * kBlockM + q * 32, (mn2 % tiles_n) * block_n, sub, nchunks);
      }
      // Everything that does not depend on the accumulator is issued before waiting for it:
      // the bias slice of this warp's chunks and the first residual / gate block.
      if (p.bias) {
        __syncwarp();
        for (int k = 0, c = sub; c < nchunks; c += kEpiWarps / 4, ++k) {
          const int col = colbase + c * 32 + lane;
          sbias[k * 32 + lane] = col < p.N ? __ldg(p.bias + col) : 0.f;
        }
      }
      if (has_in && sub < nchunks) {
        stg_acquire(p, lane);
        epi_prefetch(p, stg, lane, row0, colbase + sub * 32);
      }
      mbar_wait(&tfull_bar[acc], acc_phase);
      __syncwarp();
      tc_fence_after();
      const uint32_t t_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                              static_cast<uint32_t>(acc * block_n);
      uint32_t r[32];
      for (int c = sub, k = 0; c < nchunks && m_blk < tiles_m; c += kEpiWarps / 4, ++k) {
        tmem_ld32(t_base + static_cast<uint32_t>(c * 32), r);
        tmem_ld_wait();
        const int cn = c + kEpiWarps / 4;
        gemm_epilogue_chunk(p, r, stg, stg, sbias + k * 32, lane, row0, colbase + c * 32,
                            cn < nchunks ? colbase + cn * 32 : -1, dkey, &tmO32, &tmO16);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (pair) mbar_arrive_cluster(&tempty_bar[acc], 0);
        else      mbar_arrive(&tempty_bar[acc]);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
    if (p.tma_store && lane == 0) tma_store_wait_all();   // shared memory stays valid until the engine has read it
  }

  tc_fence_before();
  __syncwarp();
  if constexpr (pair) cluster_sync_all();   // the partner may still read this CTA's smem, signal its barriers, write its TMEM
  else __syncthreads();
  if (warp == 2) {
    if constexpr (pair) tmem_dealloc_pair(tmem_base, tmem_cols);
    else      tmem_dealloc(tmem_base, tmem_cols);
  }
}

static constexpr size_t kSmemLimit = 232448;
static size_t gemm_fixed_smem(int stg_bytes, int colsum_k) {   // alignment pad, staging, barriers (<= 8 stages), TMEM slot,
  return 1024 + static_cast<size_t>(kEpiWarps) * stg_bytes + (3 * 8 + 4) * sizeof(uint64_t) + 32 +   // column sums
         2 * sizeof(float) * static_cast<size_t>(colsum_k);
}

template <bool A_MN, bool B_MN, bool PAIR>
static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO32,
                       const CUtensorMap& tmO16, const GemmParams& p, int grid, size_t smem, cudaStream_t stream) {
  static bool configured = false;
  if (!configured) {
    TT_CHECK_CUDA(cudaFuncSetAttribute(gemm_bf16_kernel<A_MN, B_MN, PAIR>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    configured = true;
  }
  TT_REQUIRE(smem <= kSmemLimit, "tt_gemm_bf16: %zu B of shared memory requested", smem);
  if (PAIR) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    TT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_bf16_kernel<A_MN, B_MN, PAIR>, tmA, tmB, tmO32, tmO16, p));
  } else {
    TT_CHECK_CUDA(launch_k(gemm_bf16_kernel<A_MN, B_MN, PAIR>, dim3(grid), dim3(kGemmThreads), smem, stream, tmA, tmB, tmO32, tmO16, p));
  }
  TT_LAUNCH_CHECK();
  return TT_OK;
}

template <bool A_MN, bool B_MN>
static int launch_gemm_mode(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO32,
                            const CUtensorMap& tmO16, const GemmParams& p, int grid, size_t smem, cudaStream_t stream) {
  return p.pair ? launch_gemm<A_MN, B_MN, true>(tmA, tmB, tmO32, tmO16, p, grid, smem, stream)
                : launch_gemm<A_MN, B_MN, false>(tmA, tmB, tmO32, tmO16, p, grid, smem, stream);
}

}  // namespace tt

extern "C" int tt_gemm_bf16(const tt_gemm_args* a, void* stream_) {
  using namespace tt;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(a != nullptr, "tt_gemm_bf16: null args");
  TT_REQUIRE(a->A && a->B, "tt_gemm_bf16: null operand");
  TT_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0, "tt_gemm_bf16: empty problem %d x %d x %d", a->M,
             a->N, a->K);
  TT_REQUIRE(a->out_f32 || a->out_bf16, "tt_gemm_bf16: no output");
  TT_REQUIRE(a->lda % 8 == 0 && a->ldb % 8 == 0, "tt_gemm_bf16: lda/ldb must be multiples of 8");
  // MN-major operands are fetched in 64-wide chunks: a ragged last chunk reads up to 63 elements
  // past M (resp. N) inside each K row (results there are never stored), so the dimension must be
  // a multiple of 8 and the buffer readable up to the next multiple of 64 on its last row.
  TT_REQUIRE(!a->a_mn || a->M % 8 == 0, "tt_gemm_bf16: MN-major A needs M %% 8 == 0 (M=%d)", a->M);
  TT_REQUIRE(!a->b_mn || a->N % 8 == 0, "tt_gemm_bf16: MN-major B needs N %% 8 == 0 (N=%d)", a->N);
  TT_REQUIRE(!a->out_f32 || a->ld_f32 % 4 == 0, "tt_gemm_bf16: ld_f32 must be a multiple of 4");
  TT_REQUIRE(!a->out_bf16 || a->ld_bf16 % 8 == 0, "tt_gemm_bf16: ld_bf16 must be a multiple of 8");
  TT_REQUIRE(!a->residual || a->ld_res % 4 == 0, "tt_gemm_bf16: ld_res must be a multiple of 4");
  TT_REQUIRE(!a->gate || a->ld_gate % 8 == 0, "tt_gemm_bf16: ld_gate must be a multiple of 8");
  TT_REQUIRE(a->drop_p >= 0.f && a->drop_p < 1.f, "tt_gemm_bf16: drop_p out of range");
  TT_REQUIRE(!a->out_f32 || a->N % 4 == 0, "tt_gemm_bf16: fp32 output needs N %% 4 == 0 (N=%d)", a->N);
  TT_REQUIRE(!(a->out_bf16 || a->gate) || a->N % 8 == 0, "tt_gemm_bf16: bf16 output / gate need N %% 8 == 0 (N=%d)", a->N);
  TT_REQUIRE(!(a->gate && a->residual), "tt_gemm_bf16: gate and residual cannot be combined");
  TT_REQUIRE(!a->accumulate || (a->out_f32 && !a->out_bf16),
             "tt_gemm_bf16: accumulate needs an fp32-only output");

  GemmParams p;
  p.M = a->M; p.N = a->N; p.K = a->K;
  int bn = a->block_n;
  if (bn == 0) {
    if (a->accumulate) {
      // Split-K. A deep reduction (the encoder's weight gradients, K = tokens) is bound by the L2 -> smem
      // operand stream, so it wants the widest tile (half the operand bytes per flop of a 64-wide one;
      // measured 45 -> 31 us on 1024x256x51200). A shallow one wants CTAs, i.e. many small tiles.
      if (a->K >= 4096) bn = a->N >= 256 ? 256 : (a->N > 64 ? 128 : 64);
      else bn = a->N >= 512 ? 128 : 64;
    }
    else {
      // The widest tile that still gives every SM a tile; problems too small for that (the B-row GEMMs of
      // the heads and of the single-row last layer) are latency-bound and want as many CTAs as possible
      // (256x256x256: 8.1 us with one 256-wide tile per row block, 5.0 us with four 64-wide ones).
      const int tm = (a->M + kBlockM - 1) / kBlockM;
      bn = 64;
      for (int cand = 256; cand > 64; cand >>= 1) {
        if (a->N > cand / 2 && tm * ((a->N + cand - 1) / cand) >= num_sms()) { bn = cand; break; }
      }
    }
  }
  TT_REQUIRE(bn == 64 || bn == 128 || bn == 256, "tt_gemm_bf16: block_n must be 64/128/256");
  p.block_n = bn;
  const int tiles_m = (a->M + kBlockM - 1) / kBlockM;
  const int tiles_n = (a->N + bn - 1) / bn;
  const int kblocks = (a->K + kBlockK - 1) / kBlockK;
  int ks = a->k_splits;
  if (ks <= 0) {
    ks = 1;
    if (a->accumulate) {
      const int sms = num_sms();
      ks = sms / (tiles_m * tiles_n);
      if (ks < 1) ks = 1;
      // keep at least 4 k-blocks per split so the pipeline has something to stream
      if (ks > (kblocks + 3) / 4) ks = (kblocks + 3) / 4;
    }
  }
  if (ks > kblocks) ks = kblocks;
  if (ks < 1) ks = 1;
  TT_REQUIRE(ks == 1 || a->accumulate, "tt_gemm_bf16: k_splits > 1 requires accumulate");
  p.k_splits = ks;

  // CTA pairs (see the kernel) for every launch where each pair of SMs still gets (nearly) a full share of work
  // items. Measured on the c2 step with the earlier LDS + STG epilogue, the deep (K >= 512) launches gained 7-15 %
  // (dgrad 1024: 39.3 -> 33.3 us, wgrads 36.9 -> 32.8 / 45.0 -> 38.8 us) while the epilogue-bound K = 256 ones lost
  // 10-20 % to the lockstep of the pair (QKV 37.1 -> 42.9 us). Since the epilogue stores through TMA the pair no
  // longer loses on the K = 256 launches (c2 step 1.160 -> 1.146 ms with every eligible launch on pairs).
  const int pairs = num_sms() / 2 > 0 ? num_sms() / 2 : 1;
  const long pair_items = static_cast<long>((tiles_m + 1) / 2) * tiles_n * ks;
  const bool eligible = bn >= 128 && tiles_m >= 2 && pair_items * 10 >= static_cast<long>(pairs) * 9;
  p.pair = eligible ? 1 : 0;
  const size_t b_bytes = (static_cast<size_t>(bn) * kBlockK * 2) >> (p.pair ? 1 : 0);   // per CTA
  // bf16-only epilogues stage 64-byte rows: half the staging, more pipeline stages
  p.stg_bytes = static_cast<int>((a->out_f32 || a->residual) ? kStageBytesF32 : kStageBytesBf16);
  p.a_colsum = a->a_colsum;
  TT_REQUIRE(!a->a_colsum || (!a->a_mn && ks == 1 && a->K <= 2048),
             "tt_gemm_bf16: a_colsum needs a K-major A operand, no split-K and K <= 2048 (K=%d)", a->K);
  const size_t fixed = gemm_fixed_smem(p.stg_bytes + (a->bias ? static_cast<int>(kBiasBytesPerWarp) : 0),
                                       a->a_colsum ? kblocks * kBlockK : 0);
  int stages = static_cast<int>((kSmemLimit - fixed) / (kABytes + b_bytes));
  if (stages > 8) stages = 8;
  TT_REQUIRE(stages >= 2, "tt_gemm_bf16: no room for a 2-stage pipeline (block_n %d)", bn);
  p.stages = stages;

  p.alpha = a->alpha;
  p.bias = a->bias;
  p.relu = a->relu;
  p.drop_thresh = 0;
  p.drop_scale = 1.f;
  if (a->drop_p > 0.f) {
    double t = static_cast<double>(a->drop_p) * 4294967296.0;
    p.drop_thresh = t >= 4294967295.0 ? 4294967295u : static_cast<uint32_t>(t);
    if (p.drop_thresh == 0) p.drop_thresh = 1;
    p.drop_scale = 1.f / (1.f - a->drop_p);
  }
  p.drop_seed = a->drop_seed;
  p.drop_seed_dev = a->drop_seed_dev;
  p.drop_site = a->drop_site;
  p.gate = static_cast<const __nv_bfloat16*>(a->gate);
  p.ld_gate = a->ld_gate;
  p.gate_scale = a->gate_scale;
  p.residual = a->residual;
  p.ld_res = a->ld_res;
  p.out_f32 = a->out_f32;
  p.ld_f32 = a->ld_f32;
  p.out_bf16 = static_cast<__nv_bfloat16*>(a->out_bf16);
  p.ld_bf16 = a->ld_bf16;
  p.accumulate = a->accumulate;

  CUtensorMap tmA, tmB;
  int rc;
  if (a->a_mn) {
    uint64_t dims[3] = {64, static_cast<uint64_t>(a->K), static_cast<uint64_t>((a->M + 63) / 64)};
    uint64_t str[2] = {static_cast<uint64_t>(a->lda) * 2, 128};
    uint32_t box[3] = {64, kBlockK, kBlockM / 64};
    rc = make_tmap_bf16(&tmA, a->A, 3, dims, str, box);
  } else {
    uint64_t dims[2] = {static_cast<uint64_t>(a->K), static_cast<uint64_t>(a->M)};
    uint64_t str[1] = {static_cast<uint64_t>(a->lda) * 2};
    uint32_t box[2] = {kBlockK, kBlockM};
    rc = make_tmap_bf16(&tmA, a->A, 2, dims, str, box);
  }
  if (rc) return rc;
  if (a->b_mn) {
    uint64_t dims[3] = {64, static_cast<uint64_t>(a->K), static_cast<uint64_t>((a->N + 63) / 64)};
    uint64_t str[2] = {static_cast<uint64_t>(a->ldb) * 2, 128};
    uint32_t box[3] = {64, kBlockK, static_cast<uint32_t>(p.pair ? bn / 128 : bn / 64)};
    rc = make_tmap_bf16(&tmB, a->B, 3, dims, str, box);
  } else {
    uint64_t dims[2] = {static_cast<uint64_t>(a->K), static_cast<uint64_t>(a->N)};
    uint64_t str[1] = {static_cast<uint64_t>(a->ldb) * 2};
    uint32_t box[2] = {kBlockK, static_cast<uint32_t>(p.pair ? bn / 2 : bn)};
    rc = make_tmap_bf16(&tmB, a->B, 2, dims, str, box);
  }
  if (rc) return rc;

  // Output tensor maps (32 x 32 blocks, the staging tile's swizzle): plain stores only — split-K keeps red.add
  CUtensorMap tmO32 = tmA, tmO16 = tmA;   // placeholders when unused
  p.tma_store = a->accumulate ? 0 : 1;
  if (p.tma_store && a->out_f32) {
    uint64_t dims[2] = {static_cast<uint64_t>(a->N), static_cast<uint64_t>(a->M)};
    uint64_t str[1] = {static_cast<uint64_t>(a->ld_f32) * 4};
    uint32_t box[2] = {32, 32};
    rc = make_tmap(&tmO32, a->out_f32, 2, dims, str, box, 1, 128);
    if (rc) return rc;
  }
  if (p.tma_store && a->out_bf16) {
    uint64_t dims[2] = {static_cast<uint64_t>(a->N), static_cast<uint64_t>(a->M)};
    uint64_t str[1] = {static_cast<uint64_t>(a->ld_bf16) * 2};
    uint32_t box[2] = {32, 32};
    rc = make_tmap(&tmO16, a->out_bf16, 2, dims, str, box, 0, 64);
    if (rc) return rc;
  }

  int grid;
  if (p.pair) {
    grid = 2 * static_cast<int>(pair_items < pairs ? pair_items : pairs);
  } else {
    const int num_tiles = tiles_m * tiles_n * ks;
    grid = num_tiles < num_sms() ? num_tiles : num_sms();
  }
  const size_t smem = fixed + static_cast<size_t>(stages) * (kABytes + b_bytes);
  if (a->a_mn) {
    return a->b_mn ? launch_gemm_mode<true, true>(tmA, tmB, tmO32, tmO16, p, grid, smem, stream)
                   : launch_gemm_mode<true, false>(tmA, tmB, tmO32, tmO16, p, grid, smem, stream);
  }
  return a->b_mn ? launch_gemm_mode<false, true>(tmA, tmB, tmO32, tmO16, p, grid, smem, stream)
                 : launch_gemm_mode<false, false>(tmA, tmB, tmO32, tmO16, p, grid, smem, stream);
}
