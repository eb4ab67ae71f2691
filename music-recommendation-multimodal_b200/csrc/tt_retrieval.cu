// Catalog retrieval: scores = U E^T fused with a streaming per-user top-K' selection, exact
// re-scoring of the candidates, canonical ordering, cross-shard merge and Recall/NDCG.
//
// Replaces, in calculate_metrics_global (src/evaluate_metrics.py:106-192):
//   scores = user_emb @ item_embeddings.T   (:148, fp32 SGEMM, (B, V) matrix materialised)
//   scores[:, 0] = -inf                     (:152)
//   torch.topk(scores, max_k)               (:156, radix select over V-long rows)
//   per-k hit / NDCG bookkeeping            (:159-185, nonzero() syncs)
//
// tt_score_topk (tcgen05, cta_group::2): a work unit = 256 users x one contiguous item range, run by a
// PAIR of CTAs (cluster of 2). Each CTA keeps 128 of the users resident in shared memory (64 KB,
// bf16) and streams 128 of every 256-item step through an 8-stage TMA ring; the leader CTA issues
// M=256, N=256 MMAs that read both CTAs' shared memory, so per SM the tensor pipe reads 8 KB of
// operands per 128-cycle MMA instead of the 16 KB two M=128,N=128 MMAs need (the single-CTA version
// of this kernel sat at 60 % tensor-pipe activity whatever the epilogue or ring depth: shared-memory
// operand bandwidth). Accumulators: 128 lanes x 256 columns per CTA, double-buffered (512 columns).
// Sixteen epilogue warps per CTA read them with tcgen05.ld; a warp owns 32 user rows x 64 item
// columns, each thread keeps its row's running threshold in a register and appends (score, item)
// keys that beat it to a per-(range, column quarter, row) candidate list in global memory; a full
// list is pruned to its K' best by the whole warp (bitwise binary search on the 64-bit keys with
// ballot/popc + compaction). The score matrix never exists.
// Keys are totally ordered: (score descending, item index ascending) — the canonical order.
//
// tt_topk_finalize: per user, select the K' best keys over all ranges, re-score them EXACTLY
// (fp32 inputs, fp64 accumulation, rounded once to fp32), sort canonically, emit the top K and
// a certificate that no non-candidate can belong to the exact top K.
#include "../../include/tt_b200.h"
#include "tt_common.cuh"
#include <climits>
#include <math.h>

namespace tt {

static constexpr int kUT = 256;        // users per work unit: 128 per CTA of the pair (MMA M = 256, cta_group::2)
static constexpr int kIT = 256;        // items per MMA step (N = 256): 128 from each CTA's shared memory
static constexpr int kLists = 4;       // candidate lists per (range, user row): one per 64-item column quarter of a step
static constexpr int kD = 256;         // embedding dim
static constexpr int kKB = kD / 64;    // k-blocks
static constexpr uint32_t kTile16K = 128 * 64 * 2;
static constexpr int kChunks = kIT / 32; // 32-score chunks per item step
static constexpr int kBStages = 8;     // 16 KB item slices in flight per CTA
static constexpr int kTopkThreads = 640;   // TMA, MMA, TMEM-alloc, spare + 16 epilogue warps
static constexpr int kCap = 512;       // candidate list capacity per (range, row)
static constexpr int kMaxLists = 1216;  // finalize: lists per user (ranges x kLists) the offset table holds
static constexpr int kPoolCap = 4096;  // finalize: per-user key pool in shared memory
static constexpr int kExclMax = 4096;  // excluded ids per user (tt_exclusions_build: one shared-memory bitonic sort)
static constexpr int kExclWords = 128; // per-user hashed bitmap of excluded ids: 4096 bits

__device__ __forceinline__ uint32_t f2ord(float f) {
  const uint32_t u = __float_as_uint(f + 0.0f);  // -0 -> +0
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
  const uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
  return __uint_as_float(u);
}
__device__ __forceinline__ uint64_t make_key(float s, uint32_t gidx) {
  return (static_cast<uint64_t>(f2ord(s)) << 32) | static_cast<uint64_t>(0xFFFFFFFFu - gidx);
}
__device__ __forceinline__ uint32_t key_idx(uint64_t k) { return 0xFFFFFFFFu - static_cast<uint32_t>(k); }
__device__ __forceinline__ float key_score(uint64_t k) { return ord2f(static_cast<uint32_t>(k >> 32)); }

struct TopkParams {
  int U, N, item_base;
  int n_ut, n_ranges, tiles_per_range, total_tiles;
  int tile_stride;           // logical tile t of a range is physical tile t * tile_stride (sample pass: strided tiles)
  float* smax;               // non-null: SAMPLE pass — store each 32-score chunk's maximum, collect nothing
  int kprime;
  int u_pad;
  unsigned long long* cand;  // [n_ranges * kLists][u_pad][kCap]
  int* cand_cnt;             // [n_ranges * kLists][u_pad]
  unsigned long long* thr;   // [u_pad]
  int mask_item0;
  // score_topk_kernel<false, true>: per-user excluded global ids (tt_exclusions_build)
  const int* ex_ids;         // [U][ex_ld] sorted ascending, distinct
  const int* ex_cnt;         // [U]
  const uint32_t* ex_bits;   // [U][kExclWords] hashed bitmap: a clear bit proves an id is not excluded
  int ex_ld;
  // score_topk_kernel<*, *, true>: one bit per row of this shard, 1 = retired (never scored as a candidate); a
  // 64-bit word covers the 64 item columns an epilogue warp owns in one step. ceil(N / 256) * 4 words.
  const unsigned long long* retired;
};

// Bit of the exclusion bitmap that stands for global id `id` (Fibonacci hashing: the top 12 bits of id * 2^32/phi).
__device__ __forceinline__ uint32_t excl_hash(uint32_t id) { return (id * 2654435761u) >> 20; }

// Drop the keys of excluded items from one lane's candidate list buf[0, n) in place; returns the new count. A key
// whose bitmap bit is clear is kept after one L2-resident load; only the ~m/4096 others pay for a binary search of
// the sorted list. Candidates (about one score in a thousand) enter the list unchecked and the list is filtered here,
// once per work unit and before a prune — testing each candidate as it is admitted put an L2 round trip into the
// epilogue's chunk chain, whose latency bounds an item step (measured on a B200: 1.48x the plain pass at m = 50).
__device__ __noinline__ int drop_excluded(unsigned long long* buf, int n, const uint32_t* __restrict__ bits,
                                          const int* __restrict__ ids, int n_ids) {
  constexpr int kBatch = 8;   // keys whose list and bitmap loads are in flight together (the writes trail the reads)
  int w = 0;
  for (int i0 = 0; i0 < n; i0 += kBatch) {
    unsigned long long k[kBatch];
    uint32_t word[kBatch];
#pragma unroll
    for (int e = 0; e < kBatch; ++e) k[e] = i0 + e < n ? buf[i0 + e] : 0ull;
#pragma unroll
    for (int e = 0; e < kBatch; ++e) word[e] = i0 + e < n ? __ldg(bits + (excl_hash(key_idx(k[e])) >> 5)) : 0u;
#pragma unroll
    for (int e = 0; e < kBatch; ++e) {
      if (i0 + e >= n) break;
      const uint32_t gidx = key_idx(k[e]);
      bool ex = false;
      if ((word[e] >> (excl_hash(gidx) & 31u)) & 1u) {
        int lo = 0, hi = n_ids;                          // first position whose id is >= gidx
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (__ldg(ids + mid) < static_cast<int>(gidx)) lo = mid + 1; else hi = mid;
        }
        ex = lo < n_ids && __ldg(ids + lo) == static_cast<int>(gidx);
      }
      if (!ex) buf[w++] = k[e];
    }
  }
  return w;
}

__device__ __forceinline__ int drop_excluded_row(unsigned long long* buf, int n, const TopkParams& p, int row) {
  return drop_excluded(buf, n, p.ex_bits + static_cast<size_t>(row) * kExclWords,
                       p.ex_ids + static_cast<size_t>(row) * p.ex_ld, __ldg(p.ex_cnt + row));
}

// Warp-cooperative prune of one row's candidate list to its kprime largest keys.
// Returns the new count; T receives a threshold with count(keys >= T) == new count.
__device__ __noinline__ int warp_prune(unsigned long long* buf, int n, int kprime, int lane, unsigned long long& T) {
  __syncwarp();
  unsigned long long k[kCap / 32];
#pragma unroll
  for (int e = 0; e < kCap / 32; ++e) {
    const int i = e * 32 + lane;
    k[e] = i < n ? buf[i] : 0ull;
  }
  unsigned long long t = 0;
  for (int bit = 63; bit >= 0; --bit) {
    const unsigned long long cand = t | (1ull << bit);
    int c = 0;
#pragma unroll
    for (int e = 0; e < kCap / 32; ++e) c += (k[e] >= cand);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (c >= kprime) {
      t = cand;
      if (c == kprime) break;
    }
  }
  int base = 0;
  const unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int e = 0; e < kCap / 32; ++e) {
    const bool keep = k[e] >= t && k[e] != 0ull;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (keep) buf[base + __popc(m & lt)] = k[e];
    base += __popc(m);
  }
  __syncwarp();
  T = t;
  return base;
}

__device__ __forceinline__ float chunk_max(const uint32_t (&r)[32]) {
  float m = __uint_as_float(r[0]);
#pragma unroll
  for (int t = 1; t < 32; ++t) m = fmaxf(m, __uint_as_float(r[t]));
  return m;
}

// Filter one 32-score chunk of this lane's user row against the row threshold.
//
// The epilogue loop has to stay SMALL: an earlier version examined the 32 registers of a chunk with
// fully unrolled nested branches (4 096 SASS instructions in the kernel) and the ncu source page
// showed the epilogue warps stalled on instruction fetch (stall_no_inst first, ahead of every data
// dependency) whenever a chunk held a candidate — which, at ~1 candidate per 1 000 scores, is two
// chunks out of three. Now the registers only feed a max tree (one 8-bit "which 4-score groups beat
// the threshold" mask per lane and chunk), and the rare groups that do hold a candidate are RE-READ
// from TMEM four columns at a time (the TMEM address is a run-time value, a register index is not)
// in a short warp-uniform loop.
__device__ __forceinline__ uint32_t chunk_group_mask(const uint32_t (&r)[32], float thr_s) {
  uint32_t gm = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float g = fmaxf(fmaxf(__uint_as_float(r[4 * k]), __uint_as_float(r[4 * k + 1])),
                          fmaxf(__uint_as_float(r[4 * k + 2]), __uint_as_float(r[4 * k + 3])));
    gm |= (g >= thr_s) ? (1u << k) : 0u;
  }
  return gm;
}

template <bool kExclude, bool kLive>
__device__ __forceinline__ void collect_groups(uint32_t gm, uint32_t t_chunk, int idx0, const TopkParams& p, int lane,
                                               int row, unsigned long long* buf, int& cnt,
                                               unsigned long long& thr_key, float& thr_s, uint64_t retired) {
  uint32_t wm = __reduce_or_sync(0xffffffffu, gm);   // groups in which ANY lane has a candidate (warp-uniform)
#pragma unroll 1
  while (wm) {
    const int k = __ffs(wm) - 1;
    wm &= wm - 1;
    uint32_t v[4];
    tmem_ld4(t_chunk + 4u * k, v);
    tmem_ld_wait();
    if ((gm >> k) & 1u) {
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float s = __uint_as_float(v[t]);
        if (s >= thr_s) {
          const int idx = idx0 + 4 * k + t;
          const uint32_t gidx = static_cast<uint32_t>(p.item_base + idx);
          const bool live = !kLive || !((retired >> (4 * k + t)) & 1ull);
          if (idx < p.N && !(p.mask_item0 && gidx == 0u) && live) {
            const unsigned long long key = make_key(s, gidx);
            if (key > thr_key) buf[cnt++] = key;
          }
        }
      }
    }
  }
  if constexpr (kExclude) {
    if (cnt > kCap - 64) cnt = drop_excluded_row(buf, cnt, p, row);   // prune thresholds count admissible keys only
  }
  unsigned full = __ballot_sync(0xffffffffu, cnt > kCap - 64)   /* a call appends at most 64 keys per lane */;
  while (full) {
    const int src = __ffs(full) - 1;
    full &= full - 1;
    const unsigned long long bsrc = __shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(buf), src);
    const int nsrc = __shfl_sync(0xffffffffu, cnt, src);
    unsigned long long T;
    const int ncnt = warp_prune(reinterpret_cast<unsigned long long*>(bsrc), nsrc, p.kprime, lane, T);
    if (lane == src) {
      cnt = ncnt;
      thr_key = T;
      thr_s = key_score(T);
      atomicMax(p.thr + row, T);
    }
  }
}

// kExclude (main pass only): the user's excluded items are removed from its candidate lists before every prune and
// before the lists are handed over, so the pruning thresholds, finalize and its certificate all speak about the
// admissible items only.
// kLive: rows whose bit in p.retired is set are never admitted (main pass) and never own a chunk maximum (sample
// pass: their scores become -inf first, which can only lower a start threshold). A warp's 64 columns of a step share
// one 64-bit word of the bitmap; it is loaded one step ahead, so the L2 round trip stays out of the chunk chain.
template <bool kSample, bool kExclude, bool kLive>
__global__ void __launch_bounds__(kTopkThreads, 1)
score_topk_kernel(const __grid_constant__ CUtensorMap tmU, const __grid_constant__ CUtensorMap tmI,
                  const TopkParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();              // 0 = leader (issues the MMAs of the pair)
  const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

  uint8_t* sA = smem;                                   // [4 kb] x 16 KB: this CTA's 128 users
  uint8_t* sB = smem + kKB * kTile16K;                  // kBStages x 16 KB: this CTA's 128 items of a 256-item step
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + kBStages * kTile16K);
  uint64_t* a_full = bars + 0;                          // leader's copy is the live one (tx bytes of both CTAs)
  uint64_t* a_empty = bars + 1;                         // every CTA's copy is live (multicast commit)
  uint64_t* b_full = bars + 2;                          // leader's
  uint64_t* b_empty = b_full + kBStages;                // every CTA's
  uint64_t* t_full = b_empty + kBStages;                // every CTA's
  uint64_t* t_empty = t_full + 2;                       // leader's: 16 epilogue warps x 2 CTAs
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmU);
    tma_prefetch_desc(&tmI);
  }
  if (warp == 1 && elect_one()) {
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int s = 0; s < kBStages; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&t_full[a], 1); mbar_init(&t_empty[a], 32); }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc_pair(tmem_slot, 512);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  __syncwarp();           // the elected lanes above rejoin their warps: barrier.cluster is .aligned
  cluster_sync_all();     // barriers of BOTH CTAs initialised and TMEM of both allocated before anyone signals
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  const int units = p.n_ut * p.n_ranges;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0, it = 0;
      for (int unit = cluster; unit < units; unit += n_clusters, ++it) {
        const int ut = unit % p.n_ut, range = unit / p.n_ut;
        mbar_wait(a_empty, (it & 1u) ^ 1u);
        if (rank == 0) mbar_arrive_expect_tx(a_full, 2 * kKB * kTile16K);
        for (int kb = 0; kb < kKB; ++kb)
          tma_load_2d_pair(sA + kb * kTile16K, &tmU, a_full, kb * 64, ut * kUT + static_cast<int>(rank) * 128);
        const int tile0 = range * p.tiles_per_range;
        const int tile1 = min(p.total_tiles, tile0 + p.tiles_per_range);
        for (int tile = tile0; tile < tile1; ++tile) {
          for (int kb = 0; kb < kKB; ++kb) {
            mbar_wait(&b_empty[stage], phase ^ 1u);
            if (rank == 0) mbar_arrive_expect_tx(&b_full[stage], 2 * kTile16K);
            tma_load_2d_pair(sB + stage * kTile16K, &tmI, &b_full[stage], kb * 64,
                             tile * p.tile_stride * kIT + static_cast<int>(rank) * 128);
            if (++stage == kBStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0 && elect_one()) {
      const uint32_t idesc = umma_idesc_bf16(256, kIT, false, false);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0, it = 0;
      for (int unit = cluster; unit < units; unit += n_clusters, ++it) {
        const int range = unit / p.n_ut;
        const int tile0 = range * p.tiles_per_range;
        const int tile1 = min(p.total_tiles, tile0 + p.tiles_per_range);
        mbar_wait(a_full, it & 1u);
        tc_fence_after();
        for (int tile = tile0; tile < tile1; ++tile) {
          mbar_wait(&t_empty[acc], acc_phase ^ 1u);
          tc_fence_after();
          const uint32_t d = tmem_base + static_cast<uint32_t>(acc * kIT);
          for (int kb = 0; kb < kKB; ++kb) {
            mbar_wait(&b_full[stage], phase);
            tc_fence_after();
            const uint32_t a_base = smem_u32(sA + kb * kTile16K);
            const uint32_t b_base = smem_u32(sB + stage * kTile16K);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_pair(d, umma_desc_kmajor(a_base + k * 32), umma_desc_kmajor(b_base + k * 32), idesc,
                             (kb > 0 || k > 0) ? 1u : 0u);
            umma_commit_pair(&b_empty[stage]);
            if (++stage == kBStages) { stage = 0; phase ^= 1u; }
          }
          umma_commit_pair(&t_full[acc]);
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1u;
        }
        umma_commit_pair(a_empty);  // the resident user tiles may be replaced once these MMAs retire
      }
    }
  } else if (warp >= 4) {
    // Sixteen epilogue warps per CTA: TMEM lane quarter q (32 user rows) x column quarter (64 of the step's
    // 256 items = two 32-score chunks). What bounds a step is the LATENCY of the slowest warp's chunk chain
    // (TMEM load -> max tree -> vote -> rare candidate re-read), because the accumulator buffer is released
    // only when all 32 warps of the pair are done and there are just two buffers: with eight warps x four
    // chunks the pass ran at (MMA + scan) / 2 per step with both sides waiting for each other (ncu: t_full
    // and t_empty waits both hot); handing alternate steps to two sets of eight warps left that chain as
    // long as before. Two chunks per warp halve it. Warps that share a user row append to separate lists.
    const int e = warp - 4;                  // 0..15
    const int colq = e >> 2, q = e & 3;      // q == warp % 4: TMEM lane quarter
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int unit = cluster; unit < units; unit += n_clusters) {
      const int ut = unit % p.n_ut, range = unit / p.n_ut;
      const int tile0 = range * p.tiles_per_range;
      const int tile1 = min(p.total_tiles, tile0 + p.tiles_per_range);
      const int row = ut * kUT + static_cast<int>(rank) * 128 + q * 32 + lane;
      const bool active = row < p.U;
      const size_t list = static_cast<size_t>(range) * kLists + colq;
      unsigned long long* buf = p.cand + (list * p.u_pad + row) * kCap;
      unsigned long long thr_key = active ? p.thr[row] : ~0ull;
      float thr_s = thr_key == 0ull ? -INFINITY : (active ? key_score(thr_key) : INFINITY);
      int cnt = 0;
      // word of the retired bitmap for this warp's 64 columns of step `tile` (sample pass: of physical step
      // tile * tile_stride); the next step's word is in flight while this step is scanned
      const auto retired_word = [&](int tile) -> uint64_t {
        return __ldg(p.retired + static_cast<size_t>(tile) * p.tile_stride * (kIT / 64) + colq);
      };
      uint64_t rb_next = 0;
      if constexpr (kLive) rb_next = tile0 < tile1 ? retired_word(tile0) : 0ull;
      for (int tile = tile0; tile < tile1; ++tile) {
        uint64_t rb = 0;
        if constexpr (kLive) {
          rb = rb_next;
          if (tile + 1 < tile1) rb_next = retired_word(tile + 1);
        }
        mbar_wait(&t_full[acc], acc_phase);
        __syncwarp();
        tc_fence_after();
        const uint32_t t_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                                static_cast<uint32_t>(acc * kIT + colq * 64);
        uint32_t r0[32], r1[32];
        tmem_ld32(t_base, r0);
        tmem_ld32(t_base + 32, r1);
        uint32_t dead = 0;   // main pass: 4-score groups whose items are all retired (computed under the TMEM load)
        if constexpr (kLive && !kSample) {
          uint64_t x = rb & (rb >> 1);
          x &= (x >> 2) & 0x1111111111111111ull;              // bit 4g: group g fully retired
          x = (x | (x >> 3)) & 0x0303030303030303ull;
          x = (x | (x >> 6)) & 0x000F000F000F000Full;
          x = (x | (x >> 12)) & 0x000000FF000000FFull;
          dead = static_cast<uint32_t>(x | (x >> 24)) & 0xFFFFu;
        }
        if constexpr (kSample) {
          // sample pass: one float per (user, chunk) — the chunk's best score; layout [user][chunk]
          float* dst = p.smax + static_cast<size_t>(row) * (p.total_tiles * kChunks) + tile * kChunks + colq * 2;
          tmem_ld_wait();
          if (kLive && rb != 0ull) {
#pragma unroll
            for (int t = 0; t < 32; ++t) {
              if ((rb >> t) & 1ull) r0[t] = 0xFF800000u;          // -inf
              if ((rb >> (32 + t)) & 1ull) r1[t] = 0xFF800000u;
            }
          }
          dst[0] = chunk_max(r0);
          dst[1] = chunk_max(r1);
        } else {
          tmem_ld_wait();
          uint32_t gm0 = chunk_group_mask(r0, thr_s);
          uint32_t gm1 = chunk_group_mask(r1, thr_s);
          if constexpr (kLive) {   // fully retired groups leave the vote
            gm0 &= ~dead & 0xFFu;
            gm1 &= ~(dead >> 8);
          }
          if (__any_sync(0xffffffffu, (gm0 | gm1) != 0u)) {
            const int idx0 = tile * kIT + colq * 64;
            collect_groups<kExclude, kLive>(gm0 | (gm1 << 8), t_base, idx0, p, lane, row, buf, cnt, thr_key, thr_s, rb);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&t_empty[acc], 0);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
      if constexpr (kExclude) {
        if (active && cnt > 0) cnt = drop_excluded_row(buf, cnt, p, row);
      }
      if constexpr (!kSample) p.cand_cnt[list * p.u_pad + row] = active ? cnt : 0;
    }
  }

  // Neither CTA may leave while its partner can still read its shared memory (the leader's MMAs), signal
  // its barriers (multicast commits, remote arrivals) or write its TMEM.
  tc_fence_before();
  __syncwarp();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_pair(tmem_base, 512);
}

// --------------------------------------------------------------------------------------------
// Sample pass -> per-user start threshold. The sample pass scores every `tile_stride`-th item tile
// and stores, per user, the maximum of each 32-score chunk (nothing is collected, nothing pruned:
// it runs at the fast-path rate). If a fraction q = target / N of the items beat a score t, a chunk
// maximum beats it with probability p = 1 - (1-q)^32, so the rank-(p * n_chunks) chunk maximum
// estimates the score that about `target` = 4 K' items of the catalog exceed. The main pass collects
// only scores above it (no pruning, mostly the fast path). It is a heuristic STARTING point only:
// tt_topk_finalize verifies that enough candidates were found plus the exactness certificate, and
// users for which that fails go to the exact fallback. One warp per user, maxima held in registers.
// With exclusions (ex_cnt != nullptr) the sample still scores every item, and an excluded item can own a chunk
// maximum: the rank rises by the number of the user's excluded ids inside the sampled item steps (step index a
// multiple of tile_stride, below sample_tiles * tile_stride). Each lifts at most one chunk maximum, so the
// (rank + e)-th raw maximum is at most the rank-th maximum over admissible items.
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sample_threshold_kernel(const float* __restrict__ smax, int U, int n_chunks,
                                                               int rank, unsigned long long* __restrict__ thr,
                                                               const int* __restrict__ ex_ids,
                                                               const int* __restrict__ ex_cnt, int ex_ld,
                                                               int item_base, int N, int tile_stride,
                                                               int sample_tiles) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int kMaxPerLane = 32;   // up to 1024 chunk maxima per user
  const int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (u >= U) return;
  if (ex_cnt != nullptr) {
    const int* ids = ex_ids + static_cast<size_t>(u) * ex_ld;
    const int n = ex_cnt[u];
    int e = 0;
    for (int i = lane; i < n; i += 32) {
      const int local = ids[i] - item_base;
      const int tile = local / kIT;
      e += (local >= 0 && local < N && tile % tile_stride == 0 && tile < sample_tiles * tile_stride) ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
    rank += e;
  }
  const float* row = smax + static_cast<size_t>(u) * n_chunks;
  uint32_t v[kMaxPerLane];
#pragma unroll
  for (int e = 0; e < kMaxPerLane; ++e) {
    const int i = e * 32 + lane;
    v[e] = i < n_chunks ? f2ord(row[i]) : 0u;
  }
  uint32_t t = 0;
  for (int bit = 31; bit >= 0; --bit) {
    const uint32_t cand = t | (1u << bit);
    int c = 0;
#pragma unroll
    for (int e = 0; e < kMaxPerLane; ++e) c += (v[e] >= cand);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (c >= rank) t = cand;
  }
  if (lane == 0) thr[u] = static_cast<unsigned long long>(t) << 32;
}

// --------------------------------------------------------------------------------------------
// Finalize: one block (256 threads) per user.
// --------------------------------------------------------------------------------------------
struct FinalizeParams {
  int U, N, item_base, n_ranges, u_pad, kprime, K;
  const unsigned long long* cand;
  const int* cand_cnt;
  const unsigned long long* thr;  // [u_pad] published thresholds
  const float* users;   // [U, 256] fp32
  const float* items;   // [N, 256] fp32 (this shard)
  float eps;            // bound on |bf16-path score - exact score| (host value), or, when eps_stats != nullptr,
  const float* eps_stats;  // device {max ||bf16(u) - u||, max ||u||} of this pass (users_prepare_kernel):
  float ne_max, de_max;    //   eps = du * ne_max + nu * de_max + nu * ne_max * 2^-18, evaluated on the device
  int* out_idx;         // [U, ld_out] global item index, -1 padded
  float* out_score;     // [U, ld_out]
  int ld_out;           // elements between consecutive users in out_idx / out_score
  int* flags;           // [U * ld_aux] 1 = certificate failed (fallback needed)
  float* bound;         // bounded mode (non-null): [U * ld_aux] every item of the shard NOT in the list has exact score <= bound
  int ld_aux;
  int pool_cap;         // keys the shared-memory pool holds (<= kPoolCap)
};

__device__ __forceinline__ float finalize_eps(const FinalizeParams& p) {
  if (p.eps_stats == nullptr) return p.eps;
  const float du = p.eps_stats[0], nu = p.eps_stats[1];
  // Cauchy-Schwarz on the bf16 rounding errors of both operands + fp32 accumulation slack, rounded up
  return (du * p.ne_max + nu * p.de_max + nu * p.ne_max * 3.8146973e-06f) * 1.000001f;
}

__device__ __forceinline__ int block_sum_int(int v, int* s_red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  int t = 0;
  for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) t += s_red[w];
  __syncthreads();
  return t;
}

// Bitonic sort (descending) of the first `n` (a power of two <= 256) keys in shared memory by 256 threads.
__device__ __forceinline__ void bitonic_sort_desc_256(unsigned long long* keys, int n = 256) {
  const int i = threadIdx.x;
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      const int j = i ^ stride;
      if (j > i && j < n) {
        const unsigned long long a = keys[i], b = keys[j];
        const bool desc = ((i & size) == 0);
        if (desc ? (a < b) : (a > b)) { keys[i] = b; keys[j] = a; }
      }
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256, 4) topk_finalize_kernel(const FinalizeParams p) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ unsigned long long s_keys[256];
  __shared__ unsigned long long s_sel[256];
  extern __shared__ unsigned long long s_pool[];   // p.pool_cap keys (2048 for short shard lists: 8 blocks per SM)
  __shared__ int s_red[8];
  __shared__ int s_n;
  __shared__ int s_off[kMaxLists + 1];
  const int u = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // Gather this user's candidate keys into shared memory, dropping everything below a floor key
  // that is known to have at least K' keys at or above it. First floor: the published threshold
  // thr[u] (the largest "K'-th best of one work unit"). If the pool still overflows, the floor is
  // raised by a bitwise search over the keys in global memory that stops as soon as the count fits.
  unsigned long long floor_key = p.thr[u];
  int npool = 0;
  // Offsets of this user's lists (a few dozen lists of a few dozen keys each): counts are loaded in one
  // parallel round and scanned by warp 0, so that the keys can then be fetched as ONE flat array — every
  // thread's loads are independent of each other (two global-load latencies for the whole gather instead
  // of a count -> keys chain per list).
  const int n_lists = p.n_ranges;
  for (int r = tid; r < n_lists; r += 256) s_off[r + 1] = p.cand_cnt[static_cast<size_t>(r) * p.u_pad + u];
  __syncthreads();
  if (warp == 0) {
    const int per = (n_lists + 31) / 32;
    const int b0 = min(lane * per, n_lists), b1 = min(b0 + per, n_lists);
    int sum = 0;
    for (int r = b0; r < b1; ++r) sum += s_off[r + 1];
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    int run = incl - sum;
    if (lane == 0) s_off[0] = 0;
    for (int r = b0; r < b1; ++r) { run += s_off[r + 1]; s_off[r + 1] = run; }
  }
  __syncthreads();
  const int total = s_off[n_lists];
  for (int attempt = 0; attempt < 2; ++attempt) {
    if (tid == 0) s_n = 0;
    __syncthreads();
    for (int f = tid; f < total; f += 256) {
      int lo = 0, hi = n_lists - 1;          // last list r with s_off[r] <= f
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (s_off[mid] <= f) lo = mid; else hi = mid - 1;
      }
      const unsigned long long k = p.cand[(static_cast<size_t>(lo) * p.u_pad + u) * kCap + (f - s_off[lo])];
      if (k >= floor_key) {
        const int pos = atomicAdd(&s_n, 1);
        if (pos < p.pool_cap) s_pool[pos] = k;
      }
    }
    __syncthreads();
    npool = s_n;
    __syncthreads();
    if (npool <= p.pool_cap || attempt == 1) break;
    unsigned long long t = 0;
    for (int bit = 63; bit >= 0; --bit) {
      const unsigned long long cand = t | (1ull << bit);
      int c = 0;
      for (int r = 0; r < p.n_ranges; ++r) {
        const int n = p.cand_cnt[static_cast<size_t>(r) * p.u_pad + u];
        const unsigned long long* b = p.cand + (static_cast<size_t>(r) * p.u_pad + u) * kCap;
        for (int i = tid; i < n; i += 256) c += (b[i] >= cand);
      }
      c = block_sum_int(c, s_red);
      if (c >= p.kprime) {
        t = cand;
        if (c <= p.pool_cap) break;
      }
    }
    if (t > floor_key) floor_key = t;
  }
  const bool overflow = npool > p.pool_cap;   // only massive exact-tie floods: exact fallback
  const int np = min(npool, p.pool_cap);

  // K'-th largest key of the pool (bitwise binary search over shared memory)
  unsigned long long T = 0;
  if (np > p.kprime) {
    for (int bit = 63; bit >= 0; --bit) {
      const unsigned long long cand = T | (1ull << bit);
      int c = 0;
      for (int i = tid; i < np; i += 256) c += (s_pool[i] >= cand);
      c = block_sum_int(c, s_red);
      if (c >= p.kprime) {
        T = cand;
        if (c == p.kprime) break;
      }
    }
  }
  if (tid == 0) s_n = 0;
  s_keys[tid] = 0ull;
  __syncthreads();
  for (int i = tid; i < np; i += 256) {
    const unsigned long long k = s_pool[i];
    if (k >= T) {
      const int pos = atomicAdd(&s_n, 1);
      if (pos < 256) s_sel[pos] = k;
    }
  }
  __syncthreads();
  const int nsel = min(s_n, 256);
  if (T < floor_key) T = floor_key;   // every non-pool item has key <= floor_key: bound for the certificate

  // exact re-score: fp32 inputs, fp64 accumulate, one rounding to fp32
  const float* urow = p.users + static_cast<size_t>(u) * kD;
  float uf[8];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(urow) + k * 32 + lane);
    uf[4 * k] = x.x; uf[4 * k + 1] = x.y; uf[4 * k + 2] = x.z; uf[4 * k + 3] = x.w;
  }
  // Four candidates per warp iteration: their eight 16-byte loads per lane are all issued before the first
  // dependent fp64 operation (a random 1 KB row gather is latency-bound otherwise: 36 % of the HBM peak with
  // one row in flight per warp). The per-candidate operation order is unchanged, so scores are bit-identical.
  for (int c0 = warp; c0 < nsel; c0 += 32) {
    float4 x[4][2];
    uint32_t gi[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cidx = c0 + 8 * j;
      gi[j] = key_idx(s_sel[cidx < nsel ? cidx : c0]);
      const float* irow = p.items + static_cast<size_t>(gi[j] - p.item_base) * kD;
#pragma unroll
      for (int k = 0; k < 2; ++k) x[j][k] = __ldg(reinterpret_cast<const float4*>(irow) + k * 32 + lane);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double acc = 0.0;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        acc += static_cast<double>(uf[4 * k]) * x[j][k].x + static_cast<double>(uf[4 * k + 1]) * x[j][k].y +
               static_cast<double>(uf[4 * k + 2]) * x[j][k].z + static_cast<double>(uf[4 * k + 3]) * x[j][k].w;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      const int cidx = c0 + 8 * j;
      if (lane == 0 && cidx < nsel) s_keys[cidx] = make_key(static_cast<float>(acc), gi[j]);
    }
  }
  __syncthreads();
  {
    int n_sort = 32;                       // nsel <= kprime <= 256 keys, the rest of s_keys is zero
    while (n_sort < p.kprime) n_sort <<= 1;
    bitonic_sort_desc_256(s_keys, n_sort);
  }

  for (int k = tid; k < p.K; k += 256) {
    const bool ok = k < nsel;
    p.out_idx[static_cast<size_t>(u) * p.ld_out + k] = ok ? static_cast<int>(key_idx(s_keys[k])) : -1;
    p.out_score[static_cast<size_t>(u) * p.ld_out + k] = ok ? key_score(s_keys[k]) : -INFINITY;
  }
  const float eps = finalize_eps(p);
  if (tid == 0 && p.bound != nullptr) {
    // Bounded mode (sharded catalogs): the list is every candidate with bf16-path key >= T, re-scored
    // exactly; every other item of the shard has exact score <= score(T) + eps. The caller merges the
    // shards' lists and checks that the merged K-th score beats every shard's bound.
    p.bound[static_cast<size_t>(u) * p.ld_aux] = overflow ? INFINITY : (T == 0ull ? -INFINITY : key_score(T) + eps);
    p.flags[static_cast<size_t>(u) * p.ld_aux] = overflow ? 1 : 0;
  } else if (tid == 0) {
    // Certificate: every non-candidate has bf16-path key < T, hence exact score <= score(T) + eps.
    // If the exact K-th best beats that, no non-candidate can enter the top K.
    // T == 0 means every item of the shard is a candidate (tiny catalog, no threshold): exact.
    int flag = overflow ? 1 : 0;
    if (!overflow && T != 0ull) {
      if (nsel < p.K) flag = 1;   // the start threshold was too high for this user
      else flag = !(key_score(s_keys[p.K - 1]) > key_score(T) + eps);
    }
    p.flags[static_cast<size_t>(u) * p.ld_aux] = flag;
  }
}

// --------------------------------------------------------------------------------------------
// Cross-shard merge: lists [G][U][K] of (score, global idx) sorted canonically per shard ->
// top K of their union, canonical order. One block per user; G*K <= 1024.
// --------------------------------------------------------------------------------------------
// Rows of shard g / user u start at (g * U + u) * row_stride in `scores` and `idx` (two views of one packed buffer
// or two separate arrays). aux != nullptr (packed exchange buffer, retrieval.sharded_topk): aux[(g*U+u)*row_stride]
// is the shard's completeness bound (fp32 bits) and the next word its tie-flood flag; then bad[u] receives the
// merged list's certificate: 0 iff the K_out-th merged score beats every shard's bound (or every shard listed all
// of its items) and no shard flagged the user.
__global__ void __launch_bounds__(256) topk_merge_kernel(const float* __restrict__ scores, const int* __restrict__ idx,
                                                         long long row_stride, const int* __restrict__ aux,
                                                         int G, int U, int K, int K_out, float* __restrict__ out_score,
                                                         int* __restrict__ out_idx, int* __restrict__ bad) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ unsigned long long s_all[];  // G lists of K keys, each sorted descending (0 = padding, at the end)
  __shared__ unsigned long long s_kth_key;
  const int u = blockIdx.x;
  const int n = G * K;
  if (threadIdx.x == 0) s_kth_key = 0ull;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int g = i / K, k = i % K;
    const size_t o = (static_cast<size_t>(g) * U + u) * row_stride + k;
    const int id = idx[o];
    s_all[i] = id < 0 ? 0ull : make_key(scores[o], static_cast<uint32_t>(id));
  }
  // Every shard's list arrives sorted in the canonical order, so the merged rank of a key is its position in its own
  // list plus, for every other list, the number of keys ahead of it there — a binary search per list (log2 K steps)
  // instead of comparing against all G*K keys (the first version: 430 us for 10 k users x 8 shards x 64 entries)
  // and without the ~45 block-wide barriers of a bitonic sort (235 us). Keys are unique (distinct items).
  for (int k = threadIdx.x; k < K_out; k += blockDim.x) {      // default: fewer than K_out items in the union
    out_score[static_cast<size_t>(u) * K_out + k] = -INFINITY;
    out_idx[static_cast<size_t>(u) * K_out + k] = -1;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const unsigned long long key = s_all[i];
    if (key == 0ull) continue;
    const int g = i / K;
    int rank = i - g * K;
    for (int h = 0; h < G; ++h) {
      if (h == g) continue;
      const unsigned long long* list = s_all + h * K;
      int lo = 0, hi = K;                      // first position whose key is NOT greater than `key`
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (list[mid] > key) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < K_out) {
      out_score[static_cast<size_t>(u) * K_out + rank] = key_score(key);
      out_idx[static_cast<size_t>(u) * K_out + rank] = static_cast<int>(key_idx(key));
      if (rank == K_out - 1) s_kth_key = key;
    }
  }
  __syncthreads();
  if (bad != nullptr && threadIdx.x == 0) {
    float bmax = -INFINITY;
    int flagged = 0;
    for (int g = 0; g < G; ++g) {
      const size_t o = (static_cast<size_t>(g) * U + u) * row_stride;
      bmax = fmaxf(bmax, __int_as_float(aux[o]));
      flagged |= aux[o + 1];
    }
    const unsigned long long kth = s_kth_key;
    // K_out merged entries exist: the K_out-th must beat every shard's bound; fewer: fine only when every shard
    // listed ALL of its items (bound = -inf)
    const bool ok = kth != 0ull ? (key_score(kth) > bmax) : (bmax == -INFINITY);
    bad[u] = (!ok || flagged) ? 1 : 0;
  }
}

// --------------------------------------------------------------------------------------------
// Exact fallback for users whose certificate failed: brute-force fp64-accumulated scores over
// the whole shard into a key array, then K-th largest by bitwise search + sort. Slow and rare.
// --------------------------------------------------------------------------------------------
// kLive: rows whose bit in `retired` is set get key 0, like item 0 under mask_item0.
template <bool kLive>
__global__ void __launch_bounds__(256) exact_keys_kernel(const float* __restrict__ user, const float* __restrict__ items,
                                                         int N, int item_base, int mask_item0,
                                                         const uint32_t* __restrict__ retired,
                                                         unsigned long long* __restrict__ keys) {
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  float uf[8];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(user) + k * 32 + lane);
    uf[4 * k] = x.x; uf[4 * k + 1] = x.y; uf[4 * k + 2] = x.z; uf[4 * k + 3] = x.w;
  }
  for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < N; i += warps) {
    const float* irow = items + static_cast<size_t>(i) * kD;
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(irow) + k * 32 + lane);
      acc += static_cast<double>(uf[4 * k]) * x.x + static_cast<double>(uf[4 * k + 1]) * x.y +
             static_cast<double>(uf[4 * k + 2]) * x.z + static_cast<double>(uf[4 * k + 3]) * x.w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      const uint32_t gidx = static_cast<uint32_t>(item_base + i);
      bool drop = mask_item0 && gidx == 0u;
      if constexpr (kLive) drop = drop || ((__ldg(retired + (i >> 5)) >> (i & 31)) & 1u);
      keys[i] = drop ? 0ull : make_key(static_cast<float>(acc), gidx);
    }
  }
}

// Exact fallback with exclusions: zero the keys of the user's excluded ids that lie in this shard. A key of 0 is
// never selected (the same way mask_item0 removes item 0).
__global__ void __launch_bounds__(256) exact_exclude_kernel(const int* __restrict__ ex_ids, const int* __restrict__ ex_cnt,
                                                            int N, int item_base, unsigned long long* __restrict__ keys) {
  pdl_launch_dependents();
  pdl_wait();
  const int n = *ex_cnt;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int local = ex_ids[i] - item_base;
    if (local >= 0 && local < N) keys[local] = 0ull;
  }
}

__global__ void __launch_bounds__(256) exact_select_kernel(const unsigned long long* __restrict__ keys, int N, int K,
                                                           float* __restrict__ out_score, int* __restrict__ out_idx) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ unsigned long long s_keys[256];
  __shared__ int s_red[8];
  __shared__ int s_n;
  const int tid = threadIdx.x;
  unsigned long long T = 0;
  const int want = min(K, 256);
  for (int bit = 63; bit >= 0; --bit) {
    const unsigned long long cand = T | (1ull << bit);
    int c = 0;
    for (int i = tid; i < N; i += 256) c += (keys[i] >= cand);
    c = block_sum_int(c, s_red);
    if (c >= want) {
      T = cand;
      if (c == want) break;
    }
  }
  if (tid == 0) s_n = 0;
  s_keys[tid] = 0ull;
  __syncthreads();
  for (int i = tid; i < N; i += 256) {
    const unsigned long long k = keys[i];
    if (k >= T && k != 0ull) {
      const int pos = atomicAdd(&s_n, 1);
      if (pos < 256) s_keys[pos] = k;
    }
  }
  __syncthreads();
  const int nsel = min(s_n, 256);
  bitonic_sort_desc_256(s_keys);
  for (int k = tid; k < K; k += 256) {
    const bool ok = k < nsel;
    out_idx[k] = ok ? static_cast<int>(key_idx(s_keys[k])) : -1;
    out_score[k] = ok ? key_score(s_keys[k]) : -INFINITY;
  }
}

// --------------------------------------------------------------------------------------------
// Recall@k / NDCG@k per row (src/evaluate_metrics.py:159-185). gain_table[r] = 1/log2(r+2) is
// supplied by the host (computed with the same fp32 torch ops as the reference) so the per-row
// values are bit-identical; the host then takes the mean exactly like the reference.
// --------------------------------------------------------------------------------------------
__global__ void rank_metrics_kernel(const int* __restrict__ topk, const int64_t* __restrict__ targets, int U, int K,
                                    const int* __restrict__ k_list, int nk, const float* __restrict__ gain_table,
                                    float* __restrict__ recall, float* __restrict__ ndcg) {
  pdl_launch_dependents();
  pdl_wait();
  const int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (u >= U) return;
  const int target = static_cast<int>(targets[u]);
  int rank = K;  // first position where the target appears
  for (int i = lane; i < K; i += 32)
    if (topk[static_cast<size_t>(u) * K + i] == target) rank = min(rank, i);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rank = min(rank, __shfl_xor_sync(0xffffffffu, rank, o));
  for (int j = lane; j < nk; j += 32) {
    const bool hit = rank < k_list[j];
    recall[static_cast<size_t>(j) * U + u] = hit ? 1.f : 0.f;
    ndcg[static_cast<size_t>(j) * U + u] = hit ? gain_table[rank] : 0.f;
  }
}

// fp32 user rows -> bf16 operand rows, plus the two user-side terms of the scoring-error bound for THIS pass:
// stats[0] = max_u ||bf16(u) - u||_2, stats[1] = max_u ||u||_2 (non-negative floats: integer atomicMax on the bits).
__global__ void __launch_bounds__(256) users_prepare_kernel(const float* __restrict__ users, __nv_bfloat16* __restrict__ out,
                                                            int U, float* __restrict__ stats) {
  pdl_launch_dependents();
  pdl_wait();
  const int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (u >= U) return;
  float d2 = 0.f, n2 = 0.f;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(users + static_cast<size_t>(u) * kD) + k * 32 + lane);
    uint2 b;
    b.x = pack_bf16(x.x, x.y);
    b.y = pack_bf16(x.z, x.w);
    reinterpret_cast<uint2*>(out + static_cast<size_t>(u) * kD)[k * 32 + lane] = b;
    const float2 r0 = unpack_bf16(b.x), r1 = unpack_bf16(b.y);
    const float e0 = r0.x - x.x, e1 = r0.y - x.y, e2 = r1.x - x.z, e3 = r1.y - x.w;
    d2 += e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3;
    n2 += x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
  }
  d2 = warp_sum(d2);
  n2 = warp_sum(n2);
  if (lane == 0) {
    // rounded up by a few ulps: these feed an upper bound
    atomicMax(reinterpret_cast<int*>(stats), __float_as_int(sqrtf(d2) * 1.00001f));
    atomicMax(reinterpret_cast<int*>(stats) + 1, __float_as_int(sqrtf(n2) * 1.00001f));
  }
}

// --------------------------------------------------------------------------------------------
// Per-user exclusion lists (the history masking of src/inference.py:296-302) in the form the selection epilogue
// probes: ids sorted ascending and de-duplicated, their count, and a 4096-bit hashed bitmap. One block per user;
// the row (0 = empty slot, ids <= 0 or >= vocab dropped) is padded with INT_MAX to a power of two >= 256, bitonic
// sorted in shared memory, and compacted with a block scan (each thread owns n_pad / 256 consecutive slots).
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) exclusions_build_kernel(const int64_t* __restrict__ in, int m, int ld_in,
                                                               int vocab, int n_pad, int* __restrict__ out_ids,
                                                               int ld, int* __restrict__ out_cnt,
                                                               uint32_t* __restrict__ out_bits) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ int s[kExclMax];
  __shared__ uint32_t s_bits[kExclWords];
  __shared__ int s_scan[8];
  const int u = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t* row = in + static_cast<size_t>(u) * ld_in;
  for (int i = tid; i < n_pad; i += 256) {
    const int64_t v = i < m ? row[i] : 0;
    s[i] = (v > 0 && v < vocab) ? static_cast<int>(v) : INT_MAX;
  }
  for (int i = tid; i < kExclWords; i += 256) s_bits[i] = 0u;
  for (int size = 2; size <= n_pad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int i = tid; i < n_pad; i += 256) {
        const int j = i ^ stride;
        if (j > i) {
          const int a = s[i], b = s[j];
          if (((i & size) == 0) ? (a > b) : (a < b)) { s[i] = b; s[j] = a; }
        }
      }
    }
  }
  __syncthreads();
  const int per = n_pad >> 8, b0 = tid * per;
  int c = 0;
  for (int e = 0; e < per; ++e) {
    const int i = b0 + e, v = s[i];
    c += (v != INT_MAX && (i == 0 || s[i - 1] != v)) ? 1 : 0;
  }
  int incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_scan[warp] = incl;
  __syncthreads();
  int pos = incl - c, total = 0;
  for (int w = 0; w < 8; ++w) {
    pos += w < warp ? s_scan[w] : 0;
    total += s_scan[w];
  }
  int* dst = out_ids + static_cast<size_t>(u) * ld;
  for (int e = 0; e < per; ++e) {
    const int i = b0 + e, v = s[i];
    if (v != INT_MAX && (i == 0 || s[i - 1] != v)) {
      dst[pos++] = v;
      const uint32_t h = excl_hash(static_cast<uint32_t>(v));
      atomicOr(&s_bits[h >> 5], 1u << (h & 31u));
    }
  }
  __syncthreads();
  for (int i = tid; i < kExclWords; i += 256) out_bits[static_cast<size_t>(u) * kExclWords + i] = s_bits[i];
  if (tid == 0) out_cnt[u] = total;
}

}  // namespace tt

using namespace tt;

extern "C" int tt_exclusions_build(const int64_t* ids, int U, int m, int ld_in, int vocab_size, int32_t* out_ids,
                                   int ld, int32_t* out_cnt, uint32_t* out_bits, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(out_ids && out_cnt && out_bits && U > 0 && m >= 0 && vocab_size > 0 && ld >= m && ld >= 1 &&
             (m == 0 || (ids && ld_in >= m)), "tt_exclusions_build: bad arguments");
  TT_REQUIRE(m <= kExclMax, "tt_exclusions_build: %d ids per user exceed %d", m, kExclMax);
  int n_pad = 256;
  while (n_pad < m) n_pad <<= 1;
  TT_CHECK_CUDA(launch_k(exclusions_build_kernel, dim3(U), dim3(256), 0, stream, ids, m, ld_in, vocab_size, n_pad,
                         out_ids, ld, out_cnt, out_bits));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_users_prepare(const float* users_f32, void* users_bf16, int U, float* stats, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(users_f32 && users_bf16 && stats && U > 0, "tt_users_prepare: bad arguments");
  TT_CHECK_CUDA(cudaMemsetAsync(stats, 0, 2 * sizeof(float), stream));
  TT_CHECK_CUDA(launch_k(users_prepare_kernel, dim3((U * 32 + 255) / 256), dim3(256), 0, stream, users_f32, static_cast<__nv_bfloat16*>(users_bf16), U, stats));
  TT_LAUNCH_CHECK();
  return TT_OK;
}


// persistent CTA pairs the launch will run: one per two SMs
static int num_pairs() {
  const int n = num_sms() / 2;
  return n < 1 ? 1 : n;
}

// Work units (user tile x item range) are dealt round-robin to the persistent CTA pairs, so a pass lasts
// as long as the pair with the most units: pick the number of ranges whose busiest pair scores the fewest
// item steps (e.g. 600 units on 148 workers = five units on eight of them, four on the rest: 23 % over
// the balanced time). Fewer ranges win ties (fewer candidate lists). `reload` = item steps' worth of time
// a unit spends refilling the resident user tile.
static int balanced_ranges(int n_ut, int total_tiles, int max_ranges, int reload) {
  int n_ranges = 1;
  long best = -1;
  for (int c = 1; c <= max_ranges; ++c) {
    const int tpr = (total_tiles + c - 1) / c;
    const int nr = (total_tiles + tpr - 1) / tpr;
    const long waves = (static_cast<long>(n_ut) * nr + num_pairs() - 1) / num_pairs();
    const long cost = 2 * waves * (tpr + reload) + c;   // + c/2 steps: every range adds lists to merge
    if (best < 0 || cost < best) { best = cost; n_ranges = c; }
  }
  return n_ranges;
}

extern "C" int tt_topk_plan_make(int U, int N, int kprime, tt_topk_plan* plan) {
  TT_REQUIRE(plan && U > 0 && N > 0, "tt_topk_plan_make: bad arguments");
  TT_REQUIRE(kprime >= 8 && kprime <= 256, "tt_topk_plan_make: kprime %d outside [8, 256]", kprime);
  plan->U = U; plan->N = N; plan->kprime = kprime; plan->cap = kCap;
  plan->n_ut = (U + kUT - 1) / kUT;
  const int total_tiles = (N + kIT - 1) / kIT;
  int max_ranges = (total_tiles + 31) / 32;        // at least 32 item steps (8192 items) per range
  if (max_ranges > 4 * num_pairs()) max_ranges = 4 * num_pairs();
  if (max_ranges > kMaxLists / kLists) max_ranges = kMaxLists / kLists;
  if (max_ranges < 1) max_ranges = 1;
  const int n_ranges = balanced_ranges(plan->n_ut, total_tiles, max_ranges, 2);
  plan->tiles_per_range = (total_tiles + n_ranges - 1) / n_ranges;
  plan->n_ranges = (total_tiles + plan->tiles_per_range - 1) / plan->tiles_per_range;
  const int64_t u_pad = static_cast<int64_t>(plan->n_ut) * kUT;
  plan->cand_bytes = static_cast<int64_t>(plan->n_ranges) * kLists * u_pad * kCap * 8;
  plan->cnt_bytes = static_cast<int64_t>(plan->n_ranges) * kLists * u_pad * 4;
  plan->thr_bytes = u_pad * 8;
  // Sample pass: chunk maxima of a strided subset of the item steps (see sample_threshold_kernel).
  plan->sample_stride = 0; plan->sample_rank = 0; plan->sample_tiles = 0; plan->smax_bytes = 0;
  if (total_tiles >= 128) {
    double target = 4.0 * kprime;
    if (target > N / 4.0) target = N / 4.0;
    const double q = target / N;
    const double pc = 1.0 - pow(1.0 - q, 32.0);
    int tiles = static_cast<int>(24.0 / pc / kChunks + 0.999);   // expected rank ~ 24
    if (tiles < 4) tiles = 4;
    if (tiles > total_tiles / 4) tiles = total_tiles / 4;
    if (tiles > 120) tiles = 120;                                 // <= 1024 chunk maxima per user (threshold kernel registers)
    const int stride = total_tiles / tiles;
    plan->sample_stride = stride;
    plan->sample_tiles = (total_tiles + stride - 1) / stride;
    // The threshold is the rank-th largest sampled chunk maximum. With few expected hits (huge catalogs: the
    // sample holds at most 1024 chunks, 3.2 expected hits at 10 M items) that rank statistic is noisy and
    // one user in a thousand got a start threshold above its own K'-th best score (exact fallback: a full
    // brute-force pass each). Two standard deviations of slack on small ranks costs candidates, not passes.
    double rexp = pc * plan->sample_tiles * kChunks;
    if (rexp < 16.0) rexp += 2.0 * sqrt(rexp);
    int rank = static_cast<int>(rexp + 0.5);
    if (rank < 4) rank = 4;
    plan->sample_rank = rank;
    plan->smax_bytes = static_cast<int64_t>(plan->sample_tiles) * kChunks * u_pad * 4;
  }
  return TT_OK;
}

static int launch_score_topk(const void* users_bf16, const void* items_bf16, TopkParams& p, int n_items_rows,
                             cudaStream_t stream) {
  CUtensorMap tmU, tmI;
  {
    uint64_t dims[2] = {kD, static_cast<uint64_t>(p.U)};
    uint64_t str[1] = {kD * 2};
    uint32_t box[2] = {64, 128};
    int rc = make_tmap_bf16(&tmU, users_bf16, 2, dims, str, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {kD, static_cast<uint64_t>(n_items_rows)};
    uint64_t str[1] = {kD * 2};
    uint32_t box[2] = {64, 128};
    int rc = make_tmap_bf16(&tmI, items_bf16, 2, dims, str, box);
    if (rc) return rc;
  }
  const size_t smem = 1024 + (kKB + kBStages) * kTile16K + 256;
  static bool configured = false;
  if (!configured) {
    TT_CHECK_CUDA(cudaFuncSetAttribute(score_topk_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    TT_CHECK_CUDA(cudaFuncSetAttribute(score_topk_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    TT_CHECK_CUDA(cudaFuncSetAttribute(score_topk_kernel<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    TT_CHECK_CUDA(cudaFuncSetAttribute(score_topk_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    TT_CHECK_CUDA(cudaFuncSetAttribute(score_topk_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    TT_CHECK_CUDA(cudaFuncSetAttribute(score_topk_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    configured = true;
  }
  const int units = p.n_ut * p.n_ranges;
  const int pairs = units < num_pairs() ? units : num_pairs();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(kTopkThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const bool live = p.retired != nullptr;
  if (p.smax != nullptr)
    TT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, live ? score_topk_kernel<true, false, true> : score_topk_kernel<true, false, false>, tmU, tmI, p));
  else if (p.ex_ids != nullptr)
    TT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, live ? score_topk_kernel<false, true, true> : score_topk_kernel<false, true, false>, tmU, tmI, p));
  else
    TT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, live ? score_topk_kernel<false, false, true> : score_topk_kernel<false, false, false>, tmU, tmI, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_score_topk(const void* users_bf16, const void* items_bf16, int item_base, const tt_topk_plan* plan,
                             void* cand, int32_t* cand_cnt, void* thr, void* smax, int mask_item0, void* stream_) {
  return tt_score_topk_excl(users_bf16, items_bf16, item_base, plan, cand, cand_cnt, thr, smax, mask_item0, nullptr,
                            nullptr, nullptr, 0, stream_);
}

extern "C" int tt_score_topk_excl(const void* users_bf16, const void* items_bf16, int item_base,
                                  const tt_topk_plan* plan, void* cand, int32_t* cand_cnt, void* thr, void* smax,
                                  int mask_item0, const int32_t* ex_ids, const int32_t* ex_cnt,
                                  const uint32_t* ex_bits, int ex_ld, void* stream_) {
  return tt_score_topk_live(users_bf16, items_bf16, item_base, plan, cand, cand_cnt, thr, smax, mask_item0, ex_ids,
                            ex_cnt, ex_bits, ex_ld, nullptr, stream_);
}

extern "C" int tt_score_topk_live(const void* users_bf16, const void* items_bf16, int item_base,
                                  const tt_topk_plan* plan, void* cand, int32_t* cand_cnt, void* thr, void* smax,
                                  int mask_item0, const int32_t* ex_ids, const int32_t* ex_cnt,
                                  const uint32_t* ex_bits, int ex_ld, const uint32_t* retired_bits, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(users_bf16 && items_bf16 && plan && cand && cand_cnt && thr, "tt_score_topk: null pointer");
  const bool excl = ex_ids != nullptr;
  TT_REQUIRE(excl == (ex_cnt != nullptr) && excl == (ex_bits != nullptr) && (!excl || ex_ld >= 1),
             "tt_score_topk_excl: exclusion ids, counts and bits must be given together (ex_ld >= 1)");
  TT_REQUIRE(reinterpret_cast<uintptr_t>(retired_bits) % 8 == 0, "tt_score_topk_live: retired_bits must be 8-byte aligned");
  TopkParams p;
  p.U = plan->U; p.N = plan->N; p.item_base = item_base;
  p.n_ut = plan->n_ut;
  p.total_tiles = (plan->N + kIT - 1) / kIT;
  p.kprime = plan->kprime;
  p.u_pad = plan->n_ut * kUT;
  p.cand = static_cast<unsigned long long*>(cand);
  p.cand_cnt = cand_cnt;
  p.thr = static_cast<unsigned long long*>(thr);
  p.mask_item0 = mask_item0;
  p.ex_ids = ex_ids; p.ex_cnt = ex_cnt; p.ex_bits = ex_bits; p.ex_ld = ex_ld;
  p.retired = reinterpret_cast<const unsigned long long*>(retired_bits);
  TT_CHECK_CUDA(cudaMemsetAsync(thr, 0, static_cast<size_t>(plan->thr_bytes), stream));

  // ---- sample pass: chunk maxima of every sample_stride-th item step -> per-user start thresholds
  p.smax = nullptr;
  if (plan->sample_stride > 1 && smax != nullptr && plan->sample_tiles * kChunks <= 1024) {
    const int sample_tiles = plan->sample_tiles;
    const int sr = balanced_ranges(p.n_ut, sample_tiles, sample_tiles < 16 ? sample_tiles : 16, 2);
    p.tile_stride = plan->sample_stride;
    p.tiles_per_range = (sample_tiles + sr - 1) / sr;
    p.n_ranges = (sample_tiles + p.tiles_per_range - 1) / p.tiles_per_range;
    const int total_saved = p.total_tiles;
    p.total_tiles = sample_tiles;
    p.smax = static_cast<float*>(smax);
    int rc = launch_score_topk(users_bf16, items_bf16, p, plan->N, stream);
    if (rc) return rc;
    TT_CHECK_CUDA(launch_k(sample_threshold_kernel, dim3((plan->U * 32 + 255) / 256), dim3(256), 0, stream, p.smax, plan->U, sample_tiles * kChunks, plan->sample_rank, p.thr, ex_ids, ex_cnt, ex_ld, item_base, plan->N, plan->sample_stride, sample_tiles));
    TT_LAUNCH_CHECK();
    p.total_tiles = total_saved;
    p.smax = nullptr;
  }
  // ---- main pass
  p.n_ranges = plan->n_ranges; p.tiles_per_range = plan->tiles_per_range;
  p.tile_stride = 1;
  return launch_score_topk(users_bf16, items_bf16, p, plan->N, stream);
}

struct EpsSpec { float eps; const float* stats; float ne_max, de_max; };

static int finalize_impl(const tt_topk_plan* plan, const void* cand, const int32_t* cand_cnt, const void* thr,
                         const float* users_f32, const float* items_f32, int item_base, int K, EpsSpec eps,
                         int32_t* out_idx, float* out_score, int ld_out, int32_t* flags, float* bound, int ld_aux,
                         void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(plan && cand && cand_cnt && thr && users_f32 && items_f32 && out_idx && out_score && flags,
             "tt_topk_finalize: null pointer");
  TT_REQUIRE(K > 0 && K <= plan->kprime, "tt_topk_finalize: K=%d must be in [1, kprime=%d]", K, plan->kprime);
  TT_REQUIRE(ld_out >= K && ld_aux >= 1, "tt_topk_finalize: output strides too small");
  TT_REQUIRE(plan->n_ranges * kLists <= kMaxLists, "tt_topk_finalize: %d candidate lists per user exceed %d",
             plan->n_ranges * kLists, kMaxLists);
  FinalizeParams p;
  p.U = plan->U; p.N = plan->N; p.item_base = item_base; p.n_ranges = plan->n_ranges * kLists;   // lists per row
  p.u_pad = plan->n_ut * kUT; p.kprime = plan->kprime; p.K = K;
  p.cand = static_cast<const unsigned long long*>(cand);
  p.cand_cnt = cand_cnt; p.thr = static_cast<const unsigned long long*>(thr); p.users = users_f32; p.items = items_f32;
  p.eps = eps.eps; p.eps_stats = eps.stats; p.ne_max = eps.ne_max; p.de_max = eps.de_max;
  p.out_idx = out_idx; p.out_score = out_score; p.ld_out = ld_out; p.flags = flags; p.bound = bound; p.ld_aux = ld_aux;
  p.pool_cap = plan->kprime <= 128 ? 2048 : kPoolCap;
  TT_CHECK_CUDA(launch_k(topk_finalize_kernel, dim3(plan->U), dim3(256), static_cast<size_t>(p.pool_cap) * 8, stream, p));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_topk_finalize(const tt_topk_plan* plan, const void* cand, const int32_t* cand_cnt, const void* thr,
                                const float* users_f32, const float* items_f32, int item_base, int K, float eps,
                                const float* eps_stats, float ne_max, float de_max,
                                int32_t* out_idx, float* out_score, int32_t* flags, void* stream_) {
  return finalize_impl(plan, cand, cand_cnt, thr, users_f32, items_f32, item_base, K, EpsSpec{eps, eps_stats, ne_max, de_max},
                       out_idx, out_score, K, flags, nullptr, 1, stream_);
}

extern "C" int tt_topk_finalize_bounded(const tt_topk_plan* plan, const void* cand, const int32_t* cand_cnt,
                                        const void* thr, const float* users_f32, const float* items_f32, int item_base,
                                        float eps, const float* eps_stats, float ne_max, float de_max,
                                        int32_t* out_idx, float* out_score, int ld_out, float* out_bound,
                                        int32_t* flags, int ld_aux, void* stream_) {
  TT_REQUIRE(plan && out_bound, "tt_topk_finalize_bounded: null pointer");
  return finalize_impl(plan, cand, cand_cnt, thr, users_f32, items_f32, item_base, plan->kprime,
                       EpsSpec{eps, eps_stats, ne_max, de_max}, out_idx, out_score, ld_out, flags, out_bound, ld_aux,
                       stream_);
}

static size_t merge_smem_bytes(int n) { return static_cast<size_t>(n) * 8; }

extern "C" int tt_topk_merge(const float* scores, const int32_t* idx, int G, int U, int K, float* out_score,
                             int32_t* out_idx, void* stream_) {
  return tt_topk_merge_lists(scores, idx, G, U, K, K, out_score, out_idx, stream_);
}

extern "C" int tt_topk_merge_lists(const float* scores, const int32_t* idx, int G, int U, int K_in, int K_out,
                                   float* out_score, int32_t* out_idx, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(scores && idx && out_score && out_idx && G > 0 && U > 0 && K_in > 0 && K_out > 0,
             "tt_topk_merge_lists: bad arguments");
  TT_REQUIRE(G * K_in <= 4096, "tt_topk_merge_lists: G*K_in = %d too large", G * K_in);
  TT_CHECK_CUDA(launch_k(topk_merge_kernel, dim3(U), dim3(256), merge_smem_bytes(G * K_in), stream, scores, idx, static_cast<long long>(K_in), static_cast<const int*>(nullptr), G, U, K_in, K_out, out_score, out_idx, static_cast<int*>(nullptr)));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_topk_merge_packed(const int32_t* packed, int ld, int G, int U, int K_in, int K_out, float* out_score,
                                    int32_t* out_idx, int32_t* bad, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(packed && out_score && out_idx && bad && G > 0 && U > 0 && K_in > 0 && K_out > 0 && ld >= 2 * K_in + 2,
             "tt_topk_merge_packed: bad arguments");
  TT_REQUIRE(G * K_in <= 4096, "tt_topk_merge_packed: G*K_in = %d too large", G * K_in);
  TT_CHECK_CUDA(launch_k(topk_merge_kernel, dim3(U), dim3(256), merge_smem_bytes(G * K_in), stream, reinterpret_cast<const float*>(packed), packed + K_in, static_cast<long long>(ld), packed + 2 * K_in, G, U, K_in, K_out, out_score, out_idx, bad));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_exact_topk(const float* user_f32, const float* items_f32, int N, int item_base, int mask_item0,
                             int K, void* key_scratch, float* out_score, int32_t* out_idx, void* stream_) {
  return tt_exact_topk_excl(user_f32, items_f32, N, item_base, mask_item0, K, nullptr, nullptr, key_scratch, out_score,
                            out_idx, stream_);
}

extern "C" int tt_exact_topk_excl(const float* user_f32, const float* items_f32, int N, int item_base, int mask_item0,
                                  int K, const int32_t* ex_ids, const int32_t* ex_cnt, void* key_scratch,
                                  float* out_score, int32_t* out_idx, void* stream_) {
  return tt_exact_topk_live(user_f32, items_f32, N, item_base, mask_item0, K, ex_ids, ex_cnt, nullptr, key_scratch,
                            out_score, out_idx, stream_);
}

extern "C" int tt_exact_topk_live(const float* user_f32, const float* items_f32, int N, int item_base, int mask_item0,
                                  int K, const int32_t* ex_ids, const int32_t* ex_cnt, const uint32_t* retired_bits,
                                  void* key_scratch, float* out_score, int32_t* out_idx, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(user_f32 && items_f32 && key_scratch && out_score && out_idx && N > 0 && K > 0 && K <= 256,
             "tt_exact_topk: bad arguments");
  TT_REQUIRE((ex_ids != nullptr) == (ex_cnt != nullptr), "tt_exact_topk_excl: exclusion ids and count go together");
  int grid = (N + 7) / 8;
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  if (retired_bits != nullptr)
    TT_CHECK_CUDA(launch_k(exact_keys_kernel<true>, dim3(grid), dim3(256), 0, stream, user_f32, items_f32, N, item_base, mask_item0, retired_bits, static_cast<unsigned long long*>(key_scratch)));
  else
    TT_CHECK_CUDA(launch_k(exact_keys_kernel<false>, dim3(grid), dim3(256), 0, stream, user_f32, items_f32, N, item_base, mask_item0, retired_bits, static_cast<unsigned long long*>(key_scratch)));
  TT_LAUNCH_CHECK();
  if (ex_ids != nullptr) {
    TT_CHECK_CUDA(launch_k(exact_exclude_kernel, dim3(1), dim3(256), 0, stream, ex_ids, ex_cnt, N, item_base, static_cast<unsigned long long*>(key_scratch)));
    TT_LAUNCH_CHECK();
  }
  TT_CHECK_CUDA(launch_k(exact_select_kernel, dim3(1), dim3(256), 0, stream, static_cast<const unsigned long long*>(key_scratch), N, K, out_score, out_idx));
  TT_LAUNCH_CHECK();
  return TT_OK;
}

extern "C" int tt_rank_metrics(const int32_t* topk_idx, const int64_t* targets, int U, int K, const int32_t* k_list,
                               int nk, const float* gain_table, float* recall, float* ndcg, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  TT_REQUIRE(topk_idx && targets && k_list && gain_table && recall && ndcg && U > 0 && K > 0 && nk > 0,
             "tt_rank_metrics: bad arguments");
  TT_CHECK_CUDA(launch_k(rank_metrics_kernel, dim3((U * 32 + 255) / 256), dim3(256), 0, stream, topk_idx, targets, U, K, k_list, nk, gain_table, recall, ndcg));
  TT_LAUNCH_CHECK();
  return TT_OK;
}
