// Shared device/host helpers for the sm_100a two-tower kernels.
//
// Everything here is thin: raw PTX wrappers for mbarrier / TMA / tcgen05 / TMEM,
// the UMMA shared-memory + instruction descriptor encoders, warp reductions,
// a counter-based dropout hash, and the host-side error/TMA-map helpers.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tt_b200.h"

namespace tt {

// ----------------------------------------------------------------------------
// Host-side error convention (C ABI returns int; message is thread-local)
// ----------------------------------------------------------------------------
enum : int {
  TT_OK = 0,
  TT_ERR_INVALID = 1,   // bad argument / unsupported shape
  TT_ERR_CUDA = 2,      // a CUDA runtime/driver call failed
  TT_ERR_WORKSPACE = 3, // caller workspace too small
};

void set_last_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define TT_CHECK_CUDA(expr)                                   \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return ::tt::cuda_fail(_e, #expr); \
  } while (0)

#define TT_REQUIRE(cond, ...)               \
  do {                                      \
    if (!(cond)) {                          \
      ::tt::set_last_error(__VA_ARGS__);    \
      return ::tt::TT_ERR_INVALID;          \
    }                                       \
  } while (0)

#define TT_LAUNCH_CHECK() TT_CHECK_CUDA(cudaGetLastError())

// Encode a tiled bf16 tensor map (rank 2 or 3), 128B swizzle. dims/strides are
// innermost-first; strides[] has rank-1 entries in BYTES (dim 0 is contiguous).
int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                   const uint64_t* strides_bytes, const uint32_t* box);
// The general form: bf16 or fp32 elements, 0 / 32 / 64 / 128-byte swizzle.
int make_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
              const uint32_t* box, int fp32, int swizzle_bytes);

int num_sms();

// The ID table as the sparse kernels (tt_sparse.cu) see it: one replicated table (world == 0: row `id` lives at
// base[0] + id * 256) or a table row-sharded ROUND-ROBIN over the ranks of one NVLink domain (row id lives at local
// row id / world of rank id % world; base[r] = rank r's shard as mapped into this process, symmetric arena).
// Round-robin because item popularity is Zipfian in the id (SURVEY.md §8d): contiguous ranges would put most of
// every rank's lookups on rank 0.
struct TableRef {
  float* base[16];
  int world;
#ifdef __CUDACC__
  __device__ __forceinline__ float* row(int64_t id) const {
    if (world == 0) return base[0] + static_cast<size_t>(id) * 256;
    const int64_t local = id / world;
    return base[static_cast<int>(id - local * world)] + static_cast<size_t>(local) * 256;
  }
#endif
};
int make_sharded_table(TableRef& t, const ::tt_symm_team* team, int64_t offset, const char* who);   // tt_sparse.cu

#ifdef __CUDACC__
// ----------------------------------------------------------------------------
// Programmatic dependent launch (PDL). Every kernel of the library
//   * signals `launch_dependents` as its first instruction, so the NEXT kernel of the stream (or
//     graph branch) may be scheduled while this one is still running, and
//   * executes `griddepcontrol.wait` before its first global-memory access; the wait returns only
//     when the previous kernel has completed and its writes are visible.
// What overlaps with the predecessor is therefore only launch latency and the prologue (barrier
// init, TMEM allocation, tensor-map prefetch) — semantics stay those of a serialized stream.
// launch_k sets the programmatic launch attribute only on grids of at most kPdlMaxCtas CTAs (without it
// the two instructions are no-ops). Measured on the c2 step: 1.308 ms with no programmatic launch,
// 1.326 ms with it on every launch, 1.282 ms with it on the small grids only.
// ----------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

constexpr size_t kPdlMaxCtas = 64;   // largest grid that launches programmatically

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                            Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  // Programmatic dependent launch lets this grid start (and run its prologue up to griddepcontrol.wait)
  // while the previous kernel in the stream drains. Early CTAs of a big grid would sit on SMs the
  // concurrent weight-gradient / item-tower streams could use, so only the small latency-bound
  // launches (B-row GEMMs, heads, loss), where launch + prologue latency is the cost, use it.
  const size_t ctas = static_cast<size_t>(grid.x) * grid.y * grid.z;
  cfg.numAttrs = ctas <= kPdlMaxCtas ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ----------------------------------------------------------------------------
// Small device utilities
// ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 rx;\n\t"
      ".reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, px;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}

// Counter-based dropout decision. keep-probability = 1 - p, encoded as a 32-bit threshold by
// the host (thresh = p * 2^32). Same (seed, site, idx) -> same bit in forward and backward, so
// no mask tensor is stored. The per-call key (seed, site) is loop-invariant; one 32-bit integer
// finaliser (two IMULs) is shared by four consecutive elements.
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x7feb352dU;
  x ^= x >> 15;
  x *= 0x846ca68bU;
  x ^= x >> 16;
  return x;
}
__device__ __forceinline__ uint32_t drop_key(uint64_t seed, uint32_t site) {
  return mix32(static_cast<uint32_t>(seed) ^ mix32(static_cast<uint32_t>(seed >> 32) + site * 0x9E3779B9u));
}
// One 32-bit hash decides FOUR consecutive elements: element idx uses word (idx & 3) of
// h = hash(idx >> 2), where word 0 is h itself and words 1..3 are h times three odd constants
// (a bijection of a well-mixed word; its high bits depend on every bit of h). Each word is
// compared with the full 32-bit threshold p * 2^32. Per element: 1/4 finaliser + 1 IMAD + 1 ISETP.
static constexpr uint32_t kDropMul1 = 0x9E3779B1u;
static constexpr uint32_t kDropMul2 = 0x85EBCA6Bu;
static constexpr uint32_t kDropMul3 = 0xC2B2AE35u;
__device__ __forceinline__ bool drop_keep_k(uint32_t key, uint64_t idx, uint32_t thresh) {
  const uint64_t quad = idx >> 2;
  const uint32_t x = static_cast<uint32_t>(quad) ^ (static_cast<uint32_t>(quad >> 32) * 0x85EBCA6Bu);
  const uint32_t h = mix32(x ^ key);
  const uint32_t j = static_cast<uint32_t>(idx) & 3u;
  const uint32_t mul = j == 0 ? 1u : (j == 1 ? kDropMul1 : (j == 2 ? kDropMul2 : kDropMul3));
  return h * mul >= thresh;
}
__device__ __forceinline__ bool drop_keep(uint64_t seed, uint32_t site, uint64_t idx, uint32_t thresh) {
  return drop_keep_k(drop_key(seed, site), idx, thresh);
}
// Pair form for an EVEN 32-bit index: k0 = keep(idx_even), k1 = keep(idx_even + 1), one hash.
__device__ __forceinline__ void drop_keep_pair(uint32_t key, uint32_t idx_even, uint32_t thresh, bool& k0, bool& k1) {
  const uint32_t h = mix32((idx_even >> 2) ^ key);
  const bool hi = (idx_even & 2u) != 0;
  k0 = h * (hi ? kDropMul2 : 1u) >= thresh;
  k1 = h * (hi ? kDropMul3 : kDropMul1) >= thresh;
}
// Quad form for a 32-bit index that is a multiple of 4: k[j] = keep(idx4 + j), one hash.
__device__ __forceinline__ void drop_keep_quad(uint32_t key, uint32_t idx4, uint32_t thresh, bool (&k)[4]) {
  const uint32_t h = mix32((idx4 >> 2) ^ key);
  k[0] = h >= thresh;
  k[1] = h * kDropMul1 >= thresh;
  k[2] = h * kDropMul2 >= thresh;
  k[3] = h * kDropMul3 >= thresh;
}
// 64-bit forms of the two above, bit-equal to drop_keep_k at every index (the 32-bit forms agree with it only below
// 2^32): the high word of the quad number enters the hash exactly as in drop_keep_k.
__device__ __forceinline__ uint32_t drop_quad_hash64(uint32_t key, uint64_t idx) {
  const uint64_t quad = idx >> 2;
  return mix32((static_cast<uint32_t>(quad) ^ (static_cast<uint32_t>(quad >> 32) * 0x85EBCA6Bu)) ^ key);
}
__device__ __forceinline__ void drop_keep_pair64(uint32_t key, uint64_t idx_even, uint32_t thresh, bool& k0, bool& k1) {
  const uint32_t h = drop_quad_hash64(key, idx_even);
  const bool hi = (idx_even & 2u) != 0;
  k0 = h * (hi ? kDropMul2 : 1u) >= thresh;
  k1 = h * (hi ? kDropMul3 : kDropMul1) >= thresh;
}
__device__ __forceinline__ void drop_keep_quad64(uint32_t key, uint64_t idx4, uint32_t thresh, bool (&k)[4]) {
  const uint32_t h = drop_quad_hash64(key, idx4);
  k[0] = h >= thresh;
  k[1] = h * kDropMul1 >= thresh;
  k[2] = h * kDropMul2 >= thresh;
  k[3] = h * kDropMul3 >= thresh;
}
// Packed fp32 pairs (sm_100 FFMA2 / FMUL2): d = a * b + c on two lanes in one issue slot.
__device__ __forceinline__ void ffma2(float& a0, float& a1, float b0, float b1, float c0, float c1) {
  uint64_t d;
  asm("{\n\t"
      ".reg .b64 ra, rb, rc;\n\t"
      "mov.b64 ra, {%1, %2};\n\t"
      "mov.b64 rb, {%3, %4};\n\t"
      "mov.b64 rc, {%5, %6};\n\t"
      "fma.rn.f32x2 %0, ra, rb, rc;\n\t"
      "}\n"
      : "=l"(d)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1), "f"(c0), "f"(c1));
  a0 = __uint_as_float(static_cast<uint32_t>(d));
  a1 = __uint_as_float(static_cast<uint32_t>(d >> 32));
}
__device__ __forceinline__ void fadd2(float& a0, float& a1, float b0, float b1) {
  uint64_t d;
  asm("{\n\t"
      ".reg .b64 ra, rb;\n\t"
      "mov.b64 ra, {%1, %2};\n\t"
      "mov.b64 rb, {%3, %4};\n\t"
      "add.rn.f32x2 %0, ra, rb;\n\t"
      "}\n"
      : "=l"(d)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
  a0 = __uint_as_float(static_cast<uint32_t>(d));
  a1 = __uint_as_float(static_cast<uint32_t>(d >> 32));
}
__device__ __forceinline__ void fmul2(float& a0, float& a1, float b0, float b1) {
  uint64_t d;
  asm("{\n\t"
      ".reg .b64 ra, rb;\n\t"
      "mov.b64 ra, {%1, %2};\n\t"
      "mov.b64 rb, {%3, %4};\n\t"
      "mul.rn.f32x2 %0, ra, rb;\n\t"
      "}\n"
      : "=l"(d)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
  a0 = __uint_as_float(static_cast<uint32_t>(d));
  a1 = __uint_as_float(static_cast<uint32_t>(d >> 32));
}
// 16-byte vector reduction into global memory (sm_90+: one RED instead of four)
__device__ __forceinline__ void red_add_f32x4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

// Register re-partitioning between warpgroups (setmaxnreg): every warp of a warpgroup (4 consecutive
// warps) executes the same instruction; the increase blocks until other warpgroups released enough.
template <int N>
__device__ __forceinline__ void reg_alloc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void reg_dealloc() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// ----------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (reported as a launch failure) instead of
// hanging the GPU forever.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) __trap();
  }
}

// ----------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor) loads into shared memory, completing on an mbarrier
// ----------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1), "r"(c2)
      : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (UMMA / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// TMA tensor store shared -> global (bulk async-group completion): the issuing thread commits the group and later
// waits either for the engine to have READ the shared tile (it may be overwritten) or for full completion.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }


// ----------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate; single thread issues.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all previously issued tcgen05.mma of this thread retire.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32"
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
      " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31},"
      "[%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&r)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32"
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15},"
      "[%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// ----------------------------------------------------------------------------
// CTA pair (cluster of 2, tcgen05 cta_group::2): one elected thread of the even-ranked ("leader") CTA
// issues M=256 MMAs that read A/B from BOTH CTAs' shared memory (same offsets) and write 128 lanes
// of TMEM in each CTA. Both CTAs run TMA producers whose transaction bytes land on the LEADER's
// full barrier; MMA completion is multicast to the barrier at the same offset in both CTAs.
// ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// In the shared::cluster window bit 24 of a CTA-local shared address selects the odd CTA of the pair;
// clearing it addresses the same offset in the leader.
static constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* leader_bar,
                                                 int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(leader_bar) & kPeerBitMask),
        "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* leader_bar,
                                                 int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(leader_bar) & kPeerBitMask),
        "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// arrive on the barrier at this offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
      "}\n"
      :
      : "r"(smem_u32(bar)), "r"(cta)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the barrier at this offset in BOTH CTAs receives one arrival once all MMAs issued so far retire
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// ----------------------------------------------------------------------------
// UMMA descriptors (bf16 operands, 128B swizzle, 1024B-aligned tiles)
//
// K-major operand tile  : rows = M/N index, 64 K-elements (128 B) per row, 8-row
//                         swizzle atoms of 1024 B  -> SBO = 1024, LBO unused (1).
// MN-major operand tile : rows = K index, 64 MN-elements (128 B) per row, 8 K-rows
//                         per 1024 B atom -> SBO = 1024 (next 8 K rows),
//                         LBO = byte distance between consecutive 64-wide MN chunks.
// ----------------------------------------------------------------------------
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ULL << 46;  // descriptor version (Blackwell)
  d |= 2ULL << 61;  // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ uint64_t umma_desc_kmajor(uint32_t smem_addr) {
  return umma_smem_desc(smem_addr, 16, 1024);
}
__device__ __forceinline__ uint64_t umma_desc_mnmajor(uint32_t smem_addr, uint32_t chunk_stride) {
  return umma_smem_desc(smem_addr, chunk_stride, 1024);
}
// kind::f16 instruction descriptor: bf16 x bf16 -> fp32, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n, bool a_mn, bool b_mn) {
  return (1u << 4)                        // D format fp32
         | (1u << 7)                      // A bf16
         | (1u << 10)                     // B bf16
         | ((a_mn ? 1u : 0u) << 15)       // A major
         | ((b_mn ? 1u : 0u) << 16)       // B major
         | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
#endif  // __CUDACC__

}  // namespace tt
