// Shared device/host helpers for the crowdmod B200 (sm_100a) hot path.
//
// PTX wrappers for mbarrier, TMA (tiled + im2col), tcgen05 (alloc / mma / commit / ld),
// plus error plumbing used by every translation unit.  sm_100a only — no fallbacks.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

namespace cm {

// ------------------------------------------------------------------------------------------
// error plumbing (host)
// ------------------------------------------------------------------------------------------
void set_error(const std::string& msg);          // api.cu
const char* get_error();

#define CM_CUDA(expr)                                                                        \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      char _b[512];                                                                          \
      snprintf(_b, sizeof(_b), "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                 \
               cudaGetErrorString(_e));                                                      \
      cm::set_error(_b);                                                                     \
      return 1;                                                                              \
    }                                                                                        \
  } while (0)

#define CM_CHECK(cond, ...)                                                                  \
  do {                                                                                       \
    if (!(cond)) {                                                                           \
      char _b[512];                                                                          \
      int _n = snprintf(_b, sizeof(_b), "%s:%d: check failed (%s): ", __FILE__, __LINE__,    \
                        #cond);                                                              \
      snprintf(_b + _n, sizeof(_b) - _n, __VA_ARGS__);                                       \
      cm::set_error(_b);                                                                     \
      return 2;                                                                              \
    }                                                                                        \
  } while (0)

// device-side "a wait timed out / something impossible happened" flag, checked by the host
// after tests (never read on the hot path).  One int per process.
int* device_error_flag();                        // api.cu (lazily cudaMalloc'ed, zeroed)

// ------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.0f + __expf(-x)); }

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

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
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
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug becomes a reported error (flag != 0) instead of a hung GPU.
// Returns false on timeout.  ~2^22 polls of a HW-suspending try_wait is seconds, far beyond
// any legitimate wait in these kernels.
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* err_flag, int code) {
  if (mbar_try_wait(bar, parity)) return true;
#pragma unroll 1
  for (uint32_t it = 0; it < (1u << 22); ++it) {
    if (mbar_try_wait(bar, parity)) return true;
  }
  if (err_flag) atomicExch(err_flag, code);
  return false;
}

// ------------------------------------------------------------------------------------------
// TMA
// ------------------------------------------------------------------------------------------
// 1-D bulk copy global -> shared (no tensor map): 16-byte aligned, size a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
// 2-D tiled load (weights): coords (c0 = innermost).
__device__ __forceinline__ void tma_load_2d(const void* desc, uint64_t* bar, void* smem, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(const void* desc, uint64_t* bar, void* smem, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "r"(c2)
      : "memory");
}
// 5-D im2col load (activations, NDHWC): coords {c, w, h, d, n} = first pixel of the column in
// bounding-box coordinates, offsets {w, h, d} = filter tap.
__device__ __forceinline__ void tma_load_im2col_5d(const void* desc, uint64_t* bar, void* smem,
                                                   int c, int w, int h, int d, int n,
                                                   uint16_t ow, uint16_t oh, uint16_t od) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2], {%8, %9, %10};"
      :
      : "r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c),
        "r"(w), "r"(h), "r"(d), "r"(n), "h"(ow), "h"(oh), "h"(od)
      : "memory");
}

// ------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
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
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (fp16/bf16 operands, fp32 accumulate)
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Lean form for the single issuing thread: descriptors as (lo, hi) 32-bit halves so that the
// per-MMA work is two integer adds (the hi halves are kernel constants).
__device__ __forceinline__ void umma_f16_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo,
                                              uint32_t desc_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}\n"
      :
      : "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TS form: the A operand (128 rows x 16 fp16 = 8 packed 32-bit columns per k16 step) is read from tensor memory, where
// tcgen05.cp (or tcgen05.st) put it; B stays a shared-memory descriptor.  Measured (tools/utccp_microbench.cu): an SS-mode
// MMA whose A tile differs from its predecessor's pays ~131 cycles for the A fetch whatever N is.
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t desc_hi,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}\n"
      :
      : "r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// shared memory -> tensor memory: 128 rows x 256 bits (one k16 slice of a K-major fp16 tile, same descriptor as the MMA's
// A operand) into lanes 0..127 x 8 columns at taddr.  Asynchronous; ordered with later tcgen05.mma of the same thread.
__device__ __forceinline__ void tmem_cp_128x256b(uint32_t taddr, uint32_t desc_lo, uint32_t desc_hi) {
  asm volatile(
      "{\n\t.reg .b64 ds;\n\t"
      "mov.b64 ds, {%1, %2};\n\t"
      "tcgen05.cp.cta_group::1.128x256b [%0], ds;\n\t}\n"
      :
      : "r"(taddr), "r"(desc_lo), "r"(desc_hi)
      : "memory");
}
__host__ __device__ constexpr uint32_t kmajor_desc_hi(int row_bytes) {
  return static_cast<uint32_t>(((8 * row_bytes) >> 4) & 0x3FFF) | (1u << 14) |
         (static_cast<uint32_t>(row_bytes == 128 ? 2 : 4) << 29);
}
__device__ __forceinline__ uint32_t kmajor_desc_lo(uint32_t smem_addr) {
  return ((smem_addr >> 4) & 0x3FFFu) | (1u << 16);
}

// arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::
                   "r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread (thread i <-> lane i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// 256-bit global stores (STG.E.256, sm_100+; p 32-byte aligned): a row-per-thread epilogue moves a full 32-byte sector per
// instruction instead of half of one
__device__ __forceinline__ void st_global_v8(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t* u) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]),
               "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7])
               : "memory");
}

// four consecutive fp32 adds into global memory as ONE reduction (REDG.E.ADD.F32x4, sm_90+; p 16-byte aligned): a quarter of
// the L2 atomic operations of four scalar atomicAdd() calls
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// same, without the wait: issue several loads, then tmem_ld_wait() once
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, float (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]),
        "=f"(v[8]), "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major shared-memory matrix descriptor for a TMA-written tile whose rows are `row_bytes`
// (128 -> SWIZZLE_128B, 64 -> SWIZZLE_64B) wide.  SBO = 8 rows; LBO unused (=1) for swizzled
// K-major; version = 1 (Blackwell).  Layout-type encoding: 2 = SW128, 4 = SW64.
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr, int row_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>(1) << 16;                                    // LBO (ignored)
  d |= static_cast<uint64_t>(((8 * row_bytes) >> 4) & 0x3FFF) << 32;      // SBO
  d |= static_cast<uint64_t>(1) << 46;                                    // version
  d |= static_cast<uint64_t>(row_bytes == 128 ? 2 : 4) << 61;             // swizzle mode
  return d;
}
// kind::f16 instruction descriptor: fp16 A/B (K-major both), fp32 D, M x N tile.
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// ------------------------------------------------------------------------------------------
// Philox4x32-10 counter RNG + Box-Muller (noise for the reverse chain in throughput mode).
// counter = (element index lo, element index hi, step, 0), key = seed: invariant to how the
// sample batch is sharded over GPUs.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  // u from the top 24 bits (+0.5): exact in fp32, u1 in (0,1) strictly (never rounds to 1.0, so -2 ln(u1) > 0
  // even with the ~2^-21 absolute error of __logf near 1: fmaxf guards the sqrt all the same), u2 in (0,1)
  float u1 = (static_cast<float>(a >> 8) + 0.5f) * 5.9604644775390625e-8f;
  float u2 = (static_cast<float>(b >> 8) + 0.5f) * 5.9604644775390625e-8f;
  float r = sqrtf(fmaxf(0.0f, -2.0f * __logf(u1)));
  float s, c;
  __sincosf(6.283185307179586f * u2, &s, &c);
  return make_float2(r * c, r * s);
}

}  // namespace cm
