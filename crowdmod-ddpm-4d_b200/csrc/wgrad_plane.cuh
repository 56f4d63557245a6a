// Weight gradient of the full-resolution k3 s1 p1 convs with 32 output channels (cuDNN backward-filter of
// encoder_blocks.0.conv_1/2 and the conv_1 / conv_2 of the two finest decoder blocks under loss.backward(); reference
// models/backbones/layers.py:32,43, models/diffusion/ddpm.py:143), plane / halo operand scheme, tcgen05 / TMEM / TMA, sm_100a.
//
//   G[(tap, ci), co] = sum_p  A[p + tap, ci] * dOut[p, co]
//
// wgrad_umma_kernel<32,32,32> fetches one im2col tile per (tap, 128 pixels): every tap re-reads the whole activation tensor
// (27 x 22 MB at the HERMES shape) and every M tile re-reads dOut -- 750 MB through L2 for a 19 GFLOP launch, 221 us, the top
// kernel of the training backward.  Here a unit is HB rows of one plane ((HB+2) * (W+2) a multiple of 16): ONE haloed box
// {32 ch, W+2, HB+3} per td plane and ONE dOut box {32 co, W+2, HB} (both zero-filled outside the tensor, so the pad columns
// and ragged row blocks contribute nothing) serve all 27 taps:
//   * both operands are MN-major (the reduction index = pixel is the strided one), rows of 64 bytes, SWIZZLE_64B;
//   * the three tw taps are the M dimension's 32-channel chunks at a leading-dimension byte offset of ONE box row (64 B):
//     M = 128 = (tw 0..3, ci), the fourth chunk is discarded (the UMMA swizzle is a function of the absolute shared-memory
//     address, so overlapping / row-offset views read correctly);
//   * the three th taps are stacked along N by shifting dOut instead of A: with p' = p + th*(W+2),
//     sum_p A[p + th*(W+2) + tw] dOut[p] = sum_p' A[p' + tw] dOut[p' - th*(W+2)], so N = 96 = (th = 2, 1, 0; co) are three
//     views of the dOut box one grid row apart (leading-dimension byte offset (W+2)*64) into a slot whose rows above and
//     below the box are zero (written once, never touched by TMA): ONE 128 x 96 x 16 MMA per (td, 16 pixels) -- an MN-major
//     MMA costs ~160 cycles here whatever N is (measured with the N = 32 version: 131 us per launch);
//   * three accumulators (td) of 96 columns live in TMEM for the whole launch: a persistent CTA adds all its units into
//     them and writes them out once (fp32 atomics into the packed-K G, as wgrad_umma_kernel; deterministic (DET): plain
//     stores of the CTA's 27 x 32 x 32 partial into `part`, summed in CTA order by wgrad_run_enqueue over a grid of
//     WP_DET_CTAS that depends on the shape only).
// One launch covers one 32-channel chunk of the source (c0); wider sources take one launch per chunk.
#pragma once
#include "common.cuh"
#include "conv_plane.cuh"
#include "wgrad_umma.cuh"

namespace cm {

constexpr int WP_THREADS = 192;     // warp0 TMA, warp1 MMA, warps2-5 epilogue
constexpr int WP_MAX_STAGES = 4;
constexpr int WP_DET_CTAS = 148;    // deterministic grid: min(units, this), a constant rather than the device's SM count
constexpr int WP_PART = 27 * 32 * 32;   // floats of one CTA's partial [tap][ci][co]

struct WgradPlaneParams {
  CUtensorMap amap;      // activations, tiled 5-D (C, W, H, D, N), box {32, W+2, HB+3, 1, 1}
  CUtensorMap gmap;      // dOut, tiled 5-D, box {32, W+2, HB, 1, 1}
  int H, W, D, Wp, HB;
  int hblocks;           // ceil(H / HB)
  int units_per_sample;  // D * hblocks
  int n_units;           // B * units_per_sample
  int c0;                // first channel of this launch's 32-channel chunk
  int ksteps;            // (HB + 2) * Wp / 16: pixels p' of the unit and of the two row blocks the th shifts reach
  int a_box_bytes, a_slot_bytes, g_box_bytes, stage_bytes, stages;
  int g_data_off;        // byte offset of the dOut box inside its slot (zero guard rows in front, 1024-byte aligned)
  int g_slot_bytes;      // guard + box + guard
  int cin;               // channels of the whole main source: G row = tap * cin + c0 + ci
  float* G;              // [27 * cin (+ extra rows)][32] fp32, zeroed by the caller
  float* part;           // DET only: [gridDim.x][27][32][32]
  int* err_flag;
};

template <int COUT, bool DET>   // COUT always 32 (a template keeps the definition in this header; instantiated in conv_umma.cu)
__global__ void __launch_bounds__(WP_THREADS, 1) wgrad_plane_kernel(const __grid_constant__ WgradPlaneParams P) {
  static_assert(COUT == 32, "one 32-column accumulator per (td, th)");
  constexpr uint32_t IDESC = make_idesc_f16_mn(128, 96);
  constexpr uint32_t DESC_HI = kmajor_desc_hi(64);           // SBO = 8 rows of 64 B, version, SWIZZLE_64B
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  const int S = P.stages;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S * P.stage_bytes);
  uint64_t* empty_bar = full_bar + WP_MAX_STAGES;
  uint64_t* tmem_full = empty_bar + WP_MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&P.amap);
    tma_prefetch_desc(&P.gmap);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);                 // three accumulators of 96 columns (288 -> 512)
  // zero guard rows of every stage's dOut slot (generic proxy, once; the TMA boxes land between them)
  for (int s = 0; s < S; ++s) {
    uint4* g = reinterpret_cast<uint4*>(smem + s * P.stage_bytes + 3 * P.a_slot_bytes);
    const int front = P.g_data_off / 16, back0 = (P.g_data_off + P.g_box_bytes) / 16, total = P.g_slot_bytes / 16;
    for (int i = threadIdx.x; i < front; i += blockDim.x) g[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = back0 + threadIdx.x; i < total; i += blockDim.x) g[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const bool has_work = static_cast<int>(blockIdx.x) < P.n_units;

  if (warp == 0) {
    // ===================== TMA producer =====================
    int s = 0;
    uint32_t ph = 0;
    const uint32_t tx = static_cast<uint32_t>(3 * P.a_box_bytes + P.g_box_bytes);
    for (int u = blockIdx.x; u < P.n_units; u += gridDim.x) {
      if (!mbar_wait(&empty_bar[s], ph ^ 1, P.err_flag, 211)) break;
      if (elect_one()) {
        const int n = u / P.units_per_sample;
        const int v = u - n * P.units_per_sample;
        const int d = v / P.hblocks;
        const int h0 = (v - d * P.hblocks) * P.HB;
        uint8_t* sa = smem + s * P.stage_bytes;
        mbar_expect_tx(&full_bar[s], tx);
#pragma unroll
        for (int td = 0; td < 3; ++td)
          tma_load_tile_5d(&P.amap, &full_bar[s], sa + td * P.a_slot_bytes, P.c0, -1, h0 - 1, d + td - 1, n);
        tma_load_tile_5d(&P.gmap, &full_bar[s], sa + 3 * P.a_slot_bytes + P.g_data_off, 0, 0, h0, d, n);
      }
      __syncwarp();
      if (++s == S) { s = 0; ph ^= 1; }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0 && has_work) {
      int s = 0;
      uint32_t ph = 0, first = 0;                            // first = 0: the accumulators are overwritten by the first unit
      bool alive = true;
      for (int u = blockIdx.x; u < P.n_units && alive; u += gridDim.x) {
        if (!mbar_wait(&full_bar[s], ph, P.err_flag, 212)) { alive = false; break; }
        tc_fence_after();
        const uint32_t base = smem_u32(smem + s * P.stage_bytes);
        // N chunks (th = 2, 1, 0) one grid row apart, starting two grid rows above the dOut box
        const uint32_t g_lo0 = mnmajor_desc_lo(base + 3 * P.a_slot_bytes + P.g_data_off - 2 * P.Wp * 64, P.Wp * 64);
#pragma unroll
        for (int td = 0; td < 3; ++td) {
          // M chunks (tw = 0..3) one box row (64 B) apart
          const uint32_t a_lo = mnmajor_desc_lo(base + td * P.a_slot_bytes, 64);
          const uint32_t d_tmem = tmem_base + td * 96;
          // 16 pixels (= 16 rows of 64 B = 64 descriptor units) per MMA
          umma_f16_lohi(d_tmem, a_lo, g_lo0, DESC_HI, IDESC, first);
          int j = 1;
          for (; j + 4 <= P.ksteps; j += 4) {
#pragma unroll
            for (int q = 0; q < 4; ++q) umma_f16_lohi(d_tmem, a_lo + (j + q) * 64, g_lo0 + (j + q) * 64, DESC_HI, IDESC, 1u);
          }
          for (; j < P.ksteps; ++j) umma_f16_lohi(d_tmem, a_lo + j * 64, g_lo0 + j * 64, DESC_HI, IDESC, 1u);
        }
        umma_commit(&empty_bar[s]);
        first = 1;
        if (++s == S) { s = 0; ph ^= 1; }
      }
      umma_commit(tmem_full);
    }
  } else if (has_work) {
    // ===================== epilogue (warps 2..5): TMEM -> fp32 atomics into G =====================
    const int tw = warp & 3;                                 // TMEM lane quarter = M chunk = tw (3: the discarded chunk)
    if (mbar_wait(tmem_full, 0, P.err_flag, 213)) {
      tc_fence_after();
      const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(tw * 32) << 16);
      // every CTA adds into the same 27 x 32 rows: start at a different (td, th) block per CTA so that the CTAs finishing
      // together spread over nine times as many L2 lines, one 128-byte row per thread as eight 16-byte reductions
      const int a0 = static_cast<int>(blockIdx.x % 9u);
#pragma unroll 1
      for (int aa = 0; aa < 9; ++aa) {                       // (td, N chunk j): th = 2 - j
        const int a = aa + a0 < 9 ? aa + a0 : aa + a0 - 9;
        const int td = a / 3, th = 2 - (a - td * 3);
        float v0[16], v1[16];
        tmem_ld16_async(t_lane + a * 32, v0);
        tmem_ld16_async(t_lane + a * 32 + 16, v1);
        tmem_ld_wait();
        if (DET && tw < 3) {
          float4* gp = reinterpret_cast<float4*>(P.part + static_cast<size_t>(blockIdx.x) * WP_PART +
                                                 (static_cast<size_t>((td * 3 + th) * 3 + tw) * 32 + lane) * 32);
#pragma unroll
          for (int i = 0; i < 16; i += 4) gp[i / 4] = make_float4(v0[i], v0[i + 1], v0[i + 2], v0[i + 3]);
#pragma unroll
          for (int i = 0; i < 16; i += 4) gp[4 + i / 4] = make_float4(v1[i], v1[i + 1], v1[i + 2], v1[i + 3]);
        } else if (tw < 3) {
          float* gp = P.G + (static_cast<size_t>((td * 3 + th) * 3 + tw) * P.cin + P.c0 + lane) * 32;
#pragma unroll
          for (int i = 0; i < 16; i += 4) red_add_v4(gp + i, v0[i], v0[i + 1], v0[i + 2], v0[i + 3]);
#pragma unroll
          for (int i = 0; i < 16; i += 4) red_add_v4(gp + 16 + i, v1[i], v1[i + 1], v1[i + 2], v1[i + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

struct WgradPlaneLaunch {
  WgradPlaneParams p;
  dim3 grid;
  size_t smem;
  bool ok;               // false: shape not covered, use wgrad_umma_kernel
  int det_ctas;          // grid of the deterministic variant: min(units, WP_DET_CTAS)
};

// One 32-channel chunk (channels [c0, c0 + 32) of a source whose pixel rows hold act_ld elements) of a k3 s1 p1 conv with
// cout == 32.  dout: fp16 rows of dout_ld elements (the first 32 are read).  G as wgrad_prepare (zeroed by the caller).
int wgrad_plane_prepare(WgradPlaneLaunch* L, const __half* act, int B, int D, int H, int W, int cin, int act_ld, int c0,
                        const __half* dout, int dout_ld, int cout, float* G);
int wgrad_plane_enqueue(const WgradPlaneLaunch& L, cudaStream_t st);
int wgrad_plane_init();

}  // namespace cm
