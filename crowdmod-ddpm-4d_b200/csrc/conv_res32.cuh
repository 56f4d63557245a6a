// Weights-resident plane conv for the 32 -> 32 channel k3 s1 p1 layers (UNet.first, encoder_blocks.0.conv_1/2,
// the conv_2 of the two finest decoder blocks with their fused 1x1x1 match_input; reference:
// models/backbones/layers.py:32,43,46, unet.py:32), tcgen05 / TMEM / TMA, sm_100a.
//
// Why a third conv kernel (measured on B200, tools/umma_microbench.cu + profiles/r2_res32_trace_*.txt, DESIGN.md 3.1):
//   * one thread cannot issue tcgen05.mma faster than one per ~55 cycles, and a 128 x 96 x 16 SS-mode MMA
//     reads 7 KB of operands from shared memory for 48 cycles of tensor-pipe work: the N = 96 MMAs of
//     conv_plane_kernel run at 67-73 cycles inside the kernel (shared-memory bandwidth: operand reads +
//     the TMA writes of the streamed weights), the hi and lo weight terms being two such MMAs.  A
//     128 x 192 x 16 MMA runs AT the pipe floor when issued back to back (95-97 cycles measured, floor 96).
//   * so: stack the three tw taps AND the hi|lo weight terms along N (N = 3*2*32 = 192, one MMA per
//     (td, th, k16)): half the MMA instructions and 29 % less operand traffic.  TMEM then holds 192
//     accumulator columns per 128-row tile, so a unit is ONE tile (HB rows of one plane, HB*(W+2) <= 128)
//     with two accumulator buffers (384 of 512 columns);
//   * one-tile units would double the weight traffic per output row, so the 27-tap weights of both terms
//     (110.6 KB for 32 -> 32) stay RESIDENT in shared memory for the whole launch: a CTA loads them once,
//     then only activations stream (one haloed plane box {32 ch, W+2, HB+2} per td, 12 KB);
//   * the epilogue is a two-stage pipeline through a double-buffered transpose buffer: 8 drain warps
//     (TMEM -> hi+lo sum -> tw row shifts -> shared memory: ~400 cycles per unit) and 8 store warps
//     (residual, bias / time embedding, GroupNorm records, coalesced fp32 + fp16 stores: ~950 cycles), so
//     neither adds to the unit period (3 600 cycles, set by the MMA issuer: 6 MMAs in ~700 cycles, then
//     ~330 cycles of commit / barrier wait per stage -- profiles/r2_res32_trace_32to32.txt).
// Measured (B200, ATC level 0, B = 64): 31.3 us against 37.2 us for conv_plane_kernel; B = 1280: 517 us against 815 us.
// Operand / epilogue semantics are those of conv_plane_kernel (mode 0 + optional 1x1x1 K-slab); hi and lo
// products are accumulated separately in fp32 and added in the epilogue (deterministic, fixed order).
#pragma once
#include "common.cuh"
#include "conv_plane.cuh"

namespace cm {

constexpr int R32_THREADS = 640;       // warp0 TMA, warp1 MMA (one thread), warp2 TMEM alloc, warp3 idle, warps4-11 drain, warps12-19 store
constexpr int R32_DRAIN_W0 = 4;        // first drain warp (warp % 4 = TMEM lane quarter)
constexpr int R32_STORE_W0 = 12;       // first store warp
constexpr int R32_MAX_STAGES = 8;
constexpr int R32_NJ = 4;              // store rows per store thread (32 rows per pass)
constexpr int R32_C = 32;              // cin (main) = cout = 32
constexpr int R32_NST = 192;           // accumulator columns: (tw, term, co)
constexpr int R32_TLD = R32_C + 4;     // transpose-buffer row (floats)
constexpr int R32_WBLK = 2 * 3 * R32_C * 64;   // bytes of one (td, th) weight block: [tw][term][co] rows of 64 B
constexpr int R32_WX = 2 * R32_C * 64;         // bytes of one 1x1x1 chunk: [term][co] rows of 64 B

struct Res32Params {
  CUtensorMap amap;      // main source, tiled 5-D (C, W, H, D, N), box {32, W+2, HB+2, 1, 1}
  CUtensorMap xmap;      // optional 1x1x1 source over the same grid, box {32, W+2, HB, 1, 1}
  CUtensorMap wmap;      // packed weights [2*32 rows][Ktot] viewed as (k within slab, row, slab), box {32, 64, 3}
  CUtensorMap wxmap;     // the same weights 2-D (k, row), box {32, 64}: the 1x1x1 K-slab at k = 27*32 + chunk*32
  int H, W, D, Wp, HB;   // plane geometry, Wp = W + 2; unit = HB rows of one plane
  int P;                 // positions per unit = HB*Wp <= 128
  int units_per_sample;  // D * (H / HB)
  int n_units;           // B * units_per_sample
  int nx;                // 1x1x1 chunks of 32 channels (0..3)
  int stages, stage_bytes;
  ConvEpilogue epi;      // rows of 32 channels, no hi|lo operand pairs; GroupNorm records over HB*W rows
  int* err_flag;
};

template <int TERMS>   // always 2 (a template keeps the definition in this header; instantiated in conv_umma.cu only)
__global__ void __launch_bounds__(R32_THREADS, 1) conv_res32_kernel(const __grid_constant__ Res32Params P) {
  static_assert(TERMS == 2, "hi|lo weight terms stacked along N");
  constexpr int C = R32_C;
  constexpr uint32_t IDESC = make_idesc_f16(128, R32_NST);
  constexpr uint32_t IDESC_X = make_idesc_f16(128, 2 * C);      // 1x1x1 source: centre tap, hi|lo columns 64..127
  constexpr uint32_t DESC_HI = kmajor_desc_hi(64);
  constexpr int TLD = R32_TLD;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  const int S = P.stages;
  uint8_t* wsm = smem;                                       // [9 (td, th)][R32_WBLK] resident main weights
  uint8_t* wxsm = wsm + 9 * R32_WBLK;                        // [nx][R32_WX]
  uint8_t* ring = wxsm + P.nx * R32_WX;                      // [S][stage_bytes] activation boxes
  uint8_t* tail = ring + S * P.stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + R32_MAX_STAGES;
  uint64_t* tmem_full = empty_bar + R32_MAX_STAGES;          // [2]
  uint64_t* tmem_empty = tmem_full + 2;                      // [2]
  uint64_t* ybuf_full = tmem_empty + 2;                      // [2]
  uint64_t* ybuf_empty = ybuf_full + 2;                      // [2]
  uint64_t* wbar = ybuf_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wbar + 1);
  float* cvs = reinterpret_cast<float*>(tail + 256);         // [2][C] per-column constants (GroupNorm record shift)
  float* sred = cvs + 2 * C;                                 // [2][8 store warps][C][2]
  float* side = sred + 2 * 8 * C * 2;                        // [2][5 blocks][3][C] block-boundary rows
  float* ybuf = side + 2 * 5 * 3 * C;                        // [2][128][TLD]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nks = 3 + P.nx;                                  // ring stages per unit: td = 0..2, then the 1x1x1 chunks
  const int hblocks = P.H / P.HB;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&P.amap);
    tma_prefetch_desc(&P.wmap);
    if (P.nx) {
      tma_prefetch_desc(&P.xmap);
      tma_prefetch_desc(&P.wxmap);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 8);                          // one arrival per drain warp
      mbar_init(&ybuf_full[b], 8);
      mbar_init(&ybuf_empty[b], 8);                          // one arrival per store warp
    }
    mbar_init(wbar, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      // resident weights: nine (td, th) blocks of [tw][hi|lo][co] rows, then the 1x1x1 chunks
      mbar_expect_tx(wbar, static_cast<uint32_t>(9 * R32_WBLK + P.nx * R32_WX));
      for (int b = 0; b < 9; ++b) tma_load_3d(&P.wmap, wbar, wsm + b * R32_WBLK, 0, 0, b * 3);
      for (int x = 0; x < P.nx; ++x) tma_load_2d(&P.wxmap, wbar, wxsm + x * R32_WX, 27 * C + x * C, 0);
    }
    __syncwarp();
    const uint32_t a_bytes = static_cast<uint32_t>((P.HB + 2) * P.Wp * 64);
    const uint32_t x_bytes = static_cast<uint32_t>(P.P * 64);
    int s = 0;
    uint32_t ph = 0;
    bool alive = true;
    for (int u = blockIdx.x; u < P.n_units && alive; u += gridDim.x) {
      const int n = u / P.units_per_sample;
      const int v = u - n * P.units_per_sample;
      const int d = v / hblocks;
      const int h0 = (v - d * hblocks) * P.HB;
      for (int ks = 0; ks < nks; ++ks) {
        if (!mbar_wait(&empty_bar[s], ph ^ 1, P.err_flag, 501)) { alive = false; break; }
        if (elect_one()) {
          uint8_t* sa = ring + s * P.stage_bytes;
          if (ks < 3) {
            mbar_expect_tx(&full_bar[s], a_bytes);
            tma_load_tile_5d(&P.amap, &full_bar[s], sa, 0, -1, h0 - 1, d + ks - 1, n);
          } else {
            mbar_expect_tx(&full_bar[s], x_bytes);
            tma_load_tile_5d(&P.xmap, &full_bar[s], sa, (ks - 3) * C, -1, h0, d, n);
          }
        }
        __syncwarp();
        if (++s == S) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    // tcgen05.mma issue is effectively synchronous (the issuing thread is held while the tensor pipe works off its one
    // queued MMA), so every instruction the issuer executes between two MMAs of different stages is tensor-pipe idle
    // time: the per-stage wait / commit / descriptor code of the first version cost ~330 cycles per stage, 3 600 cycles
    // per unit against 1 728 of MMA work (profiles/r2_res32_trace_32to32.txt).  This version keeps the issuer's instruction stream
    // minimal: ONE thread (no elect / warp-sync per stage), the four barriers a unit depends on (accumulator buffer free,
    // the three td planes loaded) polled TOGETHER up front with independent try_waits (64 cycles for three against 158 for
    // one bounded wait loop, tools/umma_microbench.cu), then the 18 MMAs of the unit straight-line with compile-time
    // weight offsets, the per-stage commits (slot release) in between.  Variants measured and rejected: a second issuing
    // warp alternating units (32.3 us against 35.2 with the old loop: each issuer owns one accumulator buffer, so the two
    // alternate instead of overlapping), a scout warp publishing barrier phases through shared memory (35.3 us).
    if (lane == 0) {
      bool alive = mbar_wait(wbar, 0, P.err_flag, 505);
      const uint32_t w_lo0 = kmajor_desc_lo(smem_u32(wsm));
      const uint32_t wx_lo0 = kmajor_desc_lo(smem_u32(wxsm));
      const uint32_t ring_lo = kmajor_desc_lo(smem_u32(ring));
      const uint32_t stage16 = static_cast<uint32_t>(P.stage_bytes) >> 4;
      const uint32_t th_step = (static_cast<uint32_t>(P.Wp) * 64) >> 4;   // one grid row of the halo box
      const uint32_t full0 = smem_u32(full_bar);
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int u = blockIdx.x; u < P.n_units && alive; u += gridDim.x, ++it) {
        const int buf = it & 1;
        // slots / parities of the unit's three main stages
        int sl[3];
        uint32_t pr[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          sl[k] = s;
          pr[k] = ph;
          if (++s == S) { s = 0; ph ^= 1; }
        }
        {
          // fast path: all four phases already complete (the producer runs a ring ahead, the drain warps a unit ahead)
          const uint32_t te = it >= 2 ? smem_u32(&tmem_empty[buf]) : full0 + sl[0] * 8;
          const uint32_t tp = it >= 2 ? static_cast<uint32_t>(((it >> 1) - 1) & 1) : pr[0];
          uint32_t ok;
          asm volatile(
              "{\n\t.reg .pred P0, P1, P2, P3;\n\t"
              "mbarrier.try_wait.parity.shared::cta.b64 P0, [%1], %5;\n\t"
              "mbarrier.try_wait.parity.shared::cta.b64 P1, [%2], %6;\n\t"
              "mbarrier.try_wait.parity.shared::cta.b64 P2, [%3], %7;\n\t"
              "mbarrier.try_wait.parity.shared::cta.b64 P3, [%4], %8;\n\t"
              "and.pred P0, P0, P1;\n\tand.pred P2, P2, P3;\n\tand.pred P0, P0, P2;\n\t"
              "selp.u32 %0, 1, 0, P0;\n\t}\n"
              : "=r"(ok)
              : "r"(te), "r"(full0 + sl[0] * 8), "r"(full0 + sl[1] * 8), "r"(full0 + sl[2] * 8), "r"(tp), "r"(pr[0]),
                "r"(pr[1]), "r"(pr[2])
              : "memory");
          if (!ok) {
            if (it >= 2 && !mbar_wait(&tmem_empty[buf], ((it >> 1) - 1) & 1, P.err_flag, 504)) break;
#pragma unroll
            for (int k = 0; k < 3; ++k)
              if (alive && !mbar_wait(&full_bar[sl[k]], pr[k], P.err_flag, 502)) alive = false;
            if (!alive) break;
          }
        }
        tc_fence_after();
        const uint32_t d_base = tmem_base + buf * R32_NST;
#pragma unroll
        for (int ks = 0; ks < 3; ++ks) {
          const uint32_t a_lo0 = ring_lo + sl[ks] * stage16;
#pragma unroll
          for (int th = 0; th < 3; ++th) {
            const uint32_t b_lo = w_lo0 + (((ks * 3 + th) * R32_WBLK) >> 4);
            const uint32_t a_lo = a_lo0 + th * th_step;
            umma_f16_lohi(d_base, a_lo, b_lo, DESC_HI, IDESC, (ks == 0 && th == 0) ? 0u : 1u);
            umma_f16_lohi(d_base, a_lo + 2, b_lo + 2, DESC_HI, IDESC, 1u);
          }
          umma_commit(&empty_bar[sl[ks]]);
        }
        // fused 1x1x1 chunks: one stage each, centre-tap columns
        for (int x = 0; x < P.nx; ++x) {
          if (!mbar_wait(&full_bar[s], ph, P.err_flag, 502)) { alive = false; break; }
          tc_fence_after();
          const uint32_t a_lo0 = ring_lo + s * stage16;
          const uint32_t b_lo = wx_lo0 + ((x * R32_WX) >> 4);
          umma_f16_lohi(d_base + 2 * C, a_lo0, b_lo, DESC_HI, IDESC_X, 1u);
          umma_f16_lohi(d_base + 2 * C, a_lo0 + 2, b_lo + 2, DESC_HI, IDESC_X, 1u);
          umma_commit(&empty_bar[s]);
          if (++s == S) { s = 0; ph ^= 1; }
        }
        if (!alive) break;
        umma_commit(&tmem_full[buf]);                          // accumulator of this unit complete
      }
    }
  } else if (warp >= R32_DRAIN_W0 && warp < R32_STORE_W0) {
    // ===================== drain warps: TMEM -> (hi + lo, tw row shifts) -> transpose buffer =====================
    // out[row] = Y0[row] + Y1[row + 1] + Y2[row + 2] with Yt = hi_t + lo_t.  Rows are TMEM lanes: the shifts are
    // warp shuffles; the two rows a 32-row block needs from the next block travel through `side`.
    const int quarter = warp & 3;
    const int c = (warp - R32_DRAIN_W0) >> 2;                // 16-column chunk of the 32 output channels
    const int row = quarter * 32 + lane;
    int it = 0;
    for (int u = blockIdx.x; u < P.n_units; u += gridDim.x, ++it) {
      const int buf = it & 1;
      if (!mbar_wait(&tmem_full[buf], (it >> 1) & 1, P.err_flag, 503)) break;
      tc_fence_after();
      if (it >= 2 && !mbar_wait(&ybuf_empty[buf], ((it >> 1) - 1) & 1, P.err_flag, 506)) break;
      const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + buf * R32_NST + c * 16;
      float* yb = ybuf + static_cast<size_t>(buf) * 128 * TLD;
      float* sd = side + (static_cast<size_t>(buf) * 5 + quarter) * 3 * C;
      float y0[16], y1[16], y2[16];
      {
        float l0[16], l1[16];
        tmem_ld16_async(t_lane, y0);
        tmem_ld16_async(t_lane + C, l0);
        tmem_ld16_async(t_lane + 2 * C, y1);
        tmem_ld16_async(t_lane + 3 * C, l1);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) { y0[i] += l0[i]; y1[i] += l1[i]; }
      }
      {
        float l2[16];
        tmem_ld16_async(t_lane + 4 * C, y2);
        tmem_ld16_async(t_lane + 5 * C, l2);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) y2[i] += l2[i];
      }
      // the accumulator has been read by this warp: hand it back to the MMA issuer
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);
      if (lane < 2) {
        float4* s1v = reinterpret_cast<float4*>(sd + c * 16);
        float4* s2v = reinterpret_cast<float4*>(sd + (lane == 0 ? C : 2 * C) + c * 16);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (lane == 0) s1v[i] = make_float4(y1[4 * i], y1[4 * i + 1], y1[4 * i + 2], y1[4 * i + 3]);
          s2v[i] = make_float4(y2[4 * i], y2[4 * i + 1], y2[4 * i + 2], y2[4 * i + 3]);
        }
      }
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float s1 = __shfl_down_sync(0xffffffffu, y1[i], 1);
        const float s2 = __shfl_down_sync(0xffffffffu, y2[i], 2);
        y0[i] += (lane < 31 ? s1 : 0.f) + (lane < 30 ? s2 : 0.f);
      }
      float4* dst = reinterpret_cast<float4*>(yb + static_cast<size_t>(row) * TLD + c * 16);
#pragma unroll
      for (int i = 0; i < 4; ++i) dst[i] = make_float4(y0[4 * i], y0[4 * i + 1], y0[4 * i + 2], y0[4 * i + 3]);
      __syncwarp();
      if (lane == 0) mbar_arrive(&ybuf_full[buf]);            // release: this warp's rows / side rows are written
    }
  } else if (warp >= R32_STORE_W0) {
    // ===================== store warps: transpose buffer -> residual / constants / records -> global =====================
    constexpr int LPR = C / 4;                               // lanes per row
    constexpr int RPP = 256 / LPR;                           // rows per pass of the 256 store threads
    constexpr int NJ = R32_NJ;
    const int st = threadIdx.x - R32_STORE_W0 * 32;          // 0..255
    const int sw = st >> 5;                                  // store warp 0..7
    const int sub_r = st / LPR, sub_c = (st % LPR) * 4;
    const bool temb_uniform = P.epi.temb != nullptr && P.epi.temb_bstride == 0;
    // unit-independent: offset of each of this thread's store rows inside a unit (-1: pad column / beyond the unit)
    int roff[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int q = sub_r + j * RPP;
      const int hl = q / P.Wp, w = q - hl * P.Wp;
      roff[j] = (q < P.P && w < P.W) ? hl * P.W + w : -1;
    }
    const int trow_u = (temb_uniform && P.epi.t_dev) ? *P.epi.t_dev : 0;
    auto load_cv = [&](int n) {
      float4 cc = make_float4(0.f, 0.f, 0.f, 0.f), b2 = cc, t4 = cc;
      if (P.epi.bias) cc = *reinterpret_cast<const float4*>(P.epi.bias + sub_c);
      if (P.epi.bias2) b2 = *reinterpret_cast<const float4*>(P.epi.bias2 + sub_c);
      if (P.epi.temb) {
        const size_t trow = temb_uniform ? static_cast<size_t>(trow_u) * P.epi.temb_ld : static_cast<size_t>(n) * P.epi.temb_bstride;
        t4 = *reinterpret_cast<const float4*>(P.epi.temb + trow + sub_c);
      }
      cc.x += b2.x; cc.y += b2.y; cc.z += b2.z; cc.w += b2.w;
      cc.x += t4.x; cc.y += t4.y; cc.z += t4.z; cc.w += t4.w;
      return cc;
    };
    const bool cv_const = P.epi.temb == nullptr || temb_uniform;
    float4 cv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cv_const) cv = load_cv(0);
    int it = 0;
    for (int u = blockIdx.x; u < P.n_units; u += gridDim.x, ++it) {
      const int buf = it & 1;
      const int n = u / P.units_per_sample;
      const int v = u - n * P.units_per_sample;
      const int d = v / hblocks;
      const int h0 = (v - d * hblocks) * P.HB;
      if (!cv_const) cv = load_cv(n);
      int mi[NJ];
      float4 rv[NJ];
      float4 rk = make_float4(0.f, 0.f, 0.f, 0.f);   // residual of the unit's first row (GroupNorm record shift)
      {
        const int base = ((n * P.D + d) * P.H + h0) * P.W;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          mi[j] = roff[j] < 0 ? -1 : base + roff[j];
          rv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (mi[j] >= 0 && P.epi.resid)
            rv[j] = *reinterpret_cast<const float4*>(P.epi.resid + static_cast<size_t>(mi[j]) * C + sub_c);
        }
        if (P.epi.stats_rec && P.epi.resid)
          rk = *reinterpret_cast<const float4*>(P.epi.resid + static_cast<size_t>(base) * C + sub_c);
      }
      if (!mbar_wait(&ybuf_full[buf], (it >> 1) & 1, P.err_flag, 507)) break;
      const float* yb = ybuf + static_cast<size_t>(buf) * 128 * TLD;
      const float* sdb = side + static_cast<size_t>(buf) * 5 * 3 * C;
      // GroupNorm records are shifted by the unit's first value k0, a sample of the data (see conv_plane_kernel)
      float4 k0 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (P.epi.stats_rec) {
        k0 = *reinterpret_cast<const float4*>(yb + sub_c);
        k0.x += rk.x; k0.y += rk.y; k0.z += rk.z; k0.w += rk.w;
      }
      float4 st1 = make_float4(0.f, 0.f, 0.f, 0.f), st2 = st1;   // GroupNorm partial sums of (v - cv - k0)
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        if (mi[j] < 0) continue;
        const int q = sub_r + j * RPP;
        float4 vv = *reinterpret_cast<const float4*>(yb + static_cast<size_t>(q) * TLD + sub_c);
        const int ln = q & 31;
        if (ln >= 30) {
          const float* sn = sdb + static_cast<size_t>((q >> 5) + 1) * 3 * C + sub_c;
          if (ln == 31) {
            const float4 a = *reinterpret_cast<const float4*>(sn);            // Y1 of the next block's lane 0
            const float4 b2 = *reinterpret_cast<const float4*>(sn + 2 * C);   // Y2 of its lane 1
            vv.x += a.x + b2.x; vv.y += a.y + b2.y; vv.z += a.z + b2.z; vv.w += a.w + b2.w;
          } else {
            const float4 b1 = *reinterpret_cast<const float4*>(sn + C);       // Y2 of its lane 0
            vv.x += b1.x; vv.y += b1.y; vv.z += b1.z; vv.w += b1.w;
          }
        }
        vv.x += rv[j].x; vv.y += rv[j].y; vv.z += rv[j].z; vv.w += rv[j].w;
        {
          const float dx = vv.x - k0.x, dy = vv.y - k0.y, dz = vv.z - k0.z, dw = vv.w - k0.w;
          st1.x += dx; st1.y += dy; st1.z += dz; st1.w += dw;
          st2.x = fmaf(dx, dx, st2.x); st2.y = fmaf(dy, dy, st2.y);
          st2.z = fmaf(dz, dz, st2.z); st2.w = fmaf(dw, dw, st2.w);
        }
        vv.x += cv.x; vv.y += cv.y; vv.z += cv.z; vv.w += cv.w;
        const size_t m = static_cast<size_t>(mi[j]);
        if (P.epi.out32) *reinterpret_cast<float4*>(P.epi.out32 + m * C + sub_c) = vv;
        if (P.epi.out16) {
          __half2 h0v = __floats2half2_rn(vv.x, vv.y), h1v = __floats2half2_rn(vv.z, vv.w);
          uint2 uu;
          uu.x = *reinterpret_cast<uint32_t*>(&h0v);
          uu.y = *reinterpret_cast<uint32_t*>(&h1v);
          *reinterpret_cast<uint2*>(P.epi.out16 + m * C + sub_c) = uu;
        }
      }
      // this warp has read its rows of the transpose buffer: hand it back to the drain warps
      __syncwarp();
      if (lane == 0) mbar_arrive(&ybuf_empty[buf]);
      if (P.epi.stats_rec) {
        // lanes that share a channel quad (same lane % LPR) hold different rows: butterfly over them
#pragma unroll
        for (int wd = LPR; wd < 32; wd <<= 1) {
          st1.x += __shfl_xor_sync(0xffffffffu, st1.x, wd); st1.y += __shfl_xor_sync(0xffffffffu, st1.y, wd);
          st1.z += __shfl_xor_sync(0xffffffffu, st1.z, wd); st1.w += __shfl_xor_sync(0xffffffffu, st1.w, wd);
          st2.x += __shfl_xor_sync(0xffffffffu, st2.x, wd); st2.y += __shfl_xor_sync(0xffffffffu, st2.y, wd);
          st2.z += __shfl_xor_sync(0xffffffffu, st2.z, wd); st2.w += __shfl_xor_sync(0xffffffffu, st2.w, wd);
        }
        float* sr = sred + static_cast<size_t>(buf) * 8 * C * 2;
        if (lane < LPR) {
          float* dd = sr + (sw * C + sub_c) * 2;
          dd[0] = st1.x; dd[1] = st2.x; dd[2] = st1.y; dd[3] = st2.y;
          dd[4] = st1.z; dd[5] = st2.z; dd[6] = st1.w; dd[7] = st2.w;
        }
        // the shift: cv + k0 == the stored value of the unit's first row, bit for bit
        if (st < LPR)
          *reinterpret_cast<float4*>(cvs + buf * C + sub_c) = make_float4(k0.x + cv.x, k0.y + cv.y, k0.z + cv.z, k0.w + cv.w);
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (st < C) {
          float a1 = 0.f, a2 = 0.f;
#pragma unroll
          for (int wv = 0; wv < 8; ++wv) {                     // fixed order over the store warps
            a1 += sr[(wv * C + st) * 2];
            a2 += sr[(wv * C + st) * 2 + 1];
          }
          float4* rec = reinterpret_cast<float4*>(P.epi.stats_rec) + (static_cast<size_t>(n) * P.units_per_sample + v) * C + st;
          *rec = make_float4(cvs[buf * C + st], a1, a2, 0.f);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

struct Res32Launch {
  Res32Params p;
  dim3 grid;
  size_t smem;
  bool ok;               // false: shape not covered
};

// Fills L for a k3 s1 p1 conv with cin = cout = 32, two weight terms (+ optional 1x1x1 source of 32/64/96
// channels).  Returns 0 with L->ok = false when the shape is outside what this kernel covers; refuses an
// epilogue with hi|lo operand pairs or fp16 rows wider than 32 channels.
int res32_prepare(Res32Launch* L, const __half* act, int B, int D, int H, int W, int cin, const __half* extra,
                  int cin_extra, const __half* wpacked, int cout, int terms, const ConvEpilogue& epi);
int res32_enqueue(const Res32Launch& L, cudaStream_t st);
int res32_init();

}  // namespace cm
