// "Plane-tile" implicit-GEMM 3-D convolution (k3 s1 p1) on tcgen05 / TMEM, sm_100a.
//
// Why a second conv kernel.  Measured on B200 (DESIGN.md 3.1, profiles/), conv_umma_kernel
// (conv_umma.cuh) is bound by what one SM can pull out of L2 (~32-45 B/clk): it re-fetches its A
// tile for each of the 27 taps (TMA im2col) and its weight tile for every 128-pixel M tile; and a
// 128 x 32 tcgen05.mma re-reads its 4 KB A operand from shared memory for only 32 output columns,
// so narrow layers are shared-memory-bandwidth bound inside the tensor pipe as well.  This kernel
//   * gives a work unit R whole planes (or a block of HB rows of one plane) of one sample: with W
//     padded to W+2 the unit is a flat array of P = R*HB*(W+2) "positions" and ONE tiled TMA box
//     {BK ch, W+2, HB, R} (zero-filled halo) per (td, th, channel chunk) serves all three tw taps
//     -> 9 A loads per channel chunk, not 27;
//   * stacks the three tw taps along N: Y[row, (tw, co)] = X[row, :] . W[(tw, co), :] is ONE
//     128 x (3*BN) MMA per k16 step (hi and lo weight terms are two MMAs into the same
//     accumulator).  A 128-row SS-mode tcgen05.mma costs >= ~64 cycles whatever N is (measured:
//     it re-reads its 4 KB A operand from shared memory), so 3x wider MMAs = 3x fewer of them.
//     The epilogue forms out[h, w] = Y0[row] + Y1[row+1] + Y2[row+2] (row = h*(W+2) + w) with a
//     row-shifted accumulation in shared memory; rows on the two pad columns are dropped.
//     (An earlier variant expressed the tw shift as a +1/+2 row offset of the A descriptor --
//     it is correct, the UMMA swizzle being a function of the absolute shared-memory address, so
//     an offset start needs no base_offset -- but it needs 3x the MMA instructions.)
//   * keeps ceil(P/128) accumulators in TMEM, so every weight tile is loaded once per unit and
//     reused by all of its M tiles;
//   * is persistent: one CTA per SM walks the units; TMEM is double-buffered, so the epilogue of
//     unit i (coalesced through a shared-memory transpose) overlaps the main loop of unit i+1.
// Same operands, same packed weights, same epilogue semantics as conv_umma_kernel (mode 0 with
// the optional fused 1x1x1 match_input K-slab).
#pragma once
#include "common.cuh"
#include "conv_umma.cuh"

namespace cm {

constexpr int PL_THREADS = 576;      // warp0 TMA, warp1 MMA, warps2-17 epilogue (four warps per TMEM lane quarter)
constexpr int PL_EPI = 512;          // epilogue threads: with th3 stages the epilogue chain of a unit is longer than
                                     // its main loop, so it gets 4 warps per scheduler instead of 2
constexpr int PL_NJ = 4;             // store rows per epilogue thread (host: ntiles*128 <= PL_NJ * rows per pass)
constexpr int PL_MAX_STAGES = 6;

struct PlaneParams {
  CUtensorMap amap;      // main source, tiled 5-D (C, W, H, D, N), box {BK, W+2, HB, R, 1}
  CUtensorMap xmap;      // optional 1x1x1 source over the same grid (same box)
  CUtensorMap bmap;      // packed weights [terms*cout][Ktot], K-major (as conv_umma)
  CUtensorMap bmap3;     // th3 mode: the same weights as (k within slab, row, (td,th,tw) slab), box {BK, BN, 9}
  int th3;               // 1: a stage = one (td, channel chunk): ONE A box with an H halo {BK, W+2, HB+2} whose
                         // three th taps are row-offset descriptor views (+th*(W+2) rows), and the nine (th, tw)
                         // weight slabs of each term in one 3-D TMA -> 3x fewer stages, 1/3 of the A ingest
                         // (measured: every pipeline stage costs ~0.16 us on top of its MMAs)
  int a_box_bytes;       // bytes one A load delivers (expect_tx)
  int H, W, D, Wp;       // plane geometry, Wp = W + 2
  int R, HB;             // unit = R planes x HB rows (R > 1 only with HB == H)
  int P;                 // positions per unit = R*HB*Wp
  int ntiles;            // ceil(P / 128) accumulators per unit
  int units_per_sample;  // (D / R) * (H / HB)
  int n_units;           // B * units_per_sample * (cout / BN)
  int n_ntiles;          // cout / BN
  int a_stage_bytes;     // bytes reserved for the A box per stage (covers ntiles*128 + 2 rows)
  int cin_main, cin_extra, cout, terms, stages;
  ConvEpilogue epi;      // GroupNorm records over the unit's R*HB*W valid rows
  int* err_flag;
};

__device__ __forceinline__ void tma_load_tile_5d(const void* desc, uint64_t* bar, void* smem, int c0,
                                                 int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      :
      : "r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

struct PlaneUnit {
  int n, d0, h0, n_tile;
};
__device__ __forceinline__ PlaneUnit plane_unit(const PlaneParams& P, int u) {
  PlaneUnit r;
  r.n_tile = u % P.n_ntiles;
  int v = u / P.n_ntiles;
  r.n = v / P.units_per_sample;
  v -= r.n * P.units_per_sample;
  const int hblocks = P.H / P.HB;
  const int db = v / hblocks;
  r.d0 = db * P.R;
  r.h0 = (v - db * hblocks) * P.HB;
  return r;
}

template <int BN, int BK, int TERMS>
__global__ void __launch_bounds__(PL_THREADS, 1)
conv_plane_kernel(const __grid_constant__ PlaneParams P) {
  constexpr int ROWB = BK * 2;
  constexpr int NST = 3 * BN;                        // N of one MMA = accumulator columns per M tile: (tw, co)
  constexpr int B_TAP = BN * ROWB;                   // weight bytes of one (term, tw) slab
  constexpr int B_TERM = 3 * B_TAP;                  // one term: tw0 | tw1 | tw2 slabs, contiguous
  constexpr int B_STAGE = TERMS * B_TERM;
  constexpr uint32_t IDESC = make_idesc_f16(128, NST);
  constexpr uint32_t IDESC_X = make_idesc_f16(128, BN);   // fused 1x1x1 source: centre (tw = 1) block only
  constexpr int TLD = BN + 4;                        // accumulation-buffer row (floats)

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  const int S = P.stages;
  const int b_term = (P.th3 ? 9 : 3) * B_TAP;              // bytes of one weight term per stage
  const int stage_bytes = P.a_stage_bytes + TERMS * b_term;   // multiple of 1024
  uint8_t* tail = smem + S * stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + PL_MAX_STAGES;
  uint64_t* tmem_full = empty_bar + PL_MAX_STAGES;         // [2]
  uint64_t* tmem_empty = tmem_full + 2;                    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* colv = reinterpret_cast<float*>(tail + 256);      // [BN]
  float* side = reinterpret_cast<float*>(tail + 256 + 512);       // [ntiles*4 + 1][3][BN] block-boundary rows
  float* ybuf = side + (P.ntiles * 4 + 1) * 3 * BN;               // [ntiles*128][TLD]
  float* sred = ybuf + (P.ntiles * 128 + 2) * TLD;                // [epilogue warps][BN][2] + [BN] shifts

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ncm = P.cin_main / BK;
  const int nks_main = (P.th3 ? 3 : 9) * ncm;         // (td, th, chunk) steps; th3: (td, chunk)
  const int nks = nks_main + P.cin_extra / BK;
  const uint32_t buf_cols = static_cast<uint32_t>(P.ntiles * NST);
  uint32_t tmem_cols = 32;
  while (tmem_cols < 2 * buf_cols) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&P.amap);
    tma_prefetch_desc(&P.bmap);
    if (P.th3) tma_prefetch_desc(&P.bmap3);
    if (P.cin_extra) tma_prefetch_desc(&P.xmap);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], PL_EPI / 32);         // one arrival per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    const uint32_t a_bytes = static_cast<uint32_t>(P.P) * ROWB;
    int s = 0;
    uint32_t ph = 0;
    bool alive = true;
    for (int u = blockIdx.x; u < P.n_units && alive; u += gridDim.x) {
      const PlaneUnit U = plane_unit(P, u);
      int td = 0, th = 0, cc = 0;
      for (int ks = 0; ks < nks; ++ks) {
        if (!mbar_wait(&empty_bar[s], ph ^ 1, P.err_flag, 401)) { alive = false; break; }
        uint8_t* sa = smem + s * stage_bytes;
        uint8_t* sb = sa + P.a_stage_bytes;
        if (elect_one()) {
          if (ks < nks_main && P.th3) {
            mbar_expect_tx(&full_bar[s], (uint32_t)P.a_box_bytes + (uint32_t)(TERMS * b_term));
            tma_load_tile_5d(&P.amap, &full_bar[s], sa, cc * BK, -1, U.h0 - 1, U.d0 + td - 1, U.n);
#pragma unroll
            for (int t = 0; t < TERMS; ++t)
              tma_load_3d(&P.bmap3, &full_bar[s], sb + t * b_term, cc * BK, U.n_tile * BN + t * P.cout, td * 9);
          } else if (ks < nks_main) {
            mbar_expect_tx(&full_bar[s], a_bytes + (uint32_t)B_STAGE);
            tma_load_tile_5d(&P.amap, &full_bar[s], sa, cc * BK, -1, U.h0 + th - 1, U.d0 + td - 1, U.n);
            const int kcol = ((td * 3 + th) * 3) * P.cin_main + cc * BK;
#pragma unroll
            for (int t = 0; t < TERMS; ++t)
#pragma unroll
              for (int tw = 0; tw < 3; ++tw)
                tma_load_2d(&P.bmap, &full_bar[s], sb + t * B_TERM + tw * B_TAP, kcol + tw * P.cin_main,
                            U.n_tile * BN + t * P.cout);
          } else {
            // fused 1x1x1 source: centre tap only (tw = 1 against a box that starts at w = -1)
            const int xc = ks - nks_main;
            mbar_expect_tx(&full_bar[s], a_bytes + TERMS * B_TAP);
            tma_load_tile_5d(&P.xmap, &full_bar[s], sa, xc * BK, -1, U.h0, U.d0, U.n);
#pragma unroll
            for (int t = 0; t < TERMS; ++t)
              tma_load_2d(&P.bmap, &full_bar[s], sb + t * b_term + 1 * B_TAP, 27 * P.cin_main + xc * BK,
                          U.n_tile * BN + t * P.cout);
          }
        }
        if (++cc == ncm) {
          cc = 0;
          if (P.th3) ++td;
          else if (++th == 3) { th = 0; ++td; }
        }
        if (++s == S) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // (a one-thread issuer with the stage's 12 MMA groups unrolled, as in conv_res32_kernel, was measured here: the
    // 96 -> 32 layer 79.7 -> 75.8 us, but the level-1 instantiations (N = 192 MMAs, BN = 64) 49.1 -> 55.1 / 28.7 -> 31.8 us
    // and the 1 280-sample chain 81.2 -> 76.4 seq/s: not kept)
    constexpr uint32_t DESC_HI = kmajor_desc_hi(ROWB);
    constexpr uint32_t TILE_LO = (128 * ROWB) >> 4;          // descriptor step between M tiles
    int s = 0;
    uint32_t ph = 0;
    int it = 0;
    bool alive = true;
    const int lo_from = P.epi.lo_from > 0 ? P.epi.lo_from : 0x40000000;
    const int lo_from_x = P.epi.lo_from_x > 0 ? P.epi.lo_from_x : 0x40000000;
    for (int u = blockIdx.x; u < P.n_units && alive; u += gridDim.x, ++it) {
      const int buf = it & 1;
      int cc = 0;
      // wait until the epilogue has drained this accumulator buffer (first two units: free)
      if (it >= 2 && !mbar_wait(&tmem_empty[buf], ((it >> 1) - 1) & 1, P.err_flag, 404)) break;
      tc_fence_after();
      const uint32_t d_base = tmem_base + buf * buf_cols;
      for (int ks = 0; ks < nks; ++ks) {
        if (!mbar_wait(&full_bar[s], ph, P.err_flag, 402)) { alive = false; break; }
        tc_fence_after();
        const int rel = ks < nks_main ? cc * BK - lo_from : (ks - nks_main) * BK - lo_from_x;
        if (++cc == ncm) cc = 0;
        if (elect_one()) {
          const uint32_t a_addr = smem_u32(smem + s * stage_bytes);
          const uint32_t a_lo0 = kmajor_desc_lo(a_addr);
          const uint32_t b_lo0 = kmajor_desc_lo(a_addr + P.a_stage_bytes);
          if (ks < nks_main) {
            uint32_t first = (ks == 0) ? 0u : 1u;
            const int nth = P.th3 ? 3 : 1;
            const uint32_t th_step = (static_cast<uint32_t>(P.Wp) * ROWB) >> 4;   // one grid row of the halo box
            for (int th = 0; th < nth; ++th) {
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
#pragma unroll
                for (int t = 0; t < TERMS; ++t) {
                  if (t == 1 && rel + k * 16 >= 0) continue;          // lo activation half x lo weight term: skipped
                  const uint32_t b_lo = b_lo0 + ((t * b_term + th * 3 * B_TAP) >> 4) + 2 * k;
                  uint32_t a_lo = a_lo0 + th * th_step + 2 * k;
                  uint32_t d = d_base;
#pragma unroll 2
                  for (int r = 0; r < P.ntiles; ++r) {
                    umma_f16_lohi(d, a_lo, b_lo, DESC_HI, IDESC, first);
                    a_lo += TILE_LO;
                    d += NST;
                  }
                  first = 1u;
                }
              }
            }
          } else {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
#pragma unroll
              for (int t = 0; t < TERMS; ++t) {
                if (t == 1 && rel + k * 16 >= 0) continue;
                const uint32_t b_lo = b_lo0 + ((t * b_term + B_TAP) >> 4) + 2 * k;
                uint32_t a_lo = a_lo0 + 2 * k;
                uint32_t d = d_base + BN;
#pragma unroll 2
                for (int r = 0; r < P.ntiles; ++r) {
                  umma_f16_lohi(d, a_lo, b_lo, DESC_HI, IDESC_X, 1u);
                  a_lo += TILE_LO;
                  d += NST;
                }
              }
            }
          }
          umma_commit(&empty_bar[s]);
          if (ks == nks - 1) umma_commit(&tmem_full[buf]);     // accumulators of this unit complete
        }
        __syncwarp();
        if (++s == S) { s = 0; ph ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (warps 2..17) =====================
    // TMEM lane quarter = warp % 4; the four warps of a quarter split the (M tile, 16-column chunk) items.
    const int quarter = warp & 3;
    const int group = (warp - 2) >> 2;                     // 0..3
    const int et = threadIdx.x - 64;
    const bool temb_uniform = P.epi.temb != nullptr && P.epi.temb_bstride == 0;
    constexpr int LPR = BN / 4;                            // lanes per row in the store phase
    constexpr int RPP = PL_EPI / LPR;                      // rows per store pass of the epilogue threads
    constexpr int NJ = PL_NJ;                              // store rows per thread (host: ntiles*128 <= NJ*RPP)
    constexpr int NCH = BN / 16;                           // 16-column chunks per accumulator block
    constexpr int NG = PL_EPI / 128;                       // warps per TMEM lane quarter
    const int plane = P.HB * P.Wp;
    const int sub_r = et / LPR, sub_c = (et % LPR) * 4;
    // Unit-independent part of the read-out, computed once per thread (measured, profiles/r2_plane_trace_32to32.txt: the
    // per-unit index divisions and the dependent loads of the column constants were 2100 of the 6800
    // cycles of a unit's epilogue chain): the offset of each of this thread's NJ store rows inside a
    // unit (-1: pad column / beyond the unit), and the per-column constants when they do not depend on
    // the unit (one N tile, batch-uniform or no time embedding).
    int roff[NJ];
    {
      int q = sub_r;
      int dl = q / plane;
      int rem = q - dl * plane;
      int hl = rem / P.Wp;
      int w = rem - hl * P.Wp;
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        roff[j] = (q < P.P && w < P.W) ? (dl * P.H + hl) * P.W + w : -1;
        q += RPP;
        w += RPP;
        while (w >= P.Wp) {
          w -= P.Wp;
          if (++hl == P.HB) { hl = 0; ++dl; }
        }
      }
    }
    const int trow_u = (temb_uniform && P.epi.t_dev) ? *P.epi.t_dev : 0;
    auto load_cv = [&](int nn, int n) {
      float4 c = make_float4(0.f, 0.f, 0.f, 0.f), b2 = c, t4 = c;
      if (P.epi.bias) c = *reinterpret_cast<const float4*>(P.epi.bias + nn);
      if (P.epi.bias2) b2 = *reinterpret_cast<const float4*>(P.epi.bias2 + nn);
      if (P.epi.temb) {
        const size_t trow = temb_uniform ? static_cast<size_t>(trow_u) * P.epi.temb_ld : static_cast<size_t>(n) * P.epi.temb_bstride;
        t4 = *reinterpret_cast<const float4*>(P.epi.temb + trow + nn);
      }
      c.x += b2.x; c.y += b2.y; c.z += b2.z; c.w += b2.w;      // same order as before: (bias + bias2) + temb
      c.x += t4.x; c.y += t4.y; c.z += t4.z; c.w += t4.w;
      return c;
    };
    const bool cv_const = P.n_ntiles == 1 && (P.epi.temb == nullptr || temb_uniform);
    float4 cv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cv_const) cv = load_cv(sub_c, 0);
    int it = 0;
    bool alive = true;
    for (int u = blockIdx.x; u < P.n_units && alive; u += gridDim.x, ++it) {
      const PlaneUnit U = plane_unit(P, u);
      const int buf = it & 1;
      const int nn0 = U.n_tile * BN;
      // Everything that does not depend on the accumulators is fetched before waiting for them: the
      // residual values of this thread's NJ store rows (and the column constants when they vary).
      if (!cv_const) cv = load_cv(nn0 + sub_c, U.n);
      int mi[NJ];
      float4 rv[NJ];
      {
        const int base = ((U.n * P.D + U.d0) * P.H + U.h0) * P.W;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          mi[j] = roff[j] < 0 ? -1 : base + roff[j];
          rv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (mi[j] >= 0 && P.epi.resid)
            rv[j] = *reinterpret_cast<const float4*>(P.epi.resid + static_cast<size_t>(mi[j]) * P.cout + nn0 + sub_c);
        }
      }
      if (!mbar_wait(&tmem_full[buf], (it >> 1) & 1, P.err_flag, 403)) { alive = false; break; }
      tc_fence_after();
      // out[row] = Y0[row] + Y1[row + 1] + Y2[row + 2].  Rows are TMEM lanes: the +1 / +2 shifts are
      // warp shuffles; the two rows a 32-row block needs from the NEXT block travel through `side`
      // (Y1 of its lane 0, Y2 of its lanes 0 and 1) and are added at read-out.  Fixed order -> the
      // result is deterministic.
#pragma unroll 1
      for (int item = group; item < P.ntiles * NCH; item += NG) {
        const int r = item / NCH, c = item - r * NCH;
        const int blk = r * 4 + quarter;
        const int row = blk * 32 + lane;
        const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + buf * buf_cols + r * NST;
        float* sd = side + static_cast<size_t>(blk) * 3 * BN;
        {
          float y0[16], y1[16], y2[16];
          tmem_ld16_async(t_lane + c * 16, y0);
          tmem_ld16_async(t_lane + BN + c * 16, y1);
          tmem_ld16_async(t_lane + 2 * BN + c * 16, y2);
          tmem_ld_wait();
          if (lane < 2) {                                  // 128-bit stores (side is 16-byte aligned, BN % 16 == 0)
            float4* s1v = reinterpret_cast<float4*>(sd + c * 16);
            float4* s2v = reinterpret_cast<float4*>(sd + (lane == 0 ? BN : 2 * BN) + c * 16);
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
          float4* dst = reinterpret_cast<float4*>(ybuf + static_cast<size_t>(row) * TLD + c * 16);
#pragma unroll
          for (int i = 0; i < 4; ++i) dst[i] = make_float4(y0[4 * i], y0[4 * i + 1], y0[4 * i + 2], y0[4 * i + 3]);
        }
      }
      // every accumulator of this buffer has been read by this warp: hand it back
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);
      asm volatile("bar.sync 1, 512;" ::: "memory");
      // coalesced read-out: RPP rows per pass, LPR lanes per row
      float4 st1 = make_float4(0.f, 0.f, 0.f, 0.f), st2 = st1;   // GroupNorm partial sums of (v - cv)
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        if (mi[j] < 0) continue;
        const int q = sub_r + j * RPP;
        float4 v = *reinterpret_cast<const float4*>(ybuf + static_cast<size_t>(q) * TLD + sub_c);
        const int ln = q & 31;
        if (ln >= 30) {
          const float* sn = side + static_cast<size_t>((q >> 5) + 1) * 3 * BN + sub_c;
          if (ln == 31) {
            const float4 a = *reinterpret_cast<const float4*>(sn);            // Y1 of the next block's lane 0
            const float4 b2 = *reinterpret_cast<const float4*>(sn + 2 * BN);  // Y2 of its lane 1
            v.x += a.x + b2.x; v.y += a.y + b2.y; v.z += a.z + b2.z; v.w += a.w + b2.w;
          } else {
            const float4 b1 = *reinterpret_cast<const float4*>(sn + BN);      // Y2 of its lane 0
            v.x += b1.x; v.y += b1.y; v.z += b1.z; v.w += b1.w;
          }
        }
        v.x += rv[j].x; v.y += rv[j].y; v.z += rv[j].z; v.w += rv[j].w;
        st1.x += v.x; st1.y += v.y; st1.z += v.z; st1.w += v.w;
        st2.x = fmaf(v.x, v.x, st2.x); st2.y = fmaf(v.y, v.y, st2.y);
        st2.z = fmaf(v.z, v.z, st2.z); st2.w = fmaf(v.w, v.w, st2.w);
        v.x += cv.x; v.y += cv.y; v.z += cv.z; v.w += cv.w;
        const size_t m = static_cast<size_t>(mi[j]);
        if (P.epi.out32) *reinterpret_cast<float4*>(P.epi.out32 + m * P.epi.out_ld + nn0 + sub_c) = v;
        if (P.epi.out16) {
          __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
          uint2 uu;
          uu.x = *reinterpret_cast<uint32_t*>(&h0);
          uu.y = *reinterpret_cast<uint32_t*>(&h1);
          __half* o16 = P.epi.out16 + m * (P.epi.out16_ld > 0 ? P.epi.out16_ld : P.epi.out_ld) + nn0 + sub_c;
          *reinterpret_cast<uint2*>(o16) = uu;
          if (P.epi.out16_lo > 0) {
            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
            __half2 l0 = __floats2half2_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2half2_rn(v.z - f1.x, v.w - f1.y);
            uu.x = *reinterpret_cast<uint32_t*>(&l0);
            uu.y = *reinterpret_cast<uint32_t*>(&l1);
            *reinterpret_cast<uint2*>(o16 + P.epi.out16_lo) = uu;
          }
        }
      }
      if (P.epi.stats_rec) {
        // lanes that share a channel quad (same lane % LPR) hold different rows: butterfly over them
#pragma unroll
        for (int w = LPR; w < 32; w <<= 1) {
          st1.x += __shfl_xor_sync(0xffffffffu, st1.x, w); st1.y += __shfl_xor_sync(0xffffffffu, st1.y, w);
          st1.z += __shfl_xor_sync(0xffffffffu, st1.z, w); st1.w += __shfl_xor_sync(0xffffffffu, st1.w, w);
          st2.x += __shfl_xor_sync(0xffffffffu, st2.x, w); st2.y += __shfl_xor_sync(0xffffffffu, st2.y, w);
          st2.z += __shfl_xor_sync(0xffffffffu, st2.z, w); st2.w += __shfl_xor_sync(0xffffffffu, st2.w, w);
        }
        if (lane < LPR) {
          float* d = sred + ((et >> 5) * BN + sub_c) * 2;
          d[0] = st1.x; d[1] = st2.x; d[2] = st1.y; d[3] = st2.y;
          d[4] = st1.z; d[5] = st2.z; d[6] = st1.w; d[7] = st2.w;
        }
        if (et < LPR) *reinterpret_cast<float4*>(sred + (PL_EPI / 32) * BN * 2 + sub_c) = cv;
      }
      asm volatile("bar.sync 1, 512;" ::: "memory");       // ybuf / side are rewritten by the next unit
      if (P.epi.stats_rec && et < BN) {
        float a1 = 0.f, a2 = 0.f;
#pragma unroll
        for (int wv = 0; wv < PL_EPI / 32; ++wv) {             // fixed order over the epilogue warps
          a1 += sred[(wv * BN + et) * 2];
          a2 += sred[(wv * BN + et) * 2 + 1];
        }
        const int hblocks = P.H / P.HB;
        const int uis = (U.d0 / P.R) * hblocks + U.h0 / P.HB;
        float4* rec = reinterpret_cast<float4*>(P.epi.stats_rec) +
                      (static_cast<size_t>(U.n) * P.units_per_sample + uis) * P.cout + nn0 + et;
        *rec = make_float4(sred[(PL_EPI / 32) * BN * 2 + et], a1, a2, 0.f);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, tmem_cols);
}

struct PlaneLaunch {
  PlaneParams p;
  dim3 grid;
  int bn, bk;
  size_t smem;
  bool ok;               // false: geometry not covered
};

// Fills L for a k3 s1 p1 conv (+ optional 1x1x1 extra source).  Returns 0 with L->ok = false when
// the geometry is outside what this kernel covers.
int plane_prepare(PlaneLaunch* L, const __half* act, int B, int D, int H, int W, int cin,
                  const __half* extra, int cin_extra, const __half* wpacked, int cout, int terms, const ConvEpilogue& epi);
int plane_enqueue(const PlaneLaunch& L, cudaStream_t st);
int plane_init();

}  // namespace cm
