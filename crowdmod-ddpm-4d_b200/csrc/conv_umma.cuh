// Implicit-GEMM 3-D convolution on tcgen05 / TMEM fed by TMA (im2col mode), sm_100a.
//
// Replaces every nn.Conv3d the reference UNet dispatches to cuDNN except the two 3-channel
// ends (reference: models/backbones/layers.py:32,43,46,84,92-94; unet.py:32,121) and the two
// attention projections (layers.py:10,16 — a 1x1x1 "conv").
//
//   D[m, n] = sum_{tap, ci} A[pixel(m) + tap, ci] * W[n, tap, ci]      m = output pixel (NDHWC order)
//
// A (activations, fp16, channels-last [B, H, W, L, C]) is never materialised as an im2col
// matrix: each k-block is ONE cp.async.bulk.tensor.5d...im2col load of 128 consecutive output
// pixels x BK channels for one filter tap (hardware does the halo / zero padding / stride).
// W is pre-packed fp16 [terms*Cout, K] (K = taps*Cin, tap-major) and loaded with tiled TMA.
// Accumulation is fp32 in TMEM; the epilogue (4 warps, one TMEM lane quarter each) fuses
// bias, the time-embedding projection add, the residual add, fp32/fp16 stores and the
// nearest-x2-upsample scatter.
#pragma once
#include "common.cuh"

namespace cm {

constexpr int CONV_BM = 128;        // UMMA M (cta_group::1)
constexpr int CONV_THREADS = 192;   // warp0 TMA, warp1 MMA, warps2-5 epilogue
constexpr int CONV_MAX_STAGES = 8;

// Epilogue of the three forward conv kernels (conv_umma, conv_plane, conv_res32):
// out = acc + bias + bias2 + temb row + resid, stored fp32 and / or fp16.
// Field order: the int pairs (lo_from, lo_from_x), (temb_ld, temb_bstride), (out_ld, out16_ld) start at 8-byte
// boundaries, as in the parameter structs before this one existed; ptxas then emits the same code (apart, it
// loads them separately and conv_umma_kernel<., ., 1> takes up to 3 more registers).
struct ConvEpilogue {
  int lo_from, lo_from_x;   // > 0: channels >= lo_from of the main (lo_from_x: the 1x1x1) source are the lo halves of hi|lo
                            // operand pairs (training): their k16 slices skip the lo weight term (a_lo * w_lo ~ 2^-22)
  const float* bias;
  const float* bias2;
  const float* temb;     // [rows][temb_ld] projection table, nullptr = none
  const int* t_dev;      // device int: row of `temb` for the whole batch (sampling); nullptr = 0
  int temb_ld;
  int temb_bstride;      // per-sample row stride (training: temb_ld, sampling: 0)
  const float* resid;    // fp32 [M][cout] or nullptr
  float* out32;          // fp32 [rows][out_ld] or nullptr
  __half* out16;         // fp16 [rows][out16_ld] or nullptr
  int out_ld;            // set by the prepare functions (cout)
  int out16_ld, out16_lo;   // fp16 copy: row stride in elements (0 -> out_ld); out16_lo > 0: also write the lo half
                            // fp16(v - hi) out16_lo elements further (hi|lo pair operand of the training forward)
  // GroupNorm statistics records of the values the launch writes (nullptr = none), plane and res32 kernels only: per
  // (sample, unit of the sample, output channel) a float4 {shift, sum(v - shift), sum((v - shift)^2), 0} over the unit's
  // valid rows, shift = the value the unit's first row stores (a sample of the data: no cancellation in the unit's
  // variance when the values share a large offset); units belong to ONE sample, so the consumer (gn_apply2_kernel) merges them in a fixed order ->
  // bit-reproducible wherever the sample sits in the batch.
  float* stats_rec;
};

struct ConvParams {
  CUtensorMap amap[8];   // main source, one map per output phase (1 normally, 8 for upsample)
  CUtensorMap xmap;      // optional extra 1x1x1 source (match_input fused as a K-slab)
  CUtensorMap bmap;      // packed weights [terms*cout rows][Ktot], K-major
  int M;                 // rows of this launch (per phase)
  int od, oh, ow;        // GEMM-M traversal extents per sample: m = ((n*od+z)*oh+p)*ow+q
  int pps;               // od*oh*ow
  int conv_stride;       // traversal stride of the main source
  int kd, kh, kw;        // taps per dim of the main source
  int nphase;
  signed char lower[8][4];  // per phase lower corner {w,h,d}
  int cin_main, cin_extra;
  int kphase;            // packed-K elements per phase
  int terms;             // 1 = fp16 weights, 2 = hi+lo split weights
  int cout;
  int stages;
  ConvEpilogue epi;      // stats_rec unused
  // optional epilogue extras of the non-split path (the DiT plan, dit.cu): v = act(acc + bias); v *= gate[sample][n];
  // v += resid; rows of sample b land at output row b*rmap_out + rmap_off + (m - b*pps) (resid is read there too)
  int act;               // 0 none, 1 exact GELU
  const float* gate;     // fp32 [samples][gate_ld] or nullptr
  int gate_ld;
  int rmap_out, rmap_off;   // rmap_out > 0: remap output rows (samples of pps GEMM rows -> samples of rmap_out rows)
  int scatter;           // 1: rows are low-res pixels, written to (2z+pz, 2p+pp, 2q+pq)
  // split-K (M-starved deep-K layers): gridDim.z = ksplit CTAs of one thread-block cluster share
  // an output tile, each accumulating kb_per_split k-blocks; the partial tiles are reduced in a
  // fixed order through distributed shared memory (deterministic, no atomics).
  int ksplit, kb_per_split;
  // scatter (UpSample) convs: one CTA walks ppc consecutive phases of its M tile (barriers / TMEM are
  // set up once; measured: the per-CTA set-up was more than half of the 8-tap phase convs' time)
  int ppc;
  int* err_flag;
};

// at most 112 registers: three CTAs of CONV_THREADS per SM, the co-residency conv_prepare's stage budget and the UpSample
// phase convs are planned for
template <int BN, int BK, int TERMS>
__global__ void __maxnreg__(112)
conv_umma_kernel(const __grid_constant__ ConvParams P) {
  constexpr int ROWB = BK * 2;                  // bytes per smem row (swizzle span)
  constexpr int A_BYTES = CONV_BM * ROWB;
  constexpr int B_BYTES = BN * ROWB;
  // hi and lo weight terms are stacked along N (their smem tiles are adjacent): ONE 128 x (TERMS*BN)
  // MMA per k16 step.  A 128-row SS-mode tcgen05.mma costs >= ~64 cycles whatever N is (it re-reads
  // its 4 KB A operand from shared memory), so halving the instruction count halves the MMA time of
  // the narrow layers; the epilogue adds the two halves.
  constexpr int NST = BN * TERMS;
  constexpr uint32_t IDESC = make_idesc_f16(CONV_BM, NST);
  constexpr uint32_t IDESC_HI = make_idesc_f16(CONV_BM, BN);   // hi weight term only (the first BN rows of the B tile)
  constexpr uint32_t TMEM_COLS = NST < 32 ? 32 : NST;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);

  const int S = P.stages;
  constexpr int terms = TERMS;
  const int stage_bytes = A_BYTES + terms * B_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S * stage_bytes);
  uint64_t* empty_bar = full_bar + CONV_MAX_STAGES;
  uint64_t* tmem_full = empty_bar + CONV_MAX_STAGES;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 1);
  float* colv = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 192);   // [BN] per-column epilogue constants

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x;
  const int n_tile = blockIdx.y;
  const int ppc = P.ppc > 1 ? P.ppc : 1;
  const int phase0 = P.ksplit > 1 ? 0 : blockIdx.z * ppc;
  const int split = P.ksplit > 1 ? blockIdx.z : 0;

  const int ncm = P.cin_main / BK;
  const int nkb_main = P.kd * P.kh * P.kw * ncm;
  const int nkb = nkb_main + P.cin_extra / BK;
  const int kb_lo = P.ksplit > 1 ? split * P.kb_per_split : 0;
  const int kb_hi = P.ksplit > 1 ? (kb_lo + P.kb_per_split < nkb ? kb_lo + P.kb_per_split : nkb) : nkb;

  if (warp == 0 && lane == 0) {
    for (int pi = 0; pi < ppc; ++pi) tma_prefetch_desc(&P.amap[phase0 + pi]);
    tma_prefetch_desc(&P.bmap);
    if (P.cin_extra) tma_prefetch_desc(&P.xmap);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 4);        // one arrival per epilogue warp
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (whole warp runs the loop; one elected lane issues) ====
    {
      const int m0 = m_tile * CONV_BM;
      const int n0 = m0 / P.pps;
      int r = m0 - n0 * P.pps;
      const int z0 = r / (P.oh * P.ow);
      r -= z0 * P.oh * P.ow;
      const int p0 = r / P.ow;
      const int q0 = r - p0 * P.ow;
      const uint32_t tx = A_BYTES + terms * B_BYTES;
      int s = 0, git = 0;
      uint32_t ph = 0;
      bool alive = true;
      for (int pi = 0; pi < ppc && alive; ++pi) {
      const int phase = phase0 + pi;
      const int w0 = q0 * P.conv_stride + P.lower[phase][0];
      const int h0 = p0 * P.conv_stride + P.lower[phase][1];
      const int d0 = z0 * P.conv_stride + P.lower[phase][2];
      const int kbase = phase * P.kphase;
      int tw = 0, th = 0, td = 0, cc = 0;
      if (kb_lo > 0 && kb_lo < nkb_main) {          // resume the (tap, channel chunk) counters at kb_lo
        cc = kb_lo % ncm;
        const int tap = kb_lo / ncm;
        tw = tap % P.kw;
        th = (tap / P.kw) % P.kh;
        td = tap / (P.kw * P.kh);
      }
      for (int kb = kb_lo; kb < kb_hi; ++kb, ++git) {
        if (git >= S && !mbar_wait(&empty_bar[s], ph ^ 1, P.err_flag, 101)) { alive = false; break; }   // first S slots: free
        uint8_t* sa = smem + s * stage_bytes;
        if (elect_one()) {
          mbar_expect_tx(&full_bar[s], tx);
          if (kb < nkb_main) {
            tma_load_im2col_5d(&P.amap[phase], &full_bar[s], sa, cc * BK, w0, h0, d0, n0,
                               (uint16_t)tw, (uint16_t)th, (uint16_t)td);
          } else {
            tma_load_im2col_5d(&P.xmap, &full_bar[s], sa, (kb - nkb_main) * BK, q0, p0, z0, n0, 0, 0, 0);
          }
#pragma unroll
          for (int t = 0; t < terms; ++t)
            tma_load_2d(&P.bmap, &full_bar[s], sa + A_BYTES + t * B_BYTES, kbase + kb * BK,
                        n_tile * BN + t * P.cout);
        }
        // advance (channel chunk, tap) counters and the stage ring without div/mod
        if (++cc == ncm) {
          cc = 0;
          if (++tw == P.kw) {
            tw = 0;
            if (++th == P.kh) { th = 0; ++td; }
          }
        }
        if (++s == S) { s = 0; ph ^= 1; }
      }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp runs the loop; one elected lane issues) =====
    {
      constexpr uint32_t DESC_HI = kmajor_desc_hi(ROWB);
      const int lo_from = P.epi.lo_from > 0 ? P.epi.lo_from : 0x40000000;
      const int lo_from_x = P.epi.lo_from_x > 0 ? P.epi.lo_from_x : 0x40000000;
      const uint32_t lo0 = kmajor_desc_lo(smem_u32(smem));
      const uint32_t lo_stage = static_cast<uint32_t>(stage_bytes) >> 4;
      int s = 0;
      uint32_t ph = 0, acc = 0;
      bool alive = true;
      for (int pi = 0; pi < ppc && alive; ++pi) {
      if (pi > 0) {                                   // the epilogue must have drained the accumulator
        if (!mbar_wait(tmem_empty, (pi - 1) & 1, P.err_flag, 104)) break;
        tc_fence_after();
        acc = 0;
      }
      int cc = (kb_lo > 0 && kb_lo < nkb_main) ? kb_lo % ncm : 0;
      for (int kb = kb_lo; kb < kb_hi; ++kb) {
        if (!mbar_wait(&full_bar[s], ph, P.err_flag, 102)) { alive = false; break; }
        tc_fence_after();
        // first channel of this k-block relative to where the lo halves of the operand pairs start
        const int rel = kb < nkb_main ? cc * BK - lo_from : (kb - nkb_main) * BK - lo_from_x;
        if (elect_one()) {
          const uint32_t a_lo = lo0 + s * lo_stage;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint32_t idesc = (TERMS == 2 && acc && rel + k * 16 >= 0) ? IDESC_HI : IDESC;
            umma_f16_lohi(tmem_base, a_lo + 2 * k, a_lo + (A_BYTES >> 4) + 2 * k, DESC_HI, idesc, acc);
            acc = 1;
          }
          umma_commit(&empty_bar[s]);   // frees the smem slot once these MMAs retire
        }
        if (++cc == ncm) cc = 0;
        if (++s == S) { s = 0; ph ^= 1; }
      }
      if (elect_one()) umma_commit(tmem_full);       // accumulator of this phase complete
      __syncwarp();
      }
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    // Everything that does not depend on the accumulator is fetched while the mainloop runs:
    // per-column bias (+ match bias + batch-uniform time-embedding row) into shared memory,
    // the first residual chunk into registers.
    const int quarter = warp & 3;     // TMEM lane quarter this warp may access
    const int row = quarter * 32 + lane;
    const int m = m_tile * CONV_BM + row;
    const bool valid = m < P.M;
    const int et = threadIdx.x - 64;  // 0..127 within the epilogue warps
    const bool temb_uniform = P.epi.temb != nullptr && P.epi.temb_bstride == 0;
    {
      const int trow = (P.epi.temb && P.epi.t_dev) ? *P.epi.t_dev : 0;
      for (int c = et; c < BN; c += 128) {
        const int n = n_tile * BN + c;
        float v = P.epi.bias ? P.epi.bias[n] : 0.f;
        if (P.epi.bias2) v += P.epi.bias2[n];
        if (temb_uniform) v += P.epi.temb[static_cast<size_t>(trow) * P.epi.temb_ld + n];
        colv[c] = v;
      }
    }
    int b = 0, sz = 0, sp = 0, sq = 0;
    size_t orow = 0;
    if (valid) {
      b = m / P.pps;
      if (P.scatter) {
        int r = m - b * P.pps;
        sz = r / (P.oh * P.ow);
        r -= sz * P.oh * P.ow;
        sp = r / P.ow;
        sq = r - sp * P.ow;
      } else if (P.rmap_out > 0) {
        orow = static_cast<size_t>(b) * P.rmap_out + P.rmap_off + (m - b * P.pps);
      } else {
        orow = static_cast<size_t>(m);
      }
    }
    const float* gate_row = (P.gate && valid) ? P.gate + static_cast<size_t>(b) * P.gate_ld + n_tile * BN : nullptr;
    const float* temb_row = nullptr;     // per-sample rows (training): added per element
    if (P.epi.temb && !temb_uniform)
      temb_row = P.epi.temb + static_cast<size_t>(b) * P.epi.temb_bstride + n_tile * BN;
    asm volatile("bar.sync 1, 128;" ::: "memory");   // colv visible to the 4 epilogue warps

    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    for (int pi = 0; pi < ppc; ++pi) {
    if (P.scatter && valid) {
      const int phase = phase0 + pi;
      const int pq = phase & 1, pp = (phase >> 1) & 1, pz = (phase >> 2) & 1;
      orow = ((static_cast<size_t>(b) * (2 * P.od) + (2 * sz + pz)) * (2 * P.oh) + (2 * sp + pp)) *
                 (2 * P.ow) + (2 * sq + pq);
    }
    const float* rp = (P.epi.resid && valid && P.ksplit <= 1) ? P.epi.resid + orow * P.cout + n_tile * BN : nullptr;   // orow == m unless scattering
    float4 rnext[4];
    if (rp) {                      // first residual chunk in flight while the main loop finishes
#pragma unroll
      for (int i = 0; i < 4; ++i) rnext[i] = *reinterpret_cast<const float4*>(rp + 4 * i);
    }
    if (!mbar_wait(tmem_full, pi & 1, P.err_flag, 103)) break;
    tc_fence_after();

    if (P.ksplit > 1) {
      // split-K: raw partial accumulators -> this CTA's shared memory (the pipeline stages are idle:
      // every TMA landed and every MMA retired); reduced across the cluster after the barrier below
      float* ptile = reinterpret_cast<float*>(smem) + static_cast<size_t>(row) * (BN + 4);
#pragma unroll 1
      for (int c = 0; c < BN / 16; ++c) {
        float v[16];
        tmem_ld16(t_lane + c * 16, v);
        if (TERMS == 2) {
          float v2[16];
          tmem_ld16(t_lane + BN + c * 16, v2);
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += v2[i];
        }
#pragma unroll
        for (int i = 0; i < 16; i += 4)
          *reinterpret_cast<float4*>(ptile + c * 16 + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      }
    } else
#pragma unroll 1
    for (int c = 0; c < BN / 16; ++c) {
      float4 rcur[4];
      if (rp) {
#pragma unroll
        for (int i = 0; i < 4; ++i) rcur[i] = rnext[i];
        if (c + 1 < BN / 16) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            rnext[i] = *reinterpret_cast<const float4*>(rp + (c + 1) * 16 + 4 * i);
        }
      }
      float v[16];
      tmem_ld16(t_lane + c * 16, v);
      if (TERMS == 2) {
        float v2[16];
        tmem_ld16(t_lane + BN + c * 16, v2);
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] += v2[i];
      }
      if (!valid) continue;
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        const float4 t4 = *reinterpret_cast<const float4*>(colv + c * 16 + i);
        v[i] += t4.x; v[i + 1] += t4.y; v[i + 2] += t4.z; v[i + 3] += t4.w;
      }
      if (temb_row) {
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
          const float4 t4 = *reinterpret_cast<const float4*>(temb_row + c * 16 + i);
          v[i] += t4.x; v[i + 1] += t4.y; v[i + 2] += t4.z; v[i + 3] += t4.w;
        }
      }
      if (P.act == 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = 0.5f * v[i] * (1.0f + erff(v[i] * 0.70710678118654752f));
      }
      if (gate_row) {
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
          const float4 g4 = *reinterpret_cast<const float4*>(gate_row + c * 16 + i);
          v[i] *= g4.x; v[i + 1] *= g4.y; v[i + 2] *= g4.z; v[i + 3] *= g4.w;
        }
      }
      if (rp) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          v[4 * i] += rcur[i].x; v[4 * i + 1] += rcur[i].y; v[4 * i + 2] += rcur[i].z; v[4 * i + 3] += rcur[i].w;
        }
      }
      const int n = n_tile * BN + c * 16;
      // row-per-thread stores: 32 bytes (one sector) per instruction (256-bit stores; every row start and n are multiples
      // of 16 elements, so fp32 chunks are 64-byte and fp16 chunks 32-byte aligned)
      if (P.epi.out32) {
        float* op = P.epi.out32 + orow * P.epi.out_ld + n;
        st_global_v8(op, v);
        st_global_v8(op + 8, v + 8);
      }
      if (P.epi.out16) {
        __half* op = P.epi.out16 + orow * (P.epi.out16_ld > 0 ? P.epi.out16_ld : P.epi.out_ld) + n;
        uint32_t uh[8], ul[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
          uh[i] = *reinterpret_cast<const uint32_t*>(&h);
          const float2 f = __half22float2(h);
          const __half2 l = __floats2half2_rn(v[2 * i] - f.x, v[2 * i + 1] - f.y);
          ul[i] = *reinterpret_cast<const uint32_t*>(&l);
        }
        st_global_v8(op, uh);
        if (P.epi.out16_lo > 0) st_global_v8(op + P.epi.out16_lo, ul);
      }
    }
    if (pi + 1 < ppc) {          // hand the accumulator back to the MMA warp for the next phase
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty);
    }
    }
  }

  if (P.ksplit > 1) {
    // ---- deterministic split-K reduction through distributed shared memory ----
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (warp >= 2) {
      uint32_t rank;
      asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
      const int S = P.ksplit;
      const int r0 = (CONV_BM * static_cast<int>(rank)) / S, r1 = (CONV_BM * (static_cast<int>(rank) + 1)) / S;
      constexpr int LPR = BN / 4;                 // lanes per row
      constexpr int RPP = 128 / LPR;              // rows per pass of the 128 epilogue threads
      const int et = threadIdx.x - 64;
      const int sub_c = (et % LPR) * 4;
      const uint32_t local = smem_u32(smem);
      const float4 cv = *reinterpret_cast<const float4*>(colv + sub_c);
      for (int rr = r0 + et / LPR; rr < r1; rr += RPP) {
        const int m = m_tile * CONV_BM + rr;
        if (m >= P.M) break;
        float4 acc = cv;
        const uint32_t off = local + static_cast<uint32_t>((rr * (BN + 4) + sub_c) * 4);
        const int n = n_tile * BN + sub_c;
        // all peer loads (and the residual) in flight together, then a fixed-order sum
        float4 pv[8];
        float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (P.epi.resid) r4 = *reinterpret_cast<const float4*>(P.epi.resid + static_cast<size_t>(m) * P.cout + n);
#pragma unroll
        for (int sidx = 0; sidx < 8; ++sidx) {
          pv[sidx] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (sidx < S) {
            uint32_t remote;
            asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(off), "r"(sidx));
            asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(pv[sidx].x), "=f"(pv[sidx].y), "=f"(pv[sidx].z), "=f"(pv[sidx].w)
                         : "r"(remote));
          }
        }
#pragma unroll
        for (int sidx = 0; sidx < 8; ++sidx) {
          acc.x += pv[sidx].x; acc.y += pv[sidx].y; acc.z += pv[sidx].z; acc.w += pv[sidx].w;
        }
        if (P.epi.temb && P.epi.temb_bstride != 0) {
          const float4 t4 = *reinterpret_cast<const float4*>(P.epi.temb + static_cast<size_t>(m / P.pps) * P.epi.temb_bstride + n);
          acc.x += t4.x; acc.y += t4.y; acc.z += t4.z; acc.w += t4.w;
        }
        acc.x += r4.x; acc.y += r4.y; acc.z += r4.z; acc.w += r4.w;
        if (P.epi.out32) *reinterpret_cast<float4*>(P.epi.out32 + static_cast<size_t>(m) * P.epi.out_ld + n) = acc;
        if (P.epi.out16) {
          __half2 h0 = __floats2half2_rn(acc.x, acc.y), h1 = __floats2half2_rn(acc.z, acc.w);
          uint2 u;
          u.x = *reinterpret_cast<uint32_t*>(&h0);
          u.y = *reinterpret_cast<uint32_t*>(&h1);
          __half* o16 = P.epi.out16 + static_cast<size_t>(m) * (P.epi.out16_ld > 0 ? P.epi.out16_ld : P.epi.out_ld) + n;
          *reinterpret_cast<uint2*>(o16) = u;
          if (P.epi.out16_lo > 0) {
            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
            __half2 l0 = __floats2half2_rn(acc.x - f0.x, acc.y - f0.y), l1 = __floats2half2_rn(acc.z - f1.x, acc.w - f1.y);
            u.x = *reinterpret_cast<uint32_t*>(&l0);
            u.y = *reinterpret_cast<uint32_t*>(&l1);
            *reinterpret_cast<uint2*>(o16 + P.epi.out16_lo) = u;
          }
        }
      }
    }
    // peers may still be reading this CTA's partial tile
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

// -------------------------------- host side --------------------------------
struct ConvLaunch {
  ConvParams p;
  dim3 grid;
  int bn, bk;
  size_t smem;
};

// Fill amap/xmap/bmap + geometry.  `mode`: 0 = k3 s1 p1 ("same"), 1 = k3 s2 p1 (DownSample),
// 2 = nearest-x2 + k3 p1 decomposed into 8 phase convs with 2x2x2 combined taps (UpSample),
// 3 = 1x1x1.  Extra source: 1x1x1 over the OUTPUT grid with cin_extra channels.  epi.stats_rec is dropped.
int conv_prepare(ConvLaunch* L, int mode, const __half* act, int B, int D, int H, int W, int cin,
                 const __half* extra, int cin_extra, const __half* wpacked, int cout, int terms, const ConvEpilogue& epi,
                 bool allow_splitk = true);
int conv_enqueue(const ConvLaunch& L, cudaStream_t st);
size_t conv_packed_k(int mode, int cin, int cin_extra);   // K elements of the packed weight rows

}  // namespace cm
