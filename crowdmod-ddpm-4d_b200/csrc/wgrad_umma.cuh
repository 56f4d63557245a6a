// Weight gradient of the implicit-GEMM 3-D convolutions on tcgen05 / TMEM, sm_100a.
//
// Replaces the cuDNN backward-filter calls autograd issues for every nn.Conv3d of the
// reference UNet during DDPM_model._train_step (models/diffusion/ddpm.py:111-121,143;
// models/backbones/layers.py:32,43,46,84,92-94 and the two attention projections :10,16).
//
//   G[(tap, ci), co] = sum_p  A[p + tap, ci] * dOut[p, co]          p = output pixel
//
// i.e. a GEMM whose reduction runs over the B*L*H*W output pixels.  Both operands live in
// HBM channels-last ([pixel][channel], fp16), so in GEMM terms they are MN-major (the K
// index = pixel is the strided one).  Neither is transposed in memory: each k-block is a set
// of TMA im2col loads of 128 consecutive output pixels x 32|64 channels -- exactly the tiles the
// forward conv loads -- and the UMMA shared-memory descriptors + instruction descriptor mark
// both operands MN-major, so the tensor core does the transposition.
//
//   M tile (128 TMEM lanes) = 128/BKC "atoms"; an atom = (filter tap, channel chunk of BKC) of
//                             the main source, or a channel chunk of the fused 1x1x1
//                             match_input source.  One TMA im2col load per atom per k-block.
//   N tile                  = BN output channels of dOut (BN/BNC loads of BNC channels).
//   K                       = pixels, split across gridDim.y CTAs; partial sums are combined with
//                             fp32 atomics into G (zeroed by the caller), or, deterministic (DET), stored
//                             per split into `part` [split][phase][krows][cout] and summed in split order
//                             by wgrad_run_enqueue.
//
// G is [phase][taps*cin + cin_extra][cout] fp32 ("packed-K" row order, identical to the
// forward weight packing); unpack_wgrad_kernel (backward.cu) turns it into the nn.Conv3d
// weight layout.
#pragma once
#include "common.cuh"

namespace cm {

constexpr int WG_KT = 128;          // pixels per k-block (= TMA im2col pixelsPerColumn)
constexpr int WG_THREADS = 192;     // warp0 TMA, warp1 MMA, warps2-5 epilogue
constexpr int WG_MAX_STAGES = 4;

struct WgradParams {
  CUtensorMap amap[8];   // main source (forward conv input), one per output phase
  CUtensorMap xmap;      // fused 1x1x1 source (match_input), k=1 over the output grid
  CUtensorMap gmap[8];   // dOut, k=1; per phase for the UpSample conv (stride-2 gather)
  int M;                 // pixels per phase (GEMM K extent)
  int od, oh, ow, pps;   // pixel traversal extents per sample
  int conv_stride;       // traversal stride in the main source
  int gstride;           // traversal stride in dOut (2 for UpSample phases, else 1)
  int kd, kh, kw, nphase;
  signed char lower[8][4];    // main-source lower corner {w,h,d} per phase
  signed char glower[8][4];   // dOut lower corner per phase
  int cin_main, cin_extra, cout;
  int ncm;               // channel chunks of the main source
  int atoms_main, atoms_total, apt;   // apt = atoms per M tile = 128 / BKC
  int n_tiles, splits, kb_total, kb_per_split;
  int krows;             // rows of G per phase
  int stages;
  float* G;
  float* part;           // DET only: splits * nphase * krows * cout floats
  int* err_flag;
};

// MN-major K-advance: one UMMA consumes 16 pixels = 16 smem rows of ROWB bytes.
__host__ __device__ constexpr uint32_t make_idesc_f16_mn(int M, int N) {
  return (1u << 4) | (1u << 15) | (1u << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// low word of an MN-major descriptor: start address + LBO (byte distance between
// consecutive 32|64-channel blocks along M/N)
__device__ __forceinline__ uint32_t mnmajor_desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}

template <int BKC, int BNC, int BN, bool DET>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_umma_kernel(const __grid_constant__ WgradParams P) {
  constexpr int ROWA = BKC * 2, ROWB = BNC * 2;          // smem row bytes (swizzle span)
  constexpr int A_ATOM = WG_KT * ROWA, B_ATOM = WG_KT * ROWB;
  constexpr int APT = 128 / BKC, BPT = BN / BNC;
  constexpr int STAGE = APT * A_ATOM + BPT * B_ATOM;
  constexpr uint32_t IDESC = make_idesc_f16_mn(128, BN);
  constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  const int S = P.stages;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S * STAGE);
  uint64_t* empty_bar = full_bar + WG_MAX_STAGES;
  uint64_t* tmem_full = empty_bar + WG_MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x;
  const int n_tile = blockIdx.y % P.n_tiles;
  const int split = blockIdx.y / P.n_tiles;
  const int phase = blockIdx.z;
  const int kb0 = split * P.kb_per_split;
  const int kb1 = min(P.kb_total, kb0 + P.kb_per_split);
  const int nkb = kb1 - kb0;       // >= 1 by construction of the grid

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&P.amap[phase]);
    tma_prefetch_desc(&P.gmap[phase]);
    if (P.cin_extra) tma_prefetch_desc(&P.xmap);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    int natoms = P.atoms_total - m_tile * APT;
    natoms = natoms < APT ? natoms : APT;
    const uint32_t tx = natoms * A_ATOM + BPT * B_ATOM;
    int s = 0;
    uint32_t ph = 0;
    for (int kb = kb0; kb < kb1; ++kb) {
      if (!mbar_wait(&empty_bar[s], ph ^ 1, P.err_flag, 201)) break;
      if (elect_one()) {
        uint8_t* sa = smem + s * STAGE;
        const int m0 = kb * WG_KT;
        const int n0 = m0 / P.pps;
        int r = m0 - n0 * P.pps;
        const int z0 = r / (P.oh * P.ow);
        r -= z0 * P.oh * P.ow;
        const int p0 = r / P.ow;
        const int q0 = r - p0 * P.ow;
        mbar_expect_tx(&full_bar[s], tx);
        for (int la = 0; la < natoms; ++la) {
          const int ga = m_tile * APT + la;
          if (ga < P.atoms_main) {
            const int tap = ga / P.ncm, cc = ga - tap * P.ncm;
            const int tw = tap % P.kw, th = (tap / P.kw) % P.kh, td = tap / (P.kw * P.kh);
            tma_load_im2col_5d(&P.amap[phase], &full_bar[s], sa + la * A_ATOM, cc * BKC,
                               q0 * P.conv_stride + P.lower[phase][0],
                               p0 * P.conv_stride + P.lower[phase][1],
                               z0 * P.conv_stride + P.lower[phase][2], n0, (uint16_t)tw,
                               (uint16_t)th, (uint16_t)td);
          } else {
            tma_load_im2col_5d(&P.xmap, &full_bar[s], sa + la * A_ATOM, (ga - P.atoms_main) * BKC,
                               q0, p0, z0, n0, 0, 0, 0);
          }
        }
#pragma unroll
        for (int j = 0; j < BPT; ++j)
          tma_load_im2col_5d(&P.gmap[phase], &full_bar[s], sa + APT * A_ATOM + j * B_ATOM,
                             n_tile * BN + j * BNC, q0 * P.gstride + P.glower[phase][0],
                             p0 * P.gstride + P.glower[phase][1],
                             z0 * P.gstride + P.glower[phase][2], n0, 0, 0, 0);
      }
      __syncwarp();
      if (++s == S) { s = 0; ph ^= 1; }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t HI_A = kmajor_desc_hi(ROWA);   // SBO = 8 rows, version, swizzle mode
    constexpr uint32_t HI_B = kmajor_desc_hi(ROWB);
    int s = 0;
    uint32_t ph = 0, acc = 0;
    for (int kb = 0; kb < nkb; ++kb) {
      if (!mbar_wait(&full_bar[s], ph, P.err_flag, 202)) break;
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a_addr = smem_u32(smem + s * STAGE);
        const uint32_t a_lo = mnmajor_desc_lo(a_addr, A_ATOM);
        const uint32_t b_lo = mnmajor_desc_lo(a_addr + APT * A_ATOM, B_ATOM);
#pragma unroll
        for (int k = 0; k < WG_KT / 16; ++k) {
          const uint64_t da = (static_cast<uint64_t>(HI_A) << 32) | (a_lo + ((k * 16 * ROWA) >> 4));
          const uint64_t db = (static_cast<uint64_t>(HI_B) << 32) | (b_lo + ((k * 16 * ROWB) >> 4));
          umma_f16(tmem_base, da, db, IDESC, acc);
          acc = 1;
        }
        umma_commit(&empty_bar[s]);
      }
      __syncwarp();
      if (++s == S) { s = 0; ph ^= 1; }
    }
    if (elect_one()) umma_commit(tmem_full);
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2..5): TMEM -> fp32 atomics into G =================
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int la = row / BKC, ch = row - la * BKC;
    const int ga = m_tile * APT + la;
    const bool valid = ga < P.atoms_total;
    size_t krow = 0;
    if (valid) {
      if (ga < P.atoms_main) {
        const int tap = ga / P.ncm, cc = ga - tap * P.ncm;
        krow = static_cast<size_t>(tap) * P.cin_main + cc * BKC + ch;
      } else {
        krow = static_cast<size_t>(P.kd * P.kh * P.kw) * P.cin_main + (ga - P.atoms_main) * BKC + ch;
      }
    }
    float* gp = (DET ? P.part + static_cast<size_t>(split) * P.nphase * P.krows * P.cout : P.G) +
                (static_cast<size_t>(phase) * P.krows + krow) * P.cout + n_tile * BN;
    mbar_wait(tmem_full, 0, P.err_flag, 203);
    tc_fence_after();
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
#pragma unroll 1
    for (int c = 0; c < BN / 16; ++c) {
      float v[16];
      tmem_ld16(t_lane + c * 16, v);
      if (!valid) continue;
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        if constexpr (DET) *reinterpret_cast<float4*>(gp + c * 16 + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        else red_add_v4(gp + c * 16 + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

struct WgradLaunch {
  WgradParams p;
  dim3 grid;
  int bkc, bnc, bn;
  size_t smem;
};

// `mode` = forward conv mode (0 k3 s1, 1 k3 s2, 2 nearest-x2 + k3 as 8 phases, 3 1x1x1).
// act: forward input [B,D,H,W,cin]; extra: [B,od,oh,ow,cin_extra] or null; dout: fp16
// [B,od',oh',ow',cout] (the forward output grid).  G: fp32 [nphase][krows][cout], pre-zeroed.
// dout_ld: channel stride of a dOut pixel row (0 -> cout; 2*cout for a K-concatenated hi|lo pair, hi half read)
int wgrad_prepare(WgradLaunch* L, int mode, const __half* act, int B, int D, int H, int W, int cin,
                  const __half* extra, int cin_extra, const __half* dout, int cout, float* G, int dout_ld = 0,
                  int act_ld = 0, int extra_ld = 0);   // row strides of act / extra (hi half of hi|lo pair rows)
int wgrad_enqueue(const WgradLaunch& L, cudaStream_t st);
int wgrad_init();
size_t wgrad_g_elems(int mode, int cin, int cin_extra, int cout);

int make_act_map(CUtensorMap* map, const __half* base, int B, int D, int H, int W, int C, int bk,
                 int lower_w, int lower_h, int lower_d, int stride, int upper_delta, int ld = 0);

}  // namespace cm
