// Attention core for sequences longer than 128 tokens and for head dims above 64 (attn_uses_long in kernels.cuh; the
// rest stays on attn_mma_kernel and attn_core_backward_kernel).  Contracts in kernels.cuh (forward) and backward.cuh
// (backward).
//
// Forward (attn_long_kernel): one CTA per (128-query tile, sample * head); keys stream in tiles of 128 with the
// online softmax (running max m and sum l per query row).  Numerics follow attn_mma_kernel:
//   scores  one tcgen05 product with K = 3 * DHP:  A rows [Qh | Ql | Qh] . B rows [Kh | Kh | Kl]
//           (fp16 hi + lo splits, fp32 accumulation: fp32-accurate scores).  Q is pre-scaled by log2(e) / sqrt(dh),
//           so the scores are in the log2 domain and each exponential is one ex2.approx.
//   P . V   P = 2^(s - m) in [0, 1] and V as single fp16 operands, a second tcgen05 product with N = DHP.
// Only the hi and lo halves are stored; the concatenation is three descriptor streams over them.  DHP is the head
// dim padded to 16 / 32 / 64 / 128.
//   warps 0-3  softmax: thread t owns query row t (TMEM lane t); per key tile it reads the scores from TMEM twice
//              (row max, then exponentials), writes P to shared memory, and folds the previous tile's P.V product
//              into O (registers) as O = O * alpha + PV.  The Q tile is staged by these warps once.
//   warps 4-5  producer: K and V rows (fp32) -> fp16 hi / lo K rows and V^T, 128-byte swizzled K-major, 2 stages.
//              At DHP = 128 two K stages do not fit next to Q (227 KB): K has one buffer, refilled once S(j-1) is done
//              (the s_full commit), and only V has two.
//   warp  6    MMA issuer (one elected thread).
// Per key tile j the issuer runs PV(j-1) then S(j) and commits once: that commit tells the softmax warps both that
// S(j) is in TMEM and that PV(j-1) has finished reading P, so P and the PV columns are single-buffered.  256 TMEM
// columns (S: 128, PV: DHP) let two CTAs share an SM at DHP <= 32, so one CTA's softmax overlaps the other's MMAs.
// At DHP = 128 S and PV fill all 256 columns, and O (128 floats a row) stays in the softmax threads' registers.
//
// Backward: two deterministic fp32 SIMT kernels (no atomics) that recompute P = exp(s - lse) from qkv and the
// forward's row log-sum-exp.  attn_long_dq_kernel walks one 64-query tile per CTA over all key tiles (twice: first the
// row sums D_i = sum_j P_ij dP_ij, then dQ); attn_long_dkdv_kernel walks one 64-key tile over all query tiles.
#include "backward.cuh"
#include "common.cuh"
#include "kernels.cuh"

namespace cm {

namespace {

constexpr int AL_THREADS = 224;
constexpr uint32_t AL_TMEM_COLS = 256;
constexpr int AL_STAGES = 2;

template <int DHP>
struct AlCfg {
  static constexpr int KCH = (2 * DHP + 63) / 64;                          // 64-column chunks of a [hi | lo] row
  static constexpr uint32_t Q_BYTES = KCH * 128u * 128u;                    // 128 query rows
  static constexpr uint32_t K_BYTES = KCH * 128u * 128u;                    // 128 key rows
  static constexpr uint32_t V_BYTES = 2u * DHP * 128u;                      // V^T: 2 chunks of 64 keys x DHP rows
  static constexpr uint32_t P_BYTES = 2u * 128u * 128u;                     // 128 rows x 2 chunks of 64 keys
  static constexpr uint32_t STAGE_BYTES = K_BYTES + V_BYTES;
  static constexpr bool K_SOLO = DHP > 64;                                  // one K buffer, two V buffers
  static constexpr uint32_t KV_BYTES = K_SOLO ? K_BYTES + AL_STAGES * V_BYTES : AL_STAGES * STAGE_BYTES;
  static constexpr uint32_t SMEM = 1024 + Q_BYTES + KV_BYTES + P_BYTES + 256;
  // stage s: K rows at s * K_STRIDE, V^T at s * V_STRIDE + K_BYTES in the K / V region
  static constexpr uint32_t K_STRIDE = K_SOLO ? 0u : STAGE_BYTES;
  static constexpr uint32_t V_STRIDE = K_SOLO ? V_BYTES : STAGE_BYTES;
};

// byte offset of element (row, col) in a K-major operand of `rows` rows stored as 64-column chunks with the 128-byte
// swizzle (16-byte unit index XOR row % 8; chunk bases 1024-aligned)
__device__ __forceinline__ uint32_t swz(int row, int col, int rows) {
  return static_cast<uint32_t>((col >> 6) * rows * 128 + row * 128 + ((((col >> 3) & 7) ^ (row & 7)) << 4) + (col & 7) * 2);
}

__device__ __forceinline__ void al_split(float x, float y, uint32_t* hi, uint32_t* lo) {
  const __half hx = __float2half_rn(x), hy = __float2half_rn(y);
  __half2 h = __halves2half2(hx, hy);
  __half2 l = __floats2half2_rn(x - __half2float(hx), y - __half2float(hy));
  *hi = *reinterpret_cast<uint32_t*>(&h);
  *lo = *reinterpret_cast<uint32_t*>(&l);
}
__device__ __forceinline__ uint32_t al_pack(float x, float y) {
  __half2 h = __floats2half2_rn(x, y);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int DHP>
__global__ void __launch_bounds__(AL_THREADS, DHP <= 32 ? 2 : 1)
attn_long_kernel(const float* __restrict__ qkv, __half* __restrict__ ctx, float* __restrict__ lse, int S, int C,
                 int heads, int dup, int* err) {
  using Cfg = AlCfg<DHP>;
  constexpr uint32_t IDESC_S = make_idesc_f16(128, 128);
  constexpr uint32_t IDESC_O = make_idesc_f16(128, DHP);
  constexpr uint32_t DESC_HI = kmajor_desc_hi(128);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* Qs = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  uint8_t* KVs = Qs + Cfg::Q_BYTES;
  uint8_t* Ps = KVs + Cfg::KV_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(Ps + Cfg::P_BYTES);
  uint64_t* q_full = bars;                  // count 128: Q tile staged
  uint64_t* kv_full = bars + 1;             // [2] count 64: K / V stage written
  uint64_t* kv_empty = bars + 3;            // [2] tcgen05.commit: the stage's MMAs are done
  uint64_t* s_full = bars + 5;              // tcgen05.commit: S(j) in TMEM and PV(j-1) done (once more after the last PV)
  uint64_t* p_full = bars + 6;              // count 128: P(j) in shared memory, PV(j-1) read out of TMEM
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int warp = threadIdx.x >> 5;
  const int qt = blockIdx.x, bh = blockIdx.y;
  const int b = bh / heads, hd = bh - b * heads;
  const int dh = C / heads;
  const int nkt = (S + 127) >> 7;
  const float* base = qkv + (size_t)b * S * 3 * C + hd * dh;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 128);
    mbar_init(&kv_full[0], 64);
    mbar_init(&kv_full[1], 64);
    mbar_init(&kv_empty[0], 1);
    mbar_init(&kv_empty[1], 1);
    mbar_init(s_full, 1);
    mbar_init(p_full, 128);
    fence_mbar_init();
  }
  if (warp == 6) tmem_alloc(tmem_slot, AL_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ===================== softmax warps =====================
    const int r = threadIdx.x;                       // query row of the tile = TMEM lane
    const int qi = qt * 128 + r;
    {
      const float qscale = 1.4426950408889634f * rsqrtf((float)dh);
#pragma unroll
      for (int g = 0; g < DHP / 8; ++g) {
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; e += 2) {
          const int d = g * 8 + e;
          float2 f = make_float2(0.f, 0.f);
          if (qi < S && d < dh) f = *reinterpret_cast<const float2*>(base + (size_t)qi * 3 * C + d);
          v[e] = f.x * qscale;
          v[e + 1] = f.y * qscale;
        }
        uint4 h, l;
        al_split(v[0], v[1], &h.x, &l.x);
        al_split(v[2], v[3], &h.y, &l.y);
        al_split(v[4], v[5], &h.z, &l.z);
        al_split(v[6], v[7], &h.w, &l.w);
        *reinterpret_cast<uint4*>(Qs + swz(r, g * 8, 128)) = h;
        *reinterpret_cast<uint4*>(Qs + swz(r, DHP + g * 8, 128)) = l;
      }
      fence_proxy_async();
      mbar_arrive(q_full);
    }
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    float o[DHP];
#pragma unroll
    for (int d = 0; d < DHP; ++d) o[d] = 0.f;
    float m = -INFINITY, l = 0.f, alpha_prev = 0.f;
    bool alive = true;
    for (int j = 0; j < nkt; ++j) {
      if (!mbar_wait(s_full, j & 1, err, 601)) { alive = false; break; }
      tc_fence_after();
      const int kbase = j * 128;
      float mx = -INFINITY;
#pragma unroll 1                                // unrolled, these two passes spill at the two-CTA budget of 128 registers
      for (int c = 0; c < 8; ++c) {
        float v[16];
        tmem_ld16(t_lane + c * 16, v);
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (kbase + c * 16 + i < S) mx = fmaxf(mx, v[i]);
      }
      const float m_new = fmaxf(m, mx);
      const float alpha = ex2(m - m_new);
      if (j > 0) {                                   // O = O * alpha(j-1) + P(j-1) V(j-1)
#pragma unroll
        for (int c = 0; c < DHP / 16; ++c) {
          float v[16];
          tmem_ld16(t_lane + 128 + c * 16, v);
#pragma unroll
          for (int i = 0; i < 16; ++i) o[c * 16 + i] = fmaf(o[c * 16 + i], alpha_prev, v[i]);
        }
      }
      float lsum = 0.f;
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        float v[16];
        tmem_ld16(t_lane + c * 16, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          v[i] = kbase + c * 16 + i < S ? ex2(v[i] - m_new) : 0.f;
          lsum += v[i];
        }
        uint4 p0, p1;
        p0.x = al_pack(v[0], v[1]); p0.y = al_pack(v[2], v[3]); p0.z = al_pack(v[4], v[5]); p0.w = al_pack(v[6], v[7]);
        p1.x = al_pack(v[8], v[9]); p1.y = al_pack(v[10], v[11]); p1.z = al_pack(v[12], v[13]); p1.w = al_pack(v[14], v[15]);
        *reinterpret_cast<uint4*>(Ps + swz(r, c * 16, 128)) = p0;
        *reinterpret_cast<uint4*>(Ps + swz(r, c * 16 + 8, 128)) = p1;
      }
      l = fmaf(l, alpha, lsum);
      m = m_new;
      alpha_prev = alpha;
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(p_full);
    }
    if (alive && mbar_wait(s_full, nkt & 1, err, 602)) {
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < DHP / 16; ++c) {
        float v[16];
        tmem_ld16(t_lane + 128 + c * 16, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) o[c * 16 + i] = fmaf(o[c * 16 + i], alpha_prev, v[i]);
      }
    }
    if (qi < S) {
      const float inv = 1.0f / l;
      const int Cd = C * dup;                        // dup = 2: hi | lo pair per token (training forward)
      __half* ob = ctx + ((size_t)b * S + qi) * Cd + hd * dh;
#pragma unroll
      for (int d = 0; d < DHP; d += 2) {
        if (d >= dh) break;
        if (dup == 2) {
          uint32_t hi, lo;
          al_split(o[d] * inv, o[d + 1] * inv, &hi, &lo);
          *reinterpret_cast<uint32_t*>(ob + d) = hi;
          *reinterpret_cast<uint32_t*>(ob + C + d) = lo;
        } else {
          *reinterpret_cast<uint32_t*>(ob + d) = al_pack(o[d] * inv, o[d + 1] * inv);
        }
      }
      // natural-log log-sum-exp of the scores q.k / sqrt(dh): (m + log2 l) * ln 2
      if (lse) lse[(size_t)bh * S + qi] = (m + log2f(l)) * 0.6931471805599453f;
    }
  } else if (warp < 6) {
    // ===================== producer: K / V tiles =====================
    const int pt = threadIdx.x - 128;
    constexpr int PAIRS = DHP / 2;
    const float* kb = base + C;
    for (int j = 0; j < nkt; ++j) {
      const int s = j & 1;
      if (j >= AL_STAGES && !mbar_wait(&kv_empty[s], ((j >> 1) - 1) & 1, err, 603)) break;
      if (Cfg::K_SOLO && j > 0 && !mbar_wait(s_full, (j - 1) & 1, err, 608)) break;   // S(j-1) has read K
      uint8_t* Ks = KVs + s * Cfg::K_STRIDE;
      uint8_t* Vt = KVs + s * Cfg::V_STRIDE + Cfg::K_BYTES;
#pragma unroll 4
      for (int idx = pt; idx < 128 * PAIRS; idx += 64) {
        const int key = idx / PAIRS, d = (idx - key * PAIRS) * 2;
        const int kj = j * 128 + key;
        float2 kv = make_float2(0.f, 0.f), vv = kv;
        if (kj < S && d < dh) {
          kv = *reinterpret_cast<const float2*>(kb + (size_t)kj * 3 * C + d);
          vv = *reinterpret_cast<const float2*>(kb + (size_t)kj * 3 * C + C + d);
        }
        uint32_t hi, lo;
        al_split(kv.x, kv.y, &hi, &lo);
        *reinterpret_cast<uint32_t*>(Ks + swz(key, d, 128)) = hi;
        *reinterpret_cast<uint32_t*>(Ks + swz(key, DHP + d, 128)) = lo;
        *reinterpret_cast<__half*>(Vt + swz(d, key, DHP)) = __float2half_rn(vv.x);
        *reinterpret_cast<__half*>(Vt + swz(d + 1, key, DHP)) = __float2half_rn(vv.y);
      }
      fence_proxy_async();
      mbar_arrive(&kv_full[s]);
    }
  } else {
    // ===================== MMA issuer =====================
    const uint32_t q_lo = kmajor_desc_lo(smem_u32(Qs));
    const uint32_t kv_lo = kmajor_desc_lo(smem_u32(KVs));
    const uint32_t p_lo = kmajor_desc_lo(smem_u32(Ps));
    const uint32_t t_s = tmem_base, t_o = tmem_base + 128;
    constexpr int KS = DHP / 16;                     // k16 steps per segment
    // descriptor offset (16-byte units) of column `col` in a 128-row [hi | lo] operand
    auto col_lo = [](int col) -> uint32_t { return ((static_cast<uint32_t>(col >> 6) * 128u * 128u) >> 4) + 2u * ((col & 63) >> 4); };
    auto issue_pv = [&](int jj) {                    // O(TMEM) = P . V(jj): 8 k16 steps over 128 keys
      const uint32_t v_lo = kv_lo + (((jj & 1) * Cfg::V_STRIDE + Cfg::K_BYTES) >> 4);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        umma_f16_lohi(t_o, p_lo + (((k >> 2) * 128u * 128u) >> 4) + 2 * (k & 3),
                      v_lo + (((k >> 2) * DHP * 128u) >> 4) + 2 * (k & 3), DESC_HI, IDESC_O, k > 0);
      umma_commit(&kv_empty[jj & 1]);
    };
    bool alive = mbar_wait(q_full, 0, err, 604);
    tc_fence_after();
    for (int j = 0; j < nkt && alive; ++j) {
      if (!mbar_wait(&kv_full[j & 1], (j >> 1) & 1, err, 605)) { alive = false; break; }
      if (j > 0 && !mbar_wait(p_full, (j - 1) & 1, err, 606)) { alive = false; break; }
      tc_fence_after();
      if (elect_one()) {
        if (j > 0) issue_pv(j - 1);
        const uint32_t k_lo = kv_lo + (((j & 1) * Cfg::K_STRIDE) >> 4);
#pragma unroll
        for (int seg = 0; seg < 3; ++seg)            // [Qh | Ql | Qh] . [Kh | Kh | Kl]
#pragma unroll
          for (int k = 0; k < KS; ++k) {
            const int ca = (seg == 1 ? DHP : 0) + k * 16, cb = (seg == 2 ? DHP : 0) + k * 16;
            umma_f16_lohi(t_s, q_lo + col_lo(ca), k_lo + col_lo(cb), DESC_HI, IDESC_S, seg + k > 0);
          }
        umma_commit(s_full);
      }
      __syncwarp();
    }
    if (alive && mbar_wait(p_full, (nkt - 1) & 1, err, 607)) {
      tc_fence_after();
      if (elect_one()) {
        issue_pv(nkt - 1);
        umma_commit(s_full);
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 6) tmem_dealloc(tmem_base, AL_TMEM_COLS);
}

template <int DHP>
int al_launch(const float* qkv, __half* ctx, float* lse, int B, int S, int C, int heads, int dup, cudaStream_t st) {
  const dim3 grid((S + 127) / 128, B * heads);
  attn_long_kernel<DHP><<<grid, AL_THREADS, AlCfg<DHP>::SMEM, st>>>(qkv, ctx, lse, S, C, heads, dup, device_error_flag());
  CM_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// backward (fp32 SIMT, 64 x 64 tiles, 256 threads as 16 x 16: thread (ty, tx) owns rows ty + 16 r, columns tx + 16 c)
// ---------------------------------------------------------------------------------------------
constexpr int BT = 64;
constexpr int BLD = BT + 1;

template <int DH>
struct BwdSmem {
  static constexpr int LD = DH + 1;
  static constexpr size_t bytes() { return ((size_t)4 * BT * LD + (size_t)2 * BT * BLD + 2 * BT) * sizeof(float); }
};

// rows [r0, r0 + 64) of q | k | v (col0 = 0 | C | 2C) -> smem [64][DH + 1], zero beyond S and dh
template <int DH>
__device__ __forceinline__ void bw_stage(float* dst, const float* src, int ld_src, int r0, int S, int dh) {
  constexpr int LD = DH + 1;
  for (int idx = threadIdx.x; idx < BT * DH; idx += blockDim.x) {
    const int r = idx / DH, d = idx - r * DH;
    dst[r * LD + d] = (r0 + r < S && d < dh) ? src[(size_t)(r0 + r) * ld_src + d] : 0.f;
  }
}

// lse and D of query rows [i0, i0 + 64) from global memory (zero past S)
__device__ __forceinline__ void bw_rowstats(float* ls, float* Ds, const float* lse_bh, const float* dsum_bh, int i0, int S) {
  for (int r = threadIdx.x; r < BT; r += blockDim.x) {
    const bool ok = i0 + r < S;
    ls[r] = ok ? lse_bh[i0 + r] : 0.f;
    if (dsum_bh) Ds[r] = ok ? dsum_bh[i0 + r] : 0.f;
  }
}

// P and dP of the thread's 4 x 4 entries (rows ty + 16 r, columns tx + 16 c) of one 64 x 64 (query, key) tile; P = 0 past S
template <int DH>
__device__ __forceinline__ void bw_scores(float (&p)[4][4], float (&dp)[4][4], const float* Qs, const float* Ks,
                                          const float* dOs, const float* Vs, const float* ls, int i0, int j0, int S,
                                          float scale) {
  constexpr int LD = DH + 1;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float s[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) s[r][c] = dp[r][c] = 0.f;
#pragma unroll 4
  for (int d = 0; d < DH; ++d) {
    float q[4], g[4], k[4], v[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      q[r] = Qs[(ty + 16 * r) * LD + d];
      g[r] = dOs[(ty + 16 * r) * LD + d];
      k[r] = Ks[(tx + 16 * r) * LD + d];
      v[r] = Vs[(tx + 16 * r) * LD + d];
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        s[r][c] = fmaf(q[r], k[c], s[r][c]);
        dp[r][c] = fmaf(g[r], v[c], dp[r][c]);
      }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c)
      p[r][c] = (i0 + ty + 16 * r < S && j0 + tx + 16 * c < S) ? expf(fmaf(s[r][c], scale, -ls[ty + 16 * r])) : 0.f;
}

// P and dS = P o (dP - D) of one tile into Ps / dSs
template <int DH>
__device__ __forceinline__ void bw_tile(float* Ps, float* dSs, const float* Qs, const float* Ks, const float* dOs,
                                        const float* Vs, const float* ls, const float* Ds, int i0, int j0, int S,
                                        float scale) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float p[4][4], dp[4][4];
  bw_scores<DH>(p, dp, Qs, Ks, dOs, Vs, ls, i0, j0, S, scale);
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i = ty + 16 * r;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int j = tx + 16 * c;
      Ps[i * BLD + j] = p[r][c];
      dSs[i * BLD + j] = p[r][c] * (dp[r][c] - Ds[i]);
    }
  }
}

// acc[r][c] += sum_k A(row = ty + 16 r, k) * Bm[k][tx + 16 c];  A(row, k) = At[k * BLD + row] (transposed) or
// A[row * BLD + k]
template <int DH, bool TRANS>
__device__ __forceinline__ void bw_acc(float (&acc)[4][DH / 16], const float* A, const float* Bm) {
  constexpr int LD = DH + 1;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll 4
  for (int k = 0; k < BT; ++k) {
    float a[4], bv[DH / 16];
#pragma unroll
    for (int r = 0; r < 4; ++r) a[r] = TRANS ? A[k * BLD + ty + 16 * r] : A[(ty + 16 * r) * BLD + k];
#pragma unroll
    for (int c = 0; c < DH / 16; ++c) bv[c] = Bm[k * LD + tx + 16 * c];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < DH / 16; ++c) acc[r][c] = fmaf(a[r], bv[c], acc[r][c]);
  }
}

template <int DH>
__device__ __forceinline__ void bw_store(float* dst, const float (&acc)[4][DH / 16], float mul, int r0, int S, int dh,
                                         int ld) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i = r0 + ty + 16 * r;
    if (i >= S) continue;
#pragma unroll
    for (int c = 0; c < DH / 16; ++c) {
      const int d = tx + 16 * c;
      if (d < dh) dst[(size_t)i * ld + d] = acc[r][c] * mul;
    }
  }
}

struct BwdArgs {
  const float* qkv;
  const float* dctx;
  const float* lse;
  float* dsum;      // [B][heads][S]: D_i, written by attn_long_dq_kernel, read by attn_long_dkdv_kernel
  float* dqkv;
  int S, C, heads;
};

// One 64-query tile: pass 1 over all key tiles forms D_i = sum_j P_ij dP_ij (fp32, fixed order) and stores it for
// attn_long_dkdv_kernel; pass 2 forms dS and dQ_i = scale * sum_j dS_ij K_j.  D is taken from the recomputed P and dP
// rather than as dO_i . O_i: the forward's O carries its fp16 P . V rounding (~3e-4), which D would pass on to dQ.
template <int DH>
__global__ void __launch_bounds__(256) attn_long_dq_kernel(const BwdArgs a) {
  constexpr int LD = DH + 1;
  extern __shared__ __align__(16) float bsm[];
  float* Qs = bsm;
  float* dOs = Qs + BT * LD;
  float* Ks = dOs + BT * LD;
  float* Vs = Ks + BT * LD;
  float* Ps = Vs + BT * LD;
  float* dSs = Ps + BT * BLD;
  float* ls = dSs + BT * BLD;
  float* Ds = ls + BT;
  const int S = a.S, C = a.C, dh = C / a.heads;
  const int bh = blockIdx.y, b = bh / a.heads, hd = bh - b * a.heads;
  const int i0 = blockIdx.x * BT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const float scale = rsqrtf((float)dh);
  const float* qb = a.qkv + (size_t)b * S * 3 * C + hd * dh;
  const float* gb = a.dctx + (size_t)b * S * C + hd * dh;
  bw_stage<DH>(Qs, qb, 3 * C, i0, S, dh);
  bw_stage<DH>(dOs, gb, C, i0, S, dh);
  bw_rowstats(ls, Ds, a.lse + (size_t)bh * S, nullptr, i0, S);
  float dacc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int j0 = 0; j0 < S; j0 += BT) {
    __syncthreads();
    bw_stage<DH>(Ks, qb + C, 3 * C, j0, S, dh);
    bw_stage<DH>(Vs, qb + 2 * C, 3 * C, j0, S, dh);
    __syncthreads();
    float p[4][4], dp[4][4];
    bw_scores<DH>(p, dp, Qs, Ks, dOs, Vs, ls, i0, j0, S, scale);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      float t = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) t = fmaf(p[r][c], dp[r][c], t);
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);   // the 16 tx lanes of row ty
      dacc[r] += t;
    }
  }
  if (tx == 0)
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = ty + 16 * r;
      Ds[i] = dacc[r];
      if (i0 + i < S) a.dsum[(size_t)bh * S + i0 + i] = dacc[r];
    }
  float dq[4][DH / 16];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < DH / 16; ++c) dq[r][c] = 0.f;
  for (int j0 = 0; j0 < S; j0 += BT) {
    __syncthreads();
    bw_stage<DH>(Ks, qb + C, 3 * C, j0, S, dh);
    bw_stage<DH>(Vs, qb + 2 * C, 3 * C, j0, S, dh);
    __syncthreads();
    bw_tile<DH>(Ps, dSs, Qs, Ks, dOs, Vs, ls, Ds, i0, j0, S, scale);
    __syncthreads();
    bw_acc<DH, false>(dq, dSs, Ks);                   // dQ_i += sum_j dS_ij K_j   (times scale at the store)
  }
  bw_store<DH>(a.dqkv + (size_t)b * S * 3 * C + hd * dh, dq, scale, i0, S, dh, 3 * C);
}

// One 64-key tile over all query tiles: dV_j = sum_i P_ij dO_i, dK_j = scale * sum_i dS_ij Q_i
template <int DH>
__global__ void __launch_bounds__(256) attn_long_dkdv_kernel(const BwdArgs a) {
  constexpr int LD = DH + 1;
  extern __shared__ __align__(16) float bsm[];
  float* Ks = bsm;
  float* Vs = Ks + BT * LD;
  float* Qs = Vs + BT * LD;
  float* dOs = Qs + BT * LD;
  float* Ps = dOs + BT * LD;
  float* dSs = Ps + BT * BLD;
  float* ls = dSs + BT * BLD;
  float* Ds = ls + BT;
  const int S = a.S, C = a.C, dh = C / a.heads;
  const int bh = blockIdx.y, b = bh / a.heads, hd = bh - b * a.heads;
  const int j0 = blockIdx.x * BT;
  const float scale = rsqrtf((float)dh);
  const float* qb = a.qkv + (size_t)b * S * 3 * C + hd * dh;
  const float* gb = a.dctx + (size_t)b * S * C + hd * dh;
  bw_stage<DH>(Ks, qb + C, 3 * C, j0, S, dh);
  bw_stage<DH>(Vs, qb + 2 * C, 3 * C, j0, S, dh);
  float dk[4][DH / 16], dv[4][DH / 16];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < DH / 16; ++c) dk[r][c] = dv[r][c] = 0.f;
  for (int i0 = 0; i0 < S; i0 += BT) {
    __syncthreads();                                  // previous tile's Qs / dOs / Ps / dSs fully consumed
    bw_stage<DH>(Qs, qb, 3 * C, i0, S, dh);
    bw_stage<DH>(dOs, gb, C, i0, S, dh);
    bw_rowstats(ls, Ds, a.lse + (size_t)bh * S, a.dsum + (size_t)bh * S, i0, S);
    __syncthreads();
    bw_tile<DH>(Ps, dSs, Qs, Ks, dOs, Vs, ls, Ds, i0, j0, S, scale);
    __syncthreads();
    bw_acc<DH, true>(dv, Ps, dOs);                    // dV_j += sum_i P_ij dO_i
    bw_acc<DH, true>(dk, dSs, Qs);                    // dK_j += sum_i dS_ij Q_i   (times scale at the store)
  }
  float* db = a.dqkv + (size_t)b * S * 3 * C + hd * dh;
  bw_store<DH>(db + C, dk, scale, j0, S, dh, 3 * C);
  bw_store<DH>(db + 2 * C, dv, 1.f, j0, S, dh, 3 * C);
}

template <int DH>
int al_bwd_launch(const BwdArgs& a, int B, cudaStream_t st) {
  const size_t smem = BwdSmem<DH>::bytes();
  const dim3 grid((a.S + BT - 1) / BT, B * a.heads);
  attn_long_dq_kernel<DH><<<grid, 256, smem, st>>>(a);        // also writes D for the dK / dV kernel
  CM_CUDA(cudaGetLastError());
  attn_long_dkdv_kernel<DH><<<grid, 256, smem, st>>>(a);
  CM_CUDA(cudaGetLastError());
  return 0;
}

template <int DHP>
int al_attr() {
  CM_CUDA(cudaFuncSetAttribute(attn_long_kernel<DHP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AlCfg<DHP>::SMEM));
  CM_CUDA(cudaFuncSetAttribute(attn_long_dkdv_kernel<DHP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)BwdSmem<DHP>::bytes()));
  CM_CUDA(cudaFuncSetAttribute(attn_long_dq_kernel<DHP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)BwdSmem<DHP>::bytes()));
  return 0;
}

}  // namespace

int attn_long_init() {
  static bool done = false;
  if (done) return 0;
  if (int rc = al_attr<16>()) return rc;
  if (int rc = al_attr<32>()) return rc;
  if (int rc = al_attr<64>()) return rc;
  if (int rc = al_attr<128>()) return rc;
  CM_CHECK(device_error_flag() != nullptr, "device error flag allocation failed");
  done = true;
  return 0;
}

int attn_long_enqueue(const float* qkv, __half* ctx, float* lse, int B, int S, int C, int heads, int dup,
                      cudaStream_t st) {
  const int dh = C / heads;
  if (dh <= 16) return al_launch<16>(qkv, ctx, lse, B, S, C, heads, dup, st);
  if (dh <= 32) return al_launch<32>(qkv, ctx, lse, B, S, C, heads, dup, st);
  if (dh <= 64) return al_launch<64>(qkv, ctx, lse, B, S, C, heads, dup, st);
  return al_launch<128>(qkv, ctx, lse, B, S, C, heads, dup, st);
}

int attn_long_backward_enqueue(const float* qkv, const float* dctx, const float* lse, float* dsum, float* dqkv, int B,
                               int S, int C, int heads, cudaStream_t st) {
  const BwdArgs a{qkv, dctx, lse, dsum, dqkv, S, C, heads};
  const int dh = C / heads;
  if (dh <= 16) return al_bwd_launch<16>(a, B, st);
  if (dh <= 32) return al_bwd_launch<32>(a, B, st);
  if (dh <= 64) return al_bwd_launch<64>(a, B, st);
  return al_bwd_launch<128>(a, B, st);
}

}  // namespace cm
