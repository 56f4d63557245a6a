// Bandwidth / small-op kernels of the UNet hot path.  See kernels.cuh for the contracts and
// the reference lines each one replaces.
#include "kernels.cuh"
#include "conv_umma.cuh"
#include "pack.cuh"

#include <cooperative_groups.h>


namespace cm {

// =============================================================================================
// weight packing
// =============================================================================================
__global__ void pack_conv_weights_kernel(const float* __restrict__ w, const float* __restrict__ wx,
                                         __half* __restrict__ dst, int cout, int cin, int cinx,
                                         int taps, int terms, int perm, int cin_src, int dup) {
  pack_conv_body(w, wx, dst, cout, cin, cinx, taps, terms, perm, cin_src, dup,
                 blockIdx.x * (size_t)blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
}

// every packed cache of a plan in one launch: blockIdx.y = job (pack.cuh)
__global__ void __launch_bounds__(256) pack_all_kernel(const PackJob* __restrict__ jobs) {
  const PackJob j = jobs[blockIdx.y];
  const size_t i0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x, istep = (size_t)gridDim.x * blockDim.x;
  if (j.kind == 0) pack_conv_body(j.w, j.wx, j.dst, j.cout, j.cin, j.cinx, j.taps, j.terms, j.perm, j.cin_src, j.dup, i0, istep);
  else if (j.kind == 1) pack_upsample_body(j.w, j.dst, j.cout, j.cin, j.terms, j.perm, j.dup, i0, istep);
  else pack_dgrad_body(j.mode, j.w, j.dst, j.cout, j.cin, j.terms, j.perm, j.dup, (size_t)j.ktot, i0, istep);
}
int pack_all_enqueue(const PackJob* d_jobs, int njobs, cudaStream_t st) {
  if (njobs <= 0) return 0;
  pack_all_kernel<<<dim3(48, njobs), 256, 0, st>>>(d_jobs);
  CM_CUDA(cudaGetLastError());
  return 0;
}

int pack_conv_weights(const float* w, const float* wx, __half* dst, int cout, int cin, int cinx,
                      int taps, int terms, int perm, cudaStream_t st, int dup) {
  const size_t total = (size_t)cout * ((size_t)taps * cin + cinx) * dup;
  const int blocks = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  pack_conv_weights_kernel<<<blocks, 256, 0, st>>>(w, wx, dst, cout, cin, cinx, taps, terms, perm, cin, dup);
  CM_CUDA(cudaGetLastError());
  return 0;
}

int pack_conv_weights_padded(const float* w, __half* dst, int cout, int cin_src, int cin_packed, int terms,
                             int perm, cudaStream_t st) {
  const size_t total = (size_t)cout * 27 * cin_packed;
  const int blocks = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  pack_conv_weights_kernel<<<blocks, 256, 0, st>>>(w, nullptr, dst, cout, cin_packed, 0, 27, terms, perm, cin_src, 1);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// API tensors (future [B,C,H,W,F] | past [B,C,H,W,P], time fastest) -> channels 0..C-1 of the fp16
// channels-last, time-major operand [B, P+F, H, W, 32] of the first conv (the other channels stay
// zero from the arena's initialisation).  One thread per pixel, one 8-byte store.
__global__ void pack_first_input_kernel(const float* __restrict__ x, const float* __restrict__ past,
                                        __half* __restrict__ out, int B, int H, int W, int P, int F, int cin, int dup) {
  const int L = P + F;
  const size_t total = (size_t)B * L * H * W;
  for (size_t pix = blockIdx.x * (size_t)blockDim.x + threadIdx.x; pix < total; pix += (size_t)gridDim.x * blockDim.x) {
    const int wc = (int)(pix % W);
    size_t r = pix / W;
    const int h = (int)(r % H);
    r /= H;
    const int l = (int)(r % L);
    const int b = (int)(r / L);
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    for (int ci = 0; ci < cin; ++ci) {
      const size_t pl = ((size_t)(b * cin + ci) * H + h) * W + wc;
      v[ci] = (l < P) ? past[pl * P + l] : x[pl * F + (l - P)];
    }
    __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&h0);
    u.y = *reinterpret_cast<uint32_t*>(&h1);
    *reinterpret_cast<uint2*>(out + pix * 32 * dup) = u;
    if (dup == 2) {
      const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
      __half2 l0 = __floats2half2_rn(v[0] - f0.x, v[1] - f0.y), l1 = __floats2half2_rn(v[2] - f1.x, v[3] - f1.y);
      u.x = *reinterpret_cast<uint32_t*>(&l0);
      u.y = *reinterpret_cast<uint32_t*>(&l1);
      *reinterpret_cast<uint2*>(out + pix * 64 + 32) = u;
    }
  }
}
int pack_first_input_enqueue(const float* x, const float* past, __half* out16, int B, int H, int W, int P, int F,
                             int cin, int dup, cudaStream_t st) {
  CM_CHECK(cin >= 1 && cin <= 4, "first conv supports 1..4 input channels (got %d)", cin);
  const size_t total = (size_t)B * (P + F) * H * W;
  const int blocks = (int)((total + 255) / 256 < 2368 ? (total + 255) / 256 : 2368);
  CM_CHECK(dup == 1 || dup == 2, "pack_first_input: dup must be 1 or 2");
  pack_first_input_kernel<<<blocks, 256, 0, st>>>(x, past, out16, B, H, W, P, F, cin, dup);
  CM_CUDA(cudaGetLastError());
  return 0;
}

__global__ void pack_upsample_weights_kernel(const float* __restrict__ w, __half* __restrict__ dst,
                                             int cout, int cin, int terms, int perm, int dup) {
  pack_upsample_body(w, dst, cout, cin, terms, perm, dup, blockIdx.x * (size_t)blockDim.x + threadIdx.x,
                     (size_t)gridDim.x * blockDim.x);
}

int pack_upsample_weights(const float* w, __half* dst, int cout, int cin, int terms, int perm,
                          cudaStream_t st, int dup) {
  const size_t total = (size_t)cout * 64 * cin * dup;
  const int blocks = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  pack_upsample_weights_kernel<<<blocks, 256, 0, st>>>(w, dst, cout, cin, terms, perm, dup);
  CM_CUDA(cudaGetLastError());
  return 0;
}

__global__ void cast_f32_to_f16_kernel(const float* __restrict__ s, __half* __restrict__ d, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    d[i] = __float2half_rn(s[i]);
}
int cast_f32_to_f16(const float* src, __half* dst, size_t n, cudaStream_t st) {
  const int blocks = (int)((n + 255) / 256 < 8192 ? (n + 255) / 256 : 8192);
  cast_f32_to_f16_kernel<<<blocks ? blocks : 1, 256, 0, st>>>(src, dst, n);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// 4 consecutive channels of one pixel -> the fp16 operand row: hi at dst, and (dup == 2) lo = fp16(v - hi) at
// dst + lo_off (the K-concatenated hi|lo pair the training forward multiplies, exact to 2^-22)
__device__ __forceinline__ void store_h4(__half* dst, int lo_off, float y0, float y1, float y2, float y3) {
  __half2 h0 = __floats2half2_rn(y0, y1), h1 = __floats2half2_rn(y2, y3);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&h0);
  u.y = *reinterpret_cast<uint32_t*>(&h1);
  *reinterpret_cast<uint2*>(dst) = u;
  if (lo_off) {
    const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
    __half2 l0 = __floats2half2_rn(y0 - f0.x, y1 - f0.y), l1 = __floats2half2_rn(y2 - f1.x, y3 - f1.y);
    u.x = *reinterpret_cast<uint32_t*>(&l0);
    u.y = *reinterpret_cast<uint32_t*>(&l1);
    *reinterpret_cast<uint2*>(dst + lo_off) = u;
  }
}

// =============================================================================================
// GroupNorm(8) + SiLU -> fp16, as two fully parallel, fully coalesced kernels:
//   gn_stats_kernel : CTA = (sample, pixel slice), all channels.  Exact two-pass (mean, centred
//                     M2) statistics of the slice per group from a register-cached copy.
//   gn_apply_kernel : combines the slice statistics of its sample with Chan's formula in a
//                     fixed order (bit-reproducible), then normalise + affine + SiLU (+ Dropout3d
//                     scale) -> fp16 operand (and optional raw fp16 copy for match_input).
// Thread count is a multiple of C/4, so a thread always handles the same 4 channels (same
// group, gamma, beta) and consecutive threads touch consecutive 16 bytes.
// =============================================================================================
constexpr int GN_CACHE = 8;          // float4 cached per thread

struct GnGeom {
  int Q, vpp, cg, C, T, chunks;
};

__device__ __forceinline__ void gn_slice(const GnParams& p, int chunks, int chunk, int* px0, int* px1) {
  *px0 = (int)(((long long)p.pixels * chunk) / chunks);
  *px1 = (int)(((long long)p.pixels * (chunk + 1)) / chunks);
}

// per-group sums of the per-thread partials of one CTA -> out8[g] valid in all threads after sync
__device__ __forceinline__ void gn_group_reduce(float v, float* part, float* out8, int T, int Q, int vpp) {
  const int tid = threadIdx.x;
  part[tid] = v;
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31, nwarps = T >> 5;
  for (int gi = warp; gi < 8; gi += nwarps) {
    const int RP = T / Q;
    float a = 0.f;
    for (int idx = lane; idx < RP * vpp; idx += 32) {
      const int rr = idx / vpp, o = idx - rr * vpp;
      a += part[rr * Q + gi * vpp + o];
    }
    a = warp_sum(a);
    if (lane == 0) out8[gi] = a;
  }
  __syncthreads();
}

// Single-launch variant: one thread-block cluster (GN_CLUSTER CTAs) per sample; the slice
// statistics are exchanged through distributed shared memory instead of global scratch, so a
// GroupNorm is ONE kernel (the per-launch latency floor matters: there are 27 per step).
constexpr int GN_CLUSTER = 8;

__global__ void __launch_bounds__(384) gn_fused_kernel(const GnParams p) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ float part[2][384];
  __shared__ float slice_stat[8][2];       // this CTA's (mean, M2) per group, read by peers
  __shared__ float all_stat[GN_CLUSTER][8][2];
  __shared__ float stat[2][8];
  const int CS = (int)cluster.num_blocks();
  const int chunk = (int)cluster.block_rank();
  const int b = blockIdx.x / CS;
  const int C = p.c0 + p.c1, cg_ch = C >> 3, vpp = cg_ch >> 2, Q = C >> 2;
  const int T = blockDim.x, tid = threadIdx.x;
  const int c = (tid % Q) * 4;
  const int g = c / cg_ch;
  int px0, px1;
  gn_slice(p, CS, chunk, &px0, &px1);
  const int nvec = (px1 - px0) * Q;
  const size_t pix_base = (size_t)b * p.pixels + px0;
  const bool from0 = c < p.c0;
  const float* src = from0 ? p.src0 + pix_base * p.c0 + c : p.src1 + pix_base * p.c1 + (c - p.c0);
  const int src_ld = from0 ? p.c0 : p.c1;

  // Single pass over the slice with SHIFTED sums: k = first element of this group in the slice
  // (a sample of the distribution, so (mean - k)^2 ~ var and the subtraction below is benign).
  float kshift = 0.f;
  if (nvec > 0) {
    const int cgf = g * cg_ch;
    kshift = (cgf < p.c0) ? p.src0[pix_base * p.c0 + cgf] : p.src1[pix_base * p.c1 + (cgf - p.c0)];
  }
  float4 cache[GN_CACHE];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int j = 0; j < GN_CACHE; ++j) {
    const int i = tid + j * T;
    if (i < nvec) {
      cache[j] = *reinterpret_cast<const float4*>(src + (size_t)(i / Q) * src_ld);
      const float dx = cache[j].x - kshift, dy = cache[j].y - kshift, dz = cache[j].z - kshift,
                  dw = cache[j].w - kshift;
      s1 += (dx + dy) + (dz + dw);
      s2 += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
  }
  for (int i = tid + GN_CACHE * T; i < nvec; i += T) {
    const float4 v = *reinterpret_cast<const float4*>(src + (size_t)(i / Q) * src_ld);
    const float dx = v.x - kshift, dy = v.y - kshift, dz = v.z - kshift, dw = v.w - kshift;
    s1 += (dx + dy) + (dz + dw);
    s2 += (dx * dx + dy * dy) + (dz * dz + dw * dw);
  }
  part[0][tid] = s1;
  part[1][tid] = s2;
  __syncthreads();
  {
    const int warp = tid >> 5, lane = tid & 31, nwarps = T >> 5;
    for (int gi = warp; gi < 8; gi += nwarps) {
      const int RP = T / Q;
      float a1 = 0.f, a2 = 0.f;
      for (int idx = lane; idx < RP * vpp; idx += 32) {
        const int rr = idx / vpp, o = idx - rr * vpp;
        a1 += part[0][rr * Q + gi * vpp + o];
        a2 += part[1][rr * Q + gi * vpp + o];
      }
      a1 = warp_sum(a1);
      a2 = warp_sum(a2);
      if (lane == 0) {
        const float n_slice = fmaxf((float)(px1 - px0) * (float)cg_ch, 1.f);
        const float d = a1 / n_slice;                       // slice mean - k
        // every thread of group gi used the same k: recover it from the first channel of the group
        const int cgf = gi * cg_ch;
        float k = 0.f;
        if (nvec > 0) k = (cgf < p.c0) ? p.src0[pix_base * p.c0 + cgf] : p.src1[pix_base * p.c1 + (cgf - p.c0)];
        slice_stat[gi][0] = k + d;                          // slice mean
        slice_stat[gi][1] = fmaxf(a2 - a1 * d, 0.f);        // slice M2 = S2 - n d^2
      }
    }
  }
  cluster.sync();
  for (int idx = tid; idx < CS * 16; idx += T) {   // parallel DSMEM gather of every slice's statistics
    const int k = idx >> 4, e = idx & 15;
    (&all_stat[k][0][0])[e] = cluster.map_shared_rank(&slice_stat[0][0], k)[e];
  }
  __syncthreads();
  if (tid < 8) {
    // Chan et al. combination over the cluster's slices, fixed order (bit-reproducible)
    float n_tot = 0.f, mean = 0.f, m2 = 0.f;
    for (int k = 0; k < CS; ++k) {
      int a0, a1;
      gn_slice(p, CS, k, &a0, &a1);
      const float nk = (float)(a1 - a0) * (float)cg_ch;
      if (nk == 0.f) continue;
      const float mk = all_stat[k][tid][0], m2k = all_stat[k][tid][1];
      const float nn = n_tot + nk;
      const float delta = mk - mean;
      mean += delta * (nk / nn);
      m2 += m2k + delta * delta * (n_tot * nk / nn);
      n_tot = nn;
    }
    stat[0][tid] = mean;
    stat[1][tid] = 1.0f / sqrtf(m2 / n_tot + p.eps);
    if (p.stats && chunk == 0) {
      p.stats[(b * 8 + tid) * 2 + 0] = mean;
      p.stats[(b * 8 + tid) * 2 + 1] = stat[1][tid];
    }
  }
  __syncthreads();
  const float mean = stat[0][g], rstd = stat[1][g];
  const float4 ga = *reinterpret_cast<const float4*>(p.gamma + c);
  const float4 be = *reinterpret_cast<const float4*>(p.beta + c);
  float4 ds = make_float4(1.f, 1.f, 1.f, 1.f);
  if (p.drop_scale) ds = *reinterpret_cast<const float4*>(p.drop_scale + (size_t)b * p.drop_ld + c);
  const float4 sc = make_float4(rstd * ga.x, rstd * ga.y, rstd * ga.z, rstd * ga.w);
  const float4 sh = make_float4(be.x - mean * sc.x, be.y - mean * sc.y, be.z - mean * sc.z,
                                be.w - mean * sc.w);
  const int dup = p.dup == 2 ? 2 : 1, lo_off = dup == 2 ? C : 0;
  __half* on = p.out_norm + pix_base * C * dup + c;
  __half* orw = p.out_raw ? p.out_raw + pix_base * C * dup + c : nullptr;
  auto emit = [&](int i, const float4& v) {
    float y0 = fmaf(v.x, sc.x, sh.x), y1 = fmaf(v.y, sc.y, sh.y), y2 = fmaf(v.z, sc.z, sh.z),
          y3 = fmaf(v.w, sc.w, sh.w);
    if (p.silu) { y0 = silu_f(y0); y1 = silu_f(y1); y2 = silu_f(y2); y3 = silu_f(y3); }
    y0 *= ds.x; y1 *= ds.y; y2 *= ds.z; y3 *= ds.w;
    const size_t o = (size_t)(i / Q) * C * dup;
    store_h4(on + o, lo_off, y0, y1, y2, y3);
    if (orw) store_h4(orw + o, lo_off, v.x, v.y, v.z, v.w);
  };
#pragma unroll
  for (int j = 0; j < GN_CACHE; ++j) {
    const int i = tid + j * T;
    if (i < nvec) emit(i, cache[j]);
  }
  for (int i = tid + GN_CACHE * T; i < nvec; i += T)
    emit(i, *reinterpret_cast<const float4*>(src + (size_t)(i / Q) * src_ld));
  cluster.sync();   // peers may still be reading slice_stat through DSMEM
}


// =============================================================================================
// GroupNorm as two fully parallel streaming kernels (the cluster kernel above serves calls without a
// partial-statistics buffer and tensors of more than 4 * GN2_T channels):
//   gn_stats2_kernel : CTA = (pixel slice, sample).  Every thread accumulates shifted sums of its
//                      (fixed) channel quad, converts them to (n, mean, M2) and the CTA merges
//                      the triples per group with Chan's formula in a fixed tree -> partial[b][slice][g].
//   gn_apply2_kernel : CTA = (pixel slice, sample).  Merges the sample's slice statistics in slice
//                      order, then one pass  fp32 -> normalise/affine/SiLU(/Dropout3d) -> fp16.
// The slicing depends only on the pixel index inside the sample, so a sample's result is
// bit-identical wherever it sits in the batch (and on whichever GPU its shard runs).
// =============================================================================================
constexpr int GN2_T = 256;
constexpr int GN2_MAX_SLICES = 32;
constexpr int GN3_V = 4;                  // float4 per sweeping thread per ring stage (stage = T*64 B <= 16 KB)
constexpr int GN3_NS = 3;                 // ring depth: up to 48 KB of bulk copies in flight per CTA
constexpr int GN3_SMEM = GN3_NS * GN2_T * GN3_V * 16;
constexpr int GN3_CTAS_PER_SM = 4;

// slice boundaries of a sample's pixel range (32-bit: pixels * slices < 2^31 for every supported grid)
__device__ __forceinline__ int gn2_px(int pixels, int slice, int slices) {
  return (int)(((unsigned)pixels * (unsigned)slice) / (unsigned)slices);
}
// SiLU from the pre-scaled exponent argument z = -y*log2(e): y / (1 + 2^z); two MUFU ops, no range fix-ups
// (2^z overflow -> rcp(inf) = 0 -> y*0 = -0, underflow -> y)
__device__ __forceinline__ float silu_ex2(float y, float z) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return y * r;
}

struct Chan3 {
  float n, mean, m2;
};
__device__ __forceinline__ Chan3 chan_merge(const Chan3 a, const Chan3 b) {
  if (b.n == 0.f) return a;
  if (a.n == 0.f) return b;
  const float nn = a.n + b.n;
  const float delta = b.mean - a.mean;
  const float w = __fdividef(b.n, nn);                 // one fast division per merge (these chains are serial)
  Chan3 r;
  r.n = nn;
  r.mean = a.mean + delta * w;
  r.m2 = a.m2 + b.m2 + delta * delta * (a.n * w);
  return r;
}

// Streaming skeleton shared by the statistics and the apply kernel: the CTA's pixel slice of one
// sample is a contiguous byte range of each source, so one thread feeds a ring of shared-memory
// stages with 1-D bulk copies (cp.async.bulk + mbarrier complete_tx) and the CTA consumes them.
// Memory-level parallelism is then set by the ring (64 KB per CTA, 192 KB per SM) and not by how
// many loads a thread can keep in registers (the register-batched version reached 20-40 % of HBM).
struct GnRing {
  float* ring;
  uint64_t* bar;
  const float* g0;     // first row of this CTA's slice in source 0 / 1
  const float* g1;
  int c0, c1, RS, stage_floats, rows, total;
  __device__ __forceinline__ void issue(int s) const {          // one thread
    const int slot = s % GN3_NS;
    const int row0 = s * RS;
    const int nr = (rows - row0) < RS ? (rows - row0) : RS;
    float* dst = ring + (size_t)slot * stage_floats;
    const uint32_t b0 = (uint32_t)nr * c0 * 4u, b1 = (uint32_t)nr * c1 * 4u;
    mbar_expect_tx(&bar[slot], b0 + b1);
    bulk_g2s(dst, g0 + (size_t)row0 * c0, b0, &bar[slot]);
    if (c1) bulk_g2s(dst + (size_t)RS * c0, g1 + (size_t)row0 * c1, b1, &bar[slot]);
  }
};

__global__ void __launch_bounds__(GN2_T) gn_stats2_kernel(const GnParams p, int slices, float* __restrict__ partial) {
  extern __shared__ __align__(128) unsigned char gn_dyn[];
  __shared__ uint64_t full_bar[GN3_NS];
  __shared__ float tri[GN2_T][3];
  const int C = p.c0 + p.c1, Q = C >> 2, vpp = Q >> 3;
  // blockDim.x == GN2_T; the first T = floor(GN2_T/Q)*Q threads sweep the data (fixed channel quad)
  const int tid = threadIdx.x;
  const int T = (GN2_T / Q) * Q;
  const int b = blockIdx.y, slice = blockIdx.x;
  const int px0 = gn2_px(p.pixels, slice, slices), px1 = gn2_px(p.pixels, slice + 1, slices);
  const int r = (int)((unsigned)tid / (unsigned)Q);
  const int c = (tid - r * Q) * 4;
  const int rpi = T / Q;
  GnRing rg;
  rg.ring = reinterpret_cast<float*>(gn_dyn);
  rg.bar = full_bar;
  rg.c0 = p.c0; rg.c1 = p.c1;
  rg.RS = rpi * GN3_V;
  rg.stage_floats = T * GN3_V * 4;
  rg.rows = px1 - px0;
  rg.total = (rg.rows + rg.RS - 1) / rg.RS;
  rg.g0 = p.src0 + ((size_t)b * p.pixels + px0) * p.c0;
  rg.g1 = p.c1 ? p.src1 + ((size_t)b * p.pixels + px0) * p.c1 : nullptr;
  if (tid == 0) {
    for (int i = 0; i < GN3_NS; ++i) mbar_init(&full_bar[i], 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (tid == 0)
    for (int s = 0; s < GN3_NS && s < rg.total; ++s) rg.issue(s);
  const bool from0 = c < p.c0;
  const int ld = from0 ? p.c0 : p.c1;
  const int soff = from0 ? c : rg.RS * p.c0 + (c - p.c0);
  float s1 = 0.f, s2 = 0.f, k = 0.f, cnt = 0.f;
  bool first = true;
  for (int s = 0; s < rg.total; ++s) {
    const int slot = s % GN3_NS;
    mbar_wait(&full_bar[slot], (uint32_t)((s / GN3_NS) & 1), nullptr, 0);
    const int nr = (rg.rows - s * rg.RS) < rg.RS ? (rg.rows - s * rg.RS) : rg.RS;
    if (tid < T) {
      const float* sb = rg.ring + (size_t)slot * rg.stage_floats + soff;
#pragma unroll
      for (int j = 0; j < GN3_V; ++j) {
        const int row = r + j * rpi;
        if (row < nr) {
          const float4 v = *reinterpret_cast<const float4*>(sb + row * ld);
          if (first) { k = v.x; first = false; }
          const float dx = v.x - k, dy = v.y - k, dz = v.z - k, dw = v.w - k;
          s1 += (dx + dy) + (dz + dw);
          s2 += (dx * dx + dy * dy) + (dz * dz + dw * dw);
          cnt += 4.f;
        }
      }
    }
    if (s + GN3_NS < rg.total) {
      __syncthreads();                                   // every thread is done with this slot
      if (tid == 0) rg.issue(s + GN3_NS);
    }
  }
  {
    const float d = cnt > 0.f ? s1 / cnt : 0.f;
    tri[tid][0] = cnt;
    tri[tid][1] = k + d;
    tri[tid][2] = fmaxf(s2 - s1 * d, 0.f);
  }
  __syncthreads();
  // warp gi merges the threads of group gi: t = r*Q + gi*vpp + o  (r < T/Q, o < vpp)
  const int warp = tid >> 5, lane = tid & 31;
  if (warp < 8) {
    const int members = (T / Q) * vpp;            // = T/8 <= 32
    Chan3 a{0.f, 0.f, 0.f};
    if (lane < members) {
      const int rr = lane / vpp, o = lane - rr * vpp;
      const int t = rr * Q + warp * vpp + o;
      a = Chan3{tri[t][0], tri[t][1], tri[t][2]};
    }
#pragma unroll
    for (int w = 1; w < 32; w <<= 1) {
      Chan3 o;
      o.n = __shfl_xor_sync(0xffffffffu, a.n, w);
      o.mean = __shfl_xor_sync(0xffffffffu, a.mean, w);
      o.m2 = __shfl_xor_sync(0xffffffffu, a.m2, w);
      // merge (lower lane, upper lane) in that order on both sides: identical results
      a = (lane & w) ? chan_merge(o, a) : chan_merge(a, o);
    }
    if (lane == 0) {
      float* o = partial + (((size_t)b * GN2_MAX_SLICES + slice) * 8 + warp) * 3;
      o[0] = a.n;
      o[1] = a.mean;
      o[2] = a.m2;
    }
  }
}

__global__ void __launch_bounds__(GN2_T) gn_apply2_kernel(const GnParams p, int slices, int stat_slices,
                                                          const float* __restrict__ partial) {
  extern __shared__ __align__(128) unsigned char gn_dyn[];
  __shared__ uint64_t full_bar[GN3_NS];
  __shared__ float stat[2][8];
  __shared__ float ptri[GN2_MAX_SLICES * 8 * 3];
  __shared__ float chst[512][2];                            // per-channel (mean, M2) from records
  const int C = p.c0 + p.c1, cg_ch = C >> 3, Q = C >> 2;
  const int tid = threadIdx.x;
  const int T = (GN2_T / Q) * Q;
  const int b = blockIdx.y, slice = blockIdx.x;
  const int px0 = gn2_px(p.pixels, slice, slices), px1 = gn2_px(p.pixels, slice + 1, slices);
  const int rpi = T / Q;
  GnRing rg;
  rg.ring = reinterpret_cast<float*>(gn_dyn);
  rg.bar = full_bar;
  rg.c0 = p.c0; rg.c1 = p.c1;
  rg.RS = rpi * GN3_V;
  rg.stage_floats = T * GN3_V * 4;
  rg.rows = px1 - px0;
  rg.total = (rg.rows + rg.RS - 1) / rg.RS;
  rg.g0 = p.src0 + ((size_t)b * p.pixels + px0) * p.c0;
  rg.g1 = p.c1 ? p.src1 + ((size_t)b * p.pixels + px0) * p.c1 : nullptr;
  if (tid == 0) {
    for (int i = 0; i < GN3_NS; ++i) mbar_init(&full_bar[i], 1);
    fence_mbar_init();
  }
  __syncthreads();
  // the data stream starts before the statistics prologue; the last ring slot doubles as the
  // staging buffer of the producers' records and joins the ring after the prologue
  if (tid == 0)
    for (int s = 0; s < GN3_NS - 1 && s < rg.total; ++s) rg.issue(s);
  float4 gb[2];
  {
    const int cq = (tid - (int)((unsigned)tid / (unsigned)Q) * Q) * 4;
    gb[0] = *reinterpret_cast<const float4*>(p.gamma + cq);
    gb[1] = *reinterpret_cast<const float4*>(p.beta + cq);
  }
  const bool from_rec = p.rec0.rec != nullptr;
  if (from_rec) {
    // statistics from the producing convs' records: channel c merges its units in unit order, then
    // the 8 group threads merge their channels in channel order (fixed tree -> deterministic).
    // The records of a source are staged through shared memory in one coalesced round trip per
    // chunk (a per-thread serial walk over the units exposed one L2 latency per unit).
    float4* rstage = reinterpret_cast<float4*>(rg.ring + (size_t)(GN3_NS - 1) * rg.stage_floats);
    const int rcap = rg.stage_floats / 4;                   // float4 capacity of the slot
    for (int src = 0; src < (p.c1 ? 2 : 1); ++src) {
      const GnRec& r = src ? p.rec1 : p.rec0;
      const int cs = src ? p.c1 : p.c0, cbase = src ? p.c0 : 0;
      const float4* rp = reinterpret_cast<const float4*>(r.rec) + ((size_t)b * r.units) * cs;
      const float nk = (float)r.nvalid;
      const int uchunk = rcap / cs;
      // every unit of a source covers the same number of rows, so the units of a channel combine without
      // a serial chain of divisions: with d_k = mean_k - mean_0,  mean = mean_0 + sum(d_k)/U  and
      // M2 = sum(M2_k) + n_unit * (sum(d_k^2) - sum(d_k)^2 / U)   (shifted -> no cancellation), fixed order.
      // A thread owns channels tid and tid + GN2_T of the source (C <= 512); the sums stay in registers.
      const float inv_nk = 1.0f / nk;
      float m0[2] = {0.f, 0.f}, s1[2] = {0.f, 0.f}, s2[2] = {0.f, 0.f}, q[2] = {0.f, 0.f};
      for (int u0 = 0; u0 < r.units; u0 += uchunk) {
        const int un = (r.units - u0) < uchunk ? (r.units - u0) : uchunk;
        __syncthreads();
        for (int i = tid; i < un * cs; i += GN2_T) rstage[i] = rp[(size_t)u0 * cs + i];
        __syncthreads();
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int cl = tid + e * GN2_T;
          if (cl >= cs) break;
          if (u0 == 0) {
            const float4 v = rstage[cl];
            m0[e] = v.x + v.y * inv_nk;
          }
          for (int uidx = 0; uidx < un; ++uidx) {
            const float4 v = rstage[uidx * cs + cl];
            const float d = v.y * inv_nk;                       // unit mean - unit shift
            const float dk = (v.x + d) - m0[e];
            s1[e] += dk;
            s2[e] = fmaf(dk, dk, s2[e]);
            q[e] += fmaxf(v.z - v.y * d, 0.f);
          }
        }
      }
      const float invU = 1.0f / (float)r.units;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int cl = tid + e * GN2_T;
        if (cl >= cs) break;
        chst[cbase + cl][0] = m0[e] + s1[e] * invU;
        chst[cbase + cl][1] = q[e] + nk * fmaxf(s2[e] - s1[e] * s1[e] * invU, 0.f);
      }
    }
  } else {
    for (int i = tid; i < stat_slices * 24; i += GN2_T)     // all slice statistics in one round trip
      ptri[i] = partial[(size_t)b * GN2_MAX_SLICES * 24 + i];
  }
  __syncthreads();
  if (tid == 0 && GN3_NS - 1 < rg.total) {
    fence_proxy_async();                                    // generic writes to the slot -> bulk copy
    rg.issue(GN3_NS - 1);
  }
  if (tid < 8) {
    Chan3 a{0.f, 0.f, 0.f};
    if (from_rec) {
      // the channels of a group all hold p.pixels values: same shifted equal-count combination
      const float nc = (float)p.pixels, m0 = chst[tid * cg_ch][0];
      float s1 = 0.f, s2 = 0.f, q = 0.f;
      for (int k2 = 0; k2 < cg_ch; ++k2) {
        const float dk = chst[tid * cg_ch + k2][0] - m0;
        s1 += dk;
        s2 = fmaf(dk, dk, s2);
        q += chst[tid * cg_ch + k2][1];
      }
      a.n = nc * (float)cg_ch;
      a.mean = m0 + s1 / (float)cg_ch;
      a.m2 = q + nc * fmaxf(s2 - s1 * s1 / (float)cg_ch, 0.f);
    } else
    for (int sidx = 0; sidx < stat_slices; ++sidx) {
      const float* o = ptri + (sidx * 8 + tid) * 3;
      a = chan_merge(a, Chan3{o[0], o[1], o[2]});
    }
    stat[0][tid] = a.mean;
    stat[1][tid] = 1.0f / sqrtf(a.m2 / a.n + p.eps);
    if (p.stats && slice == 0) {
      p.stats[(b * 8 + tid) * 2 + 0] = a.mean;
      p.stats[(b * 8 + tid) * 2 + 1] = stat[1][tid];
    }
  }
  __syncthreads();
  const int r = (int)((unsigned)tid / (unsigned)Q);
  const int c = (tid - r * Q) * 4;
  const int g = (int)((unsigned)c / (unsigned)cg_ch);
  const float mean = stat[0][g], rstd = stat[1][g];
  const float4 ga = gb[0], be = gb[1];                      // fetched before the prologue
  const bool drop = p.drop_scale != nullptr;
  float4 ds = make_float4(1.f, 1.f, 1.f, 1.f);
  if (drop) ds = *reinterpret_cast<const float4*>(p.drop_scale + (size_t)b * p.drop_ld + c);
  const float4 sc = make_float4(rstd * ga.x, rstd * ga.y, rstd * ga.z, rstd * ga.w);
  const float4 sh = make_float4(be.x - mean * sc.x, be.y - mean * sc.y, be.z - mean * sc.z, be.w - mean * sc.w);
  // exponent argument of the SiLU as its own affine map of the input (off the y dependency chain)
  constexpr float NL2E = -1.4426950408889634f;
  const float4 zc = make_float4(sc.x * NL2E, sc.y * NL2E, sc.z * NL2E, sc.w * NL2E);
  const float4 zh = make_float4(sh.x * NL2E, sh.y * NL2E, sh.z * NL2E, sh.w * NL2E);
  const bool from0 = c < p.c0;
  const int ld = from0 ? p.c0 : p.c1;
  const int soff = from0 ? c : rg.RS * p.c0 + (c - p.c0);
  const int dup = p.dup == 2 ? 2 : 1, lo_off = dup == 2 ? C : 0;
  const int Cd = C * dup;                                   // elements per output pixel row
  const size_t out_base = ((size_t)b * p.pixels + px0) * Cd + c;
  __half* on = p.out_norm + out_base;
  __half* orw = p.out_raw ? p.out_raw + out_base : nullptr;
  const bool silu = p.silu != 0;
  const int ostep = rpi * Cd;                               // output elements between a thread's rows
  for (int s = 0; s < rg.total; ++s) {
    const int slot = s % GN3_NS;
    mbar_wait(&full_bar[slot], (uint32_t)((s / GN3_NS) & 1), nullptr, 0);
    const int nr = (rg.rows - s * rg.RS) < rg.RS ? (rg.rows - s * rg.RS) : rg.RS;
    if (tid < T) {
      const float* sb = rg.ring + (size_t)slot * rg.stage_floats + soff + r * ld;
      const int sstep = rpi * ld;
      float4 v[GN3_V];
#pragma unroll
      for (int j = 0; j < GN3_V; ++j)
        if (r + j * rpi < nr) v[j] = *reinterpret_cast<const float4*>(sb + j * sstep);
      __half* o = on + (size_t)(s * rg.RS + r) * Cd;
      __half* orr = orw ? orw + (size_t)(s * rg.RS + r) * Cd : nullptr;
#pragma unroll
      for (int j = 0; j < GN3_V; ++j) {
        if (r + j * rpi < nr) {
          float y0 = fmaf(v[j].x, sc.x, sh.x), y1 = fmaf(v[j].y, sc.y, sh.y), y2 = fmaf(v[j].z, sc.z, sh.z),
                y3 = fmaf(v[j].w, sc.w, sh.w);
          if (silu) {
            y0 = silu_ex2(y0, fmaf(v[j].x, zc.x, zh.x));
            y1 = silu_ex2(y1, fmaf(v[j].y, zc.y, zh.y));
            y2 = silu_ex2(y2, fmaf(v[j].z, zc.z, zh.z));
            y3 = silu_ex2(y3, fmaf(v[j].w, zc.w, zh.w));
          }
          if (drop) { y0 *= ds.x; y1 *= ds.y; y2 *= ds.z; y3 *= ds.w; }
          store_h4(o + j * ostep, lo_off, y0, y1, y2, y3);
          if (orr) store_h4(orr + j * ostep, lo_off, v[j].x, v[j].y, v[j].z, v[j].w);
        }
      }
    }
    if (s + GN3_NS < rg.total) {
      __syncthreads();                                   // every thread is done with this slot
      if (tid == 0) rg.issue(s + GN3_NS);
    }
  }
}


// Small tensors (coarse levels): ONE kernel, one CTA per sample, the sample lives in registers
// between the statistics and the apply phase (<= GNS_CACHE float4 per thread).
constexpr int GNS_CACHE = 8;

__global__ void __launch_bounds__(1024) gn_small_kernel(const GnParams p) {
  __shared__ float tri[1024][3];
  __shared__ float stat[2][8];
  const int C = p.c0 + p.c1, cg_ch = C >> 3, Q = C >> 2, vpp = Q >> 3;
  const int tid = threadIdx.x;
  const int T = (blockDim.x / Q) * Q;            // sweeping threads (fixed channel quad each)
  const int b = blockIdx.x;
  const int c = (tid % Q) * 4;
  const int rows_per_iter = T / Q;
  const bool from0 = c < p.c0;
  const int src_ld = from0 ? p.c0 : p.c1;
  const size_t pix_base = (size_t)b * p.pixels;
  const float* src = (from0 ? p.src0 + c : p.src1 + (c - p.c0)) + pix_base * src_ld;
  float4 v[GNS_CACHE];
  float s1 = 0.f, s2 = 0.f, k = 0.f, cnt = 0.f;
  const int px0 = tid / Q;
  if (tid < T) {
#pragma unroll
    for (int j = 0; j < GNS_CACHE; ++j) {
      const int pj = px0 + j * rows_per_iter;
      if (pj < p.pixels) v[j] = *reinterpret_cast<const float4*>(src + (size_t)pj * src_ld);
    }
    if (px0 < p.pixels) k = v[0].x;
#pragma unroll
    for (int j = 0; j < GNS_CACHE; ++j) {
      if (px0 + j * rows_per_iter < p.pixels) {
        const float dx = v[j].x - k, dy = v[j].y - k, dz = v[j].z - k, dw = v[j].w - k;
        s1 += (dx + dy) + (dz + dw);
        s2 += (dx * dx + dy * dy) + (dz * dz + dw * dw);
        cnt += 4.f;
      }
    }
  }
  {
    const float d = cnt > 0.f ? s1 / cnt : 0.f;
    tri[tid][0] = cnt;
    tri[tid][1] = k + d;
    tri[tid][2] = fmaxf(s2 - s1 * d, 0.f);
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  if (warp < 8) {
    const int members = (T / Q) * vpp;            // = T/8 <= 128
    Chan3 a{0.f, 0.f, 0.f};
    for (int m = lane; m < members; m += 32) {    // fixed order: lane-strided, then the butterfly
      const int r = m / vpp, o = m - r * vpp;
      const int t = r * Q + warp * vpp + o;
      a = chan_merge(a, Chan3{tri[t][0], tri[t][1], tri[t][2]});
    }
#pragma unroll
    for (int w = 1; w < 32; w <<= 1) {
      Chan3 o;
      o.n = __shfl_xor_sync(0xffffffffu, a.n, w);
      o.mean = __shfl_xor_sync(0xffffffffu, a.mean, w);
      o.m2 = __shfl_xor_sync(0xffffffffu, a.m2, w);
      a = (lane & w) ? chan_merge(o, a) : chan_merge(a, o);
    }
    if (lane == 0) {
      stat[0][warp] = a.mean;
      stat[1][warp] = 1.0f / sqrtf(a.m2 / a.n + p.eps);
      if (p.stats) {
        p.stats[(b * 8 + warp) * 2 + 0] = a.mean;
        p.stats[(b * 8 + warp) * 2 + 1] = stat[1][warp];
      }
    }
  }
  __syncthreads();
  if (tid >= T) return;
  const int g = c / cg_ch;
  const float mean = stat[0][g], rstd = stat[1][g];
  const float4 ga = *reinterpret_cast<const float4*>(p.gamma + c);
  const float4 be = *reinterpret_cast<const float4*>(p.beta + c);
  float4 ds = make_float4(1.f, 1.f, 1.f, 1.f);
  if (p.drop_scale) ds = *reinterpret_cast<const float4*>(p.drop_scale + (size_t)b * p.drop_ld + c);
  const float4 sc = make_float4(rstd * ga.x, rstd * ga.y, rstd * ga.z, rstd * ga.w);
  const float4 sh = make_float4(be.x - mean * sc.x, be.y - mean * sc.y, be.z - mean * sc.z, be.w - mean * sc.w);
  constexpr float NL2E = -1.4426950408889634f;
  const float4 zc = make_float4(sc.x * NL2E, sc.y * NL2E, sc.z * NL2E, sc.w * NL2E);
  const float4 zh = make_float4(sh.x * NL2E, sh.y * NL2E, sh.z * NL2E, sh.w * NL2E);
  const bool silu = p.silu != 0, drop = p.drop_scale != nullptr;
  const int dup = p.dup == 2 ? 2 : 1, lo_off = dup == 2 ? C : 0;
  __half* on = p.out_norm + pix_base * C * dup + c;
  __half* orw = p.out_raw ? p.out_raw + pix_base * C * dup + c : nullptr;
#pragma unroll
  for (int j = 0; j < GNS_CACHE; ++j) {
    const int pj = px0 + j * rows_per_iter;
    if (pj >= p.pixels) break;
    float y0 = fmaf(v[j].x, sc.x, sh.x), y1 = fmaf(v[j].y, sc.y, sh.y), y2 = fmaf(v[j].z, sc.z, sh.z),
          y3 = fmaf(v[j].w, sc.w, sh.w);
    if (silu) {
      y0 = silu_ex2(y0, fmaf(v[j].x, zc.x, zh.x));
      y1 = silu_ex2(y1, fmaf(v[j].y, zc.y, zh.y));
      y2 = silu_ex2(y2, fmaf(v[j].z, zc.z, zh.z));
      y3 = silu_ex2(y3, fmaf(v[j].w, zc.w, zh.w));
    }
    if (drop) { y0 *= ds.x; y1 *= ds.y; y2 *= ds.z; y3 *= ds.w; }
    const size_t o = (size_t)pj * C * dup;
    store_h4(on + o, lo_off, y0, y1, y2, y3);
    if (orw) store_h4(orw + o, lo_off, v[j].x, v[j].y, v[j].z, v[j].w);
  }
}

static int gcd_i(int a, int b) { return b ? gcd_i(b, a % b) : a; }

int gn_chunks(int pixels, int C) { (void)pixels; (void)C; return GN_CLUSTER; }

int gn_silu_enqueue(const GnParams& p, float* partial, cudaStream_t st, int* launches) {
  if (launches) *launches = 1;
  const int C = p.c0 + p.c1;
  CM_CHECK(C % 32 == 0 && p.c0 % 4 == 0, "GroupNorm channels must be a multiple of 32 (C=%d)", C);
  if (partial && C / 4 <= GN2_T && C <= 512 && p.rec0.rec && (p.c1 == 0 || p.rec1.rec)) {
    // statistics come from the producing convs: one streaming apply kernel, no statistics pass
    const int Q = C / 4;
    const long nvec = (long)p.pixels * Q;
    int slices = (148 * GN3_CTAS_PER_SM) / p.B;
    const int max_slices = (int)((nvec + 4 * GN2_T - 1) / (4 * GN2_T));
    if (slices > max_slices) slices = max_slices;
    if (slices > GN2_MAX_SLICES) slices = GN2_MAX_SLICES;
    if (slices < 1) slices = 1;
    gn_apply2_kernel<<<dim3(slices, p.B), GN2_T, GN3_SMEM, st>>>(p, slices, 0, partial);
    CM_CUDA(cudaGetLastError());
    return 0;
  }
  if (partial && C / 4 <= GN2_T) {
    const int Q = C / 4;
    const long nvec = (long)p.pixels * Q;                       // float4 per sample
    if (nvec <= 1024L * GNS_CACHE) {
      // one CTA per sample: threads = a multiple of 32 covering nvec/GNS_CACHE, >= Q
      int T = (int)((nvec + GNS_CACHE - 1) / GNS_CACHE);
      if (T < Q) T = Q;
      T = (T + 31) / 32 * 32;
      if (T < 256) T = 256;
      while ((long)(T / Q) * Q * GNS_CACHE < nvec) T += 32;      // sweeping threads are floor(T/Q)*Q
      if (T <= 1024) {
        gn_small_kernel<<<p.B, T, 0, st>>>(p);
        CM_CUDA(cudaGetLastError());
        return 0;
      }
    }
    // slices: one wave of <= 4 CTAs per SM over the batch, >= 4 vectors per thread
    int slices = (148 * GN3_CTAS_PER_SM) / p.B;
    const int max_slices = (int)((nvec + 4 * GN2_T - 1) / (4 * GN2_T));
    if (slices > max_slices) slices = max_slices;
    if (slices > GN2_MAX_SLICES) slices = GN2_MAX_SLICES;
    if (slices < 1) slices = 1;
    gn_stats2_kernel<<<dim3(slices, p.B), GN2_T, GN3_SMEM, st>>>(p, slices, partial);
    CM_CUDA(cudaGetLastError());
    gn_apply2_kernel<<<dim3(slices, p.B), GN2_T, GN3_SMEM, st>>>(p, slices, slices, partial);
    CM_CUDA(cudaGetLastError());
    if (launches) *launches = 2;
    return 0;
  }
  const int Q = C / 4;
  const int L = Q / gcd_i(Q, 32) * 32;                 // lcm(Q, 32)
  CM_CHECK(L <= 384, "GroupNorm: too many channels (C=%d)", C);
  int CS = GN_CLUSTER;
  while (CS > 1 && p.pixels < 2 * CS) CS >>= 1;
  // threads: a multiple of lcm(C/4, 32); ~GN_CACHE cached vectors per thread, 512 at most
  const long nvec_cta = ((long)(p.pixels + CS - 1) / CS) * Q;
  int T = (int)(((nvec_cta + GN_CACHE - 1) / GN_CACHE + L - 1) / L * L);
  if (T < L) T = L;
  if (T < 128 && 128 % L == 0) T = 128;
  if (T > 384) T = 384 / L * L;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(p.B * CS);
  cfg.blockDim = dim3(T);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CM_CUDA(cudaLaunchKernelEx(&cfg, gn_fused_kernel, p));
  return 0;
}

// =============================================================================================
// first conv (K = 27*cin is tiny; memory-bound).  One CTA = a 4x4 block of grid sites x all L
// frames; the haloed fp32 input patch and the weights are staged in shared memory once, then
// every thread produces all couts of one output pixel (128 contiguous bytes per 32 couts).
// =============================================================================================
constexpr int FC_TS = 4;   // sites per tile edge

template <int CIN>
__global__ void __launch_bounds__(256)
first_conv_kernel(const float* __restrict__ x, const float* __restrict__ past,
                  const float* __restrict__ w, const float* __restrict__ bias,
                  float* __restrict__ out, int B, int H, int W, int P, int F, int cout) {
  extern __shared__ float sm[];
  constexpr int K = 27 * CIN;
  const int L = P + F;
  const int Lp = L + 2;
  float* ws = sm;                                   // [K][cout], k = ci*27 + tap
  float* patch = sm + K * cout;                     // [CIN][TS+2][TS+2][L+2]
  const int tiles_w = (W + FC_TS - 1) / FC_TS, tiles_h = (H + FC_TS - 1) / FC_TS;
  int bid = blockIdx.x;
  const int tw_i = bid % tiles_w;
  bid /= tiles_w;
  const int th_i = bid % tiles_h;
  const int b = bid / tiles_h;
  const int h0 = th_i * FC_TS, w0 = tw_i * FC_TS;

  for (int idx = threadIdx.x; idx < K * cout; idx += blockDim.x) {
    const int k = idx / cout, co = idx - k * cout;
    ws[idx] = w[(size_t)co * K + k];
  }
  const int patch_n = CIN * (FC_TS + 2) * (FC_TS + 2) * Lp;
  for (int idx = threadIdx.x; idx < patch_n; idx += blockDim.x) {
    int r = idx;
    const int ll = r % Lp - 1;
    r /= Lp;
    const int ww = w0 + r % (FC_TS + 2) - 1;
    r /= (FC_TS + 2);
    const int hh = h0 + r % (FC_TS + 2) - 1;
    const int ci = r / (FC_TS + 2);
    float v = 0.f;
    if (hh >= 0 && hh < H && ww >= 0 && ww < W && ll >= 0 && ll < L) {
      const size_t plane = ((size_t)(b * CIN + ci) * H + hh) * W + ww;
      v = (ll < P) ? past[plane * P + ll] : x[plane * F + (ll - P)];
    }
    patch[idx] = v;
  }
  __syncthreads();

  const int l = threadIdx.x % L;
  const int site = threadIdx.x / L;
  const int sh = site / FC_TS, sw = site % FC_TS;
  const int h = h0 + sh, wc = w0 + sw;
  if (h >= H || wc >= W) return;
  float in[K];
#pragma unroll
  for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
    for (int td = 0; td < 3; ++td)
#pragma unroll
      for (int th = 0; th < 3; ++th)
#pragma unroll
        for (int tw = 0; tw < 3; ++tw)
          in[ci * 27 + (td * 3 + th) * 3 + tw] =
              patch[((ci * (FC_TS + 2) + sh + td) * (FC_TS + 2) + sw + th) * Lp + l + tw];
  const size_t m = (((size_t)b * L + l) * H + h) * W + wc;      // internal layout [B, L, H, W, C]
  for (int co0 = 0; co0 < cout; co0 += 32) {
    float acc[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) acc[j] = bias[co0 + j];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float a = in[k];
      const float4* wr = reinterpret_cast<const float4*>(ws + k * cout + co0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 w4 = wr[j];
        acc[4 * j + 0] = fmaf(a, w4.x, acc[4 * j + 0]);
        acc[4 * j + 1] = fmaf(a, w4.y, acc[4 * j + 1]);
        acc[4 * j + 2] = fmaf(a, w4.z, acc[4 * j + 2]);
        acc[4 * j + 3] = fmaf(a, w4.w, acc[4 * j + 3]);
      }
    }
    float4* op = reinterpret_cast<float4*>(out + m * cout + co0);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      op[j] = make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
  }
}

int first_conv_enqueue(const float* x, const float* past, const float* w, const float* bias,
                       float* out, int B, int H, int W, int P, int F, int cin, int cout,
                       cudaStream_t st) {
  CM_CHECK(cin >= 1 && cin <= 4, "first conv supports 1..4 input channels (got %d)", cin);
  CM_CHECK(cout % 32 == 0, "first conv cout must be a multiple of 32");
  const int L = P + F;
  const int threads = FC_TS * FC_TS * L;
  CM_CHECK(threads <= 256, "first conv: past+future frames must be <= 16 (got %d)", L);
  const int blocks = B * ((H + FC_TS - 1) / FC_TS) * ((W + FC_TS - 1) / FC_TS);
  const size_t smem = ((size_t)27 * cin * cout + (size_t)cin * (FC_TS + 2) * (FC_TS + 2) * (L + 2)) * sizeof(float);
#define CM_FIRST(CI)                                                                           \
  case CI:                                                                                     \
    first_conv_kernel<CI><<<blocks, threads, smem, st>>>(x, past, w, bias, out, B, H, W, P, F, cout); \
    break;
  switch (cin) {
    CM_FIRST(1) CM_FIRST(2) CM_FIRST(3) CM_FIRST(4)
  }
#undef CM_FIRST
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// final conv (N = 3 is tiny; memory-bound) + reverse-step update.
// 4 lanes per output pixel, each lane owns 8-channel slices; only future frames are produced.
// =============================================================================================
constexpr int FIN_FC = 3;   // output frames per 4-lane group: taps along time share the group's 5 input planes

template <int COUT>
__global__ void __launch_bounds__(256) final_conv_kernel(const FinalParams p) {
  // weights as [h tap][w tap][ci][time tap][co]: the 8 channels x 3 time taps x COUT outputs a lane needs
  // for one spatial tap are contiguous (vector loads, broadcast across the warp's sites)
  extern __shared__ __align__(16) float ws[];
  const int cin = p.cin;
  for (int idx = threadIdx.x; idx < 27 * cin * COUT; idx += blockDim.x) {
    const int co = idx % COUT;
    int r = idx / COUT;
    const int tl = r % 3;
    r /= 3;
    const int ci = r % cin, sp = r / cin;             // sp = th*3 + tw (rows, cols)
    ws[idx] = p.w[((size_t)co * cin + ci) * 27 + sp * 3 + tl];
  }
  __syncthreads();
  const int F = p.L - p.P;
  const int nchunk = (F + FIN_FC - 1) / FIN_FC;
  const size_t sites = (size_t)p.B * p.H * p.W;
  const size_t total = sites * nchunk;                 // 4-lane groups
  // grid-stride over groups of 256 lanes (= 64 (site, frame chunk) groups): the weights are staged once
  // per CTA and the grid is sized to at most one resident wave
  for (size_t gbase = blockIdx.x * (size_t)blockDim.x; gbase < total * 4; gbase += (size_t)gridDim.x * blockDim.x) {
  const size_t gid = gbase + threadIdx.x;
  const size_t grp = gid >> 2;
  const int sub = (int)(gid & 3);
  const bool active = grp < total;
  int f0 = 0, wc = 0, h = 0, b = 0;
  if (active) {
    f0 = (int)(grp % nchunk) * FIN_FC;
    size_t r = grp / nchunk;
    wc = (int)(r % p.W);
    r /= p.W;
    h = (int)(r % p.H);
    b = (int)(r / p.H);
  }
  float acc3[FIN_FC][COUT];
#pragma unroll
  for (int j = 0; j < FIN_FC; ++j)
#pragma unroll
    for (int co = 0; co < COUT; ++co) acc3[j][co] = 0.f;
  if (active) {
    const int l0 = p.P + f0 - 1;                       // first of the FIN_FC + 2 input planes
    const int ald = p.act_ld > 0 ? p.act_ld : cin;     // pixel row stride (2*cin for hi|lo pair operands)
    const size_t pstride = (size_t)p.H * p.W * ald;    // elements per (b, l) plane
    for (int th = 0; th < 3; ++th) {
      const int hh = h + th - 1;
      if (hh < 0 || hh >= p.H) continue;
      for (int tw = 0; tw < 3; ++tw) {
        const int ww = wc + tw - 1;
        if (ww < 0 || ww >= p.W) continue;
        const __half* ap = p.act + (((size_t)b * p.L * p.H + hh) * p.W + ww) * ald;
        for (int c0 = sub * 8; c0 < cin; c0 += 32) {
          float a[FIN_FC + 2][8];
#pragma unroll
          for (int q = 0; q < FIN_FC + 2; ++q) {
            const int ll = l0 + q;
            uint4 u = make_uint4(0u, 0u, 0u, 0u), ul = u;
            // planes past the chunk's last valid frame + 1 are never multiplied into a stored output
            if (ll >= 0 && ll < p.L) {
              u = *reinterpret_cast<const uint4*>(ap + (size_t)ll * pstride + c0);
              if (p.act_lo > 0) ul = *reinterpret_cast<const uint4*>(ap + (size_t)ll * pstride + p.act_lo + c0);
            }
            const __half2* h2 = reinterpret_cast<const __half2*>(&u);
            const __half2* l2 = reinterpret_cast<const __half2*>(&ul);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 a2 = __half22float2(h2[e]);
              const float2 b2 = __half22float2(l2[e]);
              a[q][2 * e] = a2.x + b2.x;
              a[q][2 * e + 1] = a2.y + b2.y;
            }
          }
          const float4* wp4 = reinterpret_cast<const float4*>(ws + ((size_t)(th * 3 + tw) * cin + c0) * 3 * COUT);
          float wv[8 * 3 * COUT];
#pragma unroll
          for (int q = 0; q < (8 * 3 * COUT) / 4; ++q) {
            const float4 t4 = wp4[q];
            wv[4 * q] = t4.x; wv[4 * q + 1] = t4.y; wv[4 * q + 2] = t4.z; wv[4 * q + 3] = t4.w;
          }
#pragma unroll
          for (int e = 0; e < 8; ++e)
#pragma unroll
            for (int tl = 0; tl < 3; ++tl)
#pragma unroll
              for (int co = 0; co < COUT; ++co) {
                const float wgt = wv[(e * 3 + tl) * COUT + co];
#pragma unroll
                for (int j = 0; j < FIN_FC; ++j) acc3[j][co] = fmaf(a[j + tl][e], wgt, acc3[j][co]);
              }
        }
      }
    }
  }
  float acc[COUT];
#pragma unroll
  for (int co = 0; co < COUT; ++co) acc[co] = 0.f;
#pragma unroll
  for (int j = 0; j < FIN_FC; ++j)
#pragma unroll
    for (int co = 0; co < COUT; ++co) {
      float v = acc3[j][co];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      if (j == sub) acc[co] = v;                       // lane j of the group finalises frame f0 + j
    }
  const int f = f0 + sub;
  if (!active || sub >= FIN_FC || f >= F) continue;

  const size_t plane = (size_t)p.H * p.W * F;                       // elements per (b, c)
  const size_t e0 = ((size_t)b * COUT) * plane + ((size_t)h * p.W + wc) * F + f;
  float eps[COUT];
#pragma unroll
  for (int co = 0; co < COUT; ++co) eps[co] = acc[co] + p.bias[co];
  if (p.eps_out) {
#pragma unroll
    for (int co = 0; co < COUT; ++co) p.eps_out[e0 + co * plane] = eps[co];
  }
  if (!p.x) continue;

  const int step = *p.step_dev;
  const float* cf = p.coef + (size_t)step * 8;
  const size_t nelem = (size_t)p.B * COUT * plane;
  float z[4] = {0.f, 0.f, 0.f, 0.f};
  const float zc = (p.mode == 0) ? cf[2] : cf[4];
  if (zc != 0.f) {
    if (p.noise) {
#pragma unroll
      for (int co = 0; co < COUT; ++co) z[co] = p.noise[(size_t)step * nelem + e0 + co * plane];
    } else {
      const unsigned long long seed = p.chain_dev ? p.chain_dev[0] : p.seed;
      const long long soff = p.chain_dev ? static_cast<long long>(p.chain_dev[1]) : p.sample_offset;
      const unsigned long long gp =
          ((unsigned long long)(soff + b)) * (unsigned long long)(p.H * p.W * F) +
          ((size_t)h * p.W + wc) * F + f;
      const uint4 rnd = philox4x32_10(
          make_uint4((uint32_t)gp, (uint32_t)(gp >> 32), (uint32_t)step, 0u),
          make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
      const float2 n0 = box_muller(rnd.x, rnd.y), n1 = box_muller(rnd.z, rnd.w);
      z[0] = n0.x; z[1] = n0.y; z[2] = n1.x; z[3] = n1.y;
    }
  }
#pragma unroll
  for (int co = 0; co < COUT; ++co) {
    const size_t e = e0 + co * plane;
    const float xv = p.x[e];
    float xn;
    if (p.mode == 0) {
      // ddpm.py:33-37: one_by_sqrt_alpha * (x - (beta/sqrt(1-abar)) * eps) + sqrt(beta) * z
      xn = cf[0] * (xv - cf[1] * eps[co]) + cf[2] * z[co];
    } else {
      // ddpm.py:262-265 (DDIM eq. 12)
      const float x0 = (xv - cf[0] * eps[co]) / cf[1];
      xn = cf[2] * x0 + cf[3] * eps[co] + cf[4] * z[co];
    }
    if (co == 0 && cf[5] != 0.f) {
      // guidance.py:4-8 + ddpm.py:223-226: x[:,0] -= lambda*sigma*sign(x[:,0])
      const float sg = (xn > 0.f) ? 1.f : ((xn < 0.f) ? -1.f : 0.f);
      xn -= cf[5] * sg;
    }
    p.x[e] = xn;
    if (p.history) p.history[(size_t)(step + 1) * nelem + e] = xn;
  }
  }
}

int final_conv_enqueue(const FinalParams& p, cudaStream_t st) {
  CM_CHECK(p.cout >= 1 && p.cout <= 4, "final conv supports 1..4 output channels (got %d)", p.cout);
  CM_CHECK(p.cin % 32 == 0, "final conv cin must be a multiple of 32");
  const size_t total = (size_t)p.B * p.H * p.W * ((p.L - p.P + FIN_FC - 1) / FIN_FC) * 4;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 4) blocks = 148 * 4;          // at most one resident wave; the kernel grid-strides
  const size_t smem = (size_t)27 * p.cin * p.cout * sizeof(float);
#define CM_FINAL(CO)                                                                           \
  case CO:                                                                                     \
    final_conv_kernel<CO><<<blocks, 256, smem, st>>>(p);                                       \
    break;
  switch (p.cout) {
    CM_FINAL(1) CM_FINAL(2) CM_FINAL(3) CM_FINAL(4)
  }
#undef CM_FINAL
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// time embedding: table row -> Linear -> SiLU -> Linear -> (SiLU -> dense_1 of every block)
// =============================================================================================
// One CTA per row.  Every output is a dot product over a CONTIGUOUS weight row: a warp takes four outputs at a time, its
// lanes stride the row (coalesced 128-byte reads; the first version gave every thread its own row, 512 bytes apart, and
// took 97 us for the 13 MFLOP of a 64-row training batch), the partial sums are reduced by a fixed xor butterfly.
__device__ __forceinline__ void temb_warp_dot4(const float* __restrict__ w, int ldw, const float* __restrict__ x, int n,
                                               int j0, int jn, int lane, float (&acc)[4]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) acc[q] = 0.f;
  for (int i = lane; i < n; i += 32) {
    const float xv = x[i];
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (j0 + q < jn) acc[q] = fmaf(w[(size_t)(j0 + q) * ldw + i], xv, acc[q]);
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
  }
}

__device__ __forceinline__ float temb_pick4(const float (&acc)[4], int lane) {
  return lane == 0 ? acc[0] : (lane == 1 ? acc[1] : (lane == 2 ? acc[2] : acc[3]));
}

__global__ void __launch_bounds__(256) temb_kernel(const TembParams p) {
  extern __shared__ float sm[];   // e[base] | s1[E] | s2[E]
  float* e = sm;
  float* s1 = sm + p.base;
  float* s2 = s1 + p.E;
  const int row = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const long long t = p.t ? p.t[row] : (long long)row;
  for (int i = threadIdx.x; i < p.base; i += blockDim.x) {
    e[i] = p.table[(size_t)t * p.base + i];
    if (p.save_e) p.save_e[(size_t)row * p.base + i] = e[i];
  }
  __syncthreads();
  float acc[4];
  for (int j0 = warp * 4; j0 < p.E; j0 += nw * 4) {
    temb_warp_dot4(p.w1, p.base, e, p.base, j0, p.E, lane, acc);
    if (lane < 4 && j0 + lane < p.E) {
      const float a = p.b1[j0 + lane] + temb_pick4(acc, lane);
      s1[j0 + lane] = silu_f(a);
      if (p.save_h1) p.save_h1[(size_t)row * p.E + j0 + lane] = a;
    }
  }
  __syncthreads();
  for (int j0 = warp * 4; j0 < p.E; j0 += nw * 4) {
    temb_warp_dot4(p.w2, p.E, s1, p.E, j0, p.E, lane, acc);
    if (lane < 4 && j0 + lane < p.E) {
      const float a = p.b2[j0 + lane] + temb_pick4(acc, lane);
      s2[j0 + lane] = silu_f(a);   // every consumer applies SiLU first (layers.py:62)
      if (p.save_h2) p.save_h2[(size_t)row * p.E + j0 + lane] = a;
    }
  }
  __syncthreads();
  for (int k = 0; k < p.nblocks; ++k) {
    const float* wd = p.wd[k];
    const float* bd = p.bd[k];
    const int co_n = p.couts[k];
    float* o = p.out + (size_t)row * p.ld + p.offs[k];
    for (int c0 = warp * 4; c0 < co_n; c0 += nw * 4) {
      temb_warp_dot4(wd, p.E, s2, p.E, c0, co_n, lane, acc);
      if (lane < 4 && c0 + lane < co_n) o[c0 + lane] = bd[c0 + lane] + temb_pick4(acc, lane);
    }
  }
}

int temb_enqueue(const TembParams& p, cudaStream_t st) {
  const size_t smem = (size_t)(p.base + 2 * p.E) * sizeof(float);
  temb_kernel<<<p.rows, 256, smem, st>>>(p);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// attention core: softmax(Q K^T / sqrt(dh)) V per (sample, head) on mma.sync m16n8k16 (S is a few
// dozen tokens: far too small for a tcgen05 tile, and the scalar version was shared-memory-bound).
// One warp owns 16 query rows end to end (flash-attention register dataflow, no online rescaling
// needed since all S keys fit one pass).  Q and K enter as fp16 hi+lo pairs (3 MMAs per product:
// hi*hi + hi*lo + lo*hi), so the scores are fp32-accurate; P and V are single fp16 operands like
// every other contraction operand of the path.
// =============================================================================================
__device__ __forceinline__ void mma_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_h2(float x, float y) {
  __half2 h = __floats2half2_rn(x, y);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void split_h2(float x, float y, uint32_t* hi, uint32_t* lo) {
  const __half hx = __float2half_rn(x), hy = __float2half_rn(y);
  __half2 h = __halves2half2(hx, hy);
  __half2 l = __floats2half2_rn(x - __half2float(hx), y - __half2float(hy));
  *hi = *reinterpret_cast<uint32_t*>(&h);
  *lo = *reinterpret_cast<uint32_t*>(&l);
}

// DH = head dim padded to a multiple of 16 (16 | 32 | 64; dh = C/heads may be 8 -> zero padded),
// NT = key tiles of 8 (S_pad = 8*NT, multiple of 16)
template <int DH, int NT>
__global__ void __launch_bounds__(NT * 16) attn_mma_kernel(const float* __restrict__ qkv, __half* __restrict__ ctx,
                                                          int S, int C, int heads, int dup) {
  const int dh = C / heads;
  constexpr int SP = NT * 8;            // padded sequence length
  constexpr int KLD = DH + 8;           // smem row stride (halfs) of K  [SP][KLD]
  constexpr int VLD = SP + 8;           // smem row stride (halfs) of V^T [DH][VLD]
  extern __shared__ __align__(16) uint8_t smraw[];
  __half* Kh = reinterpret_cast<__half*>(smraw);
  __half* Kl = Kh + SP * KLD;
  __half* Vt = Kl + SP * KLD;
  const int b = blockIdx.x / heads, hd = blockIdx.x % heads;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const float* base = qkv + (size_t)b * S * 3 * C + hd * dh;
  // ---- Q fragments straight from global (issued before the K/V staging barrier) ----
  const int i0 = warp * 16 + g, i1 = i0 + 8;
  const float scale = rsqrtf((float)dh);
  uint32_t qh[DH / 16][4], ql[DH / 16][4];
#pragma unroll
  for (int kt = 0; kt < DH / 16; ++kt) {
    float2 v00 = make_float2(0.f, 0.f), v10 = v00, v01 = v00, v11 = v00;
    const bool lo_ok = kt * 16 + 2 * t < dh, hi_ok = kt * 16 + 8 + 2 * t < dh;
    if (i0 < S) {
      if (lo_ok) v00 = *reinterpret_cast<const float2*>(base + (size_t)i0 * 3 * C + kt * 16 + 2 * t);
      if (hi_ok) v01 = *reinterpret_cast<const float2*>(base + (size_t)i0 * 3 * C + kt * 16 + 8 + 2 * t);
    }
    if (i1 < S) {
      if (lo_ok) v10 = *reinterpret_cast<const float2*>(base + (size_t)i1 * 3 * C + kt * 16 + 2 * t);
      if (hi_ok) v11 = *reinterpret_cast<const float2*>(base + (size_t)i1 * 3 * C + kt * 16 + 8 + 2 * t);
    }
    split_h2(v00.x * scale, v00.y * scale, &qh[kt][0], &ql[kt][0]);
    split_h2(v10.x * scale, v10.y * scale, &qh[kt][1], &ql[kt][1]);
    split_h2(v01.x * scale, v01.y * scale, &qh[kt][2], &ql[kt][2]);
    split_h2(v11.x * scale, v11.y * scale, &qh[kt][3], &ql[kt][3]);
  }
  // ---- stage K (hi, lo) and V^T as fp16 ----
  for (int idx = tid; idx < SP * (DH / 2); idx += blockDim.x) {
    const int j = idx / (DH / 2), d = (idx - j * (DH / 2)) * 2;
    float2 kv = make_float2(0.f, 0.f), vv = kv;
    if (j < S && d < dh) {
      kv = *reinterpret_cast<const float2*>(base + (size_t)j * 3 * C + C + d);
      vv = *reinterpret_cast<const float2*>(base + (size_t)j * 3 * C + 2 * C + d);
    }
    uint32_t hi, lo;
    split_h2(kv.x, kv.y, &hi, &lo);
    *reinterpret_cast<uint32_t*>(Kh + j * KLD + d) = hi;
    *reinterpret_cast<uint32_t*>(Kl + j * KLD + d) = lo;
    Vt[d * VLD + j] = __float2half_rn(vv.x);
    Vt[(d + 1) * VLD + j] = __float2half_rn(vv.y);
  }
  __syncthreads();
  if (warp * 16 >= S) return;
  // ---- scores: 16 x SP per warp ----
  float sc[NT][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
    const int j = nt * 8 + g;
#pragma unroll
    for (int kt = 0; kt < DH / 16; ++kt) {
      const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(Kh + j * KLD + kt * 16 + 2 * t);
      const uint32_t bh1 = *reinterpret_cast<const uint32_t*>(Kh + j * KLD + kt * 16 + 8 + 2 * t);
      const uint32_t bl0 = *reinterpret_cast<const uint32_t*>(Kl + j * KLD + kt * 16 + 2 * t);
      const uint32_t bl1 = *reinterpret_cast<const uint32_t*>(Kl + j * KLD + kt * 16 + 8 + 2 * t);
      mma_16816(sc[nt], ql[kt], bh0, bh1);
      mma_16816(sc[nt], qh[kt], bl0, bl1);
      mma_16816(sc[nt], qh[kt], bh0, bh1);
    }
  }
  // ---- softmax over keys (rows g and g+8 live in the 4 lanes of a quad) ----
  float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const int j = nt * 8 + 2 * t;
    if (j >= S) sc[nt][0] = sc[nt][2] = -INFINITY;
    if (j + 1 >= S) sc[nt][1] = sc[nt][3] = -INFINITY;
    m0 = fmaxf(m0, fmaxf(sc[nt][0], sc[nt][1]));
    m1 = fmaxf(m1, fmaxf(sc[nt][2], sc[nt][3]));
  }
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    sc[nt][0] = expf(sc[nt][0] - m0);
    sc[nt][1] = expf(sc[nt][1] - m0);
    sc[nt][2] = expf(sc[nt][2] - m1);
    sc[nt][3] = expf(sc[nt][3] - m1);
    l0 += sc[nt][0] + sc[nt][1];
    l1 += sc[nt][2] + sc[nt][3];
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
  // ---- context = P V  (P normalised before the fp16 rounding) ----
  float oc[DH / 8][4];
#pragma unroll
  for (int dt = 0; dt < DH / 8; ++dt) oc[dt][0] = oc[dt][1] = oc[dt][2] = oc[dt][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < NT / 2; ++kt) {
    uint32_t pa[4];
    pa[0] = pack_h2(sc[2 * kt][0] * inv0, sc[2 * kt][1] * inv0);
    pa[1] = pack_h2(sc[2 * kt][2] * inv1, sc[2 * kt][3] * inv1);
    pa[2] = pack_h2(sc[2 * kt + 1][0] * inv0, sc[2 * kt + 1][1] * inv0);
    pa[3] = pack_h2(sc[2 * kt + 1][2] * inv1, sc[2 * kt + 1][3] * inv1);
#pragma unroll
    for (int dt = 0; dt < DH / 8; ++dt) {
      const int d = dt * 8 + g;
      const uint32_t b0 = *reinterpret_cast<const uint32_t*>(Vt + d * VLD + kt * 16 + 2 * t);
      const uint32_t b1 = *reinterpret_cast<const uint32_t*>(Vt + d * VLD + kt * 16 + 8 + 2 * t);
      mma_16816(oc[dt], pa, b0, b1);
    }
  }
  const int Cd = C * dup;                              // dup = 2: hi | lo pair per token (training forward)
  __half* ob = ctx + (size_t)b * S * Cd + hd * dh;
#pragma unroll
  for (int dt = 0; dt < DH / 8; ++dt) {
    const int d = dt * 8 + 2 * t;
    if (d >= dh) continue;
    if (dup == 2) {
      uint32_t hi, lo;
      if (i0 < S) {
        split_h2(oc[dt][0], oc[dt][1], &hi, &lo);
        *reinterpret_cast<uint32_t*>(ob + (size_t)i0 * Cd + d) = hi;
        *reinterpret_cast<uint32_t*>(ob + (size_t)i0 * Cd + C + d) = lo;
      }
      if (i1 < S) {
        split_h2(oc[dt][2], oc[dt][3], &hi, &lo);
        *reinterpret_cast<uint32_t*>(ob + (size_t)i1 * Cd + d) = hi;
        *reinterpret_cast<uint32_t*>(ob + (size_t)i1 * Cd + C + d) = lo;
      }
      continue;
    }
    if (i0 < S) *reinterpret_cast<uint32_t*>(ob + (size_t)i0 * C + d) = pack_h2(oc[dt][0], oc[dt][1]);
    if (i1 < S) *reinterpret_cast<uint32_t*>(ob + (size_t)i1 * C + d) = pack_h2(oc[dt][2], oc[dt][3]);
  }
}

template <int DH, int NT>
static int attn_launch(const float* qkv, __half* ctx, int B, int S, int C, int heads, int dup, cudaStream_t st) {
  constexpr int SP = NT * 8;
  const size_t smem = ((size_t)2 * SP * (DH + 8) + (size_t)DH * (SP + 8)) * sizeof(__half);
  attn_mma_kernel<DH, NT><<<B * heads, NT * 16, smem, st>>>(qkv, ctx, S, C, heads, dup);
  CM_CUDA(cudaGetLastError());
  return 0;
}

template <int DH>
static int attn_dispatch(const float* qkv, __half* ctx, int B, int S, int C, int heads, int dup, cudaStream_t st) {
  const int sp16 = (S + 15) / 16;       // query tiles = warps
  switch (sp16) {
    case 1: return attn_launch<DH, 2>(qkv, ctx, B, S, C, heads, dup, st);
    case 2: return attn_launch<DH, 4>(qkv, ctx, B, S, C, heads, dup, st);
    case 3: return attn_launch<DH, 6>(qkv, ctx, B, S, C, heads, dup, st);
    case 4: return attn_launch<DH, 8>(qkv, ctx, B, S, C, heads, dup, st);
    case 5: return attn_launch<DH, 10>(qkv, ctx, B, S, C, heads, dup, st);
    case 6: return attn_launch<DH, 12>(qkv, ctx, B, S, C, heads, dup, st);
    case 7: return attn_launch<DH, 14>(qkv, ctx, B, S, C, heads, dup, st);
    case 8: return attn_launch<DH, 16>(qkv, ctx, B, S, C, heads, dup, st);
    default:
      CM_CHECK(false, "attention: sequence length %d > 128 tokens is not supported", S);
  }
  return 0;
}

int attn_core_enqueue(const float* qkv, __half* ctx, int B, int S, int C, int heads,
                      cudaStream_t st, int dup, float* lse) {
  CM_CHECK(dup == 1 || dup == 2, "attention: dup must be 1 or 2");
  CM_CHECK(C % heads == 0, "embed dim %d / heads %d unsupported", C, heads);
  const int dh = C / heads;
  CM_CHECK(dh % 2 == 0 && dh <= 128, "attention: head dim %d unsupported (even, <= 128)", dh);
  if (attn_uses_long(S, dh)) return attn_long_enqueue(qkv, ctx, lse, B, S, C, heads, dup, st);
  if (dh <= 16) return attn_dispatch<16>(qkv, ctx, B, S, C, heads, dup, st);
  if (dh <= 32) return attn_dispatch<32>(qkv, ctx, B, S, C, heads, dup, st);
  return attn_dispatch<64>(qkv, ctx, B, S, C, heads, dup, st);
}

// =============================================================================================
// Fused AttentionBlock for the sampling path (layers.py:5-18): GroupNorm(8) -> in_proj -> softmax(QK^T/sqrt(dh))V
// -> out_proj -> + x, ONE launch, one CTA per sample (the block is 0.55 GFLOP for 64 samples: four
// dependent launches were pure latency).  C = 128, 4 heads, dh = 32, S <= 128 tokens.
//   phase 0  x [S][C] fp32 -> exact two-pass group statistics -> h = GN(x) as fp16 in shared memory
//   phase 1  qkv = h W_in^T + b_in   (mma.sync m16n8k16, A from smem, hi+lo fp16 weights straight from L2)
//            -> Q/sqrt(dh) and K as hi+lo fp16 pairs, V^T as fp16, all in shared memory
//   phase 2  per (head, 16-query tile) warp: fp32-accurate scores (3 MMAs), softmax, P V -> ctx fp16 (smem)
//   phase 3  out = ctx W_o^T + b_o + x -> fp32 (and fp16) global
// Same operand precisions as the unfused path (fp16 activations, hi+lo weights, hi+lo Q/K).
// =============================================================================================
constexpr int AB_C = 128, AB_HEADS = 4, AB_DH = 32, AB_THREADS = 512, AB_WARPS = 16;
constexpr int AB_LD = AB_C + 8;           // smem row stride (halfs) of h
constexpr int AB_CL = AB_C / 2;           // channels (two heads) owned by one CTA of the pair
constexpr int AB_LDL = AB_CL + 8;         // smem row stride (halfs) of Q / K / ctx (local channels)
constexpr int AB_PLD = AB_C + 4;          // smem row stride (floats) of the out_proj partial sums

struct AttnBlockParams {
  const float* x;          // [B][S][C] fp32 (block input = residual)
  const float* gamma;
  const float* beta;
  const __half* w_in;      // packed [2*3C][C]: rows 0..3C-1 hi, 3C..6C-1 lo
  const float* b_in;       // [3C]
  const __half* w_out;     // packed [2*C][C]
  const float* b_out;      // [C]
  float* out32;            // optional [B][S][C]
  __half* out16;           // optional
  int S;
  float eps;
};

// acc[MT][NTW] (+)= A[smem rows m_base + mt*16.., K = 16*KT] . W[nb[nt] + g][kcol0 + k]^T, hi and lo weight rows
template <int MT, int NTW, int KT, int ALD>
__device__ __forceinline__ void ab_gemm(const __half* __restrict__ A, int m_base, const __half* __restrict__ Whi,
                                        const __half* __restrict__ Wlo, const int (&nb)[NTW], int kcol0,
                                        float (&acc)[MT][NTW][4], int g, int t) {
  // The k index inside a 16-wide block is permuted identically for A and B (fragment slots (2t, 2t+1) and (2t+8, 2t+9) of
  // thread t take the four CONSECUTIVE physical k's 4t .. 4t+3): the product is a sum over all 16 k's either way, and every
  // fragment pair becomes one 8-byte load instead of two 4-byte ones (the kernel's top stalls were lg_throttle and
  // long_scoreboard on these weight loads, profiles/r1_attn_block_ncu_full_raw.csv).
  uint32_t bh[2][NTW][2], bl[2][NTW][2];
  auto load_b = [&](int kt, int buf) {
#pragma unroll
    for (int nt = 0; nt < NTW; ++nt) {
      const size_t o = (size_t)(nb[nt] + g) * AB_C + kcol0 + kt * 16 + 4 * t;
      const uint2 h2 = __ldg(reinterpret_cast<const uint2*>(Whi + o));
      const uint2 l2 = __ldg(reinterpret_cast<const uint2*>(Wlo + o));
      bh[buf][nt][0] = h2.x;
      bh[buf][nt][1] = h2.y;
      bl[buf][nt][0] = l2.x;
      bl[buf][nt][1] = l2.y;
    }
  };
  load_b(0, 0);
#pragma unroll
  for (int kt = 0; kt < KT; ++kt) {
    const int buf = kt & 1;
    if (kt + 1 < KT) load_b(kt + 1, buf ^ 1);
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
      const __half* ar = A + (size_t)(m_base + mt * 16 + g) * ALD + kt * 16 + 4 * t;
      const uint2 a_lo = *reinterpret_cast<const uint2*>(ar);             // row g:     physical k 4t .. 4t+3
      const uint2 a_hi = *reinterpret_cast<const uint2*>(ar + 8 * ALD);   // row g + 8
      uint32_t a[4];
      a[0] = a_lo.x;
      a[1] = a_hi.x;
      a[2] = a_lo.y;
      a[3] = a_hi.y;
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt) {
        mma_16816(acc[mt][nt], a, bl[buf][nt][0], bl[buf][nt][1]);
        mma_16816(acc[mt][nt], a, bh[buf][nt][0], bh[buf][nt][1]);
      }
    }
  }
}

// A pair of CTAs (thread-block cluster of 2) per sample: CTA r owns heads 2r, 2r+1 (channels [64r, 64r+64))
// through in_proj and the attention core; out_proj is a K-split whose two partial tiles are summed in rank
// order through distributed shared memory (deterministic), CTA r finalising output columns [64r, 64r+64).
template <int NT>   // NT = padded tokens / 8 (even): SP = 16, 32, ... 128
__global__ void __launch_bounds__(AB_THREADS, 1) attn_block_kernel(const AttnBlockParams p) {
  namespace cgr = cooperative_groups;
  cgr::cluster_group cluster = cgr::this_cluster();
  constexpr int SP = NT * 8, MTILES = SP / 16;
  constexpr int VLD = SP + 8;
  constexpr int MH = (MTILES + 1) / 2;                   // M tiles per half (phase 1 splits M over warp halves)
  extern __shared__ __align__(16) uint8_t ab_raw[];
  __half* Hs = reinterpret_cast<__half*>(ab_raw);       // [SP][AB_LD]   h
  __half* Qh = Hs + SP * AB_LD;                          // [SP][AB_LDL]  local channels
  __half* Ql = Qh + SP * AB_LDL;
  __half* Kh = Ql + SP * AB_LDL;
  __half* Kl = Kh + SP * AB_LDL;
  __half* Vt = Kl + SP * AB_LDL;                         // [AB_CL][VLD]
  __half* Cx = Vt + AB_CL * VLD;                         // [SP][AB_LDL]  ctx (local channels)
  float* Pp = reinterpret_cast<float*>(ab_raw);          // [SP][AB_PLD]  out_proj partial (aliases h/Q/K: dead by then)
  __shared__ float red[AB_WARPS][8];
  __shared__ float gstat[2][8];
  const int S = p.S;
  const int rank = (int)cluster.block_rank();
  const int b = blockIdx.x >> 1;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const float* xb = p.x + (size_t)b * S * AB_C;
  const int cl0 = rank * AB_CL;                          // first channel owned by this CTA

  // ---- phase 0: GroupNorm.  warp = row (mod 16), lane = float4 column; group = lane / 4 (16 channels) ----
  constexpr int RPT = (SP + AB_WARPS - 1) / AB_WARPS;    // rows per warp
  float4 xv[RPT];
  float s1 = 0.f;
#pragma unroll
  for (int j = 0; j < RPT; ++j) {
    const int row = warp + j * AB_WARPS;
    xv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < S) xv[j] = *reinterpret_cast<const float4*>(xb + (size_t)row * AB_C + lane * 4);
    s1 += (xv[j].x + xv[j].y) + (xv[j].z + xv[j].w);
  }
  s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
  s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
  if ((lane & 3) == 0) red[warp][lane >> 2] = s1;
  __syncthreads();
  const float cnt = (float)S * 16.f;
  if (tid < 8) {
    float a = 0.f;
    for (int w = 0; w < AB_WARPS; ++w) a += red[w][tid];
    gstat[0][tid] = a / cnt;
  }
  __syncthreads();
  const float mean = gstat[0][lane >> 2];
  float s2 = 0.f;
#pragma unroll
  for (int j = 0; j < RPT; ++j) {
    if (warp + j * AB_WARPS < S) {
      const float dx = xv[j].x - mean, dy = xv[j].y - mean, dz = xv[j].z - mean, dw = xv[j].w - mean;
      s2 += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
  }
  s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
  s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
  if ((lane & 3) == 0) red[warp][lane >> 2] = s2;     // (red was fully consumed before the second barrier)
  __syncthreads();
  if (tid < 8) {
    float a = 0.f;
    for (int w = 0; w < AB_WARPS; ++w) a += red[w][tid];
    gstat[1][tid] = 1.0f / sqrtf(a / cnt + p.eps);
  }
  __syncthreads();
  {
    const float rstd = gstat[1][lane >> 2];
    const float4 ga = *reinterpret_cast<const float4*>(p.gamma + lane * 4);
    const float4 be = *reinterpret_cast<const float4*>(p.beta + lane * 4);
#pragma unroll
    for (int j = 0; j < RPT; ++j) {
      const int row = warp + j * AB_WARPS;
      if (row >= SP) continue;
      uint2 u = make_uint2(0u, 0u);                     // padded rows are zero (finite q/k/v = bias)
      if (row < S) {
        u.x = pack_h2((xv[j].x - mean) * rstd * ga.x + be.x, (xv[j].y - mean) * rstd * ga.y + be.y);
        u.y = pack_h2((xv[j].z - mean) * rstd * ga.z + be.z, (xv[j].w - mean) * rstd * ga.w + be.w);
      }
      *reinterpret_cast<uint2*>(Hs + (size_t)row * AB_LD + lane * 4) = u;
    }
  }
  __syncthreads();

  // ---- phase 1: q|k|v (local channels) = h W_in^T + b_in: 24 n8 tiles (8 q, 8 k, 8 v).
  //      warp = (M half, group of 3 tiles) ----
  {
    const float qscale = rsqrtf((float)AB_DH);
    const int mh = warp >> 3, ng = warp & 7;
    int nb[3], wh[3], cc[3];
#pragma unroll
    for (int nt = 0; nt < 3; ++nt) {
      const int j = ng * 3 + nt;
      wh[nt] = j >> 3;                                   // 0 q, 1 k, 2 v
      cc[nt] = (j & 7) * 8;                              // local channel of the tile
      nb[nt] = wh[nt] * AB_C + cl0 + cc[nt];             // row of W_in
    }
    if (mh * MH < MTILES) {
      float acc[MH][3][4];
#pragma unroll
      for (int mt = 0; mt < MH; ++mt)
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = acc[mt][nt][2] = acc[mt][nt][3] = 0.f;
      ab_gemm<MH, 3, AB_C / 16, AB_LD>(Hs, mh * MH * 16, p.w_in, p.w_in + (size_t)3 * AB_C * AB_C, nb, 0, acc, g, t);
#pragma unroll
      for (int nt = 0; nt < 3; ++nt) {
        const float2 bi = *reinterpret_cast<const float2*>(p.b_in + nb[nt] + 2 * t);
        const int c = cc[nt] + 2 * t;
#pragma unroll
        for (int mt = 0; mt < MH; ++mt) {
          if (mh * MH + mt >= MTILES) continue;
          const int r0 = (mh * MH + mt) * 16 + g, r1 = r0 + 8;
          const float v00 = acc[mt][nt][0] + bi.x, v01 = acc[mt][nt][1] + bi.y;
          const float v10 = acc[mt][nt][2] + bi.x, v11 = acc[mt][nt][3] + bi.y;
          if (wh[nt] == 2) {
            Vt[(size_t)c * VLD + r0] = __float2half_rn(v00);
            Vt[(size_t)(c + 1) * VLD + r0] = __float2half_rn(v01);
            Vt[(size_t)c * VLD + r1] = __float2half_rn(v10);
            Vt[(size_t)(c + 1) * VLD + r1] = __float2half_rn(v11);
          } else {
            const float sc = wh[nt] == 0 ? qscale : 1.0f;
            __half* hi = wh[nt] == 0 ? Qh : Kh;
            __half* lo = wh[nt] == 0 ? Ql : Kl;
            uint32_t h, l;
            split_h2(v00 * sc, v01 * sc, &h, &l);
            *reinterpret_cast<uint32_t*>(hi + (size_t)r0 * AB_LDL + c) = h;
            *reinterpret_cast<uint32_t*>(lo + (size_t)r0 * AB_LDL + c) = l;
            split_h2(v10 * sc, v11 * sc, &h, &l);
            *reinterpret_cast<uint32_t*>(hi + (size_t)r1 * AB_LDL + c) = h;
            *reinterpret_cast<uint32_t*>(lo + (size_t)r1 * AB_LDL + c) = l;
          }
        }
      }
    }
  }
  __syncthreads();     // q/k/v complete

  // ---- phase 2: attention core, one (local head, query tile) per warp pass ----
  for (int pr = warp; pr < 2 * MTILES; pr += AB_WARPS) {
    const int hd = pr & 1, mt = pr >> 1;
    const int i0 = mt * 16 + g, i1 = i0 + 8;
    const int cb = hd * AB_DH;
    uint32_t qh[AB_DH / 16][4], ql[AB_DH / 16][4];
#pragma unroll
    for (int kt = 0; kt < AB_DH / 16; ++kt) {
      const int o0 = i0 * AB_LDL + cb + kt * 16 + 2 * t, o1 = i1 * AB_LDL + cb + kt * 16 + 2 * t;
      qh[kt][0] = *reinterpret_cast<const uint32_t*>(Qh + o0);
      qh[kt][1] = *reinterpret_cast<const uint32_t*>(Qh + o1);
      qh[kt][2] = *reinterpret_cast<const uint32_t*>(Qh + o0 + 8);
      qh[kt][3] = *reinterpret_cast<const uint32_t*>(Qh + o1 + 8);
      ql[kt][0] = *reinterpret_cast<const uint32_t*>(Ql + o0);
      ql[kt][1] = *reinterpret_cast<const uint32_t*>(Ql + o1);
      ql[kt][2] = *reinterpret_cast<const uint32_t*>(Ql + o0 + 8);
      ql[kt][3] = *reinterpret_cast<const uint32_t*>(Ql + o1 + 8);
    }
    float sc[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
      const int j = nt * 8 + g;
#pragma unroll
      for (int kt = 0; kt < AB_DH / 16; ++kt) {
        const int o = j * AB_LDL + cb + kt * 16 + 2 * t;
        const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(Kh + o);
        const uint32_t bh1 = *reinterpret_cast<const uint32_t*>(Kh + o + 8);
        const uint32_t bl0 = *reinterpret_cast<const uint32_t*>(Kl + o);
        const uint32_t bl1 = *reinterpret_cast<const uint32_t*>(Kl + o + 8);
        mma_16816(sc[nt], ql[kt], bh0, bh1);
        mma_16816(sc[nt], qh[kt], bl0, bl1);
        mma_16816(sc[nt], qh[kt], bh0, bh1);
      }
    }
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int j = nt * 8 + 2 * t;
      if (j >= S) sc[nt][0] = sc[nt][2] = -INFINITY;
      if (j + 1 >= S) sc[nt][1] = sc[nt][3] = -INFINITY;
      m0 = fmaxf(m0, fmaxf(sc[nt][0], sc[nt][1]));
      m1 = fmaxf(m1, fmaxf(sc[nt][2], sc[nt][3]));
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    float l0 = 0.f, l1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      sc[nt][0] = expf(sc[nt][0] - m0);
      sc[nt][1] = expf(sc[nt][1] - m0);
      sc[nt][2] = expf(sc[nt][2] - m1);
      sc[nt][3] = expf(sc[nt][3] - m1);
      l0 += sc[nt][0] + sc[nt][1];
      l1 += sc[nt][2] + sc[nt][3];
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
    float oc[AB_DH / 8][4];
#pragma unroll
    for (int dt = 0; dt < AB_DH / 8; ++dt) oc[dt][0] = oc[dt][1] = oc[dt][2] = oc[dt][3] = 0.f;
#pragma unroll
    for (int kt = 0; kt < NT / 2; ++kt) {
      uint32_t pa[4];
      pa[0] = pack_h2(sc[2 * kt][0] * inv0, sc[2 * kt][1] * inv0);
      pa[1] = pack_h2(sc[2 * kt][2] * inv1, sc[2 * kt][3] * inv1);
      pa[2] = pack_h2(sc[2 * kt + 1][0] * inv0, sc[2 * kt + 1][1] * inv0);
      pa[3] = pack_h2(sc[2 * kt + 1][2] * inv1, sc[2 * kt + 1][3] * inv1);
#pragma unroll
      for (int dt = 0; dt < AB_DH / 8; ++dt) {
        const int d = cb + dt * 8 + g;
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(Vt + (size_t)d * VLD + kt * 16 + 2 * t);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(Vt + (size_t)d * VLD + kt * 16 + 8 + 2 * t);
        mma_16816(oc[dt], pa, b0, b1);
      }
    }
#pragma unroll
    for (int dt = 0; dt < AB_DH / 8; ++dt) {
      const int d = cb + dt * 8 + 2 * t;
      *reinterpret_cast<uint32_t*>(Cx + (size_t)i0 * AB_LDL + d) = pack_h2(oc[dt][0], oc[dt][1]);
      *reinterpret_cast<uint32_t*>(Cx + (size_t)i1 * AB_LDL + d) = pack_h2(oc[dt][2], oc[dt][3]);
    }
  }
  __syncthreads();     // ctx complete; h / Q / K are dead -> partial-sum tile

  // ---- phase 3: partial[S][C] = ctx_local W_o[:, local channels]^T.  Warp w owns columns [8w, 8w+8) ----
  {
    constexpr int MC = MTILES < 4 ? MTILES : 4;
    const int nb1[1] = {warp * 8};
    for (int m0 = 0; m0 < MTILES; m0 += MC) {
      float acc[MC][1][4];
#pragma unroll
      for (int mt = 0; mt < MC; ++mt) acc[mt][0][0] = acc[mt][0][1] = acc[mt][0][2] = acc[mt][0][3] = 0.f;
      ab_gemm<MC, 1, AB_CL / 16, AB_LDL>(Cx, m0 * 16, p.w_out, p.w_out + (size_t)AB_C * AB_C, nb1, cl0, acc, g, t);
#pragma unroll
      for (int mt = 0; mt < MC; ++mt) {
        if (m0 + mt >= MTILES) continue;
        const int r0 = (m0 + mt) * 16 + g;
        *reinterpret_cast<float2*>(Pp + (size_t)r0 * AB_PLD + warp * 8 + 2 * t) = make_float2(acc[mt][0][0], acc[mt][0][1]);
        *reinterpret_cast<float2*>(Pp + (size_t)(r0 + 8) * AB_PLD + warp * 8 + 2 * t) =
            make_float2(acc[mt][0][2], acc[mt][0][3]);
      }
    }
  }
  cluster.sync();
  // ---- out[:, cl0 .. cl0+64) = partial(rank 0) + partial(rank 1) + b_o + x, fixed order ----
  {
    const float* P0 = cluster.map_shared_rank(Pp, 0);
    const float* P1 = cluster.map_shared_rank(Pp, 1);
    for (int idx = tid; idx < S * (AB_CL / 4); idx += AB_THREADS) {
      const int r = idx / (AB_CL / 4), c = cl0 + (idx - r * (AB_CL / 4)) * 4;
      const float4 a = *reinterpret_cast<const float4*>(P0 + (size_t)r * AB_PLD + c);
      const float4 bq = *reinterpret_cast<const float4*>(P1 + (size_t)r * AB_PLD + c);
      const float4 bo = *reinterpret_cast<const float4*>(p.b_out + c);
      const size_t o = ((size_t)b * S + r) * AB_C + c;
      const float4 xr = *reinterpret_cast<const float4*>(p.x + o);
      float4 y;
      y.x = (a.x + bq.x) + bo.x + xr.x; y.y = (a.y + bq.y) + bo.y + xr.y;
      y.z = (a.z + bq.z) + bo.z + xr.z; y.w = (a.w + bq.w) + bo.w + xr.w;
      if (p.out32) *reinterpret_cast<float4*>(p.out32 + o) = y;
      if (p.out16) {
        uint2 u;
        u.x = pack_h2(y.x, y.y);
        u.y = pack_h2(y.z, y.w);
        *reinterpret_cast<uint2*>(p.out16 + o) = u;
      }
    }
  }
  cluster.sync();      // the peer may still be reading this CTA's partial tile
}

template <int NT>
static size_t attn_block_smem() {
  constexpr int SP = NT * 8;
  const size_t halfs = ((size_t)SP * AB_LD + (size_t)5 * SP * AB_LDL + (size_t)AB_CL * (SP + 8)) * sizeof(__half);
  const size_t part = (size_t)SP * AB_PLD * sizeof(float);        // aliases the front of the half buffers
  return halfs > part ? halfs : part;
}
template <int NT>
static int attn_block_launch(const AttnBlockParams& p, int B, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * B);
  cfg.blockDim = dim3(AB_THREADS);
  cfg.dynamicSmemBytes = attn_block_smem<NT>();
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  CM_CUDA(cudaLaunchKernelEx(&cfg, attn_block_kernel<NT>, p));
  return 0;
}

bool attn_block_supported(int S, int C, int heads) {
  return C == AB_C && heads == AB_HEADS && S >= 1 && S <= 128;
}

int attn_block_enqueue(const float* x, const float* gamma, const float* beta, const __half* w_in, const float* b_in,
                       const __half* w_out, const float* b_out, float* out32, __half* out16, int B, int S, int C,
                       int heads, float eps, cudaStream_t st) {
  CM_CHECK(attn_block_supported(S, C, heads), "fused attention block: C=%d heads=%d S=%d not covered", C, heads, S);
  AttnBlockParams p{x, gamma, beta, w_in, b_in, w_out, b_out, out32, out16, S, eps};
  switch ((S + 15) / 16) {
    case 1: return attn_block_launch<2>(p, B, st);
    case 2: return attn_block_launch<4>(p, B, st);
    case 3: return attn_block_launch<6>(p, B, st);
    case 4: return attn_block_launch<8>(p, B, st);
    case 5: return attn_block_launch<10>(p, B, st);
    case 6: return attn_block_launch<12>(p, B, st);
    case 7: return attn_block_launch<14>(p, B, st);
    default: return attn_block_launch<16>(p, B, st);
  }
}

template <int NT>
static int attn_block_attr() {
  CM_CUDA(cudaFuncSetAttribute(attn_block_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)attn_block_smem<NT>()));
  return 0;
}

// pre-set the shared-memory attribute of every attention instantiation outside stream capture
template <int DH, int NT>
static int attn_attr() {
  CM_CUDA(cudaFuncSetAttribute(attn_mma_kernel<DH, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
  return 0;
}
static int attn_init() {
#define CM_AT(NT) if (int rc = attn_attr<16, NT>()) return rc; if (int rc = attn_attr<32, NT>()) return rc; if (int rc = attn_attr<64, NT>()) return rc;
  CM_AT(2) CM_AT(4) CM_AT(6) CM_AT(8) CM_AT(10) CM_AT(12) CM_AT(14) CM_AT(16)
#undef CM_AT
#define CM_AB(NT) if (int rc = attn_block_attr<NT>()) return rc;
  CM_AB(2) CM_AB(4) CM_AB(6) CM_AB(8) CM_AB(10) CM_AB(12) CM_AB(14) CM_AB(16)
#undef CM_AB
  return 0;
}

int kernels_init() {
  static bool done = false;
  if (done) return 0;
  const int big = 160 * 1024;
  CM_CUDA(cudaFuncSetAttribute(first_conv_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  CM_CUDA(cudaFuncSetAttribute(first_conv_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  CM_CUDA(cudaFuncSetAttribute(first_conv_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  CM_CUDA(cudaFuncSetAttribute(first_conv_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  CM_CUDA(cudaFuncSetAttribute(final_conv_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  CM_CUDA(cudaFuncSetAttribute(final_conv_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  CM_CUDA(cudaFuncSetAttribute(final_conv_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  CM_CUDA(cudaFuncSetAttribute(final_conv_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  CM_CUDA(cudaFuncSetAttribute(gn_stats2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GN3_SMEM));
  CM_CUDA(cudaFuncSetAttribute(gn_apply2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GN3_SMEM));
  if (int rc = attn_init()) return rc;
  if (int rc = attn_long_init()) return rc;
  if (int rc = conv_init()) return rc;
  done = true;
  return 0;
}

// =============================================================================================
// chain bookkeeping
// =============================================================================================
__global__ void advance_step_kernel(int* step_dev, int* t_dev, const int* tsteps, int nsteps) {
  const int s = *step_dev + 1;
  *step_dev = s;
  *t_dev = tsteps[s < nsteps ? s : nsteps - 1];
}
int advance_step_enqueue(int* step_dev, int* t_dev, const int* tsteps, int nsteps, cudaStream_t st) {
  advance_step_kernel<<<1, 1, 0, st>>>(step_dev, t_dev, tsteps, nsteps);
  CM_CUDA(cudaGetLastError());
  return 0;
}
__global__ void advance_step_cond_kernel(int* step_dev, int* t_dev, const int* tsteps, int nsteps,
                                         cudaGraphConditionalHandle h) {
  const int s = *step_dev + 1;
  *step_dev = s;
  *t_dev = tsteps[s < nsteps ? s : nsteps - 1];
  cudaGraphSetConditional(h, s < nsteps ? 1u : 0u);
}
int advance_step_cond_enqueue(int* step_dev, int* t_dev, const int* tsteps, int nsteps, cudaGraphConditionalHandle h,
                              cudaStream_t st) {
  advance_step_cond_kernel<<<1, 1, 0, st>>>(step_dev, t_dev, tsteps, nsteps, h);
  CM_CUDA(cudaGetLastError());
  return 0;
}
__global__ void chain_begin_kernel(int* step_dev, int* t_dev, const int* tsteps, unsigned long long* chain_dev,
                                   unsigned long long seed, long long sample_offset) {
  *step_dev = 0;
  *t_dev = tsteps[0];
  chain_dev[0] = seed;
  chain_dev[1] = static_cast<unsigned long long>(sample_offset);
}
int chain_begin_enqueue(int* step_dev, int* t_dev, const int* tsteps, unsigned long long* chain_dev,
                        unsigned long long seed, long long sample_offset, cudaStream_t st) {
  chain_begin_kernel<<<1, 1, 0, st>>>(step_dev, t_dev, tsteps, chain_dev, seed, sample_offset);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// test-only scalar restatement of conv_umma (same packed fp16 operands, fp32 accumulate)
// =============================================================================================
__global__ void conv_ref_kernel(const ConvParams p, const __half* __restrict__ act,
                                const __half* __restrict__ extra, const __half* __restrict__ wp,
                                int B, int D, int H, int W) {
  const size_t total = (size_t)p.nphase * p.M * p.cout;
  const int taps = p.kd * p.kh * p.kw;
  const size_t ktot = (p.nphase > 1) ? (size_t)p.nphase * p.kphase
                                     : (size_t)taps * p.cin_main + p.cin_extra;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int n = (int)(idx % p.cout);
    size_t r = idx / p.cout;
    const int m = (int)(r % p.M);
    const int phase = (int)(r / p.M);
    const int b = m / p.pps;
    int rr = m - b * p.pps;
    const int z = rr / (p.oh * p.ow);
    rr -= z * p.oh * p.ow;
    const int pp_ = rr / p.ow;
    const int q = rr - pp_ * p.ow;
    float acc = 0.f;
    for (int t = 0; t < p.terms; ++t) {
      const __half* wrow = wp + ((size_t)t * p.cout + n) * ktot + (size_t)phase * p.kphase;
      for (int tap = 0; tap < taps; ++tap) {
        const int tw = tap % p.kw, th = (tap / p.kw) % p.kh, td = tap / (p.kw * p.kh);
        const int w = q * p.conv_stride + p.lower[phase][0] + tw;
        const int h = pp_ * p.conv_stride + p.lower[phase][1] + th;
        const int d = z * p.conv_stride + p.lower[phase][2] + td;
        if (w < 0 || w >= W || h < 0 || h >= H || d < 0 || d >= D) continue;
        const __half* ap = act + ((((size_t)b * D + d) * H + h) * W + w) * p.cin_main;
        const __half* wk = wrow + (size_t)tap * p.cin_main;
        for (int c = 0; c < p.cin_main; ++c) acc = fmaf(__half2float(ap[c]), __half2float(wk[c]), acc);
      }
      if (p.cin_extra) {
        const __half* ap = extra + (size_t)m * p.cin_extra;
        const __half* wk = wrow + (size_t)taps * p.cin_main;
        for (int c = 0; c < p.cin_extra; ++c) acc = fmaf(__half2float(ap[c]), __half2float(wk[c]), acc);
      }
    }
    if (p.epi.bias) acc += p.epi.bias[n];
    if (p.epi.bias2) acc += p.epi.bias2[n];
    if (p.epi.temb) {
      const int trow = p.epi.t_dev ? *p.epi.t_dev : 0;
      acc += p.epi.temb[(size_t)trow * p.epi.temb_ld + (size_t)b * p.epi.temb_bstride + n];
    }
    size_t orow = m;
    if (p.scatter) {
      const int pq = phase & 1, pp = (phase >> 1) & 1, pz = (phase >> 2) & 1;
      orow = (((size_t)b * (2 * p.od) + (2 * z + pz)) * (2 * p.oh) + (2 * pp_ + pp)) * (2 * p.ow) +
             (2 * q + pq);
    }
    if (p.epi.resid) acc += p.epi.resid[orow * p.cout + n];
    if (p.epi.out32) p.epi.out32[orow * p.epi.out_ld + n] = acc;
    if (p.epi.out16) p.epi.out16[orow * p.epi.out_ld + n] = __float2half_rn(acc);
  }
}

int conv_ref_enqueue(const ConvParams& p, const __half* act, const __half* extra,
                     const __half* wpacked, int B, int D, int H, int W, cudaStream_t st) {
  conv_ref_kernel<<<1024, 256, 0, st>>>(p, act, extra, wpacked, B, D, H, W);
  CM_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace cm
