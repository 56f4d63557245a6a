// Backward-pass kernels of the UNet hot path (training).  Contracts in backward.cuh; the
// reference ops they differentiate are cited there and per kernel below.
#include "backward.cuh"

#include "conv_umma.cuh"
#include "kernels.cuh"
#include "pack.cuh"

namespace cm {

int wgrad_init();   // conv_umma.cu

namespace {

__device__ __forceinline__ float silu_grad(float y) {
  const float s = 1.0f / (1.0f + __expf(-y));
  return s * (1.0f + y * (1.0f - s));
}

inline int grid_for(size_t total, int threads, int cap) {
  size_t b = (total + threads - 1) / threads;
  if (b < 1) b = 1;
  return (int)(b < (size_t)cap ? b : (size_t)cap);
}

// threads per CTA for a [pixels][C] channels-last sweep in float4 units: a multiple of Q = C/4 so
// that every thread keeps the same channel quad.
inline int sweep_threads(int Q) {
  int T = Q * (256 / Q > 0 ? 256 / Q : 1);
  return T;
}

}  // namespace

// =============================================================================================
// dgrad weight packing
// =============================================================================================
int dgrad_mode_of(int fwd_mode) {
  switch (fwd_mode) {
    case 0: return 0;
    case 1: return 2;
    case 2: return 4;
    default: return 3;
  }
}
size_t dgrad_packed_k(int fwd_mode, int cout_f, int dup) {
  const size_t c = (size_t)dup * cout_f;
  switch (fwd_mode) {
    case 0: return 27 * c;
    case 1:
    case 2: return 64 * c;
    default: return c;
  }
}

__global__ void pack_dgrad_kernel(int fwd_mode, const float* __restrict__ w, __half* __restrict__ dst,
                                  int cout_f, int cin_f, int terms, int perm, int dup, size_t ktot) {
  pack_dgrad_body(fwd_mode, w, dst, cout_f, cin_f, terms, perm, dup, ktot,
                  blockIdx.x * (size_t)blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
}

int pack_dgrad_weights(int fwd_mode, const float* w, __half* dst, int cout_f, int cin_f, int terms,
                       int perm, int dup, cudaStream_t st) {
  const size_t ktot = dgrad_packed_k(fwd_mode, cout_f, dup);
  const size_t total = (size_t)cin_f * ktot;
  pack_dgrad_kernel<<<grid_for(total, 256, 4096), 256, 0, st>>>(fwd_mode, w, dst, cout_f, cin_f, terms,
                                                               perm, dup, ktot);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// loss scale
// =============================================================================================
__global__ void absmax_kernel(const float* __restrict__ x, size_t n, unsigned int* __restrict__ out) {
  float m = 0.f;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(x[i]));
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));   // non-negative floats order as uints
}
__global__ void scale_from_max_kernel(unsigned int* __restrict__ mx, float target, float* __restrict__ scale) {
  const float m = __uint_as_float(*mx);
  float s = 1.f;
  if (m > 0.f && isfinite(m)) {
    int e;
    frexpf(target / m, &e);           // target/m = f * 2^e, f in [0.5, 1)
    e = e - 1;
    e = e > 60 ? 60 : (e < -60 ? -60 : e);
    s = ldexpf(1.f, e);
  }
  scale[0] = s;
  scale[1] = 1.f / s;
  *mx = 0u;                            // ready for the next call
}
int auto_scale_enqueue(const float* x, size_t n, float target, float* scale_dev, unsigned int* max_scratch,
                       cudaStream_t st) {
  absmax_kernel<<<grid_for(n, 256, 592), 256, 0, st>>>(x, n, max_scratch);
  scale_from_max_kernel<<<1, 1, 0, st>>>(max_scratch, target, scale_dev);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// dOut preparation: fp32 -> fp16 operand (+ residual fan-out, per-sample channel sums)
// =============================================================================================
__global__ void __launch_bounds__(1024)
cast_colsum_kernel(const float* __restrict__ src, __half* __restrict__ dst16, int dup, float* __restrict__ acc_dst,
                   int acc_init, float* __restrict__ colsum, int colsum_ld, int pixels, int C, int chunks,
                   int* __restrict__ err_flag) {
  extern __shared__ float red[];   // [T][4]
  const int Q = C >> 2, T = blockDim.x, tid = threadIdx.x;
  const int b = blockIdx.y, chunk = blockIdx.x;
  const int px0 = (int)(((long long)pixels * chunk) / chunks);
  const int px1 = (int)(((long long)pixels * (chunk + 1)) / chunks);
  const int nvec = (px1 - px0) * Q;
  const size_t base = ((size_t)b * pixels + px0) * C;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  bool sat = false;
  for (int i = tid; i < nvec; i += T) {
    const float4 v = *reinterpret_cast<const float4*>(src + base + (size_t)i * 4);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    if (dst16) {
      const float lim = 65504.f;
      float4 c = make_float4(fminf(fmaxf(v.x, -lim), lim), fminf(fmaxf(v.y, -lim), lim),
                             fminf(fmaxf(v.z, -lim), lim), fminf(fmaxf(v.w, -lim), lim));
      sat = sat || c.x != v.x || c.y != v.y || c.z != v.z || c.w != v.w;
      __half2 h0 = __floats2half2_rn(c.x, c.y), h1 = __floats2half2_rn(c.z, c.w);
      uint2 u;
      u.x = *reinterpret_cast<uint32_t*>(&h0);
      u.y = *reinterpret_cast<uint32_t*>(&h1);
      if (dup == 1) {
        *reinterpret_cast<uint2*>(dst16 + base + (size_t)i * 4) = u;
      } else {
        // hi | lo pair, K-concatenated per pixel: [pixel][2C], hi in [0, C), lo = fp16(v - hi) in [C, 2C)
        const int px = i / Q, cq = (i - px * Q) * 4;
        __half* row = dst16 + (((size_t)b * pixels + px0 + px) * 2) * C + cq;
        *reinterpret_cast<uint2*>(row) = u;
        const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
        __half2 l0 = __floats2half2_rn(c.x - f0.x, c.y - f0.y), l1 = __floats2half2_rn(c.z - f1.x, c.w - f1.y);
        u.x = *reinterpret_cast<uint32_t*>(&l0);
        u.y = *reinterpret_cast<uint32_t*>(&l1);
        *reinterpret_cast<uint2*>(row + C) = u;
      }
    }
    if (acc_dst) {
      float4* ap = reinterpret_cast<float4*>(acc_dst + base + (size_t)i * 4);
      if (acc_init) *ap = v;
      else {
        float4 a = *ap;
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        *ap = a;
      }
    }
  }
  if (sat && err_flag) atomicExch(err_flag, 301);   // fp16 overflow of a scaled gradient
  if (!colsum) return;
  reinterpret_cast<float4*>(red)[tid] = s;
  __syncthreads();
  if (tid < Q) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = tid; r < T; r += Q) {
      const float4 v = reinterpret_cast<float4*>(red)[r];
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    float* cp = colsum + (size_t)b * colsum_ld + tid * 4;
    atomicAdd(cp + 0, a.x);
    atomicAdd(cp + 1, a.y);
    atomicAdd(cp + 2, a.z);
    atomicAdd(cp + 3, a.w);
  }
}

int cast_colsum_enqueue(const float* src, __half* dst16, int dup, float* acc_dst, int acc_init, float* colsum,
                        int colsum_ld, int B, int pixels, int C, cudaStream_t st) {
  CM_CHECK(C % 4 == 0 && C / 4 <= 1024, "cast_colsum: bad channel count %d", C);
  CM_CHECK(dup == 1 || dup == 2, "cast_colsum: dup must be 1 or 2");
  const int Q = C / 4;
  const int T = sweep_threads(Q);
  int chunks = 592 / B;
  if (chunks < 1) chunks = 1;
  if (chunks > (pixels + 7) / 8) chunks = (pixels + 7) / 8;
  if (chunks < 1) chunks = 1;
  cast_colsum_kernel<<<dim3(chunks, B), T, (size_t)T * 16, st>>>(src, dst16, dup, acc_dst, acc_init, colsum,
                                                                colsum_ld, pixels, C, chunks,
                                                                device_error_flag());
  CM_CUDA(cudaGetLastError());
  return 0;
}

__global__ void rowsum_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int C, int ld,
                              int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float a = 0.f;
  for (int b = 0; b < B; ++b) a += in[(size_t)b * ld + c];
  out[c] = accumulate ? out[c] + a : a;
}
int rowsum_enqueue(const float* in, float* out, int B, int C, int ld, int accumulate, cudaStream_t st) {
  rowsum_kernel<<<(C + 127) / 128, 128, 0, st>>>(in, out, B, C, ld, accumulate);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// G -> nn.Conv3d weight-gradient layout
// =============================================================================================
__device__ __forceinline__ void unpack_wgrad_body(int fwd_mode, const float* __restrict__ G, float* __restrict__ dw,
                                                  float* __restrict__ dwx, int cout_arg, int cin_arg, int cinx, int perm) {
  // cout_arg = cout | (cout_g << 16) likewise: columns per row of G (the final conv's d_eps packed into 32 columns)
  const int cout_w = cout_arg & 0xffff;
  const int cout = (cout_arg >> 16) ? (cout_arg >> 16) : cout_w;
  // cin_arg = cin | (cin_g << 16): cin_g = channels per tap of G when it is wider than the weight (the first conv's packed
  // 32-channel operand), 0 = the same
  const int cin = cin_arg & 0xffff;
  const int cin_g = (cin_arg >> 16) ? (cin_arg >> 16) : cin;
  const int taps = (fwd_mode == 3) ? 1 : 27;
  const size_t n_main = (size_t)cout_w * cin * taps;
  const size_t total = n_main + (size_t)cout_w * cinx;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    if (idx >= n_main) {
      const size_t r = idx - n_main;
      const int co = (int)(r / cinx), cx = (int)(r - (size_t)co * cinx);
      dwx[r] = G[((size_t)taps * cin + cx) * cout + co];
      continue;
    }
    const int st = (int)(idx % taps);            // source tap index (reference weight layout)
    const size_t r = idx / taps;
    const int ci = (int)(r % cin), co = (int)(r / cin);
    float v = 0.f;
    if (fwd_mode == 3) {
      v = G[(size_t)ci * cout + co];
    } else {
      // source tap -> activation-order tap (d, h, w)
      int td, th, tw;
      if (perm) { td = st % 3; tw = (st / 3) % 3; th = st / 9; }
      else { tw = st % 3; th = (st / 3) % 3; td = st / 9; }
      if (fwd_mode != 2) {
        v = G[((size_t)((td * 3 + th) * 3 + tw) * cin_g + ci) * cout + co];
      } else {
        // fold the 8 phases x 8 taps: original tap k of one dim lives in (p, a) pairs
        //   k=0: (0,0),(1,0)   k=1: (0,1),(1,0)   k=2: (0,1),(1,1)
        const int kk[3] = {tw, th, td};
        const size_t krows = (size_t)8 * cin;
        for (int sel = 0; sel < 8; ++sel) {
          int phase = 0, tap8 = 0;
#pragma unroll
          for (int d = 0; d < 3; ++d) {
            const int which = (sel >> d) & 1;
            int p, a;
            if (kk[d] == 0) { p = which; a = 0; }
            else if (kk[d] == 1) { p = which; a = which ? 0 : 1; }
            else { p = which; a = 1; }
            phase |= p << d;
            tap8 |= a << d;
          }
          v += G[((size_t)phase * krows + (size_t)tap8 * cin + ci) * cout + co];
        }
      }
    }
    dw[idx] = v;
  }
}
__global__ void unpack_wgrad_kernel(int fwd_mode, const float* __restrict__ G, float* __restrict__ dw,
                                    float* __restrict__ dwx, int cout, int cin, int cinx, int perm) {
  unpack_wgrad_body(fwd_mode, G, dw, dwx, cout, cin, cinx, perm);
}
// every conv of the plan in one launch (blockIdx.y = conv): tab[e] = {fwd_mode, G offset, dw offset,
// dwx offset or -1, cout, cin, cinx, perm}; offsets in floats from Gbase / grads
__global__ void unpack_wgrad_all_kernel(const long long* __restrict__ tab, const float* __restrict__ Gbase,
                                        float* __restrict__ grads) {
  const long long* t = tab + (size_t)blockIdx.y * 8;
  unpack_wgrad_body((int)t[0], Gbase + t[1], grads + t[2], t[3] >= 0 ? grads + t[3] : nullptr, (int)t[4], (int)t[5],
                    (int)t[6], (int)t[7]);
}
int unpack_wgrad_all_enqueue(const long long* tab, int n, const float* Gbase, float* grads, cudaStream_t st) {
  unpack_wgrad_all_kernel<<<dim3(64, n), 256, 0, st>>>(tab, Gbase, grads);
  CM_CUDA(cudaGetLastError());
  return 0;
}

int unpack_wgrad_enqueue(int fwd_mode, const float* G, float* dw, float* dwx, int cout, int cin,
                         int cinx, int perm, cudaStream_t st) {
  const size_t total = (size_t)cout * cin * (fwd_mode == 3 ? 1 : 27) + (size_t)cout * cinx;
  unpack_wgrad_kernel<<<grid_for(total, 256, 4096), 256, 0, st>>>(fwd_mode, G, dw, dwx, cout, cin, cinx,
                                                                 perm);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// scalar restatement of the weight gradient (same fp16 operands, same G layout; test oracle)
// =============================================================================================
__global__ void wgrad_ref_kernel(int fwd_mode, const __half* __restrict__ act, const __half* __restrict__ extra,
                                 const __half* __restrict__ dout, float* __restrict__ G, int B, int D, int H,
                                 int W, int cin, int cinx, int cout) {
  int k = 3, stride = 1, od = D, oh = H, ow = W, nphase = 1;
  if (fwd_mode == 1) { stride = 2; od = (D - 1) / 2 + 1; oh = (H - 1) / 2 + 1; ow = (W - 1) / 2 + 1; }
  else if (fwd_mode == 2) { k = 2; nphase = 8; }
  else if (fwd_mode == 3) k = 1;
  const int taps = k * k * k;
  const size_t krows = (size_t)taps * cin + cinx;
  const size_t total = (size_t)nphase * krows * cout;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int co = (int)(idx % cout);
    size_t r = idx / cout;
    const int krow = (int)(r % krows);
    const int phase = (int)(r / krows);
    float acc = 0.f;
    const bool main = krow < taps * cin;
    const int tap = main ? krow / cin : 0;
    const int ci = main ? krow - tap * cin : krow - taps * cin;
    const int tw = tap % k, th = (tap / k) % k, td = tap / (k * k);
    int lw = -1, lh = -1, ld = -1;
    if (fwd_mode == 2) { lw = (phase & 1) ? 0 : -1; lh = (phase & 2) ? 0 : -1; ld = (phase & 4) ? 0 : -1; }
    else if (fwd_mode == 3) lw = lh = ld = 0;
    for (int b = 0; b < B; ++b)
      for (int z = 0; z < od; ++z)
        for (int p = 0; p < oh; ++p)
          for (int q = 0; q < ow; ++q) {
            float a;
            if (main) {
              const int w = q * stride + lw + tw, h = p * stride + lh + th, d = z * stride + ld + td;
              if (w < 0 || w >= W || h < 0 || h >= H || d < 0 || d >= D) continue;
              a = __half2float(act[((((size_t)b * D + d) * H + h) * W + w) * cin + ci]);
            } else {
              a = __half2float(extra[((((size_t)b * od + z) * oh + p) * ow + q) * cinx + ci]);
            }
            size_t orow;
            if (fwd_mode == 2)
              orow = (((size_t)b * (2 * od) + (2 * z + ((phase >> 2) & 1))) * (2 * oh) + (2 * p + ((phase >> 1) & 1))) *
                         (2 * ow) + (2 * q + (phase & 1));
            else
              orow = (((size_t)b * od + z) * oh + p) * ow + q;
            acc = fmaf(a, __half2float(dout[orow * cout + co]), acc);
          }
    G[idx] = acc;
  }
}

int wgrad_ref_enqueue(int fwd_mode, const __half* act16, const __half* extra16, const __half* dout16,
                      float* G, int B, int D, int H, int W, int cin, int cinx, int cout,
                      cudaStream_t st) {
  wgrad_ref_kernel<<<1024, 128, 0, st>>>(fwd_mode, act16, extra16, dout16, G, B, D, H, W, cin, cinx, cout);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// GroupNorm(8) [+SiLU] [+Dropout3d scale] backward
//   xhat = (x - mean) rstd, y = xhat*gamma + beta, z = silu(y) (optional), out = z * drop
//   dy = dout*drop*silu'(y);  S1[b,c] = sum_p dy, S2[b,c] = sum_p dy*xhat
//   dgamma = sum_b S2, dbeta = sum_b S1
//   per (b, group): m1 = sum_c gamma_c S1 / N, m2 = sum_c gamma_c S2 / N   (N = pixels * C/8)
//   dx = rstd * (dy*gamma - m1 - xhat*m2) (+ draw)
// =============================================================================================
struct GnBwdGeom {
  int Q, T, chunks;
};

__device__ __forceinline__ float4 gn_bwd_dy(const GnBwdParams& p, const float4 x, const float4 dn,
                                            const float mean, const float rstd, const float4 ga,
                                            const float4 be, const float4 ds, float4* xhat) {
  float4 xh = make_float4((x.x - mean) * rstd, (x.y - mean) * rstd, (x.z - mean) * rstd, (x.w - mean) * rstd);
  float4 dy = make_float4(dn.x * ds.x, dn.y * ds.y, dn.z * ds.z, dn.w * ds.w);
  if (p.silu) {
    dy.x *= silu_grad(fmaf(xh.x, ga.x, be.x));
    dy.y *= silu_grad(fmaf(xh.y, ga.y, be.y));
    dy.z *= silu_grad(fmaf(xh.z, ga.z, be.z));
    dy.w *= silu_grad(fmaf(xh.w, ga.w, be.w));
  }
  *xhat = xh;
  return dy;
}

// pass 1: partial[b][chunk][c][2]
__global__ void __launch_bounds__(1024) gn_bwd_sums_kernel(const GnBwdParams p, int chunks, float* __restrict__ partial) {
  extern __shared__ float red[];   // [T][8]
  const int C = p.c0 + p.c1, Q = C >> 2, cg_ch = C >> 3, T = blockDim.x, tid = threadIdx.x;
  const int b = blockIdx.y, chunk = blockIdx.x;
  const int px0 = (int)(((long long)p.pixels * chunk) / chunks);
  const int px1 = (int)(((long long)p.pixels * (chunk + 1)) / chunks);
  const int c = (tid % Q) * 4;
  const int g = c / cg_ch;
  const float mean = p.stats[(b * 8 + g) * 2], rstd = p.stats[(b * 8 + g) * 2 + 1];
  const float4 ga = *reinterpret_cast<const float4*>(p.gamma + c);
  const float4 be = *reinterpret_cast<const float4*>(p.beta + c);
  float4 ds = make_float4(1.f, 1.f, 1.f, 1.f);
  if (p.drop_scale) ds = *reinterpret_cast<const float4*>(p.drop_scale + (size_t)b * p.drop_ld + c);
  const bool from0 = c < p.c0;
  const float* src = from0 ? p.src0 + c : p.src1 + (c - p.c0);
  const int src_ld = from0 ? p.c0 : p.c1;
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
  const int rows_per_iter = T / Q;
  for (int px = px0 + tid / Q; px < px1; px += rows_per_iter) {
    const size_t pix = (size_t)b * p.pixels + px;
    const float4 x = *reinterpret_cast<const float4*>(src + pix * src_ld);
    const float4 dn = *reinterpret_cast<const float4*>(p.dnorm + pix * C + c);
    float4 xh;
    const float4 dy = gn_bwd_dy(p, x, dn, mean, rstd, ga, be, ds, &xh);
    s1.x += dy.x; s1.y += dy.y; s1.z += dy.z; s1.w += dy.w;
    s2.x += dy.x * xh.x; s2.y += dy.y * xh.y; s2.z += dy.z * xh.z; s2.w += dy.w * xh.w;
  }
  reinterpret_cast<float4*>(red)[tid * 2] = s1;
  reinterpret_cast<float4*>(red)[tid * 2 + 1] = s2;
  __syncthreads();
  if (tid < Q) {
    float4 a1 = make_float4(0.f, 0.f, 0.f, 0.f), a2 = a1;
    for (int r = tid; r < T; r += Q) {
      const float4 v1 = reinterpret_cast<float4*>(red)[r * 2], v2 = reinterpret_cast<float4*>(red)[r * 2 + 1];
      a1.x += v1.x; a1.y += v1.y; a1.z += v1.z; a1.w += v1.w;
      a2.x += v2.x; a2.y += v2.y; a2.z += v2.z; a2.w += v2.w;
    }
    float* o = partial + (((size_t)b * chunks + chunk) * C + c) * 2;
    o[0] = a1.x; o[1] = a2.x; o[2] = a1.y; o[3] = a2.y; o[4] = a1.z; o[5] = a2.z; o[6] = a1.w; o[7] = a2.w;
  }
}

// pass 2: combine partials (fixed order), group means, dx
__global__ void __launch_bounds__(1024) gn_bwd_apply_kernel(const GnBwdParams p, int chunks, const float* __restrict__ partial) {
  extern __shared__ float sm[];    // [C][2] gamma-weighted channel sums | [8][2] group means
  const int C = p.c0 + p.c1, Q = C >> 2, cg_ch = C >> 3, T = blockDim.x, tid = threadIdx.x;
  float* gs = sm;
  float* gm = sm + 2 * C;
  const int b = blockIdx.y, chunk = blockIdx.x;
  for (int cc = tid; cc < C; cc += T) {
    float a1 = 0.f, a2 = 0.f;
    for (int k = 0; k < chunks; ++k) {
      const float* o = partial + (((size_t)b * chunks + k) * C + cc) * 2;
      a1 += o[0];
      a2 += o[1];
    }
    if (chunk == 0) {
      p.chsum[((size_t)b * C + cc) * 2] = a1;
      p.chsum[((size_t)b * C + cc) * 2 + 1] = a2;
    }
    const float gmm = p.gamma[cc];
    gs[cc * 2] = a1 * gmm;
    gs[cc * 2 + 1] = a2 * gmm;
  }
  __syncthreads();
  if (tid < 16) {
    const int g = tid >> 1, which = tid & 1;
    float a = 0.f;
    for (int k = 0; k < cg_ch; ++k) a += gs[(g * cg_ch + k) * 2 + which];
    gm[tid] = a / ((float)p.pixels * (float)cg_ch);
  }
  __syncthreads();
  const int px0 = (int)(((long long)p.pixels * chunk) / chunks);
  const int px1 = (int)(((long long)p.pixels * (chunk + 1)) / chunks);
  const int c = (tid % Q) * 4;
  const int g = c / cg_ch;
  const float mean = p.stats[(b * 8 + g) * 2], rstd = p.stats[(b * 8 + g) * 2 + 1];
  const float m1 = gm[g * 2], m2 = gm[g * 2 + 1];
  const float4 ga = *reinterpret_cast<const float4*>(p.gamma + c);
  const float4 be = *reinterpret_cast<const float4*>(p.beta + c);
  float4 ds = make_float4(1.f, 1.f, 1.f, 1.f);
  if (p.drop_scale) ds = *reinterpret_cast<const float4*>(p.drop_scale + (size_t)b * p.drop_ld + c);
  const bool from0 = c < p.c0;
  const float* src = from0 ? p.src0 + c : p.src1 + (c - p.c0);
  float* dsrc = from0 ? p.dsrc0 + c : p.dsrc1 + (c - p.c0);
  const int src_ld = from0 ? p.c0 : p.c1;
  const int init = from0 ? p.init0 : p.init1;
  const int rows_per_iter = T / Q;
  for (int px = px0 + tid / Q; px < px1; px += rows_per_iter) {
    const size_t pix = (size_t)b * p.pixels + px;
    const float4 x = *reinterpret_cast<const float4*>(src + pix * src_ld);
    const float4 dn = *reinterpret_cast<const float4*>(p.dnorm + pix * C + c);
    float4 xh;
    const float4 dy = gn_bwd_dy(p, x, dn, mean, rstd, ga, be, ds, &xh);
    float4 dx = make_float4(rstd * (dy.x * ga.x - m1 - xh.x * m2), rstd * (dy.y * ga.y - m1 - xh.y * m2),
                            rstd * (dy.z * ga.z - m1 - xh.z * m2), rstd * (dy.w * ga.w - m1 - xh.w * m2));
    if (p.draw) {
      const float4 r = *reinterpret_cast<const float4*>(p.draw + pix * C + c);
      dx.x += r.x; dx.y += r.y; dx.z += r.z; dx.w += r.w;
    }
    float4* dp = reinterpret_cast<float4*>(dsrc + pix * src_ld);
    if (!init) {
      const float4 o = *dp;
      dx.x += o.x; dx.y += o.y; dx.z += o.z; dx.w += o.w;
    }
    *dp = dx;
  }
}

__global__ void gn_bwd_params_kernel(const float* __restrict__ chsum, int B, int C, float* __restrict__ dgamma,
                                     float* __restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float a1 = 0.f, a2 = 0.f;
  for (int b = 0; b < B; ++b) {
    a1 += chsum[((size_t)b * C + c) * 2];
    a2 += chsum[((size_t)b * C + c) * 2 + 1];
  }
  dbeta[c] = a1;
  dgamma[c] = a2;
}

int gn_bwd_chunks(int B, int pixels) {
  int chunks = 592 / B;
  if (chunks < 1) chunks = 1;
  if (chunks > 32) chunks = 32;
  if (chunks > (pixels + 3) / 4) chunks = (pixels + 3) / 4;
  if (chunks < 1) chunks = 1;
  return chunks;
}

int gn_backward_enqueue(const GnBwdParams& p, float* partial, cudaStream_t st) {
  const int C = p.c0 + p.c1;
  CM_CHECK(C % 32 == 0 && p.c0 % 4 == 0, "GroupNorm backward: channels must be a multiple of 32 (C=%d)", C);
  const int Q = C / 4;
  CM_CHECK(Q <= 1024, "GroupNorm backward: too many channels (C=%d)", C);
  const int T = sweep_threads(Q);
  const int chunks = gn_bwd_chunks(p.B, p.pixels);
  gn_bwd_sums_kernel<<<dim3(chunks, p.B), T, (size_t)T * 32, st>>>(p, chunks, partial);
  gn_bwd_apply_kernel<<<dim3(chunks, p.B), T, (size_t)(2 * C + 16) * 4, st>>>(p, chunks, partial);
  // dgamma / dbeta = batch sums of chsum: per GroupNorm here, or for all of them in one launch at the end of
  // the backward (gn_backward_params_all_enqueue) when the caller keeps one chsum region per GroupNorm
  if (p.dgamma) gn_bwd_params_kernel<<<(C + 127) / 128, 128, 0, st>>>(p.chsum, p.B, C, p.dgamma, p.dbeta);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// one CTA per GroupNorm: tab[g] = {chsum offset (floats), C, dgamma offset, dbeta offset (floats into grads)}
__global__ void gn_bwd_params_all_kernel(const float* __restrict__ chsum_base, const long long* __restrict__ tab,
                                         int B, float* __restrict__ grads) {
  const long long* t = tab + (size_t)blockIdx.x * 4;
  const float* chsum = chsum_base + t[0];
  const int C = (int)t[1];
  float* dgamma = grads + t[2];
  float* dbeta = grads + t[3];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a1 = 0.f, a2 = 0.f;
    for (int b = 0; b < B; ++b) {
      a1 += chsum[((size_t)b * C + c) * 2];
      a2 += chsum[((size_t)b * C + c) * 2 + 1];
    }
    dbeta[c] = a1;
    dgamma[c] = a2;
  }
}
// every conv's bias gradient (batch sum of its per-sample channel sums) in one launch:
// tab[e] = {source offset (floats from base), row stride, channels, gradient offset (floats into grads)}
// blockDim = (32 channels, 8 batch slices): the first version walked the batch serially per channel (64 dependent-latency
// loads per thread, 51 us for ~40 small CTAs); slice sums are added in slice order (fixed)
__global__ void __launch_bounds__(256) rowsum_all_kernel(const float* __restrict__ base, const long long* __restrict__ tab,
                                                         int B, float* __restrict__ grads) {
  __shared__ float part[8][33];
  const long long* t = tab + (size_t)blockIdx.x * 4;
  const float* src = base + t[0];
  const int ld = (int)t[1], C = (int)t[2];
  float* out = grads + t[3];
  for (int c0 = 0; c0 < C; c0 += 32) {
    const int c = c0 + threadIdx.x;
    float a = 0.f;
    if (c < C)
      for (int b = threadIdx.y; b < B; b += 8) a += src[(size_t)b * ld + c];
    part[threadIdx.y][threadIdx.x] = a;
    __syncthreads();
    if (threadIdx.y == 0 && c < C) {
      float v = 0.f;
#pragma unroll
      for (int y = 0; y < 8; ++y) v += part[y][threadIdx.x];
      out[c] = v;
    }
    __syncthreads();
  }
}
int rowsum_all_enqueue(const float* base, const long long* tab, int n, int B, float* grads, cudaStream_t st) {
  rowsum_all_kernel<<<n, dim3(32, 8), 0, st>>>(base, tab, B, grads);
  CM_CUDA(cudaGetLastError());
  return 0;
}

int gn_backward_params_all_enqueue(const float* chsum_base, const long long* tab, int n_gn, int B, float* grads,
                                   cudaStream_t st) {
  gn_bwd_params_all_kernel<<<n_gn, 256, 0, st>>>(chsum_base, tab, B, grads);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// attention core backward (one CTA per (sample, head); everything in shared memory, fp32).
// Reference: autograd of nn.MultiheadAttention's softmax(Q K^T / sqrt(dh)) V (models/backbones/layers.py:5-18).
// Five small products per (sample, head); each is a register-tiled (4 x 4 outputs per thread) shared-memory GEMM whose B
// operand is laid out with the output column contiguous (K and V are also kept transposed), so the inner loop is one
// broadcast row read + one 128-bit read per 16 FMAs.  The first version (one output per thread, two scalar shared-memory
// reads per FMA) took 0.12 ms per attention block at the HERMES shape, 0.48 ms of the 8 ms backward.
//   P = softmax(Q K^T * s)            dV = P^T dO            dP = dO V^T (formed twice: row sums D_i = sum_j dP o P, then dS)
//   dS = P o (dP - D) * s             dQ = dS K              dK = dS^T Q
// Every output element is one ascending-k fmaf chain: deterministic.
// =============================================================================================
namespace {
// C(i, j) = sum_k A(i, k) * B(k, j) for i < M, j < N (N a multiple of 4); A(i, k) = Ap[i * sai + k * sak],
// B(k, j) = Bp[k * ldb + j] with ldb a multiple of 4 and Bp 16-byte aligned; epi(i, j0, float4 of columns j0 .. j0 + 3)
template <class Epi>
__device__ __forceinline__ void smem_gemm_4x4(int M, int N, int K, const float* __restrict__ Ap, int sai, int sak,
                                              const float* __restrict__ Bp, int ldb, Epi epi) {
  const int tn = N >> 2, tm = (M + 3) >> 2;
  for (int t = threadIdx.x; t < tm * tn; t += blockDim.x) {
    const int ti = t / tn, j0 = (t - ti * tn) << 2, i0 = ti << 2;
    int ia[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) ia[r] = (i0 + r < M ? i0 + r : M - 1) * sai;
    float acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
    const float* bp = Bp + j0;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
      const float4 b = *reinterpret_cast<const float4*>(bp + (size_t)k * ldb);
      float a[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) a[r] = Ap[ia[r] + k * sak];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        acc[r][0] = fmaf(a[r], b.x, acc[r][0]);
        acc[r][1] = fmaf(a[r], b.y, acc[r][1]);
        acc[r][2] = fmaf(a[r], b.z, acc[r][2]);
        acc[r][3] = fmaf(a[r], b.w, acc[r][3]);
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (i0 + r < M) epi(i0 + r, j0, make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]));
  }
}
}  // namespace

__global__ void __launch_bounds__(256)
attn_core_backward_kernel(const float* __restrict__ qkv, const float* __restrict__ dctx,
                          float* __restrict__ dqkv, int S, int C, int heads) {
  extern __shared__ __align__(16) float sm[];
  const int dh = C / heads;                 // multiple of 4 (host-checked)
  const int ld = dh + 4;                    // row-major [S][ld] tiles: 16-byte aligned rows
  const int Sp = (S + 3) & ~3;              // padded column count of the S x S / transposed tiles
  const int lds = Sp + 4;
  const int b = blockIdx.x / heads, hd = blockIdx.x % heads;
  float* Qs = sm;                           // [S][ld]
  float* Ks = Qs + (size_t)S * ld;
  float* Os = Ks + (size_t)S * ld;          // dO
  float* Kt = Os + (size_t)S * ld;          // [dh][lds] K^T
  float* Vt = Kt + (size_t)dh * lds;        // [dh][lds] V^T
  float* Ps = Vt + (size_t)dh * lds;        // [S][lds]: P, then dS in place
  float* Dp = Ps + (size_t)S * lds;         // [S][Sp / 4] partial row sums of dP o P, one slot per column tile
  float* Dv = Dp + (size_t)S * (Sp >> 2);   // [S]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
  const float* base = qkv + (size_t)b * S * 3 * C + hd * dh;
  const float* dob = dctx + (size_t)b * S * C + hd * dh;
  for (int idx = tid; idx < S * dh; idx += blockDim.x) {
    const int j = idx / dh, d = idx - j * dh;
    const float q = base[(size_t)j * 3 * C + d], k = base[(size_t)j * 3 * C + C + d], v = base[(size_t)j * 3 * C + 2 * C + d];
    Qs[j * ld + d] = q;
    Ks[j * ld + d] = k;
    Kt[d * lds + j] = k;
    Vt[d * lds + j] = v;
    Os[j * ld + d] = dob[(size_t)j * C + d];
  }
  for (int idx = tid; idx < dh * (lds - S); idx += blockDim.x) {   // padded columns of the transposed tiles: finite zeros
    const int d = idx / (lds - S), j = S + idx % (lds - S);
    Kt[d * lds + j] = 0.f;
    Vt[d * lds + j] = 0.f;
  }
  __syncthreads();
  const float scale = rsqrtf((float)dh);
  // scores: Ps[i][j] = Q_i . K_j * scale   (columns >= S are padding: computed from the zero columns, never used)
  smem_gemm_4x4(S, Sp, dh, Qs, ld, 1, Kt, lds, [&](int i, int j0, float4 v) {
    *reinterpret_cast<float4*>(Ps + (size_t)i * lds + j0) = make_float4(v.x * scale, v.y * scale, v.z * scale, v.w * scale);
  });
  __syncthreads();
  for (int i = warp; i < S; i += nwarps) {          // row softmax
    float mx = -INFINITY;
    for (int j = lane; j < S; j += 32) mx = fmaxf(mx, Ps[(size_t)i * lds + j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < S; j += 32) {
      const float e = expf(Ps[(size_t)i * lds + j] - mx);
      Ps[(size_t)i * lds + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    for (int j = lane; j < S; j += 32) Ps[(size_t)i * lds + j] *= inv;
    for (int j = S + lane; j < lds; j += 32) Ps[(size_t)i * lds + j] = 0.f;
  }
  __syncthreads();
  float* dq = dqkv + (size_t)b * S * 3 * C + hd * dh;
  // dV[j][d] = sum_i P[i][j] dO[i][d]
  smem_gemm_4x4(S, dh, S, Ps, 1, lds, Os, ld, [&](int j, int d0, float4 v) {
    *reinterpret_cast<float4*>(dq + (size_t)j * 3 * C + 2 * C + d0) = v;
  });
  // D_i = sum_j dP[i][j] P[i][j] with dP[i][j] = dO_i . V_j: every (row, column tile) writes its own slot, the slots of a
  // row are then added in tile order (deterministic)
  smem_gemm_4x4(S, Sp, dh, Os, ld, 1, Vt, lds, [&](int i, int j0, float4 v) {
    const float4 p = *reinterpret_cast<const float4*>(Ps + (size_t)i * lds + j0);
    Dp[(size_t)i * (Sp >> 2) + (j0 >> 2)] = fmaf(v.w, p.w, fmaf(v.z, p.z, fmaf(v.y, p.y, v.x * p.x)));
  });
  __syncthreads();
  for (int i = tid; i < S; i += blockDim.x) {
    float a = 0.f;
    for (int t = 0; t < (Sp >> 2); ++t) a += Dp[(size_t)i * (Sp >> 2) + t];
    Dv[i] = a;
  }
  __syncthreads();
  // dS[i][j] = P[i][j] * (dO_i . V_j - D_i) * scale, in place over P (the scale is folded in: dQ and dK both carry it)
  smem_gemm_4x4(S, Sp, dh, Os, ld, 1, Vt, lds, [&](int i, int j0, float4 v) {
    float4* pp = reinterpret_cast<float4*>(Ps + (size_t)i * lds + j0);
    const float4 p = *pp;
    const float di = Dv[i];
    *pp = make_float4(p.x * (v.x - di) * scale, p.y * (v.y - di) * scale, p.z * (v.z - di) * scale, p.w * (v.w - di) * scale);
  });
  __syncthreads();
  // dQ[i][d] = sum_j dS[i][j] K[j][d],  dK[j][d] = sum_i dS[i][j] Q[i][d]
  smem_gemm_4x4(S, dh, S, Ps, lds, 1, Ks, ld, [&](int i, int d0, float4 v) {
    *reinterpret_cast<float4*>(dq + (size_t)i * 3 * C + d0) = v;
  });
  smem_gemm_4x4(S, dh, S, Ps, 1, lds, Qs, ld, [&](int j, int d0, float4 v) {
    *reinterpret_cast<float4*>(dq + (size_t)j * 3 * C + C + d0) = v;
  });
}

static size_t attn_bwd_smem(int S, int dh) {
  const size_t Sp = (size_t)((S + 3) & ~3), lds = Sp + 4;
  return ((size_t)3 * S * (dh + 4) + (size_t)2 * dh * lds + (size_t)S * lds + (size_t)S * (Sp >> 2) + S) * sizeof(float);
}

int attn_core_backward_enqueue(const float* qkv, const float* dctx, float* dqkv, int B, int S, int C,
                               int heads, cudaStream_t st, const float* lse, float* dsum) {
  if (attn_uses_long(S, C / heads)) {
    CM_CHECK(C % heads == 0 && (C / heads) % 2 == 0 && C / heads <= 128, "attention: head dim %d / %d unsupported (even, <= 128)",
             C, heads);
    CM_CHECK(lse && dsum, "attention backward at S=%d, dh=%d needs the forward's log-sum-exp and a row-sum workspace", S,
             C / heads);
    return attn_long_backward_enqueue(qkv, dctx, lse, dsum, dqkv, B, S, C, heads, st);
  }
  CM_CHECK(C % heads == 0 && (C / heads) % 4 == 0 && C % 4 == 0, "embed dim %d / heads %d unsupported", C, heads);
  const size_t smem = attn_bwd_smem(S, C / heads);
  CM_CHECK(smem <= 227 * 1024, "attention backward tile too large for shared memory (S=%d dh=%d)", S, C / heads);
  attn_core_backward_kernel<<<B * heads, 256, smem, st>>>(qkv, dctx, dqkv, S, C, heads);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// final conv backward (unet.py:121,165-167): only future frames carry gradient
// =============================================================================================
template <int COUT>
__global__ void __launch_bounds__(256)
final_conv_dact_kernel(const float* __restrict__ deps, const float* __restrict__ scale_dev,
                       const float* __restrict__ w, float* __restrict__ dact, int B, int H, int W, int L,
                       int P, int cin) {
  extern __shared__ float ws[];   // [27][cin][COUT]
  for (int idx = threadIdx.x; idx < 27 * cin * COUT; idx += blockDim.x) {
    const int co = idx % COUT;
    const int r = idx / COUT;
    const int ci = r % cin, tap = r / cin;
    ws[idx] = w[((size_t)co * cin + ci) * 27 + tap];
  }
  __syncthreads();
  const float scale = scale_dev ? scale_dev[0] : 1.f;
  const int F = L - P;
  const int slices = cin / 8;
  const size_t total = (size_t)B * L * H * W * slices;
  const size_t plane = (size_t)H * W * F;
  for (size_t gid = blockIdx.x * (size_t)blockDim.x + threadIdx.x; gid < total;
       gid += (size_t)gridDim.x * blockDim.x) {
    const int sl = (int)(gid % slices);
    size_t pix = gid / slices;                       // internal layout [B][L][H][W]
    const int wc = (int)(pix % W);
    size_t r = pix / W;
    const int h = (int)(r % H);
    r /= H;
    const int l = (int)(r % L);
    const int b = (int)(r / L);
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
    // forward: out[o] += w[tap] * in[o + tap - 1]  ->  in[i] receives from o = i - tap + 1
    for (int td = 0; td < 3; ++td) {
      const int oh = h - td + 1;
      if (oh < 0 || oh >= H) continue;
      for (int th = 0; th < 3; ++th) {
        const int ow = wc - th + 1;
        if (ow < 0 || ow >= W) continue;
        for (int tw = 0; tw < 3; ++tw) {
          const int ol = l - tw + 1;
          if (ol < P || ol >= L) continue;
          const int tap = (td * 3 + th) * 3 + tw;
          float d[COUT];
#pragma unroll
          for (int co = 0; co < COUT; ++co)
            d[co] = deps[((size_t)b * COUT + co) * plane + ((size_t)oh * W + ow) * F + (ol - P)] * scale;
          const float* wp = ws + ((size_t)tap * cin + sl * 8) * COUT;
#pragma unroll
          for (int e = 0; e < 8; ++e)
#pragma unroll
            for (int co = 0; co < COUT; ++co) acc[e] = fmaf(wp[e * COUT + co], d[co], acc[e]);
        }
      }
    }
    float4* op = reinterpret_cast<float4*>(dact + pix * cin + sl * 8);
    op[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    op[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  }
}

template <int COUT>
__global__ void __launch_bounds__(256)
final_conv_wgrad_kernel(const float* __restrict__ deps, const float* __restrict__ scale_dev,
                        const __half* __restrict__ act, int ald, int alo, float* __restrict__ dw,
                        float* __restrict__ db, int B, int H, int W, int L, int P, int cin, int pix_per_cta) {
  constexpr int MAXP = 8;                      // (tap, ci) pairs per thread: 27*cin <= 2048
  const float scale = scale_dev ? scale_dev[0] : 1.f;
  const int F = L - P;
  const int npairs = 27 * cin;
  const size_t total = (size_t)B * H * W * F;
  const size_t plane = (size_t)H * W * F;
  float acc[MAXP][COUT];
  float bacc[COUT];
#pragma unroll
  for (int k = 0; k < MAXP; ++k)
#pragma unroll
    for (int co = 0; co < COUT; ++co) acc[k][co] = 0.f;
#pragma unroll
  for (int co = 0; co < COUT; ++co) bacc[co] = 0.f;
  const size_t p0 = (size_t)blockIdx.x * pix_per_cta;
  const size_t p1 = p0 + pix_per_cta < total ? p0 + pix_per_cta : total;
  // per-thread (tap, ci) constants hoisted out of the pixel walk (the divisions per pixel and pair made
  // this kernel instruction-bound: 0.6 ms for 0.3 GFLOP)
  int kdh[MAXP], kdw[MAXP], kdl[MAXP];
  long long koff[MAXP];
  bool kok[MAXP];
#pragma unroll
  for (int k = 0; k < MAXP; ++k) {
    const int pr = threadIdx.x + k * 256;
    kok[k] = pr < npairs;
    const int tap = kok[k] ? pr / cin : 0, ci = kok[k] ? pr - tap * cin : 0;
    kdh[k] = tap / 9 - 1;
    kdw[k] = (tap / 3) % 3 - 1;
    kdl[k] = tap % 3 - 1;
    koff[k] = (((long long)kdl[k] * H + kdh[k]) * W + kdw[k]) * ald + ci;
  }
  int f = 0, wc = 0, h = 0, b = 0;
  if (p0 < p1) {
    f = (int)(p0 % F);
    size_t r = p0 / F;
    wc = (int)(r % W);
    r /= W;
    h = (int)(r % H);
    b = (int)(r / H);
  }
  for (size_t pix = p0; pix < p1; ++pix) {
    const int l = P + f;
    float d[COUT];
#pragma unroll
    for (int co = 0; co < COUT; ++co) {
      d[co] = deps[((size_t)b * COUT + co) * plane + ((size_t)h * W + wc) * F + f] * scale;
      bacc[co] += d[co];
    }
    const long long base = ((((long long)b * L + l) * H + h) * W + wc) * ald;
#pragma unroll
    for (int k = 0; k < MAXP; ++k) {
      if (!kok[k]) break;
      const int hh = h + kdh[k], ww = wc + kdw[k], ll = l + kdl[k];
      if (hh < 0 || hh >= H || ww < 0 || ww >= W || ll < 0 || ll >= L) continue;
      float a = __half2float(act[base + koff[k]]);
      if (alo > 0) a += __half2float(act[base + koff[k] + alo]);      // hi|lo pair operand: exact activation
#pragma unroll
      for (int co = 0; co < COUT; ++co) acc[k][co] = fmaf(a, d[co], acc[k][co]);
    }
    if (++f == F) {
      f = 0;
      if (++wc == W) {
        wc = 0;
        if (++h == H) { h = 0; ++b; }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < MAXP; ++k) {
    const int pr = threadIdx.x + k * 256;
    if (pr >= npairs) break;
    const int tap = pr / cin, ci = pr - tap * cin;
#pragma unroll
    for (int co = 0; co < COUT; ++co) atomicAdd(dw + ((size_t)co * cin + ci) * 27 + tap, acc[k][co]);
  }
  if (threadIdx.x == 0) {
#pragma unroll
    for (int co = 0; co < COUT; ++co) atomicAdd(db + co, bacc[co]);
  }
}

// d_eps * scale -> columns 0 .. cout-1 of the fp16 dOut operand [B][L][H][W][32] of the plane weight-gradient kernel (future
// frames only; everything else in the buffer stays zero) and the bias gradient (block sums, one atomic per CTA and channel)
__global__ void __launch_bounds__(256)
pack_final_dout_kernel(const float* __restrict__ deps, const float* __restrict__ scale_dev, __half* __restrict__ out,
                       float* __restrict__ db, int B, int H, int W, int L, int P, int cout) {
  __shared__ float red[8][4];
  const float scale = scale_dev ? scale_dev[0] : 1.f;
  const int F = L - P;
  const size_t total = (size_t)B * F * H * W;
  const size_t plane = (size_t)H * W * F;
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int wc = (int)(i % W);
    size_t r = i / W;
    const int h = (int)(r % H);
    r /= H;
    const int f = (int)(r % F);
    const int b = (int)(r / F);
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    for (int co = 0; co < cout; ++co) {
      v[co] = deps[((size_t)b * cout + co) * plane + ((size_t)h * W + wc) * F + f] * scale;
      s[co] += v[co];
    }
    const __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t*>(&h0);
    u.y = *reinterpret_cast<const uint32_t*>(&h1);
    const size_t pix = (((size_t)b * L + P + f) * H + h) * W + wc;
    *reinterpret_cast<uint2*>(out + pix * 32) = u;
  }
#pragma unroll
  for (int co = 0; co < 4; ++co) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[co] += __shfl_xor_sync(0xffffffffu, s[co], o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
#pragma unroll
    for (int co = 0; co < 4; ++co) red[warp][co] = s[co];
  }
  __syncthreads();
  if (threadIdx.x < cout) {
    float a = 0.f;
    for (int k = 0; k < 8; ++k) a += red[k][threadIdx.x];
    atomicAdd(db + threadIdx.x, a);
  }
}

constexpr int FCB_MAX_CIN = 256;   // the data-gradient kernel keeps all 27 * cin * cout weights in shared memory

// dout16 != nullptr: the weight gradient is left to the caller's launch over dout16 (filled here, with the bias
// gradient); nullptr: the SIMT weight-gradient kernel (cin <= 64)
int final_conv_backward_enqueue(const float* deps, const float* scale_dev, const __half* act, int act_ld, int act_lo,
                                const float* w, float* dact, float* dw, float* db, int B, int H, int W,
                                int L, int P, int cin, int cout, __half* dout16, cudaStream_t st) {
  const int ald = act_ld > 0 ? act_ld : cin;
  CM_CHECK(cout >= 1 && cout <= 4, "final conv supports 1..4 output channels (got %d)", cout);
  CM_CHECK(cin % 32 == 0 && cin <= FCB_MAX_CIN && (dout16 || 27 * cin <= 2048),
           "final conv backward: cin %d must be a multiple of 32, <= 64 (<= %d with the packed weight gradient)", cin,
           FCB_MAX_CIN);
  const size_t total = (size_t)B * L * H * W * (cin / 8);
  const int blocks = grid_for(total, 256, 148 * 16);
  const size_t smem = (size_t)27 * cin * cout * sizeof(float);
  const size_t opix = (size_t)B * H * W * (L - P);
  const int ppc = (int)((opix + 591) / 592);
  const int wblocks = (int)((opix + ppc - 1) / ppc);
#define CM_FB(CO)                                                                                   \
  case CO:                                                                                          \
    final_conv_dact_kernel<CO><<<blocks, 256, smem, st>>>(deps, scale_dev, w, dact, B, H, W, L, P, cin); \
    if (dout16)                                                                                     \
      pack_final_dout_kernel<<<592, 256, 0, st>>>(deps, scale_dev, dout16, db, B, H, W, L, P, cout); \
    else                                                                                            \
      final_conv_wgrad_kernel<CO><<<wblocks, 256, 0, st>>>(deps, scale_dev, act, ald, act_lo, dw, db, B, H, W, L, P, cin, ppc); \
    break;
  switch (cout) { CM_FB(1) CM_FB(2) CM_FB(3) CM_FB(4) }
#undef CM_FB
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// first conv weight / bias gradient (unet.py:32): dW[co][k] = sum_pixels dOut[p][co] * col[p][k],
// k = ci*27 + tap.  Persistent CTAs walk chunks of 256 pixels: every thread expands ITS pixel
// into an im2col row (84 floats, from the fp32 API tensors) and copies its dOut row to shared
// memory; then warp g accumulates k-group g (12 k's = three 128-bit broadcast loads per pixel)
// with lane = output channel.  Partial sums stay in registers across chunks; one atomicAdd per
// (CTA, output) at the end.
// =============================================================================================
constexpr int FW_PIX = 192;     // pixels per chunk
constexpr int FW_THREADS = 288; // 9 warps x 12 k's
constexpr int FW_KP = 108;      // padded K = 27 * 4 input channels

__global__ void __launch_bounds__(FW_THREADS)
first_conv_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ past,
                        const float* __restrict__ dout, float* __restrict__ dw, float* __restrict__ db,
                        int B, int H, int W, int P, int F, int cin, int cout, int nchunks) {
  extern __shared__ float sm[];
  float* col = sm;                       // [FW_PIX][FW_KP]
  float* dsm = sm + FW_PIX * FW_KP;      // [FW_PIX][cout + 1]
  const int L = P + F, K = 27 * cin;
  const size_t total = (size_t)B * L * H * W;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ldd = cout + 1;
  // accumulators: this warp's 12 k's x (cout/32) channel groups of this lane (cout <= 64)
  float acc[2][12];
  float bacc[2] = {0.f, 0.f};
#pragma unroll
  for (int g = 0; g < 2; ++g)
#pragma unroll
    for (int j = 0; j < 12; ++j) acc[g][j] = 0.f;
  const int ngrp = cout / 32;
  for (int chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
    const size_t pix = (size_t)chunk * FW_PIX + tid;
    __syncthreads();                     // previous chunk fully consumed
    float* cr = col + tid * FW_KP;
    if (tid >= FW_PIX) {
      // warps beyond the chunk's pixels only take part in the accumulation
    } else if (pix < total) {
      const int wc = (int)(pix % W);
      size_t r = pix / W;
      const int h = (int)(r % H);
      r /= H;
      const int l = (int)(r % L);
      const int b = (int)(r / L);
      for (int k = 0; k < K; ++k) {
        const int ci = k / 27, tap = k - ci * 27;
        const int hh = h + tap / 9 - 1, ww = wc + (tap / 3) % 3 - 1, ll = l + tap % 3 - 1;
        float v = 0.f;
        if (hh >= 0 && hh < H && ww >= 0 && ww < W && ll >= 0 && ll < L) {
          const size_t pl = ((size_t)(b * cin + ci) * H + hh) * W + ww;
          v = (ll < P) ? past[pl * P + ll] : x[pl * F + (ll - P)];
        }
        cr[k] = v;
      }
      for (int k = K; k < FW_KP; ++k) cr[k] = 0.f;
      for (int c = 0; c < cout; ++c) dsm[tid * ldd + c] = 0.f;
    } else {
      for (int k = 0; k < FW_KP; ++k) cr[k] = 0.f;
      for (int c = 0; c < cout; ++c) dsm[tid * ldd + c] = 0.f;
    }
    __syncthreads();
    // coalesced copy of the chunk's dOut rows: [FW_PIX][cout] contiguous in global memory
    {
      const size_t base = (size_t)chunk * FW_PIX;
      const size_t nvalid = total - base < (size_t)FW_PIX ? total - base : (size_t)FW_PIX;
      for (size_t i = tid; i < nvalid * cout; i += FW_THREADS) {
        const int pp = (int)(i / cout), c = (int)(i - (size_t)pp * cout);
        dsm[pp * ldd + c] = dout[base * cout + i];
      }
    }
    __syncthreads();
#pragma unroll 2
    for (int pp = 0; pp < FW_PIX; ++pp) {
      const float4* c4 = reinterpret_cast<const float4*>(col + pp * FW_KP + warp * 12);
      const float4 a0 = c4[0], a1 = c4[1], a2 = c4[2];
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        if (g >= ngrp) break;
        const float d = dsm[pp * ldd + g * 32 + lane];
        acc[g][0] = fmaf(a0.x, d, acc[g][0]); acc[g][1] = fmaf(a0.y, d, acc[g][1]);
        acc[g][2] = fmaf(a0.z, d, acc[g][2]); acc[g][3] = fmaf(a0.w, d, acc[g][3]);
        acc[g][4] = fmaf(a1.x, d, acc[g][4]); acc[g][5] = fmaf(a1.y, d, acc[g][5]);
        acc[g][6] = fmaf(a1.z, d, acc[g][6]); acc[g][7] = fmaf(a1.w, d, acc[g][7]);
        acc[g][8] = fmaf(a2.x, d, acc[g][8]); acc[g][9] = fmaf(a2.y, d, acc[g][9]);
        acc[g][10] = fmaf(a2.z, d, acc[g][10]); acc[g][11] = fmaf(a2.w, d, acc[g][11]);
        if (warp == 8) bacc[g] += d;
      }
    }
  }
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    if (g >= ngrp) break;
    const int co = g * 32 + lane;
#pragma unroll
    for (int j = 0; j < 12; ++j) {
      const int k = warp * 12 + j;
      if (k < K) atomicAdd(dw + (size_t)co * K + k, acc[g][j]);
    }
    if (warp == 8) atomicAdd(db + co, bacc[g]);
  }
}

int first_conv_wgrad_enqueue(const float* x, const float* past, const float* dout, float* dw, float* db,
                             int B, int H, int W, int P, int F, int cin, int cout, cudaStream_t st) {
  CM_CHECK(cout == 32 || cout == 64, "first conv wgrad: cout must be 32 or 64 (got %d)", cout);
  CM_CHECK(27 * cin <= FW_KP, "first conv wgrad: at most 4 input channels (got %d)", cin);
  const size_t total = (size_t)B * (P + F) * H * W;
  const int nchunks = (int)((total + FW_PIX - 1) / FW_PIX);
  const int blocks = nchunks < 296 ? nchunks : 296;
  const size_t smem = ((size_t)FW_PIX * FW_KP + (size_t)FW_PIX * (cout + 1)) * sizeof(float);
  static bool attr = false;
  if (!attr) {
    CM_CUDA(cudaFuncSetAttribute(first_conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 180 * 1024));
    attr = true;
  }
  first_conv_wgrad_kernel<<<blocks, FW_THREADS, smem, st>>>(x, past, dout, dw, db, B, H, W, P, F, cin, cout, nchunks);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// =============================================================================================
// tiny helpers for the time-embedding MLP backward
// =============================================================================================
__global__ void small_gemm_kernel(int M, int N, int K, const float* __restrict__ A, int sam, int sak,
                                  const float* __restrict__ Bm, int sbk, int sbn, float* __restrict__ Cm,
                                  int ldc, int accumulate) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * N) return;
  const int m = idx / N, n = idx - m * N;
  const float* ap = A + (size_t)m * sam;
  const float* bp = Bm + (size_t)n * sbn;
  // 8 independent loads in flight per operand and four accumulators (merged in a fixed order): the
  // dependent one-load-per-FMA loop exposed one L2 round trip per k
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int k = 0;
  for (; k + 8 <= K; k += 8) {
    float av[8], bv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      av[j] = ap[(size_t)(k + j) * sak];
      bv[j] = bp[(size_t)(k + j) * sbk];
    }
    a0 = fmaf(av[0], bv[0], a0); a1 = fmaf(av[1], bv[1], a1); a2 = fmaf(av[2], bv[2], a2); a3 = fmaf(av[3], bv[3], a3);
    a0 = fmaf(av[4], bv[4], a0); a1 = fmaf(av[5], bv[5], a1); a2 = fmaf(av[6], bv[6], a2); a3 = fmaf(av[7], bv[7], a3);
  }
  for (; k < K; ++k) a0 = fmaf(ap[(size_t)k * sak], bp[(size_t)k * sbk], a0);
  const float a = (a0 + a1) + (a2 + a3);
  float* o = Cm + (size_t)m * ldc + n;
  *o = accumulate ? *o + a : a;
}
int small_gemm_enqueue(int M, int N, int K, const float* A, int sam, int sak, const float* Bm, int sbk,
                       int sbn, float* Cm, int ldc, int accumulate, cudaStream_t st) {
  small_gemm_kernel<<<(M * N + 127) / 128, 128, 0, st>>>(M, N, K, A, sam, sak, Bm, sbk, sbn, Cm, ldc,
                                                         accumulate);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// Every block's dense_1 (layers.py:35,62) backward in two launches instead of three per block.
//   wgrad: CTA = one column j of dtemb (= output channel c of block k): dW_k[c][e] = sum_b dtemb[b][j] * s2[b][e],
//          db_k[c] = sum_b dtemb[b][j]                      (s2 = SiLU(h2), the dense_1 input)
//   dgrad: CTA = one sample: ds2[b][e] = sum_j dtemb[b][j] * W_cat[j][e]
__global__ void __launch_bounds__(128)
temb_dense_wgrad_kernel(const float* __restrict__ dtemb, int ld, int B, const float* __restrict__ s2, int E,
                        const int* __restrict__ couts, const int* __restrict__ offs, int nblocks,
                        float* __restrict__ grads, const long long* __restrict__ goff_w,
                        const long long* __restrict__ goff_b) {
  const int j = blockIdx.y;
  int k = 0;
  while (k + 1 < nblocks && offs[k + 1] <= j) ++k;
  const int c = j - offs[k];
  if (c >= couts[k]) return;
  const int e = blockIdx.x * 128 + threadIdx.x;
  float a0 = 0.f, a1 = 0.f, bs0 = 0.f, bs1 = 0.f;
  int b = 0;
  if (e < E) {
    for (; b + 4 <= B; b += 4) {
      const float d0 = dtemb[(size_t)b * ld + j], d1 = dtemb[(size_t)(b + 1) * ld + j];
      const float d2 = dtemb[(size_t)(b + 2) * ld + j], d3 = dtemb[(size_t)(b + 3) * ld + j];
      const float s0 = s2[(size_t)b * E + e], s1 = s2[(size_t)(b + 1) * E + e];
      const float s2v = s2[(size_t)(b + 2) * E + e], s3 = s2[(size_t)(b + 3) * E + e];
      a0 = fmaf(d0, s0, a0); a1 = fmaf(d1, s1, a1); a0 = fmaf(d2, s2v, a0); a1 = fmaf(d3, s3, a1);
      bs0 += d0 + d2; bs1 += d1 + d3;
    }
    for (; b < B; ++b) {
      const float d0 = dtemb[(size_t)b * ld + j];
      a0 = fmaf(d0, s2[(size_t)b * E + e], a0);
      bs0 += d0;
    }
    grads[goff_w[k] + (long long)c * E + e] = a0 + a1;
    if (e == 0) grads[goff_b[k] + c] = bs0 + bs1;
  }
}
// blockDim = G * E: group gq walks the dense blocks k = gq, gq + G, ... ; the G partial sums are added in
// group order (fixed) through shared memory
__global__ void temb_dense_dgrad_kernel(const float* __restrict__ dtemb, int ld, const float* const* __restrict__ wd,
                                        const int* __restrict__ couts, const int* __restrict__ offs, int nblocks,
                                        int E, int G, float* __restrict__ ds2) {
  extern __shared__ float drow[];   // [ld] | [G][E]
  float* part = drow + ld;
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < ld; i += blockDim.x) drow[i] = dtemb[(size_t)b * ld + i];
  __syncthreads();
  const int gq = threadIdx.x / E, e = threadIdx.x - gq * E;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  for (int k = gq; k < nblocks; k += G) {
    const float* w = wd[k] + e;
    const float* d = drow + offs[k];
    const int co = couts[k];
    int c = 0;
    for (; c + 4 <= co; c += 4) {
      a0 = fmaf(d[c], w[(size_t)c * E], a0);
      a1 = fmaf(d[c + 1], w[(size_t)(c + 1) * E], a1);
      a2 = fmaf(d[c + 2], w[(size_t)(c + 2) * E], a2);
      a3 = fmaf(d[c + 3], w[(size_t)(c + 3) * E], a3);
    }
    for (; c < co; ++c) a0 = fmaf(d[c], w[(size_t)c * E], a0);
  }
  part[gq * E + e] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  if (gq == 0) {
    float a = 0.f;
    for (int q = 0; q < G; ++q) a += part[q * E + e];
    ds2[(size_t)b * E + e] = a;
  }
}
int temb_dense_backward_enqueue(const float* dtemb, int ld, int B, const float* s2, int E, const float* const* wd,
                                const int* couts, const int* offs, int nblocks, float* grads,
                                const long long* goff_w, const long long* goff_b, float* ds2, cudaStream_t st) {
  CM_CHECK(E <= 1024, "time-embedding width %d > 1024 unsupported", E);
  temb_dense_wgrad_kernel<<<dim3((E + 127) / 128, ld), 128, 0, st>>>(dtemb, ld, B, s2, E, couts, offs, nblocks, grads,
                                                                    goff_w, goff_b);
  int G = 1024 / E;
  if (G > 8) G = 8;
  if (G > nblocks) G = nblocks;
  if (G < 1) G = 1;
  temb_dense_dgrad_kernel<<<B, G * E, (size_t)(ld + G * E) * sizeof(float), st>>>(dtemb, ld, wd, couts, offs, nblocks,
                                                                                  E, G, ds2);
  CM_CUDA(cudaGetLastError());
  return 0;
}

__global__ void silu_backward_kernel(const float* __restrict__ pre, const float* __restrict__ dpost,
                                     float* __restrict__ dpre, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    dpre[i] = dpost[i] * silu_grad(pre[i]);
}
int silu_backward_enqueue(const float* pre, const float* dpost, float* dpre, size_t n, cudaStream_t st) {
  silu_backward_kernel<<<grid_for(n, 256, 1024), 256, 0, st>>>(pre, dpost, dpre, n);
  CM_CUDA(cudaGetLastError());
  return 0;
}
__global__ void silu_forward_kernel(const float* __restrict__ x, float* __restrict__ y, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    y[i] = silu_f(x[i]);
}
int silu_forward_enqueue(const float* x, float* y, size_t n, cudaStream_t st) {
  silu_forward_kernel<<<grid_for(n, 256, 1024), 256, 0, st>>>(x, y, n);
  CM_CUDA(cudaGetLastError());
  return 0;
}
__global__ void scale_inplace_kernel(float* __restrict__ x, size_t n, const float* __restrict__ f) {
  const float s = *f;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    x[i] *= s;
}
int scale_inplace_enqueue(float* x, size_t n, const float* factor_dev, cudaStream_t st) {
  scale_inplace_kernel<<<grid_for(n, 256, 2048), 256, 0, st>>>(x, n, factor_dev);
  CM_CUDA(cudaGetLastError());
  return 0;
}

int temb_backward_enqueue(const TembBwdParams& p, float* grads, cudaStream_t st) {
  const int B = p.B, E = p.E;
  const size_t nE = (size_t)B * E;
  if (int e = silu_forward_enqueue(p.h1, p.s1, nE, st)) return e;
  if (int e = silu_forward_enqueue(p.h2, p.s2, nE, st)) return e;
  // (dense_1.bias gradient == the batch sum of dtemb; the conv_1 bias gradient is the same sum)
  if (int e = temb_dense_backward_enqueue(p.dtemb, p.ld, B, p.s2, E, p.wd, p.couts, p.offs, p.nblocks, grads, p.goff_w,
                                          p.goff_b, p.ds2, st))
    return e;
  if (int e = silu_backward_enqueue(p.h2, p.ds2, p.dh2, nE, st)) return e;
  if (int e = rowsum_enqueue(p.dh2, p.db2, B, E, E, 0, st)) return e;
  if (int e = small_gemm_enqueue(E, E, B, p.dh2, 1, E, p.s1, E, 1, p.dw2, E, 0, st)) return e;
  if (int e = small_gemm_enqueue(B, E, E, p.dh2, E, 1, p.w2, E, 1, p.ds1, E, 0, st)) return e;
  if (int e = silu_backward_enqueue(p.h1, p.ds1, p.dh1, nE, st)) return e;
  if (int e = rowsum_enqueue(p.dh1, p.db1, B, E, E, 0, st)) return e;
  return small_gemm_enqueue(E, p.base, B, p.dh1, 1, E, p.e, p.base, 1, p.dw1, p.base, 0, st);
}

int backward_init() {
  static bool done = false;
  if (done) return 0;
  CM_CUDA(cudaFuncSetAttribute(attn_core_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               227 * 1024));
  constexpr int fcb_smem = 27 * FCB_MAX_CIN * 4 * sizeof(float);
  CM_CUDA(cudaFuncSetAttribute(final_conv_dact_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, fcb_smem));
  CM_CUDA(cudaFuncSetAttribute(final_conv_dact_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, fcb_smem));
  CM_CUDA(cudaFuncSetAttribute(final_conv_dact_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, fcb_smem));
  CM_CUDA(cudaFuncSetAttribute(final_conv_dact_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, fcb_smem));
  if (int rc = wgrad_init()) return rc;
  done = true;
  return 0;
}

}  // namespace cm
