// Library-level C ABI: error reporting, device error flag, op-level entry points used by the
// unit tests (each wraps one kernel of the hot path; they allocate temporaries and synchronise,
// the model-level calls in unet.cu do not).
#include <stdlib.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/crowdmod_b200.h"
#include "backward.cuh"
#include "wgrad_plane.cuh"
#include "conv_plane.cuh"
#include "conv_res32.cuh"
#include "conv_umma.cuh"
#include "kernels.cuh"
#include "wgrad_umma.cuh"

namespace cm {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* get_error() { return g_err.c_str(); }

bool pdl_enabled() {
  // measured on B200 (ATC B=64, graph replay): 1.296 ms/step with PDL vs 1.269 without -> opt-in only
  static const bool on = getenv("CM_PDL") != nullptr;
  return on;
}

static int* g_flag = nullptr;
int* device_error_flag() {
  static std::once_flag once;
  std::call_once(once, [] {
    if (cudaMalloc(&g_flag, sizeof(int)) == cudaSuccess) cudaMemset(g_flag, 0, sizeof(int));
    else g_flag = nullptr;
  });
  return g_flag;
}

}  // namespace cm

using namespace cm;

extern "C" {

int cm_version(void) { return 100; }
const char* cm_last_error(void) { return get_error(); }

int cm_device_error(void) {
  int* f = device_error_flag();
  if (!f) return -1;
  int v = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return -2;
  if (cudaMemcpy(&v, f, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -3;
  cudaMemset(f, 0, sizeof(int));
  return v;
}

int cm_op_conv3d(int mode, const void* act16, int B, int D, int H, int W, int cin,
                 const void* extra16, int cin_extra, const float* w, const float* wx,
                 const float* bias, int cout, int terms, const float* resid, float* out32,
                 void* out16, int impl, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = kernels_init()) return e;
  const size_t ktot = conv_packed_k(mode, cin, cin_extra);
  __half* wp = nullptr;
  CM_CUDA(cudaMalloc(&wp, (size_t)terms * cout * ktot * sizeof(__half)));
  int rc = 0;
  if (mode == 2) rc = pack_upsample_weights(w, wp, cout, cin, terms, 0, st);
  else rc = pack_conv_weights(w, wx, wp, cout, cin, cin_extra, mode == 3 ? 1 : 27, terms, 0, st);
  ConvLaunch L;
  if (!rc && impl == 3) {
    // weights-resident 32 -> 32 kernel (conv_res32.cuh).  Fails if the shape is not covered.
    Res32Launch R;
    rc = (mode == 0) ? res32_prepare(&R, static_cast<const __half*>(act16), B, D, H, W, cin,
                                     static_cast<const __half*>(extra16), cin_extra, wp, cout, terms)
                     : 2;
    if (!rc && !R.ok) {
      set_error("weights-resident conv does not cover this shape");
      rc = 2;
    }
    if (!rc) {
      R.p.bias = bias;
      R.p.resid = resid;
      R.p.out32 = out32;
      R.p.out16 = static_cast<__half*>(out16);
      rc = res32_enqueue(R, st);
      if (const char* e = getenv("CM_DBG_REPS")) {
        const int reps = atoi(e);
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaStreamSynchronize(st);
        cudaEventRecord(a, st);
        for (int i = 0; i < reps && !rc; ++i) rc = res32_enqueue(R, st);
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        fprintf(stderr, "CM_DBG res32 B=%d D=%d H=%d W=%d cin=%d+%d cout=%d HB=%d units=%d stages=%d grid=%d smem=%zu: %.2f us/launch (%.1f TF/s)\n",
                B, D, H, W, cin, cin_extra, cout, R.p.HB, R.p.n_units, R.p.stages, R.grid.x, R.smem, ms * 1e3f / reps,
                R.flops / (ms * 1e-3 / reps) * 1e-12);
        cudaEventDestroy(a);
        cudaEventDestroy(b);
      }
    }
    if (!rc && getenv("CM_PLANE_TRACE")) {   // bring-up: event trace of CTA 0 (producer / MMA issuer / drain warp / store warp)
      const size_t n = (size_t)4 * PL_TRACE_CAP * 2;
      long long* tr = nullptr;
      cudaMalloc(&tr, n * 8);
      cudaMemset(tr, 0, n * 8);
      R.p.trace = tr;
      unsigned long long* ct = nullptr;
      cudaMalloc(&ct, (size_t)R.grid.x * 16);
      cudaMemset(ct, 0, (size_t)R.grid.x * 16);
      R.p.cta_times = ct;
      cudaStreamSynchronize(st);
      rc = res32_enqueue(R, st);
      cudaStreamSynchronize(st);
      {
        std::vector<unsigned long long> hc((size_t)R.grid.x * 2);
        cudaMemcpy(hc.data(), ct, hc.size() * 8, cudaMemcpyDeviceToHost);
        unsigned long long s0 = ~0ull, s1 = 0, e0 = ~0ull, e1 = 0, dmin = ~0ull, dmax = 0;
        for (unsigned i = 0; i < R.grid.x; ++i) {
          const unsigned long long a = hc[2 * i], b = hc[2 * i + 1];
          if (a < s0) s0 = a;
          if (a > s1) s1 = a;
          if (b < e0) e0 = b;
          if (b > e1) e1 = b;
          if (b - a < dmin) dmin = b - a;
          if (b - a > dmax) dmax = b - a;
        }
        fprintf(stderr, "CTA_TIMES ns: first start 0, last start %llu, first end %llu, last end %llu; CTA duration min %llu max %llu\n",
                s1 - s0, e0 - s0, e1 - s0, dmin, dmax);
      }
      R.p.cta_times = nullptr;
      cudaFree(ct);
      std::vector<long long> h(n);
      cudaMemcpy(h.data(), tr, n * 8, cudaMemcpyDeviceToHost);
      long long t0 = 0;
      for (size_t i = 0; i < n; i += 2)
        if (h[i] && (t0 == 0 || h[i + 1] < t0)) t0 = h[i + 1];
      static const char* role[4] = {"prod", "mma", "drain", "store"};
      for (int r = 0; r < 4; ++r) {
        long long prev = t0;
        for (int i = 0; i < PL_TRACE_CAP; ++i) {
          const long long code = h[((size_t)r * PL_TRACE_CAP + i) * 2], t = h[((size_t)r * PL_TRACE_CAP + i) * 2 + 1];
          if (!code) break;
          fprintf(stderr, "PL_TRACE %s i=%d code=%lld t=%lld dt=%lld\n", role[r], i, code, t - t0, t - prev);
          prev = t;
        }
      }
      R.p.trace = nullptr;
      cudaFree(tr);
    }
    cudaError_t se3 = cudaStreamSynchronize(st);
    cudaFree(wp);
    if (rc) return rc;
    CM_CUDA(se3);
    return 0;
  }
  if (!rc && impl == 2) {
    // plane-tile kernel (conv_plane.cuh); mode 0 only.  Fails if the geometry is not covered.
    PlaneLaunch PLn;
    rc = (mode == 0) ? plane_prepare(&PLn, static_cast<const __half*>(act16), B, D, H, W, cin,
                                     static_cast<const __half*>(extra16), cin_extra, wp, cout, terms)
                     : 2;
    if (!rc && !PLn.ok) {
      set_error("plane-tile conv does not cover this geometry");
      rc = 2;
    }
    if (!rc) {
      PLn.p.bias = bias;
      PLn.p.resid = resid;
      PLn.p.out32 = out32;
      PLn.p.out16 = static_cast<__half*>(out16);
      rc = plane_enqueue(PLn, st);
      if (const char* e = getenv("CM_DBG_REPS")) {
        const int reps = atoi(e);
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaStreamSynchronize(st);
        cudaEventRecord(a, st);
        for (int i = 0; i < reps && !rc; ++i) rc = plane_enqueue(PLn, st);
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        fprintf(stderr, "CM_DBG plane B=%d D=%d H=%d W=%d cin=%d+%d cout=%d bn=%d bk=%d R=%d HB=%d tiles=%d units=%d stages=%d grid=%d: %.2f us/launch (%.1f TF/s)\n",
                B, D, H, W, cin, cin_extra, cout, PLn.bn, PLn.bk, PLn.p.R, PLn.p.HB, PLn.p.ntiles, PLn.p.n_units,
                PLn.p.stages, PLn.grid.x, ms * 1e3f / reps, PLn.flops / (ms * 1e-3 / reps) * 1e-12);
        cudaEventDestroy(a);
        cudaEventDestroy(b);
      }
      if (!rc && getenv("CM_PLANE_TRACE")) {   // bring-up: event trace of CTA 0 (producer / MMA issuer / epilogue warp 2)
        const size_t n = (size_t)3 * PL_TRACE_CAP * 2;
        long long* tr = nullptr;
        cudaMalloc(&tr, n * 8);
        cudaMemset(tr, 0, n * 8);
        PLn.p.trace = tr;
        cudaStreamSynchronize(st);
        rc = plane_enqueue(PLn, st);
        cudaStreamSynchronize(st);
        std::vector<long long> h(n);
        cudaMemcpy(h.data(), tr, n * 8, cudaMemcpyDeviceToHost);
        long long t0 = 0;
        for (size_t i = 0; i < n; i += 2)
          if (h[i] && (t0 == 0 || h[i + 1] < t0)) t0 = h[i + 1];
        static const char* role[3] = {"prod", "mma", "epi"};
        for (int r = 0; r < 3; ++r) {
          long long prev = t0;
          for (int i = 0; i < PL_TRACE_CAP; ++i) {
            const long long code = h[((size_t)r * PL_TRACE_CAP + i) * 2], t = h[((size_t)r * PL_TRACE_CAP + i) * 2 + 1];
            if (!code) break;
            fprintf(stderr, "PL_TRACE %s i=%d code=%lld t=%lld dt=%lld\n", role[r], i, code, t - t0, t - prev);
            prev = t;
          }
        }
        PLn.p.trace = nullptr;
        cudaFree(tr);
      }
    }
    cudaError_t se2 = cudaStreamSynchronize(st);
    cudaFree(wp);
    if (rc) return rc;
    CM_CUDA(se2);
    return 0;
  }
  if (!rc) rc = conv_prepare(&L, mode, static_cast<const __half*>(act16), B, D, H, W, cin,
                             static_cast<const __half*>(extra16), cin_extra, wp, cout, terms);
  if (!rc) {
    L.p.bias = bias;
    L.p.resid = resid;
    L.p.out32 = out32;
    L.p.out16 = static_cast<__half*>(out16);
    if (impl == 0) {
      rc = conv_enqueue(L, st);
      if (getenv("CM_DBG_TRACE")) {
        unsigned long long* tr = nullptr;
        cudaMalloc(&tr, 512 * 8);
        cudaMemset(tr, 0, 512 * 8);
        L.p.trace = tr;
        cudaStreamSynchronize(st);
        conv_enqueue(L, st);
        cudaStreamSynchronize(st);
        unsigned long long h[512];
        cudaMemcpy(h, tr, sizeof(h), cudaMemcpyDeviceToHost);
        const unsigned long long t0 = h[0];
        fprintf(stderr, "CM_TRACE start=0 setup_done=%lld tmem_full=%lld epi_done=%lld end=%lld\n",
                (long long)(h[4] - t0), (long long)(h[1] - t0), (long long)(h[2] - t0), (long long)(h[3] - t0));
        for (int kb = 0; kb < 120 && h[8 + kb * 4]; ++kb)
          fprintf(stderr, "CM_TRACE kb=%d prod_wait_done=%lld prod_issued=%lld mma_wait_done=%lld mma_committed=%lld\n", kb,
                  (long long)(h[8 + kb * 4] - t0), (long long)(h[8 + kb * 4 + 1] - t0),
                  (long long)(h[8 + kb * 4 + 2] - t0), (long long)(h[8 + kb * 4 + 3] - t0));
        L.p.trace = nullptr;
        cudaFree(tr);
      }
      if (const char* e = getenv("CM_DBG_REPS")) {   // bring-up timing: avg device time of `reps` launches
        const int reps = atoi(e);
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaStreamSynchronize(st);
        cudaEventRecord(a, st);
        for (int i = 0; i < reps && !rc; ++i) rc = conv_enqueue(L, st);
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        fprintf(stderr, "CM_DBG conv mode=%d M=%d cin=%d cout=%d bn=%d bk=%d stages=%d grid=%d,%d,%d dbg=%d: %.2f us/launch\n",
                mode, L.p.M, cin, cout, L.bn, L.bk, L.p.stages, L.grid.x, L.grid.y, L.grid.z, L.p.dbg,
                ms * 1e3f / reps);
        cudaEventDestroy(a);
        cudaEventDestroy(b);
      }
    } else rc = conv_ref_enqueue(L.p, static_cast<const __half*>(act16),
                               static_cast<const __half*>(extra16), wp, B, D, H, W, st);
  }
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(wp);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_gn_silu(const float* src0, int c0, const float* src1, int c1, const float* gamma,
                  const float* beta, int B, int pixels, float eps, int silu, void* out_norm16,
                  void* out_raw16, void* stream) {
  if (int e = kernels_init()) return e;   // the streaming kernels need their dynamic shared-memory attribute
  GnParams g{};
  g.src0 = src0; g.c0 = c0; g.src1 = src1; g.c1 = c1;
  g.gamma = gamma; g.beta = beta; g.B = B; g.pixels = pixels; g.eps = eps; g.silu = silu;
  g.out_norm = static_cast<__half*>(out_norm16);
  g.out_raw = static_cast<__half*>(out_raw16);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = nullptr;
  CM_CUDA(cudaMalloc(&partial, (size_t)B * 32 * 8 * 3 * sizeof(float)));
  const int rc = gn_silu_enqueue(g, partial, st);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(partial);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_attn_core(const float* qkv, void* ctx16, int B, int S, int C, int heads, void* stream) {
  if (int e = kernels_init()) return e;
  return attn_core_enqueue(qkv, static_cast<__half*>(ctx16), B, S, C, heads,
                           static_cast<cudaStream_t>(stream));
}

int cm_op_attn_core_backward(const float* qkv, const float* dctx, float* dqkv, int B, int S, int C, int heads,
                             void* stream) {
  if (int e = backward_init()) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (S <= 128) return attn_core_backward_enqueue(qkv, dctx, dqkv, B, S, C, heads, st);
  // the long-sequence backward reads the forward's row log-sum-exp: rerun the forward into temporaries
  if (int e = kernels_init()) return e;
  CM_CHECK(C % heads == 0, "embed dim %d / heads %d unsupported", C, heads);
  __half* ctx = nullptr;
  float* lse = nullptr;      // [B][heads][S] log-sum-exp | [B][heads][S] backward row sums
  CM_CUDA(cudaMalloc(&ctx, (size_t)B * S * C * sizeof(__half)));
  if (cudaMalloc(&lse, (size_t)2 * B * heads * S * sizeof(float)) != cudaSuccess) {
    cudaFree(ctx);
    CM_CHECK(false, "attention backward: out of device memory for the log-sum-exp");
  }
  int rc = attn_core_enqueue(qkv, ctx, B, S, C, heads, st, 1, lse);
  if (!rc) rc = attn_core_backward_enqueue(qkv, dctx, dqkv, B, S, C, heads, st, lse, lse + (size_t)B * heads * S);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(ctx);
  cudaFree(lse);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_attn_block(const float* x, const float* gamma, const float* beta, const float* w_in, const float* b_in,
                     const float* w_out, const float* b_out, float* out32, void* out16, int B, int S, int C,
                     int heads, float eps, void* stream) {
  if (int e = kernels_init()) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CM_CHECK(attn_block_supported(S, C, heads), "fused attention block: C=%d heads=%d S=%d not covered", C, heads, S);
  __half* wpk = nullptr;    // hi|lo packed rows of in_proj ([2*3C][C]) then out_proj ([2*C][C])
  CM_CUDA(cudaMalloc(&wpk, (size_t)2 * 4 * C * C * sizeof(__half)));
  int rc = pack_conv_weights(w_in, nullptr, wpk, 3 * C, C, 0, 1, 2, 0, st);
  if (!rc) rc = pack_conv_weights(w_out, nullptr, wpk + (size_t)6 * C * C, C, C, 0, 1, 2, 0, st);
  if (!rc)
    rc = attn_block_enqueue(x, gamma, beta, wpk, b_in, wpk + (size_t)6 * C * C, b_out, out32,
                            static_cast<__half*>(out16), B, S, C, heads, eps, st);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(wpk);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_first_conv(const float* x, const float* past, const float* w, const float* bias,
                     float* out, int B, int H, int W, int P, int F, int cin, int cout,
                     void* stream) {
  if (int e = kernels_init()) return e;
  return first_conv_enqueue(x, past, w, bias, out, B, H, W, P, F, cin, cout,
                            static_cast<cudaStream_t>(stream));
}

int cm_op_final_conv(const void* act16, const float* w, const float* bias, float* eps_out, int B,
                     int H, int W, int L, int P, int cin, int cout, void* stream) {
  if (int e = kernels_init()) return e;
  FinalParams f{};
  f.act = static_cast<const __half*>(act16);
  f.w = w; f.bias = bias; f.B = B; f.H = H; f.W = W; f.L = L; f.P = P; f.cin = cin; f.cout = cout;
  f.eps_out = eps_out;
  return final_conv_enqueue(f, static_cast<cudaStream_t>(stream));
}


int cm_op_conv3d_dgrad(int mode, const void* dout16, int B, int D, int H, int W, int cin,
                       const float* w, int cout, int terms, float* dx32, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = kernels_init()) return e;
  if (int e = backward_init()) return e;
  CM_CHECK(mode >= 0 && mode <= 3, "bad forward conv mode %d", mode);
  int od = D, oh = H, ow = W;   // forward output grid
  if (mode == 1) { od = (D - 1) / 2 + 1; oh = (H - 1) / 2 + 1; ow = (W - 1) / 2 + 1; }
  else if (mode == 2) { od = 2 * D; oh = 2 * H; ow = 2 * W; }
  const size_t ktot = dgrad_packed_k(mode, cout);
  __half* wp = nullptr;
  CM_CUDA(cudaMalloc(&wp, (size_t)terms * cin * ktot * sizeof(__half) + 16));
  int rc = pack_dgrad_weights(mode, w, wp, cout, cin, terms, 0, 1, st);
  ConvLaunch L;
  if (!rc) rc = conv_prepare(&L, dgrad_mode_of(mode), static_cast<const __half*>(dout16), B, od, oh, ow, cout,
                             nullptr, 0, wp, cin, terms);
  if (!rc) {
    L.p.out32 = dx32;
    rc = conv_enqueue(L, st);
  }
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(wp);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_conv3d_dgrad_f32(int mode, const float* dout32, int B, int D, int H, int W, int cin,
                           const float* w, int cout, int terms, int dup, float* dx32, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = kernels_init()) return e;
  if (int e = backward_init()) return e;
  CM_CHECK(mode >= 0 && mode <= 3, "bad forward conv mode %d", mode);
  CM_CHECK(dup == 1 || dup == 2, "dup must be 1 or 2");
  int od = D, oh = H, ow = W;   // forward output grid
  if (mode == 1) { od = (D - 1) / 2 + 1; oh = (H - 1) / 2 + 1; ow = (W - 1) / 2 + 1; }
  else if (mode == 2) { od = 2 * D; oh = 2 * H; ow = 2 * W; }
  const size_t ktot = dgrad_packed_k(mode, cout, dup);
  const size_t npix = (size_t)B * od * oh * ow;
  __half* wp = nullptr;
  __half* d16 = nullptr;
  CM_CUDA(cudaMalloc(&wp, (size_t)terms * cin * ktot * sizeof(__half) + 16));
  CM_CUDA(cudaMalloc(&d16, npix * cout * dup * sizeof(__half) + 16));
  int rc = pack_dgrad_weights(mode, w, wp, cout, cin, terms, 0, dup, st);
  if (!rc) rc = cast_colsum_enqueue(dout32, d16, dup, nullptr, 0, nullptr, 0, B, od * oh * ow, cout, st);
  ConvLaunch L;
  PlaneLaunch PLn;
  PLn.ok = false;
  if (!rc) rc = conv_prepare(&L, dgrad_mode_of(mode), d16, B, od, oh, ow, dup * cout, nullptr, 0, wp, cin, terms);
  if (!rc && mode == 0 && getenv("CM_NO_PLANE") == nullptr)
    rc = plane_prepare(&PLn, d16, B, od, oh, ow, dup * cout, nullptr, 0, wp, cin, terms);
  if (!rc) {
    if (PLn.ok) {
      PLn.p.out32 = dx32;
      rc = plane_enqueue(PLn, st);
    } else {
      L.p.out32 = dx32;
      rc = conv_enqueue(L, st);
    }
  }
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(wp);
  cudaFree(d16);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_conv3d_wgrad(int mode, const void* act16, int B, int D, int H, int W, int cin,
                       const void* extra16, int cin_extra, const void* dout16, int cout, float* dw,
                       float* dwx, int impl, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = kernels_init()) return e;
  if (int e = backward_init()) return e;
  CM_CHECK(mode >= 0 && mode <= 3, "bad forward conv mode %d", mode);
  const size_t gel = wgrad_g_elems(mode, cin, cin_extra, cout);
  float* G = nullptr;
  CM_CUDA(cudaMalloc(&G, gel * sizeof(float)));
  CM_CUDA(cudaMemsetAsync(G, 0, gel * sizeof(float), st));
  int rc = 0;
  if (impl == 0) {
    WgradLaunch L;
    rc = wgrad_prepare(&L, mode, static_cast<const __half*>(act16), B, D, H, W, cin,
                       static_cast<const __half*>(extra16), cin_extra, static_cast<const __half*>(dout16),
                       cout, G);
    if (!rc) rc = wgrad_enqueue(L, st);
    if (!rc) {
      if (const char* e = getenv("CM_DBG_REPS")) {
        const int reps = atoi(e);
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaStreamSynchronize(st);
        cudaEventRecord(a, st);
        for (int i = 0; i < reps && !rc; ++i) rc = wgrad_enqueue(L, st);
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        fprintf(stderr, "CM_DBG wgrad mode=%d M=%d cin=%d cout=%d bkc=%d bn=%d splits=%d grid=%d,%d,%d: %.2f us/launch (%.1f TF/s)\n",
                mode, L.p.M, cin, cout, L.bkc, L.bn, L.p.splits, L.grid.x, L.grid.y, L.grid.z, ms * 1e3f / reps,
                L.flops / (ms * 1e-3 / reps) * 1e-12);
        cudaEventDestroy(a);
        cudaEventDestroy(b);
        cudaMemsetAsync(G, 0, gel * sizeof(float), st);
        rc = wgrad_enqueue(L, st);
      }
    }
  } else if (impl == 2) {
    // plane / halo scheme (wgrad_plane.cuh): one launch per 32-channel chunk of the main source; the fused 1x1x1 source
    // goes through wgrad_umma_kernel in 1x1x1 mode into its rows of G
    CM_CHECK(mode == 0, "plane wgrad covers k3 s1 p1 convs (mode 0), got mode %d", mode);
    WgradPlaneLaunch PL[8];
    const int nc = cin / 32;
    CM_CHECK(nc >= 1 && nc <= 8, "plane wgrad: cin %d not covered", cin);
    for (int c = 0; c < nc && !rc; ++c) {
      rc = wgrad_plane_prepare(&PL[c], static_cast<const __half*>(act16), B, D, H, W, cin, 0, c * 32,
                               static_cast<const __half*>(dout16), 0, cout, G);
      if (!rc && !PL[c].ok) {
        cm::set_error("plane wgrad does not cover this shape");
        rc = 1;
      }
    }
    WgradLaunch XL;
    if (!rc && cin_extra)
      rc = wgrad_prepare(&XL, 3, static_cast<const __half*>(extra16), B, D, H, W, cin_extra, nullptr, 0,
                         static_cast<const __half*>(dout16), cout, G + (size_t)27 * cin * cout);
    auto run = [&]() {
      int e = 0;
      for (int c = 0; c < nc && !e; ++c) e = wgrad_plane_enqueue(PL[c], st);
      if (!e && cin_extra) e = wgrad_enqueue(XL, st);
      return e;
    };
    if (!rc) rc = run();
    if (!rc) {
      if (const char* e = getenv("CM_DBG_REPS")) {
        const int reps = atoi(e);
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaStreamSynchronize(st);
        cudaEventRecord(a, st);
        for (int i = 0; i < reps && !rc; ++i) rc = run();
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        fprintf(stderr, "CM_DBG wgrad plane B=%d D=%d H=%d W=%d cin=%d+%d cout=%d HB=%d units=%d stages=%d grid=%d: %.2f us per conv (%.1f TF/s)\n",
                B, D, H, W, cin, cin_extra, cout, PL[0].p.HB, PL[0].p.n_units, PL[0].p.stages, PL[0].grid.x, ms * 1e3f / reps,
                2.0 * B * D * H * W * cout * (27.0 * cin + cin_extra) / (ms * 1e-3 / reps) * 1e-12);
        cudaEventDestroy(a);
        cudaEventDestroy(b);
        cudaMemsetAsync(G, 0, gel * sizeof(float), st);
        rc = run();
      }
    }
  } else {
    rc = wgrad_ref_enqueue(mode, static_cast<const __half*>(act16), static_cast<const __half*>(extra16),
                           static_cast<const __half*>(dout16), G, B, D, H, W, cin, cin_extra, cout, st);
  }
  if (!rc) rc = unpack_wgrad_enqueue(mode, G, dw, dwx, cout, cin, cin_extra, 0, st);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(G);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

}  // extern "C"
