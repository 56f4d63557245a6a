// Library-level C ABI: error reporting, device error flag, op-level entry points used by the
// unit tests (each wraps one kernel of the hot path; they allocate temporaries and synchronise,
// the model-level calls in unet.cu do not).
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/crowdmod_b200.h"
#include "backward.cuh"
#include "conv_run.cuh"
#include "kernels.cuh"

namespace cm {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* get_error() { return g_err.c_str(); }

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
  ConvEpilogue e{};
  e.bias = bias;
  e.resid = resid;
  e.out32 = out32;
  e.out16 = static_cast<__half*>(out16);
  const __half* a16 = static_cast<const __half*>(act16);
  const __half* x16 = static_cast<const __half*>(extra16);
  // impl: 0 conv_umma, 2 conv_plane, 3 conv_res32 (each fails if it does not cover the conv), else the scalar reference
  const unsigned kind = impl == 0 ? CONV_UMMA : impl == 2 ? CONV_PLANE : impl == 3 ? CONV_RES32 : 0;
  if (!rc && kind) {
    ConvRun R;
    rc = conv_run_prepare(&R, kind, mode, a16, B, D, H, W, cin, x16, cin_extra, wp, cout, terms, e);
    if (!rc && !R.covered()) {
      set_error("the requested conv kernel does not cover this shape");
      rc = 2;
    }
    if (!rc) rc = conv_run_enqueue(R, st);
  } else if (!rc) {
    ConvLaunch L;
    rc = conv_prepare(&L, mode, a16, B, D, H, W, cin, x16, cin_extra, wp, cout, terms, e);
    if (!rc) rc = conv_ref_enqueue(L.p, a16, x16, wp, B, D, H, W, st);
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
  CM_CHECK(heads > 0 && C % heads == 0, "embed dim %d / heads %d unsupported", C, heads);
  if (!attn_uses_long(S, C / heads)) return attn_core_backward_enqueue(qkv, dctx, dqkv, B, S, C, heads, st);
  // the streaming backward reads the forward's row log-sum-exp: rerun the forward into temporaries
  if (int e = kernels_init()) return e;
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
  ConvEpilogue e{};
  e.out32 = dx32;
  ConvRun R;
  if (!rc) rc = conv_run_prepare(&R, CONV_UMMA, dgrad_mode_of(mode), static_cast<const __half*>(dout16), B, od, oh, ow,
                                 cout, nullptr, 0, wp, cin, terms, e);
  if (!rc) rc = conv_run_enqueue(R, st);
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
  ConvEpilogue e{};
  e.out32 = dx32;
  ConvRun R;
  if (!rc)
    rc = conv_run_prepare(&R, CONV_UMMA | CONV_PLANE, dgrad_mode_of(mode), d16, B, od, oh, ow, dup * cout, nullptr, 0,
                          wp, cin, terms, e);
  if (!rc) rc = conv_run_enqueue(R, st);
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
  if (impl == 0 || impl == 2) {
    // impl 2: the plane / halo scheme (wgrad_plane.cuh), mode 0 with 32 output channels only
    WgradRun R;
    rc = wgrad_run_prepare(&R, impl == 0 ? CONV_UMMA : CONV_PLANE, mode, static_cast<const __half*>(act16), B, D, H, W,
                           cin, static_cast<const __half*>(extra16), cin_extra, static_cast<const __half*>(dout16),
                           cout, G);
    if (!rc && R.launches() == 0) {
      cm::set_error("plane wgrad does not cover this shape");
      rc = 1;
    }
    if (!rc) rc = wgrad_run_enqueue(R, st);
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

// ---- fp32 kernels of the training backward (backward.cu), one enqueue function each ----

int cm_op_gn_backward(const float* src0, int c0, const float* src1, int c1, const float* gamma, const float* beta,
                      const float* stats, const float* dnorm, const float* draw, const float* drop_scale, int drop_ld,
                      int B, int pixels, int silu, float* dsrc0, int init0, float* dsrc1, int init1, float* dgamma,
                      float* dbeta, int params_all, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CM_CHECK(B > 0 && pixels > 0, "GroupNorm backward: empty input");
  const int C = c0 + c1;
  GnBwdParams g{};
  g.src0 = src0; g.c0 = c0; g.src1 = src1; g.c1 = c1;
  g.gamma = gamma; g.beta = beta; g.stats = stats; g.dnorm = dnorm; g.draw = draw;
  g.drop_scale = drop_scale; g.drop_ld = drop_ld;
  g.B = B; g.pixels = pixels; g.silu = silu;
  g.dsrc0 = dsrc0; g.init0 = init0; g.dsrc1 = dsrc1; g.init1 = init1;
  g.dgamma = params_all ? nullptr : dgamma;
  g.dbeta = params_all ? nullptr : dbeta;
  // partial [B][chunks][C][2] | chsum [B][C][2] | params_all: grads [4][C] and its two-entry table
  const size_t n_part = (size_t)B * gn_bwd_chunks(B, pixels) * C * 2, n_ch = (size_t)B * C * 2;
  char* tmp = nullptr;
  CM_CUDA(cudaMalloc(&tmp, (n_part + n_ch + 4 * (size_t)C) * sizeof(float) + 8 * sizeof(long long)));
  float* partial = reinterpret_cast<float*>(tmp);
  g.chsum = partial + n_part;
  float* grads = g.chsum + n_ch;
  long long* tab = reinterpret_cast<long long*>(grads + 4 * (size_t)C);
  int rc = gn_backward_enqueue(g, partial, st);
  if (!rc && params_all) {
    // the model's route: one launch over a table of GroupNorms; two entries over the same sums, the second writing
    // (dbeta, dgamma) swapped into the upper half, so the second CTA's table walk is checked too
    const long long h_tab[8] = {0, C, 0, C, 0, C, 3LL * C, 2LL * C};
    rc = cudaMemcpyAsync(tab, h_tab, sizeof(h_tab), cudaMemcpyHostToDevice, st) == cudaSuccess ? 0 : 1;
    if (!rc) rc = gn_backward_params_all_enqueue(g.chsum, tab, 2, B, grads, st);
    if (!rc) rc = cudaMemcpyAsync(dgamma, grads, C * sizeof(float), cudaMemcpyDeviceToDevice, st) == cudaSuccess ? 0 : 1;
    if (!rc) rc = cudaMemcpyAsync(dbeta, grads + C, C * sizeof(float), cudaMemcpyDeviceToDevice, st) == cudaSuccess ? 0 : 1;
  }
  cudaError_t se = cudaStreamSynchronize(st);
  if (!rc && se == cudaSuccess && params_all) {
    std::vector<float> h(4 * (size_t)C);
    se = cudaMemcpy(h.data(), grads, h.size() * sizeof(float), cudaMemcpyDeviceToHost);
    if (se == cudaSuccess && memcmp(h.data(), h.data() + 3 * (size_t)C, C * sizeof(float)) +
                                     memcmp(h.data() + C, h.data() + 2 * (size_t)C, C * sizeof(float)) != 0) {
      set_error("GroupNorm backward: the two entries of the dgamma / dbeta table disagree");
      rc = 3;
    }
  }
  cudaFree(tmp);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_cast_colsum(const float* src, void* dst16, int dup, float* acc_dst, int acc_init, float* colsum,
                      int colsum_ld, int B, int pixels, int C, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int rc = cast_colsum_enqueue(src, static_cast<__half*>(dst16), dup, acc_dst, acc_init, colsum, colsum_ld, B,
                                     pixels, C, st);
  cudaError_t se = cudaStreamSynchronize(st);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_rowsum_all(const float* base, const int64_t* tab, int n, int B, float* grads, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  long long* d_tab = nullptr;
  CM_CUDA(cudaMalloc(&d_tab, (size_t)n * 4 * sizeof(long long)));
  int rc = cudaMemcpyAsync(d_tab, tab, (size_t)n * 4 * sizeof(long long), cudaMemcpyHostToDevice, st) == cudaSuccess
               ? 0 : 1;
  if (!rc) rc = rowsum_all_enqueue(base, d_tab, n, B, grads, st);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(d_tab);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_final_conv_backward(const float* deps, float scale, const void* act16, int act_ld, int act_lo,
                              const float* w, float* dact, float* dw, float* db, int B, int H, int W, int L, int P,
                              int cin, int cout, void* dout16, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = kernels_init()) return e;
  if (int e = backward_init()) return e;
  const __half* act = static_cast<const __half*>(act16);
  __half* d16 = static_cast<__half*>(dout16);
  const size_t g_elems = (size_t)27 * cin * 32;
  float* tmp = nullptr;   // scale[2] | G (packed route)
  CM_CUDA(cudaMalloc(&tmp, (4 + (d16 ? g_elems : 0)) * sizeof(float)));
  float* scale_dev = tmp;
  float* G = tmp + 4;
  const float h_scale[2] = {scale, 1.f / scale};
  int rc = cudaMemcpyAsync(scale_dev, h_scale, sizeof(h_scale), cudaMemcpyHostToDevice, st) == cudaSuccess ? 0 : 1;
  if (!rc) rc = cudaMemsetAsync(dw, 0, (size_t)cout * cin * 27 * sizeof(float), st) == cudaSuccess ? 0 : 1;
  if (!rc) rc = cudaMemsetAsync(db, 0, cout * sizeof(float), st) == cudaSuccess ? 0 : 1;
  WgradRun R;
  if (!rc && d16) {
    // as the training backward: d_eps * S packed into 32 fp16 columns, a conv weight gradient over it into G (taps in
    // activation order, 32 columns), then G -> dw [cout][cin][27]
    rc = cudaMemsetAsync(d16, 0, (size_t)B * L * H * W * 32 * sizeof(__half), st) == cudaSuccess ? 0 : 1;
    if (!rc) rc = cudaMemsetAsync(G, 0, g_elems * sizeof(float), st) == cudaSuccess ? 0 : 1;
    if (!rc) rc = wgrad_run_prepare(&R, edge_wgrad_kinds(cin), 0, act, B, L, H, W, cin, nullptr, 0, d16, 32, G, 32,
                                    act_ld);
    if (!rc && R.launches() == 0) {
      set_error("final conv backward: no weight-gradient kernel covers the packed operand at this shape");
      rc = 2;
    }
  }
  if (!rc)
    rc = final_conv_backward_enqueue(deps, scale_dev, act, act_ld, act_lo, w, dact, dw, db, B, H, W, L, P, cin, cout,
                                     d16, st);
  if (!rc && d16) rc = wgrad_run_enqueue(R, st);
  if (!rc && d16) rc = unpack_wgrad_enqueue(0, G, dw, nullptr, cout | (32 << 16), cin, 0, 1, st);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(tmp);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_first_conv_wgrad(const float* x, const float* past, const float* dout, float* dw, float* db, int B, int H,
                           int W, int P, int F, int cin, int cout, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = backward_init()) return e;
  CM_CUDA(cudaMemsetAsync(dw, 0, (size_t)cout * cin * 27 * sizeof(float), st));
  CM_CUDA(cudaMemsetAsync(db, 0, cout * sizeof(float), st));
  const int rc = first_conv_wgrad_enqueue(x, past, dout, dw, db, B, H, W, P, F, cin, cout, st);
  cudaError_t se = cudaStreamSynchronize(st);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_temb_backward(const float* e, const float* h1, const float* h2, const float* dtemb, int ld, int B, int base,
                        int E, const float* w2, const void* const* wd, const int32_t* couts, const int32_t* offs,
                        int nblocks, float* dense_grads, const int64_t* goff_w, const int64_t* goff_b, float* dw1,
                        float* db1, float* dw2, float* db2, float* ds1, float* ds2, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CM_CHECK(nblocks > 0 && B > 0, "time-embedding backward: empty input");
  // device tables: wd[nblocks] | goff_w | goff_b (8-byte entries), couts | offs (int), then scratch s1 s2 dh1 dh2 [B][E]
  const size_t tab_bytes = (size_t)nblocks * 3 * 8 + (size_t)nblocks * 2 * 4;
  const size_t nE = (size_t)B * E;
  char* tmp = nullptr;
  CM_CUDA(cudaMalloc(&tmp, ((tab_bytes + 15) & ~(size_t)15) + 4 * nE * sizeof(float)));
  std::vector<char> h(tab_bytes);
  memcpy(h.data(), wd, (size_t)nblocks * 8);
  memcpy(h.data() + (size_t)nblocks * 8, goff_w, (size_t)nblocks * 8);
  memcpy(h.data() + (size_t)nblocks * 16, goff_b, (size_t)nblocks * 8);
  memcpy(h.data() + (size_t)nblocks * 24, couts, (size_t)nblocks * 4);
  memcpy(h.data() + (size_t)nblocks * 28, offs, (size_t)nblocks * 4);
  TembBwdParams p{};
  p.e = e; p.h1 = h1; p.h2 = h2; p.dtemb = dtemb; p.ld = ld;
  p.wd = reinterpret_cast<const float* const*>(tmp);
  p.goff_w = reinterpret_cast<const long long*>(tmp + (size_t)nblocks * 8);
  p.goff_b = reinterpret_cast<const long long*>(tmp + (size_t)nblocks * 16);
  p.couts = reinterpret_cast<const int*>(tmp + (size_t)nblocks * 24);
  p.offs = reinterpret_cast<const int*>(tmp + (size_t)nblocks * 28);
  p.nblocks = nblocks;
  p.w2 = w2;
  p.dw1 = dw1; p.db1 = db1; p.dw2 = dw2; p.db2 = db2;
  float* scratch = reinterpret_cast<float*>(tmp + ((tab_bytes + 15) & ~(size_t)15));
  p.s1 = scratch; p.s2 = scratch + nE; p.dh1 = scratch + 2 * nE; p.dh2 = scratch + 3 * nE;
  p.ds1 = ds1; p.ds2 = ds2;
  p.B = B; p.E = E; p.base = base;
  int rc = cudaMemcpyAsync(tmp, h.data(), tab_bytes, cudaMemcpyHostToDevice, st) == cudaSuccess ? 0 : 1;
  if (!rc) rc = temb_backward_enqueue(p, dense_grads, st);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(tmp);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

int cm_op_loss_scale(const float* x, int64_t n, float target, float* scale_out, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned int* mx = nullptr;
  CM_CUDA(cudaMalloc(&mx, sizeof(unsigned int)));
  int rc = cudaMemsetAsync(mx, 0, sizeof(unsigned int), st) == cudaSuccess ? 0 : 1;
  if (!rc) rc = auto_scale_enqueue(x, (size_t)n, target, scale_out, mx, st);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(mx);
  if (rc) return rc;
  CM_CUDA(se);
  return 0;
}

}  // extern "C"
