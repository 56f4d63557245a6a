// Native plan of the reference's second noise-prediction backbone, DiT4D_V4 (SURVEY.md section 8 f2;
// /root/reference/models/backbones/DiT4D_V4.py:228-375, selected by --arch DDPM-DiT at models/diffusion/ddpm.py:88-104),
// behind the same C ABI style as the UNet plan: forward(future, t, past) and the fused reverse chain.
//
// Every nn.Linear / the patch-embedding Conv3d (kernel = stride: a per-patch linear map) runs on the tcgen05 implicit-GEMM
// kernel of conv_umma.cuh in its 1x1x1 mode (fp16 activations, hi + lo fp16 weights, fp32 accumulation in TMEM; bias, exact
// GELU and the gated residual adds fused into its epilogue); spatial self-attention is the attention core of kernels.cu
// (mma.sync, S = 27 tokens); what is new here are the bandwidth kernels between them: LayerNorm + AdaLN modulate -> fp16
// operand, the temporal cross-attention (future slots query the T_p <= 8 slots of their spatial patch), patch gather /
// scatter, and the DDPM / DDIM update fused into the un-patch kernel.  Sampling (eval) only: training this backbone still
// raises.
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/crowdmod_b200.h"
#include "conv_umma.cuh"
#include "kernels.cuh"

namespace cm {
namespace {

struct DitParam {
  std::string name;
  std::vector<int64_t> shape;
  const float* ptr = nullptr;
  int64_t numel() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};

// ---------------------------------------------------------------------------------------------------------------
// bandwidth kernels
// ---------------------------------------------------------------------------------------------------------------
// e16[b][:] = fp16(table[t[b]][:])   (embeddings.py:24: nn.Embedding.from_pretrained lookup)
__global__ void dit_gather_emb_kernel(const float* __restrict__ table, const long long* __restrict__ t, int D,
                                      int table_rows, __half* __restrict__ out) {
  const int b = blockIdx.x;
  long long ti = t[b];
  if (ti < 0) ti = 0;
  if (ti >= table_rows) ti = table_rows - 1;
  for (int d = threadIdx.x; d < D; d += blockDim.x) out[(size_t)b * D + d] = __float2half_rn(table[(size_t)ti * D + d]);
}

// out16 = fp16(act(in32)); act: 0 identity, 1 SiLU, 2 SiLU(SiLU(.)) (c = SiLU(time_proj), AdaLN applies SiLU again)
__device__ __forceinline__ float silu_exact(float x) { return x / (1.0f + expf(-x)); }
__global__ void dit_act16_kernel(const float* __restrict__ in, __half* __restrict__ out, size_t n4, int act) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(in)[i];
    float r[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float x = r[k];
      if (act == 1) x = silu_exact(x);
      else if (act == 2) x = silu_exact(silu_exact(x));
      r[k] = x;
    }
    __half2 h0 = __floats2half2_rn(r[0], r[1]), h1 = __floats2half2_rn(r[2], r[3]);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&h0);
    u.y = *reinterpret_cast<uint32_t*>(&h1);
    reinterpret_cast<uint2*>(out)[i] = u;
  }
}

struct PatchGeom {
  int B, C, H, W, P, F, p, pt, hp, wp, Tp, Kpad;   // K = C*pt*p*p, Kpad = K rounded up to 32
};
// A16[row = (b, slot, ph, pw)][k = ((c*pt + dt)*p + dy)*p + dx] = x[b, c, ph*p + dy, pw*p + dx, slot*pt + dt] with
// x = cat(past, future) along time (DiT4D_V4.py:356-359; PatchEmbed4D.forward :47-63: Conv3d over (T, H, W) with
// kernel = stride = (pt, p, p), weight [D][C][pt][p][p])
__global__ void dit_patchify_kernel(const float* __restrict__ future, const float* __restrict__ past, PatchGeom g,
                                    __half* __restrict__ out) {
  const int rows = g.B * g.Tp * g.hp * g.wp;
  const size_t total = (size_t)rows * g.Kpad;
  const int K = g.C * g.pt * g.p * g.p;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int row = (int)(i / g.Kpad), k = (int)(i - (size_t)row * g.Kpad);
    float v = 0.f;
    if (k < K) {
      int r = row;
      const int pw = r % g.wp; r /= g.wp;
      const int ph = r % g.hp; r /= g.hp;
      const int slot = r % g.Tp;
      const int b = r / g.Tp;
      int kk = k;
      const int dx = kk % g.p; kk /= g.p;
      const int dy = kk % g.p; kk /= g.p;
      const int dt = kk % g.pt;
      const int c = kk / g.pt;
      const int y = ph * g.p + dy, x = pw * g.p + dx, tt = slot * g.pt + dt;
      const size_t cell = ((size_t)(b * g.C + c) * g.H + y) * g.W + x;
      v = tt < g.P ? past[cell * g.P + tt] : future[cell * g.F + (tt - g.P)];
    }
    out[i] = __float2half_rn(v);
  }
}

// tokens[b][slot][s][:] += spatial_pos[s][:] + temporal_pos[slot][:]   (DiT4D_V4.py:329-346)
__global__ void dit_add_pos_kernel(float* __restrict__ x, const float* __restrict__ spatial, const float* __restrict__ temporal,
                                   int rows, int Tp, int Ns, int D) {
  const size_t total = (size_t)rows * D / 4;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int row = (int)(i / (D / 4)), d = (int)(i - (size_t)row * (D / 4)) * 4;
    const int s = row % Ns, slot = (row / Ns) % Tp;
    float4 v = reinterpret_cast<float4*>(x)[i];
    const float4 a = *reinterpret_cast<const float4*>(spatial + (size_t)s * D + d);
    const float4 c = *reinterpret_cast<const float4*>(temporal + (size_t)slot * D + d);
    v.x = v.x + a.x + c.x; v.y = v.y + a.y + c.y; v.z = v.z + a.z + c.z; v.w = v.w + a.w + c.w;   // (tokens + spatial) + temporal
    reinterpret_cast<float4*>(x)[i] = v;
  }
}

// out16[row][:] = fp16( LayerNorm(x[row][:], eps 1e-6, no affine) * (1 + scale[b][:]) + shift[b][:] ), b = row / rows_per_sample
// (DiT4D_V4.py:104-106 modulate; :116,:121,:126 the three norms; :232-234 the final layer).  One warp per row, two-pass
// statistics in fp32 (mean first, then the centred second moment).
__global__ void __launch_bounds__(256) dit_ln_mod_kernel(const float* __restrict__ x, const float* __restrict__ mods, int ld_mods,
                                                         int off_shift, int off_scale, int rows_per_sample, int rows, int D,
                                                         __half* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const float* xr = x + (size_t)warp * D;
  float s = 0.f;
  for (int d = lane * 4; d < D; d += 128) {
    const float4 v = *reinterpret_cast<const float4*>(xr + d);
    s += (v.x + v.y) + (v.z + v.w);
  }
  const float mean = warp_sum(s) / (float)D;
  float q = 0.f;
  for (int d = lane * 4; d < D; d += 128) {
    const float4 v = *reinterpret_cast<const float4*>(xr + d);
    const float a = v.x - mean, b2 = v.y - mean, c = v.z - mean, e = v.w - mean;
    q += (a * a + b2 * b2) + (c * c + e * e);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)D + 1e-6f);
  const float* mb = mods + (size_t)(warp / rows_per_sample) * ld_mods;
  for (int d = lane * 4; d < D; d += 128) {
    const float4 v = *reinterpret_cast<const float4*>(xr + d);
    const float4 sh = *reinterpret_cast<const float4*>(mb + off_shift + d);
    const float4 sc = *reinterpret_cast<const float4*>(mb + off_scale + d);
    const float y0 = (v.x - mean) * rstd * (1.0f + sc.x) + sh.x, y1 = (v.y - mean) * rstd * (1.0f + sc.y) + sh.y;
    const float y2 = (v.z - mean) * rstd * (1.0f + sc.z) + sh.z, y3 = (v.w - mean) * rstd * (1.0f + sc.w) + sh.w;
    __half2 h0 = __floats2half2_rn(y0, y1), h1 = __floats2half2_rn(y2, y3);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&h0);
    u.y = *reinterpret_cast<uint32_t*>(&h1);
    *reinterpret_cast<uint2*>(out + (size_t)warp * D + d) = u;
  }
}

// Temporal cross-attention core (DiT4D_V4.py:168-190): for every (sample, spatial patch s, head) the nq future slots
// query all Tp slots of that patch.  qkv: fp32 [B][Tp][Ns][3D] (q | k | v, heads split each D); ctx16: fp16
// [B][nq][Ns][D].  One warp per (b, iq, s, head); Tp <= 8 keys, softmax in fp32.
__global__ void __launch_bounds__(256) dit_tattn_kernel(const float* __restrict__ qkv, __half* __restrict__ ctx, int B, int Tp,
                                                        int Ns, int D, int heads, int qs) {
  const int nq = Tp - qs, dh = D / heads;
  const int total = B * nq * Ns * heads;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= total) return;
  int r = w;
  const int h = r % heads; r /= heads;
  const int s = r % Ns; r /= Ns;
  const int iq = r % nq;
  const int b = r / nq;
  const float scale = rsqrtf((float)dh);
  const float* qrow = qkv + (((size_t)b * Tp + qs + iq) * Ns + s) * 3 * D + h * dh;
  float sc[8];
  float mx = -INFINITY;
  for (int j = 0; j < Tp; ++j) {
    const float* krow = qkv + (((size_t)b * Tp + j) * Ns + s) * 3 * D + D + h * dh;
    float a = 0.f;
    for (int d = lane; d < dh; d += 32) a = fmaf(qrow[d], krow[d], a);
    a = warp_sum(a) * scale;
    sc[j] = a;
    mx = fmaxf(mx, a);
  }
  float den = 0.f;
  for (int j = 0; j < Tp; ++j) {
    sc[j] = expf(sc[j] - mx);
    den += sc[j];
  }
  const float inv = 1.0f / den;
  __half* orow = ctx + (((size_t)b * nq + iq) * Ns + s) * D + h * dh;
  for (int d = lane; d < dh; d += 32) {
    float o = 0.f;
    for (int j = 0; j < Tp; ++j) o = fmaf(sc[j] * inv, qkv[(((size_t)b * Tp + j) * Ns + s) * 3 * D + 2 * D + h * dh + d], o);
    orow[d] = __float2half_rn(o);
  }
}

struct UnpatchParams {
  const float* out;      // [rows][ld]: FinalLayer output, column = ((dt*C + c)*p + dy)*p + dx (DiT4D_V4.py:94-97)
  int ld;
  int B, C, H, W, P, F, p, pt, hp, wp, Tp;
  float* eps_out;        // optional [B][C][H][W][F]
  // reverse-step update (as FinalParams of the UNet path): all optional
  float* x;
  const float* coef;     // device [nsteps][8]
  int step;
  const int* step_dev;   // device step index (graph replay): overrides `step` when set
  int mode;
  const float* noise;
  unsigned long long seed;
  long long sample_offset;
  const unsigned long long* chain_dev;   // device {seed, sample_offset}: overrides the two fields above when set
  float* history;
};
// un-patch + slice to the future frames (DiT4D_V4.py:80-102) + DDPM.step / DDIM update / Sparsity guidance / Philox
// noise exactly as final_conv_kernel does for the UNet (ddpm.py:25-38, :262-265, guidance.py:4-8): one thread per
// (b, y, x, f) handles the C <= 4 properties (one Philox draw).
__global__ void dit_unpatch_step_kernel(UnpatchParams p) {
  const size_t total = (size_t)p.B * p.H * p.W * p.F;
  const size_t plane = (size_t)p.H * p.W * p.F;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    size_t r = i;
    const int f = (int)(r % p.F); r /= p.F;
    const int xw = (int)(r % p.W); r /= p.W;
    const int y = (int)(r % p.H);
    const int b = (int)(r / p.H);
    const int tt = p.P + f, slot = tt / p.pt, dt = tt - slot * p.pt;
    const int ph = y / p.p, dy = y - ph * p.p, pw = xw / p.p, dx = xw - pw * p.p;
    const size_t row = (((size_t)b * p.Tp + slot) * p.hp + ph) * p.wp + pw;
    float eps[4] = {0.f, 0.f, 0.f, 0.f};
    for (int c = 0; c < p.C; ++c) eps[c] = p.out[row * p.ld + ((dt * p.C + c) * p.p + dy) * p.p + dx];
    const size_t e0 = ((size_t)b * p.C) * plane + ((size_t)y * p.W + xw) * p.F + f;
    if (p.eps_out)
      for (int c = 0; c < p.C; ++c) p.eps_out[e0 + c * plane] = eps[c];
    if (!p.x) continue;
    const int step = p.step_dev ? *p.step_dev : p.step;
    const unsigned long long seed = p.chain_dev ? p.chain_dev[0] : p.seed;
    const long long soff = p.chain_dev ? static_cast<long long>(p.chain_dev[1]) : p.sample_offset;
    const float* cf = p.coef + (size_t)step * 8;
    const size_t nelem = (size_t)p.B * p.C * plane;
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    const float zc = (p.mode == 0) ? cf[2] : cf[4];
    if (zc != 0.f) {
      if (p.noise) {
        for (int c = 0; c < p.C; ++c) z[c] = p.noise[(size_t)step * nelem + e0 + c * plane];
      } else {
        const unsigned long long gp = ((unsigned long long)(soff + b)) * (unsigned long long)plane +
                                      ((size_t)y * p.W + xw) * p.F + f;
        const uint4 rnd = philox4x32_10(make_uint4((uint32_t)gp, (uint32_t)(gp >> 32), (uint32_t)step, 0u),
                                        make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        const float2 n0 = box_muller(rnd.x, rnd.y), n1 = box_muller(rnd.z, rnd.w);
        z[0] = n0.x; z[1] = n0.y; z[2] = n1.x; z[3] = n1.y;
      }
    }
    for (int c = 0; c < p.C; ++c) {
      const size_t e = e0 + c * plane;
      const float xv = p.x[e];
      float xn;
      if (p.mode == 0) {
        xn = cf[0] * (xv - cf[1] * eps[c]) + cf[2] * z[c];
      } else {
        const float x0 = (xv - cf[0] * eps[c]) / cf[1];
        xn = cf[2] * x0 + cf[3] * eps[c] + cf[4] * z[c];
      }
      if (c == 0 && cf[5] != 0.f) {
        const float sg = (xn > 0.f) ? 1.f : ((xn < 0.f) ? -1.f : 0.f);
        xn -= cf[5] * sg;
      }
      p.x[e] = xn;
      if (p.history) p.history[(size_t)(step + 1) * nelem + e] = xn;
    }
  }
}

__global__ void dit_fill_t_kernel(long long* t, int B, int value) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) t[i] = value;
}
__global__ void dit_fill_t_range_kernel(long long* t, int n, int first) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) t[i] = first + i;
}
// sampling steps are batch-uniform: the step's (shift, scale, gate) vectors of every block are ONE row of the table
// precomputed per weight load (the analogue of the UNet plan's time-embedding table); copied to mods row 0
__global__ void dit_select_mods_kernel(float* __restrict__ mods, const float* __restrict__ table, const int* __restrict__ tsteps,
                                       const int* __restrict__ step_dev, int J) {
  const float* row = table + (size_t)tsteps[*step_dev] * J;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < J / 4; i += gridDim.x * blockDim.x)
    reinterpret_cast<float4*>(mods)[i] = reinterpret_cast<const float4*>(row)[i];
}
__global__ void dit_advance_kernel(int* step_dev) { ++*step_dev; }

int grid_for(size_t work_items, int block = 256) {
  size_t b = (work_items + block - 1) / block;
  if (b > 148 * 8) b = 148 * 8;
  if (b < 1) b = 1;
  return (int)b;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace
}  // namespace cm

using namespace cm;

// one Linear of the plan: fp32 master (state_dict tensor or a stacked copy), packed fp16 hi|lo cache, GEMM launch
struct DitLinear {
  int w = -1, b = -1;            // parameter indices (w < 0: stacked buffers below)
  const float* w_dev = nullptr;  // stacked fp32 weights / bias (AdaLN of all blocks in one GEMM)
  const float* b_dev = nullptr;
  int cin = 0, cout = 0;
  size_t pack_off = 0;           // element offset into wpack
  ConvLaunch launch;
};

struct cm_dit {
  cm_dit_config cfg;
  std::vector<DitParam> params;
  std::map<std::string, int> pindex;
  int D = 0, E = 0, Dm = 0, Tp = 0, Ns = 0, hp = 0, wp = 0, qs = 0, nq = 0, tokens = 0, K = 0, Kpad = 0, Nout = 0, Jtot = 0;
  int p_table = -1, p_spatial = -1, p_temporal = -1;
  DitLinear t1, t2, tproj, adaln, patch, final_lin;
  struct Block { DitLinear s_in, s_out, t_in, t_out, fc1, fc2; };
  std::vector<Block> blocks;
  std::vector<int> adaln_w, adaln_b;   // per block (+ final) parameter indices, stacked into adaln_wbuf / adaln_bbuf
  float* adaln_wbuf = nullptr;
  float* adaln_bbuf = nullptr;
  float* patch_wbuf = nullptr;         // patch weights zero-padded to Kpad columns (when K % 32 != 0)
  __half* wpack = nullptr;
  size_t wpack_elems = 0;
  bool packed = false;
  int reserved_batch = 0, prepared_batch = 0;
  uint8_t* arena = nullptr;
  // workspace pointers
  long long* t_dev = nullptr;
  __half *e16 = nullptr, *h16 = nullptr, *a16 = nullptr, *xm16 = nullptr, *ctx16 = nullptr, *g16 = nullptr;
  float *h32 = nullptr, *h2_32 = nullptr, *c32 = nullptr, *mods = nullptr, *x32 = nullptr, *qkv32 = nullptr, *out32 = nullptr,
        *chain_x = nullptr, *chain_past = nullptr, *d_coef = nullptr;
  int coef_cap = 0;
  float* mods_table = nullptr;         // [table_steps][Jtot]: AdaLN vectors of every timestep (sampling, batch-uniform t)
  bool table_ready = false;
  int* d_step = nullptr;
  int* d_tsteps = nullptr;
  unsigned long long* d_chain = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  cm_chain_args graph_key{};
  int64_t graph_launches_per_step = 0;
  int64_t last_launches = 0;
  double flops_per_sample = 0.0;

  int add_param(const std::string& name, std::vector<int64_t> shape) {
    DitParam e;
    e.name = name;
    e.shape = std::move(shape);
    params.push_back(e);
    pindex[name] = (int)params.size() - 1;
    return (int)params.size() - 1;
  }
};

namespace {

DitLinear make_linear(cm_dit* u, const std::string& wname, const std::string& bname, int cout, int cin, std::vector<int64_t> wshape = {}) {
  DitLinear l;
  if (wshape.empty()) wshape = {cout, cin};
  l.w = u->add_param(wname, wshape);
  l.b = u->add_param(bname, {cout});
  l.cin = cin;
  l.cout = cout;
  return l;
}

void reserve_pack(cm_dit* u, DitLinear& l, int cin_packed) {
  l.pack_off = u->wpack_elems;
  u->wpack_elems += (size_t)2 * l.cout * cin_packed;
}

int build(cm_dit* u) {
  const cm_dit_config& c = u->cfg;
  CM_CHECK(c.in_channels >= 1 && c.in_channels <= 4 && c.out_channels >= 1 && c.out_channels <= 4, "in/out channels must be in 1..4");
  CM_CHECK(c.hidden % 32 == 0 && c.hidden % c.heads == 0 && c.hidden / c.heads <= 128 && (c.hidden / c.heads) % 2 == 0,
           "hidden size %d / heads %d unsupported (hidden %% 32 == 0, head dim even and <= 128)", c.hidden, c.heads);
  CM_CHECK(c.rows % c.patch == 0 && c.cols % c.patch == 0, "grid %dx%d not divisible by the patch size %d (DiT4D_V4.py:26-29)", c.rows,
           c.cols, c.patch);
  const int T = c.past_len + c.future_len;
  CM_CHECK(T % c.t_patch == 0, "T_total=%d must be divisible by t_patch=%d (DiT4D_V4.py:253-254)", T, c.t_patch);
  u->D = c.hidden;
  u->E = c.hidden * c.time_multiple;
  u->Dm = c.mlp_hidden;
  CM_CHECK(u->Dm % 32 == 0 && u->E % 32 == 0, "mlp / time-embedding widths must be multiples of 32");
  u->Tp = T / c.t_patch;
  CM_CHECK(u->Tp <= 8, "more than 8 temporal slots (%d) are not supported by the temporal attention kernel", u->Tp);
  u->hp = c.rows / c.patch;
  u->wp = c.cols / c.patch;
  u->Ns = u->hp * u->wp;
  u->qs = c.past_len / c.t_patch;
  u->nq = u->Tp - u->qs;
  CM_CHECK(u->nq >= 1, "no future temporal slot (past_len %d, t_patch %d)", c.past_len, c.t_patch);
  u->tokens = u->Tp * u->Ns;
  u->K = c.in_channels * c.t_patch * c.patch * c.patch;
  u->Kpad = (u->K + 31) / 32 * 32;
  u->Nout = c.t_patch * c.out_channels * c.patch * c.patch;
  CM_CHECK(u->Nout % 32 == 0, "t_patch*C*p*p = %d must be a multiple of 32", u->Nout);
  CM_CHECK(c.t_max_slots >= u->Tp, "temporal_pos_embed holds %d slots < T_p = %d", c.t_max_slots, u->Tp);
  const int D = u->D, E = u->E;
  // parameters: the reference's state_dict names (DiT4D_V4.__init__ :247-311; nn.MultiheadAttention / nn.Sequential keys)
  u->p_spatial = u->add_param("spatial_pos_embed", {1, u->Ns, D});
  u->p_temporal = u->add_param("temporal_pos_embed", {1, c.t_max_slots, D});
  u->p_table = u->add_param("dif_time_embeddings.time_blocks.0.weight", {c.table_steps, D});
  u->t1 = make_linear(u, "dif_time_embeddings.time_blocks.1.weight", "dif_time_embeddings.time_blocks.1.bias", E, D);
  u->t2 = make_linear(u, "dif_time_embeddings.time_blocks.3.weight", "dif_time_embeddings.time_blocks.3.bias", E, E);
  u->tproj = make_linear(u, "time_proj.0.weight", "time_proj.0.bias", D, E);
  u->patch = make_linear(u, "patch_embed.proj.weight", "patch_embed.proj.bias", D, u->Kpad,
                         {D, c.in_channels, c.t_patch, c.patch, c.patch});
  u->blocks.resize(c.depth);
  for (int i = 0; i < c.depth; ++i) {
    const std::string p = "blocks." + std::to_string(i) + ".";
    cm_dit::Block& b = u->blocks[i];
    b.s_in = make_linear(u, p + "spatial_attn.in_proj_weight", p + "spatial_attn.in_proj_bias", 3 * D, D);
    b.s_out = make_linear(u, p + "spatial_attn.out_proj.weight", p + "spatial_attn.out_proj.bias", D, D);
    b.t_in = make_linear(u, p + "temporal_attn.in_proj_weight", p + "temporal_attn.in_proj_bias", 3 * D, D);
    b.t_out = make_linear(u, p + "temporal_attn.out_proj.weight", p + "temporal_attn.out_proj.bias", D, D);
    b.fc1 = make_linear(u, p + "mlp.0.weight", p + "mlp.0.bias", u->Dm, D);
    b.fc2 = make_linear(u, p + "mlp.3.weight", p + "mlp.3.bias", D, u->Dm);
    u->adaln_w.push_back(u->add_param(p + "adaLN_modulation.1.weight", {9 * D, D}));
    u->adaln_b.push_back(u->add_param(p + "adaLN_modulation.1.bias", {9 * D}));
  }
  u->final_lin = make_linear(u, "final_layer.linear.weight", "final_layer.linear.bias", u->Nout, D);
  u->adaln_w.push_back(u->add_param("final_layer.adaLN_modulation.1.weight", {2 * D, D}));
  u->adaln_b.push_back(u->add_param("final_layer.adaLN_modulation.1.bias", {2 * D}));
  u->Jtot = c.depth * 9 * D + 2 * D;
  u->adaln.cin = D;
  u->adaln.cout = u->Jtot;
  // packed-weight cache
  reserve_pack(u, u->t1, D);
  reserve_pack(u, u->t2, E);
  reserve_pack(u, u->tproj, E);
  reserve_pack(u, u->adaln, D);
  reserve_pack(u, u->patch, u->Kpad);
  for (auto& b : u->blocks) {
    reserve_pack(u, b.s_in, D);
    reserve_pack(u, b.s_out, D);
    reserve_pack(u, b.t_in, D);
    reserve_pack(u, b.t_out, D);
    reserve_pack(u, b.fc1, D);
    reserve_pack(u, b.fc2, u->Dm);
  }
  reserve_pack(u, u->final_lin, D);
  // algorithmic FLOPs per sample (dense formulation of the reference graph)
  const double tok = u->tokens, fut = (double)u->nq * u->Ns;
  double fl = 2.0 * (D * (double)E + (double)E * E + (double)E * D + (double)D * u->Jtot) + 2.0 * tok * u->K * D;
  fl += c.depth * (2.0 * tok * D * 3 * D + 4.0 * u->Tp * (double)u->Ns * u->Ns * D + 2.0 * tok * D * D     // spatial attention
                   + 2.0 * fut * D * D + 2.0 * tok * D * 2 * D + 4.0 * fut * u->Tp * D + 2.0 * fut * D * D  // temporal cross-attention
                   + 4.0 * tok * D * (double)u->Dm);                                                     // MLP
  fl += 2.0 * tok * D * u->Nout;
  u->flops_per_sample = fl;
  return 0;
}

int check_bound(cm_dit* u) {
  for (auto& p : u->params) CM_CHECK(p.ptr != nullptr, "parameter '%s' not bound (cm_dit_bind_params)", p.name.c_str());
  return 0;
}

int pack_linear(cm_dit* u, DitLinear& l, cudaStream_t st) {
  const float* w = l.w >= 0 ? u->params[l.w].ptr : l.w_dev;
  return pack_conv_weights(w, nullptr, u->wpack + l.pack_off, l.cout, l.cin, 0, 1, 2, 0, st);
}

int pack_all(cm_dit* u, cudaStream_t st) {
  if (int e = check_bound(u)) return e;
  if (int e = kernels_init()) return e;
  const int D = u->D;
  if (!u->wpack) CM_CUDA(cudaMalloc(&u->wpack, u->wpack_elems * sizeof(__half)));
  if (!u->adaln_wbuf) {
    CM_CUDA(cudaMalloc(&u->adaln_wbuf, (size_t)u->Jtot * D * sizeof(float)));
    CM_CUDA(cudaMalloc(&u->adaln_bbuf, (size_t)u->Jtot * sizeof(float)));
  }
  // stack the AdaLN projections of every block and of the final layer: one GEMM gives every (shift, scale, gate)
  size_t row = 0;
  for (size_t i = 0; i < u->adaln_w.size(); ++i) {
    const DitParam& w = u->params[u->adaln_w[i]];
    const DitParam& b = u->params[u->adaln_b[i]];
    CM_CUDA(cudaMemcpyAsync(u->adaln_wbuf + row * D, w.ptr, (size_t)w.numel() * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CM_CUDA(cudaMemcpyAsync(u->adaln_bbuf + row, b.ptr, (size_t)b.numel() * sizeof(float), cudaMemcpyDeviceToDevice, st));
    row += (size_t)b.numel();
  }
  u->adaln.w_dev = u->adaln_wbuf;
  u->adaln.b_dev = u->adaln_bbuf;
  // patch-embedding weights [D][K] (K = C*pt*p*p in the Conv3d's own (c, dt, dy, dx) order), zero-padded to Kpad columns
  const float* pw = u->params[u->patch.w].ptr;
  if (u->Kpad != u->K) {
    if (!u->patch_wbuf) CM_CUDA(cudaMalloc(&u->patch_wbuf, (size_t)D * u->Kpad * sizeof(float)));
    CM_CUDA(cudaMemsetAsync(u->patch_wbuf, 0, (size_t)D * u->Kpad * sizeof(float), st));
    CM_CUDA(cudaMemcpy2DAsync(u->patch_wbuf, (size_t)u->Kpad * sizeof(float), pw, (size_t)u->K * sizeof(float),
                              (size_t)u->K * sizeof(float), D, cudaMemcpyDeviceToDevice, st));
    u->patch.w_dev = u->patch_wbuf;
    const int keep = u->patch.w;
    u->patch.w = -1;
    const int e = pack_linear(u, u->patch, st);
    u->patch.w = keep;
    if (e) return e;
  } else if (int e = pack_linear(u, u->patch, st)) {
    return e;
  }
  if (int e = pack_linear(u, u->t1, st)) return e;
  if (int e = pack_linear(u, u->t2, st)) return e;
  if (int e = pack_linear(u, u->tproj, st)) return e;
  if (int e = pack_linear(u, u->adaln, st)) return e;
  for (auto& b : u->blocks) {
    if (int e = pack_linear(u, b.s_in, st)) return e;
    if (int e = pack_linear(u, b.s_out, st)) return e;
    if (int e = pack_linear(u, b.t_in, st)) return e;
    if (int e = pack_linear(u, b.t_out, st)) return e;
    if (int e = pack_linear(u, b.fc1, st)) return e;
    if (int e = pack_linear(u, b.fc2, st)) return e;
  }
  if (int e = pack_linear(u, u->final_lin, st)) return e;
  u->packed = true;
  u->table_ready = false;
  return 0;
}

int reserve(cm_dit* u, int batch) {
  if (batch <= u->reserved_batch) return 0;
  if (u->graph_exec) {
    cudaGraphExecDestroy(u->graph_exec);
    u->graph_exec = nullptr;
  }
  if (u->arena) CM_CUDA(cudaFree(u->arena));
  u->arena = nullptr;
  u->prepared_batch = 0;
  const cm_dit_config& c = u->cfg;
  const size_t R = (size_t)batch * u->tokens, Rq = (size_t)batch * u->nq * u->Ns;
  const size_t Bp = (size_t)(batch + 127) / 128 * 128;      // the time-path buffers hold whole 128-row tiles (>= one table chunk)
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
  const size_t o_t = take(Bp * 8), o_e16 = take(Bp * u->D * 2), o_h16 = take(Bp * u->E * 2);
  const size_t o_h32 = take(Bp * u->E * 4), o_h2 = take(Bp * u->E * 4), o_c32 = take(Bp * u->D * 4);
  const size_t o_mods = take(Bp * u->Jtot * 4);
  const size_t o_a16 = take(R * u->Kpad * 2), o_x32 = take(R * u->D * 4), o_xm = take(R * u->D * 2);
  const size_t o_qkv = take(R * 3 * u->D * 4), o_ctx = take(R * u->D * 2);
  const size_t o_g16 = take(R * u->Dm * 2), o_out = take(R * u->Nout * 4);
  const size_t xel = (size_t)batch * c.out_channels * c.rows * c.cols * c.future_len;
  const size_t pel = (size_t)batch * c.in_channels * c.rows * c.cols * (c.past_len > 0 ? c.past_len : 1);
  const size_t o_cx = take(xel * 4), o_cp = take(pel * 4);
  (void)Rq;
  CM_CUDA(cudaMalloc(&u->arena, off));
  CM_CUDA(cudaMemset(u->arena, 0, off));
  uint8_t* a = u->arena;
  u->t_dev = reinterpret_cast<long long*>(a + o_t);
  u->e16 = reinterpret_cast<__half*>(a + o_e16);
  u->h16 = reinterpret_cast<__half*>(a + o_h16);
  u->h32 = reinterpret_cast<float*>(a + o_h32);
  u->h2_32 = reinterpret_cast<float*>(a + o_h2);
  u->c32 = reinterpret_cast<float*>(a + o_c32);
  u->mods = reinterpret_cast<float*>(a + o_mods);
  u->a16 = reinterpret_cast<__half*>(a + o_a16);
  u->x32 = reinterpret_cast<float*>(a + o_x32);
  u->xm16 = reinterpret_cast<__half*>(a + o_xm);
  u->qkv32 = reinterpret_cast<float*>(a + o_qkv);
  u->ctx16 = reinterpret_cast<__half*>(a + o_ctx);
  u->g16 = reinterpret_cast<__half*>(a + o_g16);
  u->out32 = reinterpret_cast<float*>(a + o_out);
  u->chain_x = reinterpret_cast<float*>(a + o_cx);
  u->chain_past = reinterpret_cast<float*>(a + o_cp);
  u->reserved_batch = batch;
  return 0;
}

#define DIT_LAUNCH_CHECK() CM_CUDA(cudaGetLastError())

// GEMM out32[rows][cout] = act16[rows][cin] . W^T + bias  (conv_umma 1x1x1 mode; rows = nb * d * h * w)
int prep_gemm(cm_dit* u, DitLinear& l, const __half* act, int nb, int d, int h, int w, float* out32) {
  // no split-K: the epilogue fusions (act / gate / rmap) live in the non-split path, and with K <= 1024 narrower N tiles
  // fill the SMs without the cluster reduction
  ConvEpilogue e{};
  e.bias = l.b >= 0 ? u->params[l.b].ptr : l.b_dev;
  e.out32 = out32;
  return conv_prepare(&l.launch, 3, act, nb, d, h, w, l.cin, nullptr, 0, u->wpack + l.pack_off, l.cout, 2, e, false);
}

int prepare(cm_dit* u, int batch) {
  if (u->prepared_batch == batch) return 0;
  const int Tp = u->Tp, Ns = u->Ns;
  if (int e = prep_gemm(u, u->t1, u->e16, batch, 1, 1, 1, u->h32)) return e;
  if (int e = prep_gemm(u, u->t2, u->h16, batch, 1, 1, 1, u->h2_32)) return e;
  if (int e = prep_gemm(u, u->tproj, u->h16, batch, 1, 1, 1, u->c32)) return e;
  if (int e = prep_gemm(u, u->adaln, u->e16, batch, 1, 1, 1, u->mods)) return e;
  if (int e = prep_gemm(u, u->patch, u->a16, batch, 1, Tp, Ns, u->x32)) return e;
  for (auto& b : u->blocks) {
    if (int e = prep_gemm(u, b.s_in, u->xm16, batch, 1, Tp, Ns, u->qkv32)) return e;
    if (int e = prep_gemm(u, b.s_out, u->ctx16, batch, 1, Tp, Ns, u->x32)) return e;
    if (int e = prep_gemm(u, b.t_in, u->xm16, batch, 1, Tp, Ns, u->qkv32)) return e;
    if (int e = prep_gemm(u, b.t_out, u->ctx16, batch, 1, u->nq, Ns, u->x32)) return e;
    if (int e = prep_gemm(u, b.fc1, u->xm16, batch, 1, Tp, Ns, nullptr)) return e;
    if (int e = prep_gemm(u, b.fc2, u->g16, batch, 1, Tp, Ns, u->x32)) return e;
    // epilogue fusions (ConvParams::act / gate / rmap): GELU + fp16 operand out of fc1; the three gated residuals
    // x += gate * (GEMM + bias) written in place into the token stream (the temporal one into the future slots)
    b.fc1.launch.p.act = 1;
    b.fc1.launch.p.epi.out16 = u->g16;
    for (DitLinear* l : {&b.s_out, &b.t_out, &b.fc2}) {
      l->launch.p.epi.resid = u->x32;
      l->launch.p.gate = u->mods;           // + the block's gate offset, set per launch in run_forward
    }
    b.t_out.launch.p.rmap_out = u->tokens;
    b.t_out.launch.p.rmap_off = u->qs * Ns;
  }
  if (int e = prep_gemm(u, u->final_lin, u->xm16, batch, 1, Tp, Ns, u->out32)) return e;
  if (u->graph_exec) {            // the captured step bakes the launches of the previous batch
    cudaGraphExecDestroy(u->graph_exec);
    u->graph_exec = nullptr;
  }
  u->prepared_batch = batch;
  return 0;
}

// diffusion-time conditioning of `rows` timesteps (t_dev): c = SiLU(time_proj(time_blocks(t))), then every block's AdaLN
// vectors from SiLU(c) in ONE GEMM (DiT4D_V4.py:363, :134-137, :222): 8 launches.  The four GEMM launches must have been
// prepared for `rows` rows with their outputs where the caller wants them.
int run_conditioning(cm_dit* u, int rows, DitLinear& t1, DitLinear& t2, DitLinear& tproj, DitLinear& adaln, cudaStream_t st) {
  const cm_dit_config& c = u->cfg;
  const int D = u->D, E = u->E;
  dit_gather_emb_kernel<<<rows, 128, 0, st>>>(u->params[u->p_table].ptr, u->t_dev, D, c.table_steps, u->e16);
  DIT_LAUNCH_CHECK();
  if (int e = conv_enqueue(t1.launch, st)) return e;
  dit_act16_kernel<<<grid_for((size_t)rows * E / 4), 256, 0, st>>>(u->h32, u->h16, (size_t)rows * E / 4, 1);
  DIT_LAUNCH_CHECK();
  if (int e = conv_enqueue(t2.launch, st)) return e;
  dit_act16_kernel<<<grid_for((size_t)rows * E / 4), 256, 0, st>>>(u->h2_32, u->h16, (size_t)rows * E / 4, 0);
  DIT_LAUNCH_CHECK();
  if (int e = conv_enqueue(tproj.launch, st)) return e;
  dit_act16_kernel<<<grid_for((size_t)rows * D / 4), 256, 0, st>>>(u->c32, u->e16, (size_t)rows * D / 4, 2);
  DIT_LAUNCH_CHECK();
  return conv_enqueue(adaln.launch, st);
}

// one denoiser evaluation: (t_dev |mods row 0) / future / past -> out32 (FinalLayer output), then un-patch (+ optional
// update).  ld_mods = Jtot: per-sample AdaLN vectors computed here from t_dev; ld_mods = 0: mods row 0 already holds the
// step's vectors for the whole batch (sampling: batch-uniform timestep, table row selected by the caller).
int run_forward(cm_dit* u, int B, const float* future, const float* past, UnpatchParams up, int ld_mods, cudaStream_t st,
                int64_t* launches) {
  const cm_dit_config& c = u->cfg;
  const int D = u->D, Tp = u->Tp, Ns = u->Ns, R = B * u->tokens;
  int64_t n = 0;
  if (ld_mods != 0) {
    if (int e = run_conditioning(u, B, u->t1, u->t2, u->tproj, u->adaln, st)) return e;
    n += 8;
  }
  // ---- patchify + positional embeddings
  PatchGeom g{B, c.in_channels, c.rows, c.cols, c.past_len, c.future_len, c.patch, c.t_patch, u->hp, u->wp, Tp, u->Kpad};
  dit_patchify_kernel<<<grid_for((size_t)R * u->Kpad), 256, 0, st>>>(future, past, g, u->a16);
  DIT_LAUNCH_CHECK();
  if (int e = conv_enqueue(u->patch.launch, st)) return e;
  dit_add_pos_kernel<<<grid_for((size_t)R * D / 4), 256, 0, st>>>(u->x32, u->params[u->p_spatial].ptr, u->params[u->p_temporal].ptr, R, Tp,
                                                                  Ns, D);
  DIT_LAUNCH_CHECK();
  n += 3;
  const int ln_blocks = (R * 32 + 255) / 256;
  for (int i = 0; i < c.depth; ++i) {
    cm_dit::Block& b = u->blocks[i];
    const int mo = i * 9 * D;     // chunk(9): shift1, scale1, gate1, shift2, scale2, gate2, shift3, scale3, gate3
    // 1. spatial self-attention (every temporal slot is its own sequence of Ns tokens)
    dit_ln_mod_kernel<<<ln_blocks, 256, 0, st>>>(u->x32, u->mods, ld_mods, mo, mo + D, u->tokens, R, D, u->xm16);
    DIT_LAUNCH_CHECK();
    if (int e = conv_enqueue(b.s_in.launch, st)) return e;
    if (int e = attn_core_enqueue(u->qkv32, u->ctx16, B * Tp, Ns, D, c.heads, st, 1)) return e;
    {
      ConvLaunch L = b.s_out.launch;
      L.p.gate = u->mods + mo + 2 * D;
      L.p.gate_ld = ld_mods;
      if (int e = conv_enqueue(L, st)) return e;
    }
    // 2. temporal cross-attention (future slots of every spatial patch query all of its slots)
    dit_ln_mod_kernel<<<ln_blocks, 256, 0, st>>>(u->x32, u->mods, ld_mods, mo + 3 * D, mo + 4 * D, u->tokens, R, D, u->xm16);
    DIT_LAUNCH_CHECK();
    if (int e = conv_enqueue(b.t_in.launch, st)) return e;
    {
      const int warps = B * u->nq * Ns * c.heads;
      dit_tattn_kernel<<<(warps * 32 + 255) / 256, 256, 0, st>>>(u->qkv32, u->ctx16, B, Tp, Ns, D, c.heads, u->qs);
      DIT_LAUNCH_CHECK();
    }
    {
      ConvLaunch L = b.t_out.launch;
      L.p.gate = u->mods + mo + 5 * D;
      L.p.gate_ld = ld_mods;
      if (int e = conv_enqueue(L, st)) return e;
    }
    // 3. MLP
    dit_ln_mod_kernel<<<ln_blocks, 256, 0, st>>>(u->x32, u->mods, ld_mods, mo + 6 * D, mo + 7 * D, u->tokens, R, D, u->xm16);
    DIT_LAUNCH_CHECK();
    if (int e = conv_enqueue(b.fc1.launch, st)) return e;
    {
      ConvLaunch L = b.fc2.launch;
      L.p.gate = u->mods + mo + 8 * D;
      L.p.gate_ld = ld_mods;
      if (int e = conv_enqueue(L, st)) return e;
    }
    n += 11;
  }
  // ---- final layer (chunk(2): shift, scale) + un-patch (+ reverse-step update)
  const int mo = c.depth * 9 * D;
  dit_ln_mod_kernel<<<ln_blocks, 256, 0, st>>>(u->x32, u->mods, ld_mods, mo, mo + D, u->tokens, R, D, u->xm16);
  DIT_LAUNCH_CHECK();
  if (int e = conv_enqueue(u->final_lin.launch, st)) return e;
  up.out = u->out32;
  up.ld = u->Nout;
  up.B = B; up.C = c.out_channels; up.H = c.rows; up.W = c.cols; up.P = c.past_len; up.F = c.future_len;
  up.p = c.patch; up.pt = c.t_patch; up.hp = u->hp; up.wp = u->wp; up.Tp = Tp;
  dit_unpatch_step_kernel<<<grid_for((size_t)B * c.rows * c.cols * c.future_len), 256, 0, st>>>(up);
  DIT_LAUNCH_CHECK();
  n += 3;
  if (launches) *launches += n;
  return 0;
}

// AdaLN vectors of EVERY timestep, once per weight load: the conditioning path in chunks of 128 timesteps with the last
// GEMM writing straight into the table.  Needs the arena of a batch >= 128 rows for the time-path buffers (they are
// sized for max(batch, 128) rows).
int build_mods_table(cm_dit* u, cudaStream_t st) {
  if (u->table_ready) return 0;
  const cm_dit_config& c = u->cfg;
  if (!u->mods_table) CM_CUDA(cudaMalloc(&u->mods_table, (size_t)c.table_steps * u->Jtot * sizeof(float)));
  for (int t0 = 0; t0 < c.table_steps; t0 += 128) {
    const int rows = c.table_steps - t0 < 128 ? c.table_steps - t0 : 128;
    DitLinear t1 = u->t1, t2 = u->t2, tp = u->tproj, ad = u->adaln;
    if (int e = prep_gemm(u, t1, u->e16, rows, 1, 1, 1, u->h32)) return e;
    if (int e = prep_gemm(u, t2, u->h16, rows, 1, 1, 1, u->h2_32)) return e;
    if (int e = prep_gemm(u, tp, u->h16, rows, 1, 1, 1, u->c32)) return e;
    if (int e = prep_gemm(u, ad, u->e16, rows, 1, 1, 1, u->mods_table + (size_t)t0 * u->Jtot)) return e;
    dit_fill_t_range_kernel<<<1, 128, 0, st>>>(u->t_dev, rows, t0);
    DIT_LAUNCH_CHECK();
    if (int e = run_conditioning(u, rows, t1, t2, tp, ad, st)) return e;
  }
  u->table_ready = true;
  return 0;
}

int ensure_ready(cm_dit* u, int batch, cudaStream_t st) {
  CM_CHECK(batch >= 1, "batch must be >= 1");
  CM_CHECK(u->packed, "cm_dit_pack has not been called since parameters were bound");
  (void)st;
  if (int e = reserve(u, batch)) return e;
  return prepare(u, batch);
}

}  // namespace

extern "C" {

int cm_dit_create(const cm_dit_config* cfg, cm_dit** out) {
  CM_CHECK(cfg && out, "null argument");
  cm_dit* u = new cm_dit();
  u->cfg = *cfg;
  if (int e = build(u)) {
    delete u;
    return e;
  }
  *out = u;
  return 0;
}

int cm_dit_destroy(cm_dit* u) {
  if (!u) return 0;
  if (u->arena) cudaFree(u->arena);
  if (u->wpack) cudaFree(u->wpack);
  if (u->adaln_wbuf) cudaFree(u->adaln_wbuf);
  if (u->adaln_bbuf) cudaFree(u->adaln_bbuf);
  if (u->patch_wbuf) cudaFree(u->patch_wbuf);
  if (u->d_coef) cudaFree(u->d_coef);
  if (u->d_tsteps) cudaFree(u->d_tsteps);
  if (u->d_step) cudaFree(u->d_step);
  if (u->d_chain) cudaFree(u->d_chain);
  if (u->mods_table) cudaFree(u->mods_table);
  if (u->graph_exec) cudaGraphExecDestroy(u->graph_exec);
  delete u;
  return 0;
}

int cm_dit_param_count(const cm_dit* u) { return u ? (int)u->params.size() : -1; }

int cm_dit_param_info(const cm_dit* u, int idx, char* name, int name_cap, int64_t* shape5, int* ndim) {
  CM_CHECK(u && idx >= 0 && idx < (int)u->params.size(), "parameter index out of range");
  const DitParam& p = u->params[idx];
  if (name && name_cap > 0) {
    strncpy(name, p.name.c_str(), name_cap - 1);
    name[name_cap - 1] = 0;
  }
  if (shape5)
    for (size_t i = 0; i < 5; ++i) shape5[i] = i < p.shape.size() ? p.shape[i] : 1;
  if (ndim) *ndim = (int)p.shape.size();
  return 0;
}

int cm_dit_bind_params(cm_dit* u, const void* const* ptrs, int count) {
  CM_CHECK(u && ptrs && count == (int)u->params.size(), "expected %d parameter pointers", u ? (int)u->params.size() : -1);
  for (int i = 0; i < count; ++i) {
    CM_CHECK(ptrs[i] != nullptr, "parameter '%s': null pointer", u->params[i].name.c_str());
    u->params[i].ptr = static_cast<const float*>(ptrs[i]);
  }
  u->packed = false;
  u->prepared_batch = 0;      // the GEMM launches bake bias pointers
  return 0;
}

int cm_dit_pack(cm_dit* u, void* stream) {
  CM_CHECK(u, "null handle");
  return pack_all(u, static_cast<cudaStream_t>(stream));
}

double cm_dit_flops_per_sample(const cm_dit* u) { return u ? u->flops_per_sample : 0.0; }
int64_t cm_dit_last_launches(const cm_dit* u) { return u ? u->last_launches : -1; }

int cm_dit_forward(cm_dit* u, const float* future, const int64_t* t, const float* past, float* eps_out, int batch, void* stream) {
  CM_CHECK(u && future && t && past && eps_out, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = ensure_ready(u, batch, st)) return e;
  CM_CUDA(cudaMemcpyAsync(u->t_dev, t, (size_t)batch * sizeof(long long), cudaMemcpyDeviceToDevice, st));
  UnpatchParams up{};
  up.eps_out = eps_out;
  u->last_launches = 0;
  return run_forward(u, batch, future, past, up, u->Jtot, st, &u->last_launches);
}

int cm_dit_sample(cm_dit* u, const cm_chain_args* a, void* stream) {
  CM_CHECK(u && a && a->past && a->x && a->tsteps && a->coef, "null argument");
  CM_CHECK(a->n >= 1 && a->nsteps >= 1, "n and nsteps must be >= 1");
  CM_CHECK(a->mode == 0 || a->mode == 1, "mode must be 0 (DDPM) or 1 (DDIM)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = ensure_ready(u, a->n, st)) return e;
  if (int e = build_mods_table(u, st)) return e;
  const cm_dit_config& c = u->cfg;
  for (int i = 0; i < a->nsteps; ++i)
    CM_CHECK(a->tsteps[i] >= 0 && a->tsteps[i] < c.table_steps, "timestep %d outside the table", a->tsteps[i]);
  if (a->nsteps > u->coef_cap) {
    if (u->d_coef) CM_CUDA(cudaFree(u->d_coef));
    if (u->d_tsteps) CM_CUDA(cudaFree(u->d_tsteps));
    CM_CUDA(cudaMalloc(&u->d_coef, (size_t)a->nsteps * 8 * sizeof(float)));
    CM_CUDA(cudaMalloc(&u->d_tsteps, (size_t)a->nsteps * sizeof(int)));
    u->coef_cap = a->nsteps;
    if (u->graph_exec) {
      cudaGraphExecDestroy(u->graph_exec);
      u->graph_exec = nullptr;
    }
  }
  if (!u->d_step) CM_CUDA(cudaMalloc(&u->d_step, sizeof(int)));
  if (!u->d_chain) CM_CUDA(cudaMalloc(&u->d_chain, 2 * sizeof(unsigned long long)));
  // step index, timesteps, coefficients, Philox seed / shard offset, x and past all travel through buffers the handle
  // owns: one captured step serves every chain of this (n, mode, noise, history)
  const unsigned long long chain_host[2] = {a->seed, static_cast<unsigned long long>(a->sample_offset)};
  CM_CUDA(cudaMemcpyAsync(u->d_coef, a->coef, (size_t)a->nsteps * 8 * sizeof(float), cudaMemcpyHostToDevice, st));
  CM_CUDA(cudaMemcpyAsync(u->d_tsteps, a->tsteps, (size_t)a->nsteps * sizeof(int), cudaMemcpyHostToDevice, st));
  CM_CUDA(cudaMemcpyAsync(u->d_chain, chain_host, sizeof(chain_host), cudaMemcpyHostToDevice, st));
  CM_CUDA(cudaMemsetAsync(u->d_step, 0, sizeof(int), st));
  const size_t xel = (size_t)a->n * c.out_channels * c.rows * c.cols * c.future_len;
  const size_t pel = (size_t)a->n * c.in_channels * c.rows * c.cols * c.past_len;
  CM_CUDA(cudaMemcpyAsync(u->chain_x, a->x, xel * sizeof(float), cudaMemcpyDeviceToDevice, st));
  CM_CUDA(cudaMemcpyAsync(u->chain_past, a->past, pel * sizeof(float), cudaMemcpyDeviceToDevice, st));
  UnpatchParams up{};
  up.x = u->chain_x;
  up.coef = u->d_coef;
  up.step_dev = u->d_step;
  up.mode = a->mode;
  up.noise = a->noise;
  up.chain_dev = u->d_chain;
  up.history = a->history;
  auto one_step = [&](cudaStream_t s2, int64_t* launches) -> int {
    dit_select_mods_kernel<<<8, 256, 0, s2>>>(u->mods, u->mods_table, u->d_tsteps, u->d_step, u->Jtot);
    CM_CUDA(cudaGetLastError());
    // the denoiser reads the CURRENT x (the chain's staging copy) as its `future` input
    if (int e = run_forward(u, a->n, u->chain_x, u->chain_past, up, 0, s2, launches)) return e;
    dit_advance_kernel<<<1, 1, 0, s2>>>(u->d_step);
    CM_CUDA(cudaGetLastError());
    if (launches) *launches += 2;
    return 0;
  };
  u->last_launches = 0;
  if (!a->use_graph) {
    for (int i = 0; i < a->nsteps; ++i)
      if (int e = one_step(st, &u->last_launches)) return e;
  } else {
    const cm_chain_args& k = u->graph_key;
    const bool reuse = u->graph_exec && k.n == a->n && k.mode == a->mode && k.noise == a->noise && k.history == a->history;
    if (!reuse) {
      if (u->graph_exec) {
        cudaGraphExecDestroy(u->graph_exec);
        u->graph_exec = nullptr;
      }
      cudaStream_t cs;
      CM_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
      cudaGraph_t g = nullptr;
      int64_t per_step = 0;
      cudaError_t ce = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
      int e = 0;
      if (ce == cudaSuccess) {
        e = one_step(cs, &per_step);
        ce = cudaStreamEndCapture(cs, &g);
      }
      cudaStreamDestroy(cs);
      if (e || ce != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        if (e) return e;
        CM_CUDA(ce);
      }
      CM_CUDA(cudaGraphInstantiate(&u->graph_exec, g, 0));
      cudaGraphDestroy(g);
      u->graph_key = *a;
      u->graph_launches_per_step = per_step;
    }
    for (int i = 0; i < a->nsteps; ++i) CM_CUDA(cudaGraphLaunch(u->graph_exec, st));
    u->last_launches = u->graph_launches_per_step * a->nsteps;
  }
  CM_CUDA(cudaMemcpyAsync(a->x, u->chain_x, xel * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // extern "C"
