// UNet execution plan behind the C ABI (include/crowdmod_b200.h); its reverse chain runs on the shared driver of chain.cu.
//
// The plan is a flat op list derived from the same constructor arguments the reference UNet
// takes (models/backbones/unet.py:11-122) and executed in the order of UNet.forward
// (unet.py:124-167) / ResnetBlock.forward (layers.py:55-78) / AttentionBlock.forward
// (layers.py:12-18).  torch.cat calls disappear (GroupNorm reads two sources), match_input is
// a K-slab of conv_2, residual/time-embedding adds live in conv epilogues, nearest-x2
// upsampling is folded into 8 phase convolutions, and DDPM.step (ddpm.py:25-38) is the
// epilogue of the last conv.
#include <string.h>

#include <algorithm>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/crowdmod_b200.h"
#include "backward.cuh"
#include "conv_run.cuh"
#include "kernels.cuh"
#include "pack.cuh"

namespace cm {

struct ParamEntry {
  std::string name;
  std::vector<int64_t> shape;
  const float* ptr = nullptr;
  int64_t numel() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};

struct Tens {
  int level = 0;
  int C = 0;
  bool need32 = false, need16 = false;
  float* p32 = nullptr;
  __half* p16 = nullptr;
  // GroupNorm statistics records emitted by the plane-tile conv that produces this tensor
  bool gn_src = false;      // consumed by a GroupNorm
  float* rec = nullptr;     // [batch][D*H][C] float4 (sized for the finest unit split)
  GnRec gn_rec{};           // what the producing launch writes there (units == 0: no records)
};

enum OpType { OP_FIRST, OP_GN, OP_CONV, OP_ATTN, OP_FINAL };

struct Op {
  OpType type;
  std::string tag;
  // GN
  int src0 = -1, src1 = -1, gamma = -1, beta = -1, silu = 0, out_norm = -1, out_raw = -1;
  // CONV
  int mode = 0, in = -1, extra = -1, w = -1, wx = -1, bias = -1, bias2 = -1, temb_off = -1,
      resid = -1, out = -1, cin = 0, cin_extra = 0, cout = 0, in_level = 0;
  size_t wpack_off = 0;   // element offset into the packed-weight buffer
  size_t wpack2_off = 0;  // same in the training forward's cache (hi|lo pair activation operands, K doubled)
  ConvRun fwd;
  // ATTN
  int qkv = -1, ctx = -1, heads = 4;
  // training (backward) bookkeeping
  int gn_index = -1;        // GN: slot of the saved (mean, rstd) statistics
  int drop_off = -1;        // GN normalize_2: column offset of the block's Dropout3d scales
  size_t dpack_off = 0, dxpack_off = 0;   // CONV: dgrad weight caches (main / fused 1x1 source)
  size_t g_off = 0;         // CONV: offset of the packed-K weight-gradient scratch
  size_t colsum_off = 0;    // CONV: per-sample channel sums of dOut ([B][cout])
  ConvRun dgrad, dgrad_x;   // data gradients of the main and the fused 1x1x1 source
  WgradRun wgrad;
};

struct Level {
  int D, H, W;   // frames, grid rows, grid cols: activations are stored [B, frames, rows, cols, C]
                 // (cols innermost: TMA im2col cost grows with the number of W-rows a tile spans)
  int pps() const { return D * H * W; }
};

}  // namespace cm

using namespace cm;

struct cm_unet {
  cm_unet_config cfg;
  std::vector<ParamEntry> params;
  std::map<std::string, int> pindex;
  std::vector<Tens> tens;
  std::vector<Op> ops;
  std::vector<Level> levels;
  // time embedding
  std::vector<int> temb_dense_w, temb_dense_b, temb_couts, temb_offs;
  int temb_ld = 0;
  int p_table = -1, p_w1 = -1, p_b1 = -1, p_w2 = -1, p_b2 = -1;
  int p_first_w = -1, p_first_b = -1, p_final_w = -1, p_final_b = -1;
  // first conv on the tensor cores: the 3(+)-channel input is packed into a zero-padded 32-channel fp16
  // operand and run through the plane-tile or res32 kernel (falls back to first_conv_kernel when neither covers it)
  int first_in = -1;
  size_t first_wpack_off = 0;
  ConvRun first;
  WgradRun first_wg;                   // first conv's weight gradient over the packed operand (edge_wgrad_kinds)
  size_t first_g_off = 0;              // its packed-K scratch (27 taps x 32 packed channels x base) and channel-sum slot
  int first_colsum_off = 0;
  WgradRun final_wg;                   // final conv's weight gradient the same way: d_eps packed into 32 fp16 columns
  size_t final_g_off = 0;              // its packed-K scratch (27 taps x cin x 32)
  __half* final_d16 = nullptr;         // [B * L * H * W][32]: columns >= out_channels and past frames stay zero
  // device state
  __half* wpack = nullptr;
  size_t wpack_elems = 0;
  float* temb_table = nullptr;          // [table_steps][temb_ld]
  const float** d_wd = nullptr;
  const float** d_bd = nullptr;
  long long* d_up_tab = nullptr;        // per conv weight-gradient unpack parameters
  std::vector<long long> up_tab_host;
  long long* d_rs_tab = nullptr;        // per conv bias {channel-sum offset, row stride, cout, gradient offset}
  std::vector<long long> rs_tab_host;
  long long* d_gn_tab = nullptr;        // per GroupNorm {chsum offset, C, dgamma offset, dbeta offset}
  std::vector<long long> gn_tab_host;
  long long* d_goff_w = nullptr;        // flat-gradient offsets of every block's dense_1 weight / bias
  long long* d_goff_b = nullptr;
  int* d_couts = nullptr;
  int* d_offs = nullptr;
  bool packed = false;                  // forward cache, single-operand layout, is current
  bool pack_called = false;
  // table-driven packing (pack.cuh): [forward jobs | dgrad jobs], rebuilt when parameter storage moves
  std::vector<PackJob> jobs_host;
  PackJob* d_jobs = nullptr;
  int n_jobs_fwd = 0, n_jobs_fwd2 = 0, n_jobs_dgrad = 0, jobs_cap = 0;
  bool jobs_dirty = true;
  int dgrad_dup = 2;                    // cfg.dgrad_terms: hi|lo dOut pair in every data-gradient conv
  int act_dup_train = 2;                // cfg.train_act_terms: hi|lo activation pair in the training forward
  __half* wpack2 = nullptr;             // forward weights packed against hi|lo activation rows (training)
  size_t wpack2_elems = 0, first_wpack2_off = 0;
  bool packed2 = false;
  int live_batch = 0;                   // batch the conv launches are prepared for (0: none)
  int live_dup = 1;                     // and activation-operand layout
  // workspace (per reserved batch)
  int reserved_batch = 0;
  uint8_t* arena = nullptr;
  size_t arena_bytes = 0;
  float* temb_batch = nullptr;          // [batch][temb_ld]
  float* gn_partial = nullptr;          // [batch][GN chunks][8][2] slice statistics (reused by every GN)
  float* chain_x = nullptr;             // staging copies of the caller's x / past: the graph bakes THESE pointers
  float* chain_past = nullptr;
  ChainDriver chain;                    // chain state, graph cache and stats of cm_ddpm_sample
  int64_t last_backward_launches = 0;
  double flops_per_sample = 0.0;
  // ---- training state (cm_unet_train_forward / cm_unet_backward) ----
  int n_gn = 0;
  size_t dpack_elems = 0, g_elems = 0, colsum_per_sample = 0;
  int max_gn_channels = 0;
  __half* dpack = nullptr;              // dgrad weight caches
  bool dpacked = false;
  std::vector<size_t> grad_off;         // flat gradient buffer: offset of parameter i
  size_t grad_total = 0;
  int train_reserved = 0, train_prepared = 0;
  std::vector<float*> attn_lse;         // per op, attention core with attn_uses_long: row log-sum-exp [B][heads][S], then as
                                        // many floats of backward workspace (reserve_train)
  uint8_t* tarena = nullptr;
  size_t tarena_bytes = 0;
  std::vector<float*> g32;              // per tensor: fp32 gradient [B][pixels][C]
  std::vector<__half*> g16;             // conv outputs: fp16 copy of the gradient (MMA operand)
  float* gn_stats = nullptr;            // [n_gn][B][8][2]
  float* gn_bwd_partial = nullptr;      // [B][32][Cmax][2]
  float* gn_chsum = nullptr;            // [B][Cmax][2]
  uint8_t* zero_region = nullptr;       // G scratch | colsums | dtemb | max word, zeroed per backward
  size_t zero_bytes = 0;
  float* G = nullptr;
  float* colsum = nullptr;
  float* dtemb = nullptr;
  unsigned int* max_word = nullptr;
  float* tsave_e = nullptr;             // time-MLP saves / scratch, all [B][E] except e: [B][base]
  float* tsave_h1 = nullptr; float* tsave_h2 = nullptr;
  float* ts1 = nullptr; float* ts2 = nullptr; float* tds2 = nullptr; float* tdh2 = nullptr;
  float* tds1 = nullptr; float* tdh1 = nullptr;
  float* loss_scale = nullptr;          // device {S, 1/S}
  // the forward whose activations currently sit in the arena
  int live_train_batch = 0;
  const float* live_future = nullptr;
  const float* live_past = nullptr;
  const float* live_drop = nullptr;
  // reproducible backward (cm_unet_set_deterministic): every weight-gradient and channel-sum reduction stores per-CTA
  // partials into det_part and adds them in a fixed order; det_part is allocated by the first such backward
  int deterministic = 0;
  float* det_part = nullptr;
  size_t det_part_elems = 0;

  int add_param(const std::string& name, std::vector<int64_t> shape) {
    ParamEntry e;
    e.name = name;
    e.shape = std::move(shape);
    params.push_back(e);
    pindex[name] = (int)params.size() - 1;
    return (int)params.size() - 1;
  }
  int add_tensor(int level, int C) {
    Tens t;
    t.level = level;
    t.C = C;
    tens.push_back(t);
    return (int)tens.size() - 1;
  }
};

namespace {

// ---- plan construction ---------------------------------------------------------------------

int add_gn(cm_unet* u, const std::string& prefix, int src0, int src1, int silu, bool want_raw,
           int* out_norm, int* out_raw, int drop_off = -1) {
  const int C = u->tens[src0].C + (src1 >= 0 ? u->tens[src1].C : 0);
  Op op;
  op.type = OP_GN;
  op.tag = prefix;
  op.src0 = src0;
  op.src1 = src1;
  op.gamma = u->add_param(prefix + ".weight", {C});
  op.beta = u->add_param(prefix + ".bias", {C});
  op.silu = silu;
  u->tens[src0].gn_src = true;
  if (src1 >= 0) u->tens[src1].gn_src = true;
  op.gn_index = u->n_gn++;
  op.drop_off = drop_off;
  if (C > u->max_gn_channels) u->max_gn_channels = C;
  u->tens[src0].need32 = true;
  if (src1 >= 0) u->tens[src1].need32 = true;
  op.out_norm = u->add_tensor(u->tens[src0].level, C);
  u->tens[op.out_norm].need16 = true;
  if (want_raw) {
    op.out_raw = u->add_tensor(u->tens[src0].level, C);
    u->tens[op.out_raw].need16 = true;
  }
  *out_norm = op.out_norm;
  if (out_raw) *out_raw = op.out_raw;
  u->ops.push_back(op);
  return 0;
}

// generic conv op; weight/bias params are registered by the caller (ordering of state_dict)
int add_conv(cm_unet* u, const std::string& tag, int mode, int in, int extra, int w, int wx,
             int bias, int bias2, int temb_off, int resid, int cout, int out_level) {
  Op op;
  op.type = OP_CONV;
  op.tag = tag;
  op.mode = mode;
  op.in = in;
  op.extra = extra;
  op.w = w;
  op.wx = wx;
  op.bias = bias;
  op.bias2 = bias2;
  op.temb_off = temb_off;
  op.resid = resid;
  op.cin = u->tens[in].C;
  op.cin_extra = extra >= 0 ? u->tens[extra].C : 0;
  op.cout = cout;
  op.in_level = u->tens[in].level;
  u->tens[in].need16 = true;
  if (extra >= 0) u->tens[extra].need16 = true;
  if (resid >= 0) u->tens[resid].need32 = true;
  op.out = u->add_tensor(out_level, cout);
  op.wpack_off = u->wpack_elems;
  u->wpack_elems += (size_t)u->cfg.weight_terms * cout * conv_packed_k(mode, op.cin, op.cin_extra);
  op.wpack2_off = u->wpack2_elems;
  u->wpack2_elems += (size_t)u->cfg.weight_terms * cout * conv_packed_k(mode, 2 * op.cin, 2 * op.cin_extra);
  op.dpack_off = u->dpack_elems;
  u->dpack_elems += (size_t)u->cfg.weight_terms * op.cin * dgrad_packed_k(mode, cout, u->dgrad_dup);
  op.dxpack_off = u->dpack_elems;
  u->dpack_elems += (size_t)u->cfg.weight_terms * op.cin_extra * cout * u->dgrad_dup;
  op.g_off = u->g_elems;
  u->g_elems += wgrad_g_elems(mode, op.cin, op.cin_extra, cout);
  op.colsum_off = u->colsum_per_sample;
  u->colsum_per_sample += cout;
  u->ops.push_back(op);
  return op.out;
}

int add_resblock(cm_unet* u, const std::string& prefix, int src0, int src1, int cout, bool attn) {
  const int level = u->tens[src0].level;
  const int cin = u->tens[src0].C + (src1 >= 0 ? u->tens[src1].C : 0);
  const bool has_match = cin != cout;
  const int E = u->cfg.base_channels * u->cfg.time_multiple;
  // state_dict order follows ResnetBlock.__init__ (layers.py:30-52)
  int a1, xr = -1;
  add_gn(u, prefix + ".normalize_1", src0, src1, 1, has_match, &a1, &xr);
  const int w1 = u->add_param(prefix + ".conv_1.weight", {cout, cin, 3, 3, 3});
  const int b1 = u->add_param(prefix + ".conv_1.bias", {cout});
  const int dw = u->add_param(prefix + ".dense_1.weight", {cout, E});
  const int db = u->add_param(prefix + ".dense_1.bias", {cout});
  const int temb_off = u->temb_ld;
  u->temb_dense_w.push_back(dw);
  u->temb_dense_b.push_back(db);
  u->temb_couts.push_back(cout);
  u->temb_offs.push_back(temb_off);
  u->temb_ld += cout;
  const int h1 = add_conv(u, prefix + ".conv_1", 0, a1, -1, w1, -1, b1, -1, temb_off, -1, cout, level);
  int a2;
  add_gn(u, prefix + ".normalize_2", h1, -1, 1, false, &a2, nullptr, temb_off);   // Dropout3d (layers.py:70)
  const int w2 = u->add_param(prefix + ".conv_2.weight", {cout, cout, 3, 3, 3});
  const int b2 = u->add_param(prefix + ".conv_2.bias", {cout});
  int wm = -1, bm = -1;
  if (has_match) {
    wm = u->add_param(prefix + ".match_input.weight", {cout, cin, 1, 1, 1});
    bm = u->add_param(prefix + ".match_input.bias", {cout});
  }
  if (!has_match && src1 >= 0) {
    set_error("identity residual with two sources is impossible");
    return -1;
  }
  int o = add_conv(u, prefix + ".conv_2", 0, a2, has_match ? xr : -1, w2, wm, b2, bm, -1,
                   has_match ? -1 : src0, cout, level);
  if (attn) {
    // AttentionBlock (layers.py:5-18)
    int a3;
    add_gn(u, prefix + ".attention.group_norm", o, -1, 0, false, &a3, nullptr);
    const int wi = u->add_param(prefix + ".attention.mhsa.in_proj_weight", {3 * cout, cout});
    const int bi = u->add_param(prefix + ".attention.mhsa.in_proj_bias", {3 * cout});
    const int wo = u->add_param(prefix + ".attention.mhsa.out_proj.weight", {cout, cout});
    const int bo = u->add_param(prefix + ".attention.mhsa.out_proj.bias", {cout});
    const int qkv = add_conv(u, prefix + ".attention.in_proj", 3, a3, -1, wi, -1, bi, -1, -1, -1,
                             3 * cout, level);
    u->tens[qkv].need32 = true;
    Op at;
    at.type = OP_ATTN;
    at.tag = prefix + ".attention.core";
    at.qkv = qkv;
    at.heads = 4;   // layers.py:10
    at.ctx = u->add_tensor(level, cout);
    u->tens[at.ctx].need16 = true;
    u->ops.push_back(at);
    o = add_conv(u, prefix + ".attention.out_proj", 3, at.ctx, -1, wo, -1, bo, -1, -1, o, cout, level);
  }
  return o;
}

int build_plan(cm_unet* u) {
  const cm_unet_config& c = u->cfg;
  CM_CHECK(c.num_levels >= 1 && c.num_levels <= CM_MAX_LEVELS, "num_levels out of range");
  CM_CHECK(c.base_channels % 32 == 0 && c.base_channels > 0, "base_channels must be a multiple of 32");
  CM_CHECK(c.in_channels >= 1 && c.in_channels <= 4 && c.out_channels >= 1 && c.out_channels <= 4,
           "in/out channels must be in 1..4");
  CM_CHECK(c.weight_terms == 1 || c.weight_terms == 2, "weight_terms must be 1 or 2");
  CM_CHECK(c.num_res_blocks >= 1, "num_res_blocks must be >= 1");
  const int div = 1 << (c.num_levels - 1);
  const int L = c.past_len + c.future_len;
  CM_CHECK(c.rows % div == 0 && c.cols % div == 0 && L % div == 0,
           "rows/cols/(past+future) must be divisible by 2^(levels-1)=%d (skip concat, unet.py:160)", div);
  u->levels.resize(c.num_levels);
  for (int l = 0; l < c.num_levels; ++l) u->levels[l] = {L >> l, c.rows >> l, c.cols >> l};

  const int base = c.base_channels, E = base * c.time_multiple;
  // state_dict order: time_embeddings, first, encoder, bottleneck, decoder, final (unet.py:27-122)
  u->p_table = u->add_param("time_embeddings.time_blocks.0.weight", {c.table_steps, base});
  u->p_w1 = u->add_param("time_embeddings.time_blocks.1.weight", {E, base});
  u->p_b1 = u->add_param("time_embeddings.time_blocks.1.bias", {E});
  u->p_w2 = u->add_param("time_embeddings.time_blocks.3.weight", {E, E});
  u->p_b2 = u->add_param("time_embeddings.time_blocks.3.bias", {E});
  u->p_first_w = u->add_param("first.weight", {base, c.in_channels, 3, 3, 3});
  u->p_first_b = u->add_param("first.bias", {base});

  u->first_in = u->add_tensor(0, 32);
  u->tens[u->first_in].need16 = true;
  u->first_wpack_off = u->wpack_elems;
  u->wpack_elems += (size_t)c.weight_terms * base * 27 * 32;
  u->first_wpack2_off = u->wpack2_elems;
  u->wpack2_elems += (size_t)c.weight_terms * base * 27 * 64;
  Op first;
  first.type = OP_FIRST;
  first.tag = "first";
  first.out = u->add_tensor(0, base);
  u->tens[first.out].need32 = true;
  u->ops.push_back(first);
  u->first_g_off = u->g_elems;
  u->g_elems += (size_t)27 * 32 * base;
  u->first_colsum_off = u->colsum_per_sample;
  u->colsum_per_sample += base;

  int cur = first.out;
  std::vector<int> skips{cur};
  int in_ch = base, idx = 0;
  for (int level = 0; level < c.num_levels; ++level) {
    const int out_ch = base * c.mult[level];
    for (int r = 0; r < c.num_res_blocks; ++r) {
      cur = add_resblock(u, "encoder_blocks." + std::to_string(idx++), cur, -1, out_ch, c.attn[level] != 0);
      if (cur < 0) return 3;
      in_ch = out_ch;
      skips.push_back(cur);
    }
    if (level != c.num_levels - 1) {
      const std::string p = "encoder_blocks." + std::to_string(idx++) + ".downsample";
      const int w = u->add_param(p + ".weight", {in_ch, in_ch, 3, 3, 3});
      const int b = u->add_param(p + ".bias", {in_ch});
      cur = add_conv(u, p, 1, cur, -1, w, -1, b, -1, -1, -1, in_ch, level + 1);
      skips.push_back(cur);
    }
  }
  cur = add_resblock(u, "bottleneck_blocks.0", cur, -1, in_ch, true);
  cur = add_resblock(u, "bottleneck_blocks.1", cur, -1, in_ch, false);
  idx = 0;
  for (int level = c.num_levels - 1; level >= 0; --level) {
    const int out_ch = base * c.mult[level];
    for (int r = 0; r < c.num_res_blocks + 1; ++r) {
      const int skip = skips.back();
      skips.pop_back();
      cur = add_resblock(u, "decoder_blocks." + std::to_string(idx++), cur, skip, out_ch,
                         c.attn[level] != 0);
      if (cur < 0) return 3;
      in_ch = out_ch;
    }
    if (level != 0) {
      const std::string p = "decoder_blocks." + std::to_string(idx++) + ".upsample.1";
      const int w = u->add_param(p + ".weight", {in_ch, in_ch, 3, 3, 3});
      const int b = u->add_param(p + ".bias", {in_ch});
      cur = add_conv(u, p, 2, cur, -1, w, -1, b, -1, -1, -1, in_ch, level - 1);
    }
  }
  int afin;
  add_gn(u, "final.0", cur, -1, 1, false, &afin, nullptr);
  u->p_final_w = u->add_param("final.2.weight", {c.out_channels, in_ch, 3, 3, 3});
  u->p_final_b = u->add_param("final.2.bias", {c.out_channels});
  Op fin;
  fin.type = OP_FINAL;
  fin.tag = "final.2";
  fin.in = afin;
  fin.cin = in_ch;
  u->ops.push_back(fin);
  u->final_g_off = u->g_elems;
  u->g_elems += (size_t)27 * (edge_wgrad_kinds(in_ch) ? in_ch : 32) * 32;

  // algorithmic FLOPs per sample of the reference graph (dense formulation: 27-tap upsample
  // convs, separate 1x1 match_input, attention), SURVEY.md §8(d)
  double fl = 0.0;
  {
    const Level& l0 = u->levels[0];
    fl += 2.0 * l0.pps() * base * 27.0 * c.in_channels;
    fl += 2.0 * l0.pps() * c.out_channels * 27.0 * in_ch;
  }
  for (const Op& op : u->ops) {
    if (op.type == OP_CONV) {
      const Level& lo = u->levels[u->tens[op.out].level];
      const double taps = (op.mode == 3) ? 1.0 : 27.0;
      fl += 2.0 * lo.pps() * op.cout * (taps * op.cin + op.cin_extra);
    } else if (op.type == OP_ATTN) {
      const Level& lv = u->levels[u->tens[op.qkv].level];
      const double S = lv.pps(), Ce = u->tens[op.ctx].C;
      fl += 4.0 * S * S * Ce;
    }
  }
  u->flops_per_sample = fl;
  u->grad_off.resize(u->params.size());
  size_t go = 0;
  for (size_t i = 0; i < u->params.size(); ++i) {
    u->grad_off[i] = go;
    go += (size_t)((u->params[i].numel() + 3) / 4 * 4);   // keep every gradient 16-byte aligned
  }
  u->grad_total = go;
  return 0;
}

int check_params_bound(cm_unet* u) {
  for (auto& p : u->params)
    CM_CHECK(p.ptr != nullptr, "parameter '%s' not bound (cm_unet_set_param)", p.name.c_str());
  return 0;
}

// ---- workspace ---------------------------------------------------------------------------

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int reserve(cm_unet* u, int batch) {
  if (batch <= u->reserved_batch) return 0;
  chain_drop_graph(u->chain);
  if (u->arena) CM_CUDA(cudaFree(u->arena));
  u->arena = nullptr;
  u->train_prepared = 0;   // backward launches bake forward-arena pointers
  u->live_train_batch = 0;
  size_t off = 0;
  std::vector<size_t> o32(u->tens.size(), 0), o16(u->tens.size(), 0), orec(u->tens.size(), 0);
  for (size_t i = 0; i < u->tens.size(); ++i) {
    Tens& t = u->tens[i];
    const size_t n = (size_t)batch * u->levels[t.level].pps() * t.C;
    if (t.need32) { o32[i] = off; off = align_up(off + n * 4, 1024); }
    if (t.need16) { o16[i] = off; off = align_up(off + n * 2 * u->act_dup_train, 1024); }   // hi|lo rows in training
    if (t.gn_src) {
      const Level& lv = u->levels[t.level];
      orec[i] = off;
      off = align_up(off + (size_t)batch * lv.D * lv.H * t.C * 16, 1024);
    }
  }
  const size_t temb_off = off;
  off = align_up(off + (size_t)batch * u->temb_ld * 4, 1024);
  const size_t gnp_off = off;
  off = align_up(off + (size_t)batch * 32 * 8 * 3 * 4, 1024);   // [batch][GN2_MAX_SLICES][8][3]
  const Level& lv0 = u->levels[0];
  const size_t cx_off = off;
  off = align_up(off + (size_t)batch * u->cfg.out_channels * lv0.H * lv0.W * u->cfg.future_len * 4, 1024);
  const size_t cp_off = off;
  off = align_up(off + (size_t)batch * u->cfg.in_channels * lv0.H * lv0.W * (u->cfg.past_len > 0 ? u->cfg.past_len : 1) * 4, 1024);
  CM_CUDA(cudaMalloc(&u->arena, off));
  CM_CUDA(cudaMemset(u->arena, 0, off));
  u->arena_bytes = off;
  for (size_t i = 0; i < u->tens.size(); ++i) {
    Tens& t = u->tens[i];
    t.p32 = t.need32 ? reinterpret_cast<float*>(u->arena + o32[i]) : nullptr;
    t.p16 = t.need16 ? reinterpret_cast<__half*>(u->arena + o16[i]) : nullptr;
    t.rec = t.gn_src ? reinterpret_cast<float*>(u->arena + orec[i]) : nullptr;
    t.gn_rec = GnRec{};
  }
  u->temb_batch = reinterpret_cast<float*>(u->arena + temb_off);
  u->gn_partial = reinterpret_cast<float*>(u->arena + gnp_off);
  u->chain_x = reinterpret_cast<float*>(u->arena + cx_off);
  u->chain_past = reinterpret_cast<float*>(u->arena + cp_off);
  u->reserved_batch = batch;
  return 0;
}

// conv launches depend on the live batch (grid, tensor-map extents): (re)built per call batch
// dup = 1: single fp16 activation operands (sampling / eval); dup = 2: hi|lo pair rows (training forward)
int prepare_convs(cm_unet* u, int batch, int dup) {
  const __half* wbase = dup == 2 ? u->wpack2 : u->wpack;
  // res32 only for single fp16 operands: it has no hi|lo operand pairs
  const unsigned fast = dup == 1 ? CONV_PLANE | CONV_RES32 : CONV_PLANE;
  {
    const Level& l0 = u->levels[0];
    Tens& t = u->tens[u->ops[0].out];
    ConvEpilogue e{};
    e.bias = u->params[u->p_first_b].ptr;
    e.out32 = t.p32;
    e.lo_from = dup == 2 ? 32 : 0;
    e.stats_rec = t.rec;
    if (int rc = conv_run_prepare(&u->first, fast, 0, u->tens[u->first_in].p16, batch, l0.D, l0.H, l0.W, 32 * dup,
                                  nullptr, 0, wbase + (dup == 2 ? u->first_wpack2_off : u->first_wpack_off),
                                  u->cfg.base_channels, u->cfg.weight_terms, e))
      return rc;
    t.gn_rec = conv_run_records(u->first);
  }
  for (Op& op : u->ops) {
    if (op.type != OP_CONV) continue;
    const Level& li = u->levels[op.in_level];
    Tens& t = u->tens[op.out];
    ConvEpilogue e{};
    e.bias = op.bias >= 0 ? u->params[op.bias].ptr : nullptr;
    e.bias2 = op.bias2 >= 0 ? u->params[op.bias2].ptr : nullptr;
    e.resid = op.resid >= 0 ? u->tens[op.resid].p32 : nullptr;
    e.out32 = t.p32;
    e.out16 = t.p16;
    e.out16_ld = op.cout * dup;
    e.out16_lo = dup == 2 ? op.cout : 0;
    // hi|lo operand pairs against hi+lo weight terms: the lo x lo product (2^-22 of the result) is skipped
    e.lo_from = dup == 2 ? op.cin : 0;
    e.lo_from_x = dup == 2 ? op.cin_extra : 0;
    e.stats_rec = t.rec;
    CM_CHECK(e.out32 || e.out16, "conv '%s' has no consumer", op.tag.c_str());
    if (int rc = conv_run_prepare(&op.fwd, CONV_UMMA | fast, op.mode, u->tens[op.in].p16, batch, li.D, li.H, li.W,
                                  op.cin * dup, op.extra >= 0 ? u->tens[op.extra].p16 : nullptr, op.cin_extra * dup,
                                  wbase + (dup == 2 ? op.wpack2_off : op.wpack_off), op.cout, u->cfg.weight_terms, e))
      return rc;
    t.gn_rec = conv_run_records(op.fwd);
  }
  u->live_batch = batch;
  u->live_dup = dup;
  return 0;
}

// ---- execution -----------------------------------------------------------------------------

struct RunCtx {
  int batch;
  const float* future;
  const float* past;
  // time embedding source
  const float* temb;     // table or per-batch buffer
  const int* t_dev;      // device timestep (table mode) or nullptr
  int temb_bstride;
  FinalParams fin;       // eps_out / update parameters (act, w, geometry filled here)
  bool train = false;    // save GroupNorm statistics, apply Dropout3d scales
  const float* drop_scale = nullptr;   // [batch][temb_ld] or nullptr
  int dup = 1;           // activation-operand layout: 2 = hi|lo pair rows (training forward)
};

int run_ops(cm_unet* u, RunCtx& rc, cudaStream_t st, int64_t* launches,
            cudaEvent_t* events = nullptr) {
  const cm_unet_config& c = u->cfg;
  int op_index = 0;
  int skip = 0;            // ops already covered by a fused launch (their profile events still tick)
  for (size_t oi = 0; oi < u->ops.size(); ++oi) {
    Op& op = u->ops[oi];
    if (events) CM_CUDA(cudaEventRecord(events[op_index], st));
    ++op_index;
    if (skip > 0) { --skip; continue; }
    // sampling path: the whole AttentionBlock (GroupNorm, in_proj, core, out_proj + residual) is one launch
    if (op.type == OP_GN && !rc.train && oi + 3 < u->ops.size() &&
        u->ops[oi + 2].type == OP_ATTN && u->ops[oi + 1].type == OP_CONV && u->ops[oi + 3].type == OP_CONV &&
        u->ops[oi + 1].in == op.out_norm && op.src1 < 0) {
      const Op& ip = u->ops[oi + 1];
      const Op& at = u->ops[oi + 2];
      const Op& po = u->ops[oi + 3];
      const int Cc = u->tens[op.src0].C;
      const int S = u->levels[u->tens[op.src0].level].pps();
      if (attn_block_supported(S, Cc, at.heads) && c.weight_terms == 2 && ip.mode == 3 && po.mode == 3 && po.resid == op.src0 &&
          ip.extra < 0 && po.extra < 0 && ip.cout == 3 * Cc && po.cout == Cc) {
        if (int e = attn_block_enqueue(u->tens[op.src0].p32, u->params[op.gamma].ptr, u->params[op.beta].ptr,
                                       u->wpack + ip.wpack_off, u->params[ip.bias].ptr, u->wpack + po.wpack_off,
                                       u->params[po.bias].ptr, u->tens[po.out].p32, u->tens[po.out].p16, rc.batch,
                                       S, Cc, at.heads, 1e-5f, st))
          return e;
        if (launches) ++*launches;
        skip = 3;
        continue;
      }
    }
    switch (op.type) {
      case OP_FIRST: {
        const Level& l0 = u->levels[0];
        if (u->first.covered()) {
          if (int e = pack_first_input_enqueue(rc.future, rc.past, u->tens[u->first_in].p16, rc.batch, l0.H, l0.W,
                                               c.past_len, c.future_len, c.in_channels, rc.dup, st))
            return e;
          if (int e = conv_run_enqueue(u->first, st)) return e;
          if (launches) ++*launches;
          break;
        }
        if (int e = first_conv_enqueue(rc.future, rc.past, u->params[u->p_first_w].ptr,
                                       u->params[u->p_first_b].ptr, u->tens[op.out].p32, rc.batch,
                                       l0.H, l0.W, c.past_len, c.future_len, c.in_channels,
                                       c.base_channels, st))
          return e;
      } break;
      case OP_GN: {
        GnParams g{};
        g.src0 = u->tens[op.src0].p32;
        g.c0 = u->tens[op.src0].C;
        g.src1 = op.src1 >= 0 ? u->tens[op.src1].p32 : nullptr;
        g.c1 = op.src1 >= 0 ? u->tens[op.src1].C : 0;
        g.gamma = u->params[op.gamma].ptr;
        g.beta = u->params[op.beta].ptr;
        g.B = rc.batch;
        g.pixels = u->levels[u->tens[op.src0].level].pps();
        g.eps = 1e-5f;   // nn.GroupNorm default (layers.py:9,30,41)
        g.silu = op.silu;
        g.out_norm = u->tens[op.out_norm].p16;
        g.out_raw = op.out_raw >= 0 ? u->tens[op.out_raw].p16 : nullptr;
        g.dup = rc.dup;
        {
          const GnRec r0 = u->tens[op.src0].gn_rec;
          const GnRec r1 = op.src1 >= 0 ? u->tens[op.src1].gn_rec : GnRec{};
          if (r0.units > 0 && (op.src1 < 0 || r1.units > 0)) {
            g.rec0 = r0;
            g.rec1 = r1;
          }
        }
        if (rc.train) {
          g.stats = u->gn_stats + (size_t)op.gn_index * rc.batch * 16;
          if (rc.drop_scale && op.drop_off >= 0) {
            g.drop_scale = rc.drop_scale + op.drop_off;
            g.drop_ld = u->temb_ld;
          }
        }
        int nl = 1;
        if (int e = gn_silu_enqueue(g, u->gn_partial, st, &nl)) return e;
        if (launches) *launches += nl - 1;
      } break;
      case OP_CONV: {
        ConvRun r = op.fwd;
        if (op.temb_off >= 0) {
          ConvEpilogue& ep = conv_run_epi(r);
          ep.temb = rc.temb + op.temb_off;
          ep.t_dev = rc.t_dev;
          ep.temb_ld = u->temb_ld;
          ep.temb_bstride = rc.temb_bstride;
        }
        if (int e = conv_run_enqueue(r, st)) return e;
      } break;
      case OP_ATTN: {
        const Tens& q = u->tens[op.qkv];
        const int S = u->levels[q.level].pps();
        float* lse = rc.train && oi < u->attn_lse.size() ? u->attn_lse[oi] : nullptr;   // streaming path: kept for the backward
        if (int e = attn_core_enqueue(q.p32, u->tens[op.ctx].p16, rc.batch, S, u->tens[op.ctx].C,
                                      op.heads, st, rc.dup, lse))
          return e;
      } break;
      case OP_FINAL: {
        const Level& l0 = u->levels[0];
        FinalParams f = rc.fin;
        f.act = u->tens[op.in].p16;
        f.act_ld = op.cin * rc.dup;
        f.act_lo = rc.dup == 2 ? op.cin : 0;
        f.w = u->params[u->p_final_w].ptr;
        f.bias = u->params[u->p_final_b].ptr;
        f.B = rc.batch;
        f.H = l0.H;
        f.W = l0.W;
        f.L = l0.D;
        f.P = c.past_len;
        f.cin = op.cin;
        f.cout = c.out_channels;
        if (int e = final_conv_enqueue(f, st)) return e;
      } break;
    }
    if (launches) ++*launches;
  }
  if (events) CM_CUDA(cudaEventRecord(events[op_index], st));
  return 0;
}

int build_jobs(cm_unet* u);

// dup = 1: sampling / eval (single fp16 activation operands); dup = 2: training forward (hi|lo pair rows).
// The packed-weight cache of the requested layout is (re)derived here, lazily, on `st`: one launch.
int ensure_ready(cm_unet* u, int batch, int dup, cudaStream_t st) {
  CM_CHECK(batch >= 1, "batch must be >= 1");
  if (int e = kernels_init()) return e;
  CM_CHECK(u->pack_called, "cm_unet_pack has not been called since parameters were bound");
  if (dup == 2 && !u->wpack2) {
    CM_CUDA(cudaMalloc(&u->wpack2, u->wpack2_elems * sizeof(__half)));
    u->jobs_dirty = true;
    u->packed2 = false;
  }
  if (int e = build_jobs(u)) return e;
  if (dup == 1 && !u->packed) {
    if (int e = pack_all_enqueue(u->d_jobs, u->n_jobs_fwd, st)) return e;
    u->packed = true;
  }
  if (dup == 2 && !u->packed2) {
    if (int e = pack_all_enqueue(u->d_jobs + u->n_jobs_fwd, u->n_jobs_fwd2, st)) return e;
    u->packed2 = true;
  }
  if (int e = reserve(u, batch)) return e;
  if (u->live_batch != batch || u->live_dup != dup) {
    chain_drop_graph(u->chain);
    u->train_prepared = 0;           // wgrad maps bake the activation row stride
    if (int e = prepare_convs(u, batch, dup)) return e;
  }
  return 0;
}


// ---- training: workspace, dgrad caches, backward launches -------------------------------------

int reserve_train(cm_unet* u, int batch) {
  if (batch <= u->train_reserved) return 0;
  if (u->tarena) CM_CUDA(cudaFree(u->tarena));
  u->tarena = nullptr;
  u->train_prepared = 0;
  const int E = u->cfg.base_channels * u->cfg.time_multiple;
  const int Cmax = u->max_gn_channels;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off = align_up(off + bytes, 1024);
    return o;
  };
  std::vector<size_t> o32(u->tens.size()), o16(u->tens.size(), (size_t)-1);
  std::vector<char> is_conv_out(u->tens.size(), 0);
  for (const Op& op : u->ops)
    if (op.type == OP_CONV || op.type == OP_FIRST) is_conv_out[op.out] = 1;
  for (size_t i = 0; i < u->tens.size(); ++i) {
    const Tens& t = u->tens[i];
    const size_t n = (size_t)batch * u->levels[t.level].pps() * t.C;
    o32[i] = take(n * 4);
    if (is_conv_out[i]) o16[i] = take(n * 2 * u->dgrad_dup);   // hi | lo pair per pixel when dgrad_dup == 2
  }
  const size_t o_stats = take((size_t)u->n_gn * batch * 16 * 4);
  const size_t o_part = take((size_t)batch * 32 * Cmax * 2 * 4);
  const size_t o_chsum = take((size_t)u->n_gn * batch * Cmax * 2 * 4);   // one region per GroupNorm
  const size_t o_zero = off;
  const size_t o_G = take(u->g_elems * 4);
  const size_t o_colsum = take((size_t)batch * u->colsum_per_sample * 4);
  const size_t o_dtemb = take((size_t)batch * u->temb_ld * 4);
  const size_t o_max = take(16);
  const size_t zero_end = off;
  const size_t o_e = take((size_t)batch * u->cfg.base_channels * 4);
  size_t o_t[8];
  for (int k = 0; k < 8; ++k) o_t[k] = take((size_t)batch * E * 4);
  const size_t o_scale = take(16);
  const size_t o_fd16 = take((size_t)batch * u->levels[0].pps() * 32 * 2);
  std::vector<size_t> o_lse(u->ops.size(), (size_t)-1);
  for (size_t i = 0; i < u->ops.size(); ++i) {
    const Op& op = u->ops[i];
    if (op.type != OP_ATTN) continue;
    const size_t S = u->levels[u->tens[op.qkv].level].pps();
    if (attn_uses_long((int)S, u->tens[op.ctx].C / op.heads))
      o_lse[i] = take((size_t)2 * batch * op.heads * S * 4);   // lse | backward row sums
  }
  CM_CUDA(cudaMalloc(&u->tarena, off));
  CM_CUDA(cudaMemset(u->tarena, 0, off));
  u->tarena_bytes = off;
  u->g32.assign(u->tens.size(), nullptr);
  u->g16.assign(u->tens.size(), nullptr);
  for (size_t i = 0; i < u->tens.size(); ++i) {
    u->g32[i] = reinterpret_cast<float*>(u->tarena + o32[i]);
    if (o16[i] != (size_t)-1) u->g16[i] = reinterpret_cast<__half*>(u->tarena + o16[i]);
  }
  u->gn_stats = reinterpret_cast<float*>(u->tarena + o_stats);
  u->gn_bwd_partial = reinterpret_cast<float*>(u->tarena + o_part);
  u->gn_chsum = reinterpret_cast<float*>(u->tarena + o_chsum);
  u->zero_region = u->tarena + o_zero;
  u->zero_bytes = zero_end - o_zero;
  u->G = reinterpret_cast<float*>(u->tarena + o_G);
  u->colsum = reinterpret_cast<float*>(u->tarena + o_colsum);
  u->dtemb = reinterpret_cast<float*>(u->tarena + o_dtemb);
  u->max_word = reinterpret_cast<unsigned int*>(u->tarena + o_max);
  u->tsave_e = reinterpret_cast<float*>(u->tarena + o_e);
  float** tp[8] = {&u->tsave_h1, &u->tsave_h2, &u->ts1, &u->ts2, &u->tds2, &u->tdh2, &u->tds1, &u->tdh1};
  for (int k = 0; k < 8; ++k) *tp[k] = reinterpret_cast<float*>(u->tarena + o_t[k]);
  u->loss_scale = reinterpret_cast<float*>(u->tarena + o_scale);
  u->final_d16 = reinterpret_cast<__half*>(u->tarena + o_fd16);
  u->attn_lse.assign(u->ops.size(), nullptr);
  for (size_t i = 0; i < u->ops.size(); ++i)
    if (o_lse[i] != (size_t)-1) u->attn_lse[i] = reinterpret_cast<float*>(u->tarena + o_lse[i]);
  u->train_reserved = batch;
  return 0;
}

// (Re)build the pack-job table [forward | dgrad] and the time-embedding pointer tables.  Runs when
// parameter storage moved or a cache buffer was (re)allocated; synchronous, rare.
int build_jobs(cm_unet* u) {
  if (!u->jobs_dirty) return 0;
  const int terms = u->cfg.weight_terms;
  if (!u->wpack) CM_CUDA(cudaMalloc(&u->wpack, u->wpack_elems * sizeof(__half)));
  std::vector<PackJob> jobs;
  for (Op& op : u->ops) {
    if (op.type != OP_CONV) continue;
    PackJob j{};
    j.w = u->params[op.w].ptr;
    j.wx = op.wx >= 0 ? u->params[op.wx].ptr : nullptr;
    j.dst = u->wpack + op.wpack_off;
    j.kind = op.mode == 2 ? 1 : 0;
    j.cout = op.cout; j.cin = op.cin; j.cinx = op.cin_extra; j.taps = op.mode == 3 ? 1 : 27;
    j.terms = terms;
    j.perm = 1; j.cin_src = op.cin; j.dup = 1;
    jobs.push_back(j);
  }
  {
    PackJob j{};
    j.w = u->params[u->p_first_w].ptr;
    j.dst = u->wpack + u->first_wpack_off;
    j.kind = 0;
    j.cout = u->cfg.base_channels; j.cin = 32; j.cinx = 0; j.taps = 27;
    j.terms = terms;
    j.perm = 1; j.cin_src = u->cfg.in_channels; j.dup = 1;
    jobs.push_back(j);
  }
  u->n_jobs_fwd = (int)jobs.size();
  u->n_jobs_fwd2 = 0;
  if (u->wpack2) {
    // the same forward weights against hi|lo pair activation rows (training forward): K doubled
    for (int k = 0; k < u->n_jobs_fwd; ++k) {
      PackJob j = jobs[k];
      j.dup = 2;
      jobs.push_back(j);
    }
    int k = u->n_jobs_fwd;
    for (Op& op : u->ops) {
      if (op.type != OP_CONV) continue;
      jobs[k++].dst = u->wpack2 + op.wpack2_off;
    }
    jobs[k++].dst = u->wpack2 + u->first_wpack2_off;
    u->n_jobs_fwd2 = (int)jobs.size() - u->n_jobs_fwd;
  }
  u->n_jobs_dgrad = 0;
  if (u->dpack) {
    for (Op& op : u->ops) {
      if (op.type != OP_CONV) continue;
      PackJob j{};
      j.w = u->params[op.w].ptr;
      j.dst = u->dpack + op.dpack_off;
      j.kind = 2; j.mode = op.mode;
      j.cout = op.cout; j.cin = op.cin; j.terms = terms; j.perm = 1; j.dup = u->dgrad_dup;
      j.ktot = dgrad_packed_k(op.mode, op.cout, u->dgrad_dup);
      jobs.push_back(j);
      if (op.cin_extra) {
        PackJob x{};
        x.w = u->params[op.wx].ptr;
        x.dst = u->dpack + op.dxpack_off;
        x.kind = 2; x.mode = 3;
        x.cout = op.cout; x.cin = op.cin_extra; x.terms = terms; x.perm = 1; x.dup = u->dgrad_dup;
        x.ktot = dgrad_packed_k(3, op.cout, u->dgrad_dup);
        jobs.push_back(x);
      }
    }
    u->n_jobs_dgrad = (int)jobs.size() - u->n_jobs_fwd - u->n_jobs_fwd2;
  }
  if ((int)jobs.size() > u->jobs_cap) {
    cudaFree(u->d_jobs);
    u->d_jobs = nullptr;
    CM_CUDA(cudaMalloc(&u->d_jobs, jobs.size() * sizeof(PackJob)));
    u->jobs_cap = (int)jobs.size();
  }
  CM_CUDA(cudaMemcpy(u->d_jobs, jobs.data(), jobs.size() * sizeof(PackJob), cudaMemcpyHostToDevice));
  u->jobs_host.swap(jobs);
  // per-block dense_1 pointer tables of the time-embedding kernel
  const int nb = (int)u->temb_couts.size();
  if (!u->d_wd) {
    CM_CUDA(cudaMalloc(&u->d_wd, nb * sizeof(float*)));
    CM_CUDA(cudaMalloc(&u->d_bd, nb * sizeof(float*)));
    CM_CUDA(cudaMalloc(&u->d_couts, nb * sizeof(int)));
    CM_CUDA(cudaMalloc(&u->d_offs, nb * sizeof(int)));
    CM_CUDA(cudaMalloc(&u->temb_table, (size_t)u->cfg.table_steps * u->temb_ld * sizeof(float)));
  }
  std::vector<const float*> wd(nb), bd(nb);
  for (int k = 0; k < nb; ++k) {
    wd[k] = u->params[u->temb_dense_w[k]].ptr;
    bd[k] = u->params[u->temb_dense_b[k]].ptr;
  }
  CM_CUDA(cudaMemcpy(u->d_wd, wd.data(), nb * sizeof(float*), cudaMemcpyHostToDevice));
  CM_CUDA(cudaMemcpy(u->d_bd, bd.data(), nb * sizeof(float*), cudaMemcpyHostToDevice));
  CM_CUDA(cudaMemcpy(u->d_couts, u->temb_couts.data(), nb * sizeof(int), cudaMemcpyHostToDevice));
  CM_CUDA(cudaMemcpy(u->d_offs, u->temb_offs.data(), nb * sizeof(int), cudaMemcpyHostToDevice));
  u->jobs_dirty = false;
  return 0;
}

// dgrad weight caches of every conv: one launch per optimizer step (lazily, by the next training forward)
int pack_dgrad(cm_unet* u, cudaStream_t st) {
  if (u->dpacked) return 0;
  if (!u->dpack) {
    CM_CUDA(cudaMalloc(&u->dpack, (u->dpack_elems + 8) * sizeof(__half)));
    u->jobs_dirty = true;
  }
  if (int e = build_jobs(u)) return e;
  if (int e = pack_all_enqueue(u->d_jobs + u->n_jobs_fwd + u->n_jobs_fwd2, u->n_jobs_dgrad, st)) return e;
  u->dpacked = true;
  return 0;
}

int prepare_train(cm_unet* u, int batch) {
  if (u->train_prepared == batch) return 0;
  for (Op& op : u->ops) {
    if (op.type != OP_CONV) continue;
    const Level& li = u->levels[op.in_level];
    const Level& lo = u->levels[u->tens[op.out].level];
    // data gradients: convs over dOut (geometry of the OUTPUT grid) into the fp32 gradients of the sources
    const int dup = u->dgrad_dup;
    ConvEpilogue e{};
    e.out32 = u->g32[op.in];
    e.lo_from = dup == 2 ? op.cout : 0;
    if (int rc = conv_run_prepare(&op.dgrad, CONV_UMMA | CONV_PLANE, dgrad_mode_of(op.mode), u->g16[op.out], batch, lo.D,
                                  lo.H, lo.W, dup * op.cout, nullptr, 0, u->dpack + op.dpack_off, op.cin,
                                  u->cfg.weight_terms, e))
      return rc;
    if (op.cin_extra) {
      e.out32 = u->g32[op.extra];
      if (int rc = conv_run_prepare(&op.dgrad_x, CONV_UMMA, 3, u->g16[op.out], batch, lo.D, lo.H, lo.W, dup * op.cout,
                                    nullptr, 0, u->dpack + op.dxpack_off, op.cin_extra, u->cfg.weight_terms, e))
        return rc;
    }
    // activations / the 1x1 source: the hi halves of the forward's (hi|lo pair) rows
    if (int rc = wgrad_run_prepare(&op.wgrad, CONV_UMMA | CONV_PLANE, op.mode, u->tens[op.in].p16, batch, li.D, li.H,
                                   li.W, op.cin, op.extra >= 0 ? u->tens[op.extra].p16 : nullptr, op.cin_extra,
                                   u->g16[op.out], op.cout, u->G + op.g_off, dup * op.cout, u->live_dup * op.cin,
                                   u->live_dup * op.cin_extra))
      return rc;
  }
  // first conv: its operand is the packed fp16 input [pixels][32 (x live_dup)] of the forward (channels >= in_channels are
  // zero), so its weight gradient is a conv weight gradient over the hi halves like any other layer with cin = 32
  const int base = u->cfg.base_channels;
  u->first_wg = WgradRun{};
  if (u->first.covered() && edge_wgrad_kinds(base)) {
    const Level& l0 = u->levels[0];
    const int out = u->ops[0].out;
    if (int rc = wgrad_run_prepare(&u->first_wg, edge_wgrad_kinds(base), 0, u->tens[u->first_in].p16, batch, l0.D, l0.H,
                                   l0.W, 32, nullptr, 0, u->g16[out], base, u->G + u->first_g_off, u->dgrad_dup * base,
                                   u->live_dup * 32))
      return rc;
  }
  u->final_wg = WgradRun{};
  if (u->ops.back().type == OP_FINAL && edge_wgrad_kinds(u->ops.back().cin)) {
    const Level& l0 = u->levels[0];
    const Op& fo = u->ops.back();
    if (int rc = wgrad_run_prepare(&u->final_wg, edge_wgrad_kinds(fo.cin), 0, u->tens[fo.in].p16, batch, l0.D, l0.H, l0.W,
                                   fo.cin, nullptr, 0, u->final_d16, 32, u->G + u->final_g_off, 32, u->live_dup * fo.cin))
      return rc;
  }
  u->train_prepared = batch;
  return 0;
}

void fill_temb(cm_unet* u, TembParams& tp, const int64_t* t, int batch) {
  tp = TembParams{};
  tp.table = u->params[u->p_table].ptr;
  tp.w1 = u->params[u->p_w1].ptr;
  tp.b1 = u->params[u->p_b1].ptr;
  tp.w2 = u->params[u->p_w2].ptr;
  tp.b2 = u->params[u->p_b2].ptr;
  tp.wd = u->d_wd;
  tp.bd = u->d_bd;
  tp.couts = u->d_couts;
  tp.offs = u->d_offs;
  tp.nblocks = (int)u->temb_couts.size();
  tp.base = u->cfg.base_channels;
  tp.E = u->cfg.base_channels * u->cfg.time_multiple;
  tp.t = reinterpret_cast<const long long*>(t);
  tp.rows = batch;
  tp.out = u->temb_batch;
  tp.ld = u->temb_ld;
}

// Reverse walk of the plan.  Every gradient carries the loss scale S (u->loss_scale[0]); the flat
// parameter-gradient buffer is multiplied by 1/S at the end.
// Floats of partial-sum scratch the deterministic backward needs: the largest single reduction of the plan (every one
// is summed out of the scratch by the launch that follows it, so one buffer serves them all in stream order).
size_t det_partial_elems(const cm_unet* u, int B) {
  const cm_unet_config& c = u->cfg;
  const Level& l0 = u->levels[0];
  size_t m = cast_colsum_partial_elems(B, l0.pps(), c.base_channels);
  for (const Op& op : u->ops) {
    if (op.type != OP_CONV) continue;
    m = std::max(m, cast_colsum_partial_elems(B, u->levels[u->tens[op.out].level].pps(), op.cout));
    m = std::max(m, wgrad_run_partial_elems(op.wgrad));
  }
  m = std::max(m, wgrad_run_partial_elems(u->first_wg));
  m = std::max(m, wgrad_run_partial_elems(u->final_wg));
  if (!u->first_wg.launches())
    m = std::max(m, first_conv_partial_elems(B, l0.H, l0.W, c.past_len, c.future_len, c.in_channels, c.base_channels));
  m = std::max(m, final_conv_partial_elems(B, l0.H, l0.W, l0.D, c.past_len, u->ops.back().cin, c.out_channels,
                                           u->final_wg.launches() > 0));
  return m;
}

int run_backward(cm_unet* u, const float* d_eps, float* grads, cudaStream_t st, int64_t* launches) {
  const cm_unet_config& c = u->cfg;
  const int B = u->live_train_batch;
  const int E = c.base_channels * c.time_multiple;
  auto gp = [&](int pidx) { return grads + u->grad_off[pidx]; };
  int64_t nl = 0;
  float* part = nullptr;
  if (u->deterministic) {
    const size_t need = det_partial_elems(u, B);
    if (need > u->det_part_elems) {
      CM_CUDA(cudaStreamSynchronize(st));
      CM_CUDA(cudaFree(u->det_part));
      u->det_part = nullptr;
      u->det_part_elems = 0;
      CM_CUDA(cudaMalloc(&u->det_part, need * sizeof(float)));
      u->det_part_elems = need;
    }
    part = u->det_part;
  }
  // launches each deterministic reduction adds: the ordered sums of its partials
  const int det_extra = part ? 1 : 0;
  CM_CUDA(cudaMemsetAsync(grads, 0, u->grad_total * sizeof(float), st));
  CM_CUDA(cudaMemsetAsync(u->zero_region, 0, u->zero_bytes, st));
  const Level& l0 = u->levels[0];
  const size_t n_eps = (size_t)B * c.out_channels * l0.H * l0.W * c.future_len;
  if (int e = auto_scale_enqueue(d_eps, n_eps, 64.f, u->loss_scale, u->max_word, st)) return e;
  nl += 2;
  std::vector<char> written(u->tens.size(), 0);
  std::vector<long long> gn_tab;        // {chsum offset, C, dgamma offset, dbeta offset} per GroupNorm, plan order
  std::vector<long long> up_tab;        // {mode, G offset, dw offset, dwx offset | -1, cout, cin, cinx, perm} per conv
  std::vector<long long> rs_tab;        // {channel-sum offset in the training arena, row stride, cout, bias-grad offset}
  for (int oi = (int)u->ops.size() - 1; oi >= 0; --oi) {
    Op& op = u->ops[oi];
    switch (op.type) {
      case OP_FINAL: {
        if (int e = final_conv_backward_enqueue(d_eps, u->loss_scale, u->tens[op.in].p16, u->live_dup * op.cin,
                                                u->live_dup == 2 ? op.cin : 0, u->params[u->p_final_w].ptr, u->g32[op.in], gp(u->p_final_w),
                                                gp(u->p_final_b), B, l0.H, l0.W, l0.D, c.past_len, op.cin,
                                                c.out_channels, u->final_wg.launches() ? u->final_d16 : nullptr, st,
                                                part))
          return e;
        nl += det_extra * (u->final_wg.launches() ? 1 : 2);
        if (u->final_wg.launches()) {
          if (int e = wgrad_run_enqueue(u->final_wg, st, part)) return e;
          nl += det_extra * u->final_wg.launches();
          // G is (tap, cin) x 32 packed columns: G's cout in the upper half of the cout entry
          for (long long v : {0LL, (long long)u->final_g_off, (long long)u->grad_off[u->p_final_w], -1LL,
                              (long long)c.out_channels | (32LL << 16), (long long)op.cin, 0LL, 1LL})
            up_tab.push_back(v);
          nl += u->final_wg.launches();
        }
        written[op.in] = 1;
        nl += 2;
      } break;
      case OP_GN: {
        GnBwdParams g{};
        g.src0 = u->tens[op.src0].p32;
        g.c0 = u->tens[op.src0].C;
        g.src1 = op.src1 >= 0 ? u->tens[op.src1].p32 : nullptr;
        g.c1 = op.src1 >= 0 ? u->tens[op.src1].C : 0;
        g.gamma = u->params[op.gamma].ptr;
        g.beta = u->params[op.beta].ptr;
        g.stats = u->gn_stats + (size_t)op.gn_index * B * 16;
        CM_CHECK(written[op.out_norm], "backward: gradient of '%s' output missing", op.tag.c_str());
        g.dnorm = u->g32[op.out_norm];
        g.draw = op.out_raw >= 0 ? u->g32[op.out_raw] : nullptr;
        if (u->live_drop && op.drop_off >= 0) {
          g.drop_scale = u->live_drop + op.drop_off;
          g.drop_ld = u->temb_ld;
        }
        g.B = B;
        g.pixels = u->levels[u->tens[op.src0].level].pps();
        g.silu = op.silu;
        g.dsrc0 = u->g32[op.src0];
        g.init0 = !written[op.src0];
        written[op.src0] = 1;
        if (op.src1 >= 0) {
          g.dsrc1 = u->g32[op.src1];
          g.init1 = !written[op.src1];
          written[op.src1] = 1;
        }
        // per-GroupNorm channel sums; dgamma / dbeta of all of them are reduced over the batch in ONE launch
        // after the op loop (27 tiny launches -> 1)
        g.chsum = u->gn_chsum + (size_t)op.gn_index * B * u->max_gn_channels * 2;
        g.dgamma = nullptr;
        g.dbeta = nullptr;
        gn_tab.push_back((long long)((size_t)op.gn_index * B * u->max_gn_channels * 2));
        gn_tab.push_back((long long)(u->tens[op.src0].C + (op.src1 >= 0 ? u->tens[op.src1].C : 0)));
        gn_tab.push_back((long long)u->grad_off[op.gamma]);
        gn_tab.push_back((long long)u->grad_off[op.beta]);
        if (int e = gn_backward_enqueue(g, u->gn_bwd_partial, st)) return e;
        nl += 2;
      } break;
      case OP_CONV: {
        CM_CHECK(written[op.out], "backward: gradient of '%s' output missing", op.tag.c_str());
        const int pix = u->levels[u->tens[op.out].level].pps();
        float* cs = op.temb_off >= 0 ? u->dtemb + op.temb_off : u->colsum + (size_t)B * op.colsum_off;
        const int cs_ld = op.temb_off >= 0 ? u->temb_ld : op.cout;
        float* fan = nullptr;
        int fan_init = 0;
        if (op.resid >= 0) {
          fan = u->g32[op.resid];
          fan_init = !written[op.resid];
          written[op.resid] = 1;
        }
        if (int e = cast_colsum_enqueue(u->g32[op.out], u->g16[op.out], u->dgrad_dup, fan, fan_init, cs, cs_ld, B,
                                        pix, op.cout, st, part))
          return e;
        nl += det_extra;
        // bias gradients = batch sums of the channel sums: all convs in one launch after the op loop
        for (int bidx : {op.bias, op.bias2}) {
          if (bidx < 0) continue;
          rs_tab.push_back((long long)(cs - reinterpret_cast<const float*>(u->tarena)));
          rs_tab.push_back((long long)cs_ld);
          rs_tab.push_back((long long)op.cout);
          rs_tab.push_back((long long)u->grad_off[bidx]);
        }
        {
          ConvRun r = op.dgrad;
          conv_run_epi(r).resid = written[op.in] ? u->g32[op.in] : nullptr;   // accumulate in place
          written[op.in] = 1;
          if (int e = conv_run_enqueue(r, st)) return e;
        }
        if (op.cin_extra) {
          ConvRun r = op.dgrad_x;
          conv_run_epi(r).resid = written[op.extra] ? u->g32[op.extra] : nullptr;
          written[op.extra] = 1;
          if (int e = conv_run_enqueue(r, st)) return e;
          ++nl;
        }
        if (int e = wgrad_run_enqueue(op.wgrad, st, part)) return e;
        nl += op.wgrad.launches() - 1 + det_extra * op.wgrad.launches();
        // packed-K scratch -> nn.Conv3d weight layout: all convs in one launch after the op loop
        for (long long v : {(long long)op.mode, (long long)op.g_off, (long long)u->grad_off[op.w],
                            op.wx >= 0 ? (long long)u->grad_off[op.wx] : -1LL, (long long)op.cout, (long long)op.cin,
                            (long long)op.cin_extra, 1LL})
          up_tab.push_back(v);
        nl += 3;
      } break;
      case OP_ATTN: {
        CM_CHECK(written[op.ctx], "backward: gradient of '%s' output missing", op.tag.c_str());
        const Tens& q = u->tens[op.qkv];
        const int S = u->levels[q.level].pps();
        if (int e = attn_core_backward_enqueue(q.p32, u->g32[op.ctx], u->g32[op.qkv], B, S, u->tens[op.ctx].C,
                                               op.heads, st, u->attn_lse[oi], u->attn_lse[oi] ? u->attn_lse[oi] + (size_t)B * op.heads * S : nullptr))
          return e;
        written[op.qkv] = 1;
        ++nl;
      } break;
      case OP_FIRST: {
        CM_CHECK(written[op.out], "backward: gradient of the first conv output missing");
        if (u->first_wg.launches()) {
          float* cs = u->colsum + (size_t)B * u->first_colsum_off;
          if (int e = cast_colsum_enqueue(u->g32[op.out], u->g16[op.out], u->dgrad_dup, nullptr, 0, cs, c.base_channels, B,
                                          l0.pps(), c.base_channels, st, part))
            return e;
          nl += det_extra;
          rs_tab.push_back((long long)(cs - reinterpret_cast<const float*>(u->tarena)));
          rs_tab.push_back((long long)c.base_channels);
          rs_tab.push_back((long long)c.base_channels);
          rs_tab.push_back((long long)u->grad_off[u->p_first_b]);
          if (int e = wgrad_run_enqueue(u->first_wg, st, part)) return e;
          nl += det_extra * u->first_wg.launches();
          // G rows are (tap, 32 packed channels): cin of G in the upper half of the cin entry
          for (long long v : {0LL, (long long)u->first_g_off, (long long)u->grad_off[u->p_first_w], -1LL,
                              (long long)c.base_channels, (long long)c.in_channels | (32LL << 16), 0LL, 1LL})
            up_tab.push_back(v);
          nl += u->first_wg.launches();
        } else if (int e = first_conv_wgrad_enqueue(u->live_future, u->live_past, u->g32[op.out], gp(u->p_first_w),
                                                    gp(u->p_first_b), B, l0.H, l0.W, c.past_len, c.future_len,
                                                    c.in_channels, c.base_channels, st, part)) {
          return e;
        } else {
          nl += 2 * det_extra;
        }
        ++nl;
      } break;
    }
  }
  // ---- weight gradients out of the packed-K scratch: one launch ----
  if (!up_tab.empty()) {
    if (!u->d_up_tab || u->up_tab_host != up_tab) {
      if (u->d_up_tab && u->up_tab_host.size() < up_tab.size()) {
        cudaFree(u->d_up_tab);
        u->d_up_tab = nullptr;
      }
      if (!u->d_up_tab) CM_CUDA(cudaMalloc(&u->d_up_tab, up_tab.size() * sizeof(long long)));
      CM_CUDA(cudaMemcpyAsync(u->d_up_tab, up_tab.data(), up_tab.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
      CM_CUDA(cudaStreamSynchronize(st));
      u->up_tab_host = up_tab;
    }
    if (int e = unpack_wgrad_all_enqueue(u->d_up_tab, (int)(up_tab.size() / 8), u->G, grads, st)) return e;
    ++nl;
  }
  // ---- conv bias gradients: one launch ----
  if (!rs_tab.empty()) {
    if (!u->d_rs_tab || u->rs_tab_host != rs_tab) {
      if (u->d_rs_tab && u->rs_tab_host.size() < rs_tab.size()) {
        cudaFree(u->d_rs_tab);
        u->d_rs_tab = nullptr;
      }
      if (!u->d_rs_tab) CM_CUDA(cudaMalloc(&u->d_rs_tab, rs_tab.size() * sizeof(long long)));
      CM_CUDA(cudaMemcpyAsync(u->d_rs_tab, rs_tab.data(), rs_tab.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
      CM_CUDA(cudaStreamSynchronize(st));
      u->rs_tab_host = rs_tab;
    }
    if (int e = rowsum_all_enqueue(reinterpret_cast<const float*>(u->tarena), u->d_rs_tab, (int)(rs_tab.size() / 4), B,
                                   grads, st))
      return e;
    ++nl;
  }
  // ---- dgamma / dbeta of every GroupNorm: one launch ----
  if (!gn_tab.empty()) {
    const size_t bytes = gn_tab.size() * sizeof(long long);
    if (!u->d_gn_tab || u->gn_tab_host != gn_tab) {
      if (!u->d_gn_tab) CM_CUDA(cudaMalloc(&u->d_gn_tab, (size_t)u->n_gn * 4 * sizeof(long long)));
      CM_CUDA(cudaMemcpyAsync(u->d_gn_tab, gn_tab.data(), bytes, cudaMemcpyHostToDevice, st));
      CM_CUDA(cudaStreamSynchronize(st));      // gn_tab is a local: the copy must finish before it goes away
      u->gn_tab_host = gn_tab;
    }
    if (int e = gn_backward_params_all_enqueue(u->gn_chsum, u->d_gn_tab, (int)(gn_tab.size() / 4), B, grads, st))
      return e;
    ++nl;
  }
  // ---- time-embedding MLP (embeddings.py:22-34) and the per-block dense_1 (layers.py:35,62) ----
  {
    const int nb = (int)u->temb_couts.size();
    if (!u->d_goff_w) {
      std::vector<long long> gw(nb), gb(nb);
      for (int k = 0; k < nb; ++k) {
        gw[k] = (long long)u->grad_off[u->temb_dense_w[k]];
        gb[k] = (long long)u->grad_off[u->temb_dense_b[k]];
      }
      CM_CUDA(cudaMalloc(&u->d_goff_w, nb * sizeof(long long)));
      CM_CUDA(cudaMalloc(&u->d_goff_b, nb * sizeof(long long)));
      CM_CUDA(cudaMemcpy(u->d_goff_w, gw.data(), nb * sizeof(long long), cudaMemcpyHostToDevice));
      CM_CUDA(cudaMemcpy(u->d_goff_b, gb.data(), nb * sizeof(long long), cudaMemcpyHostToDevice));
    }
    TembBwdParams tb{};
    tb.e = u->tsave_e; tb.h1 = u->tsave_h1; tb.h2 = u->tsave_h2;
    tb.dtemb = u->dtemb; tb.ld = u->temb_ld;
    tb.wd = u->d_wd; tb.couts = u->d_couts; tb.offs = u->d_offs; tb.nblocks = nb;
    tb.goff_w = u->d_goff_w; tb.goff_b = u->d_goff_b;
    tb.w2 = u->params[u->p_w2].ptr;
    tb.dw1 = gp(u->p_w1); tb.db1 = gp(u->p_b1); tb.dw2 = gp(u->p_w2); tb.db2 = gp(u->p_b2);
    tb.s1 = u->ts1; tb.s2 = u->ts2; tb.ds1 = u->tds1; tb.ds2 = u->tds2; tb.dh1 = u->tdh1; tb.dh2 = u->tdh2;
    tb.B = B; tb.E = E; tb.base = c.base_channels;
    if (int e = temb_backward_enqueue(tb, grads, st)) return e;
    nl += 11;
  }
  if (int e = scale_inplace_enqueue(grads, u->grad_total, u->loss_scale + 1, st)) return e;
  ++nl;
  if (launches) *launches = nl;
  return 0;
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int cm_unet_create(const cm_unet_config* cfg, cm_unet** out) {
  CM_CHECK(cfg && out, "null argument");
  auto u = std::make_unique<cm_unet>();
  u->cfg = *cfg;
  if (u->cfg.table_steps <= 0) u->cfg.table_steps = 1000;
  if (u->cfg.weight_terms <= 0) u->cfg.weight_terms = 2;
  CM_CHECK(u->cfg.dgrad_terms >= 0 && u->cfg.dgrad_terms <= 2, "dgrad_terms must be 0 (default), 1 or 2");
  u->dgrad_dup = u->cfg.dgrad_terms == 1 ? 1 : 2;
  u->cfg.dgrad_terms = u->dgrad_dup;
  CM_CHECK(u->cfg.train_act_terms >= 0 && u->cfg.train_act_terms <= 2, "train_act_terms must be 0 (default), 1 or 2");
  u->act_dup_train = u->cfg.train_act_terms == 1 ? 1 : 2;
  u->cfg.train_act_terms = u->act_dup_train;
  if (int e = build_plan(u.get())) return e;
  *out = u.release();
  return 0;
}

int cm_unet_destroy(cm_unet* u) {
  if (!u) return 0;
  chain_free(u->chain);
  cudaFree(u->arena);
  cudaFree(u->wpack);
  cudaFree(u->wpack2);
  cudaFree(u->temb_table);
  cudaFree(u->d_wd);
  cudaFree(u->d_bd);
  cudaFree(u->d_rs_tab);
  cudaFree(u->d_gn_tab);
  cudaFree(u->d_goff_w);
  cudaFree(u->d_goff_b);
  cudaFree(u->d_couts);
  cudaFree(u->d_offs);
  cudaFree(u->d_jobs);
  cudaFree(u->d_up_tab);
  cudaFree(u->dpack);
  cudaFree(u->tarena);
  cudaFree(u->det_part);
  delete u;
  return 0;
}

int cm_unet_param_count(const cm_unet* u) { return u ? (int)u->params.size() : -1; }

int cm_unet_param_info(const cm_unet* u, int idx, char* name, int name_cap, int64_t* shape5,
                       int* ndim) {
  CM_CHECK(u && idx >= 0 && idx < (int)u->params.size(), "bad param index %d", idx);
  const ParamEntry& p = u->params[idx];
  if (name && name_cap > 0) snprintf(name, name_cap, "%s", p.name.c_str());
  if (ndim) *ndim = (int)p.shape.size();
  if (shape5)
    for (size_t i = 0; i < p.shape.size() && i < 5; ++i) shape5[i] = p.shape[i];
  return 0;
}

static int bind_one(cm_unet* u, int idx, const float* dev_ptr) {
  ParamEntry& p = u->params[idx];
  CM_CHECK(dev_ptr != nullptr, "parameter '%s': null pointer", p.name.c_str());
  CM_CHECK((reinterpret_cast<uintptr_t>(dev_ptr) & 15) == 0, "parameter '%s' must be 16-byte aligned", p.name.c_str());
  if (p.ptr != dev_ptr) {
    p.ptr = dev_ptr;
    u->packed = false;
    u->packed2 = false;
    u->dpacked = false;
    u->pack_called = false;
    u->jobs_dirty = true;
    u->train_prepared = 0;
    chain_drop_graph(u->chain);   // baked pointers are stale
    u->live_batch = 0;   // force prepare_convs (bias pointers)
  }
  return 0;
}

int cm_unet_set_param(cm_unet* u, const char* name, const float* dev_ptr, int64_t numel) {
  CM_CHECK(u && name, "null argument");
  auto it = u->pindex.find(name);
  CM_CHECK(it != u->pindex.end(), "unknown parameter '%s'", name);
  ParamEntry& p = u->params[it->second];
  CM_CHECK(p.numel() == numel, "parameter '%s': expected %lld elements, got %lld", name,
           (long long)p.numel(), (long long)numel);
  return bind_one(u, it->second, dev_ptr);
}

int cm_unet_bind_params(cm_unet* u, const void* const* ptrs, int count) {
  CM_CHECK(u && ptrs, "null argument");
  CM_CHECK(count == (int)u->params.size(), "expected %d parameter pointers, got %d", (int)u->params.size(), count);
  for (int i = 0; i < count; ++i)
    if (int e = bind_one(u, i, static_cast<const float*>(ptrs[i]))) return e;
  return 0;
}

int cm_unet_pack(cm_unet* u, int build_time_table, void* stream) {
  CM_CHECK(u, "null handle");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = check_params_bound(u)) return e;
  // every derived cache is stale; each is re-derived by the next call that needs it, on that call's stream,
  // in one launch: the forward weights of the sampling layout by cm_unet_forward / cm_ddpm_sample, the
  // training-forward layout and the dgrad weights by cm_unet_train_forward.
  u->packed = false;
  u->packed2 = false;
  u->dpacked = false;
  u->pack_called = true;
  if (build_time_table) {
    if (int e = build_jobs(u)) return e;                    // (also refreshes the dense_1 pointer tables)
    TembParams t{};
    t.table = u->params[u->p_table].ptr;
    t.w1 = u->params[u->p_w1].ptr;
    t.b1 = u->params[u->p_b1].ptr;
    t.w2 = u->params[u->p_w2].ptr;
    t.b2 = u->params[u->p_b2].ptr;
    t.wd = u->d_wd;
    t.bd = u->d_bd;
    t.couts = u->d_couts;
    t.offs = u->d_offs;
    t.nblocks = (int)u->temb_couts.size();
    t.base = u->cfg.base_channels;
    t.E = u->cfg.base_channels * u->cfg.time_multiple;
    t.t = nullptr;
    t.rows = u->cfg.table_steps;
    t.out = u->temb_table;
    t.ld = u->temb_ld;
    if (int e = temb_enqueue(t, st)) return e;
  }
  return 0;
}

int cm_unet_reserve(cm_unet* u, int batch, int64_t* bytes) {
  CM_CHECK(u, "null handle");
  if (int e = reserve(u, batch)) return e;
  if (bytes) *bytes = (int64_t)u->arena_bytes;
  return 0;
}

int cm_unet_launches_per_forward(const cm_unet* u) {
  if (!u) return -1;
  int n = 1;   // time-embedding kernel
  n += (int)u->ops.size();
  return n;
}
double cm_unet_flops_per_sample(const cm_unet* u) { return u ? u->flops_per_sample : 0.0; }
int64_t cm_last_chain_launches(const cm_unet* u) { return u ? u->chain.launches : -1; }

int cm_unet_forward(cm_unet* u, const float* future, const int64_t* t, const float* past,
                    float* eps_out, int batch, void* stream) {
  CM_CHECK(u && future && t && past && eps_out, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = ensure_ready(u, batch, 1, st)) return e;
  u->live_train_batch = 0;   // the arena is shared: a pending training backward can no longer run
  // per-sample time embedding projections (t may differ per sample: ddpm.py:113)
  TembParams tp{};
  tp.table = u->params[u->p_table].ptr;
  tp.w1 = u->params[u->p_w1].ptr;
  tp.b1 = u->params[u->p_b1].ptr;
  tp.w2 = u->params[u->p_w2].ptr;
  tp.b2 = u->params[u->p_b2].ptr;
  tp.wd = u->d_wd;
  tp.bd = u->d_bd;
  tp.couts = u->d_couts;
  tp.offs = u->d_offs;
  tp.nblocks = (int)u->temb_couts.size();
  tp.base = u->cfg.base_channels;
  tp.E = u->cfg.base_channels * u->cfg.time_multiple;
  tp.t = reinterpret_cast<const long long*>(t);
  tp.rows = batch;
  tp.out = u->temb_batch;
  tp.ld = u->temb_ld;
  if (int e = temb_enqueue(tp, st)) return e;
  RunCtx rc{};
  rc.batch = batch;
  rc.future = future;
  rc.past = past;
  rc.temb = u->temb_batch;
  rc.t_dev = nullptr;
  rc.temb_bstride = u->temb_ld;
  rc.fin = FinalParams{};
  rc.fin.eps_out = eps_out;
  return run_ops(u, rc, st, nullptr);
}


/* ---- training ---- */
int cm_unet_grad_layout(const cm_unet* u, int64_t* offsets, int cap, int64_t* total) {
  CM_CHECK(u, "null handle");
  if (offsets) {
    CM_CHECK(cap >= (int)u->params.size(), "offsets array too small");
    for (size_t i = 0; i < u->params.size(); ++i) offsets[i] = (int64_t)u->grad_off[i];
  }
  if (total) *total = (int64_t)u->grad_total;
  return 0;
}

int cm_unet_dropout_layout(const cm_unet* u, int32_t* offsets, int32_t* channels, int cap, int32_t* ld) {
  CM_CHECK(u, "null handle");
  const int nb = (int)u->temb_couts.size();
  if (offsets || channels) CM_CHECK(cap >= nb, "arrays too small (%d blocks)", nb);
  for (int k = 0; k < nb; ++k) {
    if (offsets) offsets[k] = u->temb_offs[k];
    if (channels) channels[k] = u->temb_couts[k];
  }
  if (ld) *ld = u->temb_ld;
  return nb;
}

int cm_unet_train_forward(cm_unet* u, const float* future, const int64_t* t, const float* past,
                          float* eps_out, int batch, const float* drop_scale, void* stream) {
  CM_CHECK(u && future && t && past && eps_out, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = ensure_ready(u, batch, u->act_dup_train, st)) return e;
  if (int e = backward_init()) return e;
  if (int e = reserve_train(u, batch)) return e;
  if (int e = pack_dgrad(u, st)) return e;
  if (int e = prepare_train(u, batch)) return e;
  TembParams tp;
  fill_temb(u, tp, t, batch);
  tp.save_e = u->tsave_e;
  tp.save_h1 = u->tsave_h1;
  tp.save_h2 = u->tsave_h2;
  if (int e = temb_enqueue(tp, st)) return e;
  RunCtx rc{};
  rc.batch = batch;
  rc.future = future;
  rc.past = past;
  rc.temb = u->temb_batch;
  rc.t_dev = nullptr;
  rc.temb_bstride = u->temb_ld;
  rc.fin = FinalParams{};
  rc.fin.eps_out = eps_out;
  rc.train = true;
  rc.drop_scale = drop_scale;
  rc.dup = u->act_dup_train;
  if (int e = run_ops(u, rc, st, nullptr)) return e;
  u->live_train_batch = batch;
  u->live_future = future;
  u->live_past = past;
  u->live_drop = drop_scale;
  return 0;
}

int cm_unet_backward(cm_unet* u, const float* d_eps, float* grads, void* stream) {
  CM_CHECK(u && d_eps && grads, "null argument");
  CM_CHECK(u->live_train_batch > 0, "cm_unet_backward without a preceding cm_unet_train_forward");
  CM_CHECK((reinterpret_cast<uintptr_t>(grads) & 15) == 0, "grads must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t nl = 0;
  const int e = run_backward(u, d_eps, grads, st, &nl);
  u->live_train_batch = 0;   // activations are consumed: one backward per forward
  u->last_backward_launches = nl;
  return e;
}

int64_t cm_last_backward_launches(const cm_unet* u) { return u ? u->last_backward_launches : -1; }

int cm_unet_set_deterministic(cm_unet* u, int enabled) {
  CM_CHECK(u, "null handle");
  u->deterministic = enabled ? 1 : 0;
  return 0;
}

int cm_unet_op_count(const cm_unet* u) { return u ? (int)u->ops.size() : -1; }

int cm_unet_op_info(const cm_unet* u, int idx, char* tag, int tag_cap, int* type, double* flops_per_sample) {
  CM_CHECK(u && idx >= 0 && idx < (int)u->ops.size(), "bad op index %d", idx);
  const Op& op = u->ops[idx];
  if (tag && tag_cap > 0) snprintf(tag, tag_cap, "%s", op.tag.c_str());
  if (type) *type = (int)op.type;
  if (flops_per_sample) {
    double fl = 0.0;
    const cm_unet_config& c = u->cfg;
    if (op.type == OP_CONV) {
      const Level& lo = u->levels[u->tens[op.out].level];
      const double taps = (op.mode == 3) ? 1.0 : 27.0;
      fl = 2.0 * lo.pps() * op.cout * (taps * op.cin + op.cin_extra);
    } else if (op.type == OP_ATTN) {
      const Level& lv = u->levels[u->tens[op.qkv].level];
      fl = 4.0 * (double)lv.pps() * lv.pps() * u->tens[op.ctx].C;
    } else if (op.type == OP_FIRST) {
      fl = 2.0 * u->levels[0].pps() * c.base_channels * 27.0 * c.in_channels;
    } else if (op.type == OP_FINAL) {
      fl = 2.0 * u->levels[0].pps() * c.out_channels * 27.0 * op.cin;
    }
    *flops_per_sample = fl;
  }
  return 0;
}

int cm_unet_debug_op_tensor(const cm_unet* u, int op_idx) {
  if (!u || op_idx < 0 || op_idx >= (int)u->ops.size()) return -1;
  const Op& op = u->ops[op_idx];
  switch (op.type) {
    case OP_FIRST: return op.out;
    case OP_GN: return op.out_norm;
    case OP_CONV: return op.out;
    case OP_ATTN: return op.ctx;
    default: return -1;
  }
}

int cm_unet_debug_tensor_read(const cm_unet* u, int tensor, int kind, int sample0, int nsamples, void* dst,
                              int64_t dst_bytes, int* C, int* pixels, void* stream) {
  CM_CHECK(u && tensor >= 0 && tensor < (int)u->tens.size(), "bad tensor index %d", tensor);
  const Tens& t = u->tens[tensor];
  const int pps = u->levels[t.level].pps();
  if (C) *C = t.C;
  if (pixels) *pixels = pps;
  CM_CHECK(kind == 32 || kind == 16, "kind must be 32 or 16");
  const void* src = kind == 32 ? static_cast<const void*>(t.p32) : static_cast<const void*>(t.p16);
  if (!src) return 3;                       // this copy of the tensor does not exist in the plan
  CM_CHECK(sample0 >= 0 && nsamples >= 1 && sample0 + nsamples <= u->reserved_batch, "sample range out of bounds");
  const size_t esz = kind == 32 ? 4 : 2;
  const size_t per = (size_t)pps * t.C * esz;
  CM_CHECK(dst && (size_t)dst_bytes >= per * nsamples, "dst too small (%lld < %zu)", (long long)dst_bytes, per * nsamples);
  CM_CUDA(cudaMemcpyAsync(dst, static_cast<const uint8_t*>(src) + per * sample0, per * nsamples,
                          cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}

double cm_unet_op_exec_flops(const cm_unet* u, int idx) {
  if (!u || idx < 0 || idx >= (int)u->ops.size()) return 0.0;
  double fl = 0.0;
  cm_unet_op_info(u, idx, nullptr, 0, nullptr, &fl);
  const Op& op = u->ops[idx];
  if (op.type == OP_CONV && op.mode == 2) fl *= 8.0 / 27.0;
  return fl;
}

int cm_unet_profile_forward(cm_unet* u, const float* future, const int64_t* t, const float* past,
                            float* eps_out, int batch, void* stream, float* ms_out, int cap) {
  CM_CHECK(u && future && t && past && eps_out && ms_out, "null argument");
  CM_CHECK(cap >= (int)u->ops.size(), "ms_out too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // warm pass builds descriptors / time embedding, then the measured pass brackets every op
  if (int e = cm_unet_forward(u, future, t, past, eps_out, batch, stream)) return e;
  std::vector<cudaEvent_t> ev(u->ops.size() + 1);
  for (auto& e : ev) CM_CUDA(cudaEventCreate(&e));
  RunCtx rc{};
  rc.batch = batch;
  rc.future = future;
  rc.past = past;
  rc.temb = u->temb_batch;
  rc.t_dev = nullptr;
  rc.temb_bstride = u->temb_ld;
  rc.fin = FinalParams{};
  rc.fin.eps_out = eps_out;
  int e = run_ops(u, rc, st, nullptr, ev.data());
  cudaError_t se = cudaStreamSynchronize(st);
  if (!e && se == cudaSuccess)
    for (size_t i = 0; i < u->ops.size(); ++i) cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]);
  for (auto& x : ev) cudaEventDestroy(x);
  if (e) return e;
  CM_CUDA(se);
  return 0;
}

int cm_ddpm_sample(cm_unet* u, const cm_chain_args* a, void* stream) {
  CM_CHECK(u && a, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = ensure_ready(u, a->n, 1, st)) return e;
  u->live_train_batch = 0;   // the arena is shared: a pending training backward can no longer run
  const cm_unet_config& c = u->cfg;
  const Level& l0 = u->levels[0];
  const size_t x_bytes = (size_t)a->n * c.out_channels * l0.H * l0.W * c.future_len * sizeof(float);
  const size_t past_bytes = (size_t)a->n * c.in_channels * l0.H * l0.W * c.past_len * sizeof(float);
  RunCtx rc{};
  rc.batch = a->n;
  rc.future = u->chain_x;   // the denoiser reads the CURRENT x (the chain's staging copy)
  rc.past = u->chain_past;
  rc.temb = u->temb_table;
  return chain_run(u->chain, *a, c.table_steps, u->chain_x, x_bytes, u->chain_past, past_bytes,
                   [u, &rc](const ReverseStep& rs, const int* t_dev, cudaStream_t s, int64_t* launches) {
                     rc.t_dev = t_dev;
                     rc.fin.rs = rs;
                     return run_ops(u, rc, s, launches);
                   },
                   st);
}

int64_t cm_last_chain_graph_launches(const cm_unet* u) { return u ? u->chain.graph_launches : -1; }
int cm_last_chain_graph_rebuilt(const cm_unet* u) { return u ? u->chain.graph_rebuilt : -1; }

}  // extern "C"
