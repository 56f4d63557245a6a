// Bandwidth / small-op kernels of the UNet hot path (everything that is not the tcgen05 conv).
// Each launcher cites the reference op it replaces.
#pragma once
#include "chain.cuh"
#include "common.cuh"

namespace cm {

// ---- weight packing (fp32 torch layouts -> fp16 K-major rows, optional hi+lo split) ----
// w: [cout][cin][taps] (nn.Conv3d weight flattened; taps = 27 or 1), wx: [cout][cinx] or null.
// dst: [terms*cout][taps*cin + cinx], column = tap*cin + ci, then 27*cin + cx.
// perm = 1: w is a reference nn.Conv3d weight over (rows, cols, time) and the activations are
// stored [B, time, rows, cols, C]; perm = 0: w taps are ordered like the activation dims.
int pack_conv_weights(const float* w, const float* wx, __half* dst, int cout, int cin, int cinx,
                      int taps, int terms, int perm, cudaStream_t st, int dup = 1);
// nearest-x2 + k3 conv folded into 8 phase convs with 2x2x2 combined taps
// (layers.py:92-94).  dst: [terms*cout][64*cin], column = phase*8*cin + tap8*cin + ci.
// k3 conv weights whose cin_src (< 32) input channels are zero-padded to cin_packed packed channels
// (dup = 2: against hi|lo pair rows of 2 * cin_packed channels, as pack_conv_weights)
int pack_conv_weights_padded(const float* w, __half* dst, int cout, int cin_src, int cin_packed, int terms,
                             int perm, cudaStream_t st, int dup = 1);
// first-conv operand: API tensors -> channels 0..cin-1 of fp16 [B, P+F, H, W, 32] (other channels untouched)
// dup = 2: rows of 64 (hi | lo halves of the 32 padded channels)
int pack_first_input_enqueue(const float* x, const float* past, __half* out16, int B, int H, int W, int P, int F,
                             int cin, int dup, cudaStream_t st);
int pack_upsample_weights(const float* w, __half* dst, int cout, int cin, int terms, int perm,
                          cudaStream_t st, int dup = 1);

// ---- GroupNorm(8) [+SiLU] [+Dropout3d scale] -> fp16 operand (layers.py:30,41,57,70; :9,14) ----
// GroupNorm statistics records written by a producing plane-tile or res32 conv (ConvEpilogue::stats_rec)
struct GnRec {
  const float* rec;   // [B][units][C_src] float4 {shift, sum, sumsq, 0}; nullptr = none
  int units;          // units per sample
  int nvalid;         // rows per unit
};
struct GnParams {
  const float* src0;   // fp32 channels-last [B][pixels][c0]
  const float* src1;   // optional second source (skip concat, unet.py:160), channels c0..c0+c1
  int c0, c1;
  const float* gamma;
  const float* beta;
  int B, pixels;
  float eps;
  int silu;
  const float* drop_scale;  // [B][drop_ld] (+ channel) per-(sample,channel) multiplier or nullptr
  int drop_ld;
  __half* out_norm;         // [B][pixels][dup*C]
  __half* out_raw;          // optional raw fp16 copy of the (concatenated) input, same row layout
  int dup;                  // 1: single fp16 operand; 2: K-concatenated hi|lo pair per pixel ([0,C) = hi,
                            // [C,2C) = fp16(v - hi)): the training forward's operands are exact to 2^-22
                            // (0 is read as 1)
  float* stats;             // optional [B][8][2] (mean, rstd) for backward
  GnRec rec0, rec1;         // both sources have records -> no statistics pass over the data
};
// `partial`: scratch of B * gn_chunks(pixels, C) * 16 floats (slice statistics)
int gn_chunks(int pixels, int C);
// *launches (optional) receives the number of kernels enqueued (1 or 2)
int gn_silu_enqueue(const GnParams& p, float* partial, cudaStream_t st, int* launches = nullptr);

// ---- first conv: 3(+)->base channels straight from the API layout (unet.py:32,138,144) ----
// x: [B][cin][H][W][F] fp32, past: [B][cin][H][W][P] fp32 (virtual concat along time),
// w: [cout][cin][3][3][3], out: fp32 channels-last, time-major [B][P+F][H][W][cout].
int first_conv_enqueue(const float* x, const float* past, const float* w, const float* bias,
                       float* out, int B, int H, int W, int P, int F, int cin, int cout,
                       cudaStream_t st);

// ---- final conv base->3 fused with the DDPM/DDIM update (unet.py:118-122,165-167; ddpm.py:25-38,262-265) ----
struct FinalParams {
  const __half* act;     // fp16 channels-last, time-major [B][L][H][W][act_ld], already GN+SiLU'ed
  int act_ld;            // row stride in elements (0 -> cin); act_lo > 0: a lo half sits act_lo elements
  int act_lo;            // after the hi half of every pixel row and is added (hi|lo pair operands)
  const float* w;        // [cout][cin][27] fp32
  const float* bias;
  int B, H, W, L, P;     // L = P + F; only frames l >= P are produced
  int cin, cout;
  float* eps_out;        // optional [B][cout][H][W][F]
  ReverseStep rs;        // reverse-step update (rs.x == nullptr -> eps only)
};
int final_conv_enqueue(const FinalParams& p, cudaStream_t st);

// ---- time embedding MLP + every block's dense_1 (embeddings.py:22-34; layers.py:35,62) ----
struct TembParams {
  const float* table;    // [T][base] frozen sinusoid table
  const float* w1; const float* b1;   // [E][base]
  const float* w2; const float* b2;   // [E][E]
  const float* const* wd;  // device array [nblocks] of [cout_k][E]
  const float* const* bd;  // device array [nblocks] of [cout_k]
  const int* couts;        // device array [nblocks]
  const int* offs;         // device array [nblocks] column offsets in out
  int nblocks;
  int base, E;
  const long long* t;      // [rows] int64 timesteps, or nullptr -> t = row index
  int rows;
  float* out;              // [rows][ld]
  int ld;
  // training: optional saves for the backward pass ([rows][base], [rows][E], [rows][E])
  float* save_e; float* save_h1; float* save_h2;
};
int temb_enqueue(const TembParams& p, cudaStream_t st);

// ---- attention core softmax(QK^T/sqrt(dh))V per (sample, head) (layers.py:16) ----
// qkv: fp32 [B*S][3*C] (q | k | v), ctx: fp16 [B*S][dup*C] (dup = 2: hi | lo pair per token).  Any S; dh = C / heads
// even and <= 128.  attn_uses_long(S, dh): attn_long_kernel (attn_long.cu, keys streamed with the online softmax), which
// also writes the row log-sum-exp of the scaled scores to lse (fp32 [B][heads][S]) when lse is given: the streaming
// backward recomputes P from it.  Otherwise attn_mma_kernel (whole score row in registers).  Capturable (no
// allocation, no synchronisation).
// The one test of which kernels an attention core uses; the training plans size their lse slices by it.
inline bool attn_uses_long(int S, int dh) { return S > 128 || dh > 64; }
int attn_core_enqueue(const float* qkv, __half* ctx, int B, int S, int C, int heads,
                      cudaStream_t st, int dup = 1, float* lse = nullptr);
int attn_long_enqueue(const float* qkv, __half* ctx, float* lse, int B, int S, int C, int heads, int dup,
                      cudaStream_t st);
int attn_long_init();   // attn_long.cu: shared-memory attributes of the long-sequence kernels (called by kernels_init)

// ---- fused AttentionBlock of the sampling path (layers.py:5-18): GroupNorm -> in_proj -> attention core ->
// out_proj -> + x in one launch (one CTA per sample).  w_in / w_out: packed hi|lo fp16 rows as the 1x1 convs
// use them ([2*3C][C] and [2*C][C]).  Covers C = 128, 4 heads, S <= 128; callers fall back to the four
// separate kernels otherwise (and in training, where the backward needs the intermediates).
bool attn_block_supported(int S, int C, int heads);
int attn_block_enqueue(const float* x, const float* gamma, const float* beta, const __half* w_in, const float* b_in,
                       const __half* w_out, const float* b_out, float* out32, __half* out16, int B, int S, int C,
                       int heads, float eps, cudaStream_t st);

// ---- test-only: scalar restatement of exactly what conv_umma computes (same packed operands) ----
struct ConvParams;
int conv_ref_enqueue(const ConvParams& p, const __half* act, const __half* extra,
                     const __half* wpacked, int B, int D, int H, int W, cudaStream_t st);

// one-time cudaFuncSetAttribute calls (kept out of stream capture)
int kernels_init();
int conv_init();

int cast_f32_to_f16(const float* src, __half* dst, size_t n, cudaStream_t st);

}  // namespace cm
