// Backward-pass kernels of the UNet hot path (training: reference models/diffusion/ddpm.py:111-121,
// 142-144; SURVEY.md Appendix B lists what autograd executes for the reference graph).
//
// Data gradients of the convolutions reuse conv_umma_kernel with re-packed weights; weight
// gradients run on wgrad_umma_kernel (wgrad_umma.cuh).  This header declares the packers and
// the remaining (bandwidth / small) kernels.  All gradients flow scaled by a power-of-two loss
// scale S (device scalar) so that fp16 MMA operands do not underflow; parameter gradients are
// unscaled once at the end (scale_inplace_enqueue).
#pragma once
#include "common.cuh"

namespace cm {

// ---- dgrad weight packing: fwd weight w [cout_f][cin_f][taps] (+ optional 1x1 slab handled by a
//      separate call with fwd_mode 3) -> rows n = cin_f (x terms), K-major columns for the conv
//      mode that computes the data gradient:
//      fwd mode 0 (k3 s1)  -> mode 0 with flipped taps,           K = 27*cout_f
//      fwd mode 3 (1x1)    -> mode 3,                             K = cout_f
//      fwd mode 1 (k3 s2)  -> mode 2 (8 phases x 8 taps, scatter), K = 64*cout_f
//      fwd mode 2 (up+k3)  -> mode 4 (k4 s2),                      K = 64*cout_f
// perm as in pack_conv_weights (kernels.cuh).
// dup = 2: the dOut operand is a K-concatenated hi|lo fp16 pair (pack.cuh), K doubles.
int pack_dgrad_weights(int fwd_mode, const float* w, __half* dst, int cout_f, int cin_f, int terms,
                       int perm, int dup, cudaStream_t st);
int dgrad_mode_of(int fwd_mode);
size_t dgrad_packed_k(int fwd_mode, int cout_f, int dup = 1);

// ---- loss scale: S = 2^floor(log2(target / max|x|)) (1 if x == 0); scale[0] = S, scale[1] = 1/S ----
// max_scratch: one zero-initialised device word (left zero on return)
int auto_scale_enqueue(const float* x, size_t n, float target, float* scale_dev, unsigned int* max_scratch,
                       cudaStream_t st);

// ---- dOut preparation for one conv: fp32 grad [B][pixels][C] -> fp16 operand, optional
//      residual fan-out (acc_dst (=|+=) src) and per-sample channel sums (bias / time-embedding
//      projection gradients): colsum[b*colsum_ld + c] += sum_p src[b][p][c].  dup = 2: dst16 is the
//      K-concatenated hi|lo pair [pixel][2C] (dgrad reads both halves, wgrad the hi half) ----
// part != nullptr (deterministic): every CTA stores its channel sums into part [chunks][B][C] and one more launch adds
// them to colsum in chunk order, instead of one atomicAdd per (CTA, channel); part holds cast_colsum_partial_elems.
int cast_colsum_enqueue(const float* src, __half* dst16, int dup, float* acc_dst, int acc_init, float* colsum,
                        int colsum_ld, int B, int pixels, int C, cudaStream_t st, float* part = nullptr);
size_t cast_colsum_partial_elems(int B, int pixels, int C);
// The ordered sum of deterministic reductions: for i < n, dst[(i / seg) * dst_ld + i % seg] (=, or += when
// accumulate) sum over s = 0, 1, ..., nsplit - 1 of part[s * stride + i], added in that order.
int sum_partials_enqueue(const float* part, int nsplit, size_t stride, size_t n, size_t seg, size_t dst_ld, float* dst,
                         int accumulate, cudaStream_t st);
// out[c] (+)= sum_b in[b*ld + c]
int rowsum_enqueue(const float* in, float* out, int B, int C, int ld, int accumulate, cudaStream_t st);

// ---- G (packed-K rows, wgrad_umma.cuh) -> nn.Conv3d weight-gradient layout ----
// mode 0/1: dw[co][ci][27] (tap permuted as in pack_conv_weights) (+ dwx[co][cinx]);
// mode 3: dw[co][ci] (+dwx); mode 2: the 8x8 phase/tap gradients are folded onto the 27 taps.
int unpack_wgrad_enqueue(int fwd_mode, const float* G, float* dw, float* dwx, int cout, int cin,
                         int cinx, int perm, cudaStream_t st);

// ---- scalar restatement of the weight gradient (test oracle for wgrad_umma_kernel).  Same
//      operands, same G layout, G must be zeroed. ----
int wgrad_ref_enqueue(int fwd_mode, const __half* act16, const __half* extra16, const __half* dout16,
                      float* G, int B, int D, int H, int W, int cin, int cinx, int cout,
                      cudaStream_t st);

// ---- GroupNorm(+SiLU)(+Dropout3d scale) backward (layers.py:30,41,57,70; unet.py:119-120) ----
struct GnBwdParams {
  const float* src0; const float* src1; int c0, c1;     // forward inputs (fp32, channels-last)
  const float* gamma; const float* beta;
  const float* stats;       // [B][8][2] mean, rstd saved by the forward
  const float* dnorm;       // fp32 grad w.r.t. the normalised fp16 output [B][pixels][C]
  const float* draw;        // optional fp32 grad w.r.t. the raw fp16 copy (match_input operand)
  const float* drop_scale;  // [B][drop_ld] (+ channel) or nullptr
  int drop_ld;
  int B, pixels, silu;
  float* dsrc0; float* dsrc1;   // (=) when init flag set, else (+=)
  int init0, init1;
  float* chsum;             // scratch [B][C][2]: per-sample sum(dz), sum(dz*xhat)
  float* dgamma; float* dbeta;  // [C], written (=)
};
// partial: scratch of B * gn_bwd_chunks(B, pixels) * C * 2 floats (chunks <= 32)
int gn_bwd_chunks(int B, int pixels);
int gn_backward_enqueue(const GnBwdParams& p, float* partial, cudaStream_t st);
// dgamma / dbeta of every GroupNorm in one launch (GnBwdParams::dgamma == nullptr defers them): tab[g] =
// {chsum offset, C, dgamma offset, dbeta offset} in floats
int unpack_wgrad_all_enqueue(const long long* tab, int n, const float* Gbase, float* grads, cudaStream_t st);
int rowsum_all_enqueue(const float* base, const long long* tab, int n, int B, float* grads, cudaStream_t st);
int gn_backward_params_all_enqueue(const float* chsum_base, const long long* tab, int n_gn, int B, float* grads,
                                   cudaStream_t st);

// ---- attention core backward (layers.py:16): qkv fp32 [B*S][3C] saved by the forward,
//      dctx fp32 [B*S][C] -> dqkv fp32 [B*S][3C] (=).  One fp32 CTA per (sample, head) with the S x S tile in shared
//      memory (lse / dsum unused), unless attn_uses_long(S, dh) (attn_long.cu): two deterministic kernels that recompute P from qkv
//      and lse (fp32 [B][heads][S], the row log-sum-exp attn_core_enqueue wrote); dsum (fp32 [B][heads][S]) is their
//      workspace for the row sums D_i = sum_j P_ij dP_ij. ----
int attn_core_backward_enqueue(const float* qkv, const float* dctx, float* dqkv, int B, int S, int C,
                               int heads, cudaStream_t st, const float* lse = nullptr, float* dsum = nullptr);
int attn_long_backward_enqueue(const float* qkv, const float* dctx, const float* lse, float* dsum, float* dqkv, int B,
                               int S, int C, int heads, cudaStream_t st);

// ---- final conv backward (unet.py:121,165-167): deps API layout [B][cout][H][W][F], times *scale;
//      dact (=) fp32 [B][L][H][W][cin]; dw [cout][cin][27] / db [cout] accumulated with atomics ----
// act: fp16 [B][L][H][W][act_ld] (act_ld 0 -> cin); act_lo > 0: hi|lo pair rows, the lo half is added
// dout16 != nullptr: dw is left to the caller, which runs a conv weight gradient over dout16 (fp16 [B][L][H][W][32],
// d_eps * scale in columns 0 .. cout-1); cin <= 64 without it, <= 256 with it
// part != nullptr (deterministic): per-CTA partial sums into part (final_conv_partial_elems), dw / db (=) their sums
// in CTA order
int final_conv_backward_enqueue(const float* deps, const float* scale_dev, const __half* act, int act_ld, int act_lo,
                                const float* w, float* dact, float* dw, float* db, int B, int H, int W,
                                int L, int P, int cin, int cout, __half* dout16, cudaStream_t st,
                                float* part = nullptr);
size_t final_conv_partial_elems(int B, int H, int W, int L, int P, int cin, int cout, bool packed);
// ---- first conv weight / bias gradient (unet.py:32; inputs need no gradient) ----
// dout fp32 [B][L][H][W][cout]; dw [cout][cin][27], db [cout] accumulated with atomics, or with part != nullptr
// (deterministic) (=) the CTA-ordered sums of per-CTA partials in part (first_conv_partial_elems).
int first_conv_wgrad_enqueue(const float* x, const float* past, const float* dout, float* dw, float* db,
                             int B, int H, int W, int P, int F, int cin, int cout, cudaStream_t st,
                             float* part = nullptr);
size_t first_conv_partial_elems(int B, int H, int W, int P, int F, int cin, int cout);

// ---- time-embedding MLP backward helpers (embeddings.py:22-34; layers.py:35,62) ----
// C[m][n] (=|+=) sum_k A(m,k) * B(k,n) with arbitrary element strides (tiny matrices only)
int small_gemm_enqueue(int M, int N, int K, const float* A, int sam, int sak, const float* Bm, int sbk,
                       int sbn, float* Cm, int ldc, int accumulate, cudaStream_t st);
// every block's dense_1 weight/bias gradient and the gradient of its input (SiLU(h2)) in two launches
int temb_dense_backward_enqueue(const float* dtemb, int ld, int B, const float* s2, int E, const float* const* wd,
                                const int* couts, const int* offs, int nblocks, float* grads,
                                const long long* goff_w, const long long* goff_b, float* ds2, cudaStream_t st);
// dpre = dpost * silu'(pre)
int silu_backward_enqueue(const float* pre, const float* dpost, float* dpre, size_t n, cudaStream_t st);
// y = silu(x)
int silu_forward_enqueue(const float* x, float* y, size_t n, cudaStream_t st);
int scale_inplace_enqueue(float* x, size_t n, const float* factor_dev, cudaStream_t st);
// The whole time-embedding MLP backward (embeddings.py:22-34 and every block's dense_1): e [B][base] = table rows,
// h1 = e W1^T + b1, h2 = SiLU(h1) W2^T + b2 (the forward's saves), dtemb [B][ld] = gradient of the dense_1 outputs
// (block k: columns offs[k] .. offs[k] + couts[k]); s1, s2, ds1, ds2, dh1, dh2 are [B][E] scratch, left holding
// SiLU(h1), SiLU(h2) and the gradients w.r.t. those and h1, h2.  Parameter gradients (=): dense_1 into grads at
// goff_w / goff_b, the MLP's into dw1, db1, dw2, db2.  11 launches.
struct TembBwdParams {
  const float* e; const float* h1; const float* h2;
  const float* dtemb; int ld;
  const float* const* wd; const int* couts; const int* offs; int nblocks;   // device tables
  const long long* goff_w; const long long* goff_b;                         // device tables
  const float* w2;
  float* dw1; float* db1; float* dw2; float* db2;
  float* s1; float* s2; float* ds1; float* ds2; float* dh1; float* dh2;
  int B, E, base;
};
int temb_backward_enqueue(const TembBwdParams& p, float* grads, cudaStream_t st);

// one-time cudaFuncSetAttribute calls (kept out of stream capture)
int backward_init();

}  // namespace cm
