/*
 * crowdmod_b200.h — C ABI of the B200-native (sm_100a) hot path of marcemq/crowdmod-ddpm-4D.
 *
 * The reference has no FFI of its own (it is pure PyTorch); these entry points are what a
 * binding of its hot path consumes.  Each one names the reference interface it replaces
 * (paths relative to the reference repo root).  Plain pointers and sizes only: no torch types.
 * All device pointers are caller-owned; every call is stream-ordered on `stream` (a
 * cudaStream_t passed as void*) and never synchronises unless stated.
 *
 * Return value: 0 = ok, non-zero = error; cm_last_error() returns the message.
 *
 * Tensor conventions (reference utils/dataset.py:48-53, models/backbones/unet.py:133-138):
 *   API tensors   : fp32, contiguous, [B, C, H(rows), W(cols), L(time)], time fastest.
 *   internal      : channels-last, time-major [B, L, H, W, C]; fp32 residual stream, fp16 MMA operands.
 */
#ifndef CROWDMOD_B200_H
#define CROWDMOD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CM_MAX_LEVELS 8
#if defined(__GNUC__)
#define CM_API __attribute__((visibility("default")))
#else
#define CM_API
#endif

/* Mirrors the constructor of models/backbones/unet.py:11-25 plus the tensor geometry the
 * reference takes from cfg.MACROPROPS / cfg.DATASET (models/diffusion/ddpm.py:211). */
typedef struct cm_unet_config {
  int32_t in_channels;      /* UNet(input_channels)  = mprops_count               */
  int32_t out_channels;     /* UNet(output_channels)                              */
  int32_t num_res_blocks;   /* cfg ... UNET.NUM_RES_BLOCKS                        */
  int32_t base_channels;    /* BASE_CH (multiple of 32)                           */
  int32_t num_levels;       /* len(BASE_CH_MULT)                                  */
  int32_t mult[CM_MAX_LEVELS];   /* BASE_CH_MULT                                  */
  int32_t attn[CM_MAX_LEVELS];   /* APPLY_ATTENTION[level] (extra entries ignored)*/
  int32_t time_multiple;    /* TIME_EMB_MULT                                      */
  int32_t rows, cols;       /* MACROPROPS.ROWS / COLS                             */
  int32_t past_len, future_len;  /* DATASET.PAST_LEN / FUTURE_LEN                 */
  int32_t table_steps;      /* rows of the sinusoid table (1000, embeddings.py:7) */
  int32_t weight_terms;     /* 1: fp16 weights, 2: fp16 hi+lo split weights       */
  int32_t dgrad_terms;      /* training: dOut operand of every data-gradient conv: 1 = single fp16,
                               2 = K-concatenated hi+lo fp16 pair (0 -> 2)        */
  int32_t train_act_terms;  /* training forward: activation operand of every conv: 1 = single fp16 (as
                               in sampling), 2 = hi+lo fp16 pair (0 -> 2).  With 2 the saved activations
                               are exact to 2^-22, which is what brings EVERY parameter-gradient tensor
                               within 1e-3 of the fp32 reference (fp16-rounded activations alone put the
                               deep layers' gradients at 1.3e-3 .. 2e-3)           */
} cm_unet_config;

typedef struct cm_unet cm_unet;   /* opaque */

/* ---- library ---- */
CM_API int cm_version(void);
CM_API const char* cm_last_error(void);
/* Reads and clears the device-side protocol-error flag (0 = none).  Synchronises. */
CM_API int cm_device_error(void);

/* ---- backbone: replaces UNet.__init__/state_dict/forward (unet.py:11-167) ---- */
CM_API int cm_unet_create(const cm_unet_config* cfg, cm_unet** out);
CM_API int cm_unet_destroy(cm_unet* u);
/* state_dict mirror: number of entries, and entry i's name / shape (ndim <= 5). */
CM_API int cm_unet_param_count(const cm_unet* u);
CM_API int cm_unet_param_info(const cm_unet* u, int idx, char* name, int name_cap, int64_t* shape5,
                       int* ndim);
/* Bind the fp32 device tensor of state_dict entry `name` (not copied: must stay alive). */
CM_API int cm_unet_set_param(cm_unet* u, const char* name, const float* dev_ptr, int64_t numel);
/* Bind every state_dict entry in one call: ptrs[i] = fp32 device tensor of entry i (the order of
 * cm_unet_param_info), count = cm_unet_param_count.  Cheap when nothing moved. */
CM_API int cm_unet_bind_params(cm_unet* u, const void* const* ptrs, int count);
/* Re-derive the kernel-layout caches (fp16 packed weights, time-embedding projection table)
 * from the bound fp32 parameters: ONE table-driven launch, stream-ordered, no host synchronisation
 * (unless parameter storage moved since the last call).  Call after load_state_dict / optimizer.step. */
CM_API int cm_unet_pack(cm_unet* u, int build_time_table, void* stream);
/* Size internal workspaces + TMA descriptors for batches up to `batch` (allocates; not
 * capturable).  Returns bytes via *bytes if non-NULL. */
CM_API int cm_unet_reserve(cm_unet* u, int batch, int64_t* bytes);
/* eps = UNet.forward(future[B,C,H,W,F], t[B] int64, past[B,C,H,W,P]) (unet.py:124-167), eval mode. */
CM_API int cm_unet_forward(cm_unet* u, const float* future, const int64_t* t, const float* past,
                    float* eps_out, int batch, void* stream);
/* Number of kernel launches one forward enqueues / algorithmic conv+attention FLOPs per sample. */
CM_API int cm_unet_launches_per_forward(const cm_unet* u);
CM_API double cm_unet_flops_per_sample(const cm_unet* u);


/* ---- training: replaces what autograd executes for DDPM_model._train_step / loss.backward()
 *      (models/diffusion/ddpm.py:111-121,142-144; SURVEY.md Appendix B) ---- */
/* Flat parameter-gradient buffer: offsets[i] = element offset of state_dict entry i (the order
 * of cm_unet_param_info; every entry 16-byte aligned), *total = elements to allocate. */
CM_API int cm_unet_grad_layout(const cm_unet* u, int64_t* offsets, int cap, int64_t* total);
/* Dropout3d scale table layout (layers.py:42,70): block k of the plan (encoder, bottleneck,
 * decoder ResnetBlocks in order) reads channels[k] columns at offsets[k] of a [batch][*ld] fp32
 * table holding mask/(1-p).  Returns the number of blocks. */
CM_API int cm_unet_dropout_layout(const cm_unet* u, int32_t* offsets, int32_t* channels, int cap,
                                  int32_t* ld);
/* Training-mode UNet.forward: as cm_unet_forward, plus saves what the backward needs (GroupNorm
 * statistics, time-MLP pre-activations; every activation stays resident in the workspace) and
 * applies the optional Dropout3d scales (NULL = no dropout).  future / past / drop_scale must stay
 * alive until cm_unet_backward returns. */
CM_API int cm_unet_train_forward(cm_unet* u, const float* future, const int64_t* t, const float* past,
                                 float* eps_out, int batch, const float* drop_scale, void* stream);
/* Backward of the last cm_unet_train_forward: d_eps [B,C,H,W,F] (gradient of the loss w.r.t. the
 * predicted noise) -> grads (flat fp32, cm_unet_grad_layout; overwritten).  dgrad / wgrad of every
 * conv run on tcgen05; gradients are carried with a power-of-two loss scale chosen on the device
 * and unscaled before returning.  One backward per forward. */
CM_API int cm_unet_backward(cm_unet* u, const float* d_eps, float* grads, void* stream);
CM_API int64_t cm_last_backward_launches(const cm_unet* u);

/* Measurement support for bench.py: the plan's ops (tag, kind: 0 first conv, 1 GroupNorm+SiLU,
 * 2 tcgen05 conv, 3 attention core, 4 final conv; algorithmic FLOPs per sample in the
 * reference's dense formulation) and one forward with CUDA events around every launch
 * (ms_out[i] = device time of op i on `stream`).  Synchronises. */
CM_API int cm_unet_op_count(const cm_unet* u);
CM_API int cm_unet_op_info(const cm_unet* u, int idx, char* tag, int tag_cap, int* type,
                           double* flops_per_sample);
/* FLOPs per sample op `idx` actually EXECUTES: as cm_unet_op_info except that the UpSample convs count
 * their 8 phase convs of 2x2x2 folded taps (8/27 of the dense 27-tap formulation). */
CM_API double cm_unet_op_exec_flops(const cm_unet* u, int idx);
CM_API int cm_unet_profile_forward(cm_unet* u, const float* future, const int64_t* t, const float* past,
                                   float* eps_out, int batch, void* stream, float* ms_out, int cap);

/* Bring-up / test support: read back an intermediate tensor of the LAST forward from the workspace.
 * cm_unet_debug_op_tensor: index of the tensor op `op_idx` writes (-1 = none; GroupNorm ops: the normalised
 * fp16 operand).  cm_unet_debug_tensor_read copies samples [sample0, sample0+nsamples) of tensor `tensor` --
 * kind 32: the fp32 copy, 16: the fp16 operand -- as [nsamples][pixels][C] to the DEVICE buffer `dst`
 * (stream-ordered); returns the channel count through *C and pixels per sample through *pixels. */
CM_API int cm_unet_debug_op_tensor(const cm_unet* u, int op_idx);
CM_API int cm_unet_debug_tensor_read(const cm_unet* u, int tensor, int kind, int sample0, int nsamples, void* dst,
                                     int64_t dst_bytes, int* C, int* pixels, void* stream);

/* ---- reverse chain: replaces DDPM_model._generate_ddpm/_generate_ddim (ddpm.py:206-282)
 *      with DDPM.step (ddpm.py:25-38) fused into the last conv's epilogue ---- */
typedef struct cm_chain_args {
  const float* past;        /* [n,C,H,W,P] device                                   */
  float* x;                 /* [n,C,H,W,F] device; in: x_T, out: x_0                */
  int32_t n;                /* samples in this shard                                */
  int32_t nsteps;           /* denoiser evaluations                                 */
  const int32_t* tsteps;    /* HOST [nsteps] timestep fed to the denoiser at step i */
  const float* coef;        /* HOST [nsteps][8] per-step update coefficients:
                               mode 0 (DDPM): {1/sqrt(alpha_t), beta_t/sqrt(1-abar_t), sqrt(beta_t)|0, g, ...}
                               mode 1 (DDIM): {sqrt(1-abar_t), sqrt(abar_t), sqrt(abar_prev), dir, sigma, g, ...}
                               g = lambda*sigma for Sparsity guidance, else 0       */
  int32_t mode;             /* 0 DDPM, 1 DDIM                                       */
  const float* noise;       /* device [nsteps][n*C*H*W*F] injected z, or NULL -> Philox(seed) */
  uint64_t seed;            /* passed through device memory: a new seed re-uses the graph */
  int64_t sample_offset;    /* global index of sample 0 (shard-invariant Philox)    */
  float* history;           /* optional device [nsteps+1][n*C*H*W*F] (slot 0 = x_T by caller) */
  int32_t use_graph;        /* 0: eager launches; 1: one step captured as a CUDA graph, replayed
                               nsteps times; 2: the WHOLE chain as one graph (a conditional WHILE
                               node over the device step counter): one cudaGraphLaunch per chain */
} cm_chain_args;
/* past / x are copied into the handle's own staging buffers first (and x_0 back at the end), so the
 * cached graph depends on (n, nsteps, mode, noise, history) only; nothing synchronises. */
CM_API int cm_ddpm_sample(cm_unet* u, const cm_chain_args* args, void* stream);
/* cudaGraphLaunch calls issued by the last cm_ddpm_sample (1 in mode 2, nsteps in mode 1, 0 eager) and
 * whether that call had to (re)build its graph. */
CM_API int64_t cm_last_chain_graph_launches(const cm_unet* u);
CM_API int cm_last_chain_graph_rebuilt(const cm_unet* u);
/* kernels enqueued by the last cm_ddpm_sample call (for bench accounting) */
CM_API int64_t cm_last_chain_launches(const cm_unet* u);

/* ---- op-level entry points (unit tests / layer parity; allocate temporaries, synchronise) ---- */
/* mode: 0 k3 s1 p1, 1 k3 s2 p1, 2 nearest-x2 + k3 p1, 3 1x1x1.  act16: fp16 channels-last
 * [B,D,H,W,cin]; w: fp32 [cout,cin,taps]; wx: optional fp32 [cout,cin_extra] 1x1 slab over
 * extra16 [B,od,oh,ow,cin_extra].  impl: 0 tcgen05 kernel, 1 scalar restatement (test only). */
CM_API int cm_op_conv3d(int mode, const void* act16, int B, int D, int H, int W, int cin,
                 const void* extra16, int cin_extra, const float* w, const float* wx,
                 const float* bias, int cout, int terms, const float* resid, float* out32,
                 void* out16, int impl, void* stream);
CM_API int cm_op_gn_silu(const float* src0, int c0, const float* src1, int c1, const float* gamma,
                  const float* beta, int B, int pixels, float eps, int silu, void* out_norm16,
                  void* out_raw16, void* stream);
/* attention core softmax(Q K^T / sqrt(dh)) V per (sample, head): qkv fp32 [B][S][3C] (q | k | v), ctx16 fp16 [B][S][C]
 * out.  Any S (S > 128 streams the keys with the online softmax); dh = C / heads even and <= 64. */
CM_API int cm_op_attn_core(const float* qkv, void* ctx16, int B, int S, int C, int heads, void* stream);
/* backward of the attention core (autograd of softmax(Q K^T / sqrt(dh)) V inside nn.MultiheadAttention, reference
 * models/backbones/layers.py:5-18 under loss.backward(), ddpm.py:143): qkv fp32 [B][S][3C] (the in_proj output the
 * training forward saved), dctx fp32 [B][S][C] = gradient of the core's output, dqkv fp32 [B][S][3C] out.  Any S;
 * S <= 128 needs dh % 4 == 0, S > 128 dh even and <= 64 (the forward is rerun into temporaries for its output and
 * row log-sum-exp).  Deterministic. */
CM_API int cm_op_attn_core_backward(const float* qkv, const float* dctx, float* dqkv, int B, int S, int C, int heads,
                             void* stream);
/* whole AttentionBlock of the sampling path (reference models/backbones/layers.py:5-18: GroupNorm(8) ->
 * nn.MultiheadAttention(C, heads) self-attention -> + x) as ONE launch.  x, out32: fp32 [B][S][C] tokens
 * (channels-last); w_in [3C][C] / b_in [3C] = mhsa.in_proj_weight / in_proj_bias, w_out [C][C] / b_out [C] =
 * mhsa.out_proj.weight / .bias.  Covers C = 128, heads = 4, S <= 128 (returns an error otherwise). */
CM_API int cm_op_attn_block(const float* x, const float* gamma, const float* beta, const float* w_in,
                     const float* b_in, const float* w_out, const float* b_out, float* out32, void* out16,
                     int B, int S, int C, int heads, float eps, void* stream);
CM_API int cm_op_first_conv(const float* x, const float* past, const float* w, const float* bias,
                     float* out, int B, int H, int W, int P, int F, int cin, int cout,
                     void* stream);
CM_API int cm_op_final_conv(const void* act16, const float* w, const float* bias, float* eps_out, int B,
                     int H, int W, int L, int P, int cin, int cout, void* stream);

/* Backward op-level entry points.  Geometry arguments describe the FORWARD conv (mode, input
 * grid B,D,H,W, cin, cout); dout16 is the fp16 gradient on the forward output grid.
 * dgrad: dx32 fp32 [B,D,H,W,cin] (overwritten).  wgrad: dw fp32 [cout,cin,taps] with taps in
 * activation-dim order, dwx fp32 [cout,cin_extra] or NULL; impl 0 = tcgen05 kernel, 1 = scalar
 * restatement (test only). */
CM_API int cm_op_conv3d_dgrad(int mode, const void* dout16, int B, int D, int H, int W, int cin,
                              const float* w, int cout, int terms, float* dx32, void* stream);
/* As cm_op_conv3d_dgrad from the fp32 gradient: casts to the fp16 operand (dup = 1) or to the
 * K-concatenated hi|lo pair (dup = 2) exactly as the training backward does. */
CM_API int cm_op_conv3d_dgrad_f32(int mode, const float* dout32, int B, int D, int H, int W, int cin,
                                  const float* w, int cout, int terms, int dup, float* dx32, void* stream);
CM_API int cm_op_conv3d_wgrad(int mode, const void* act16, int B, int D, int H, int W, int cin,
                              const void* extra16, int cin_extra, const void* dout16, int cout,
                              float* dw, float* dwx, int impl, void* stream);

/* fp32 kernels of the training backward, one enqueue function each (tests compare them with float64 autograd).
 * Channels-last fp32 tensors [B][pixels][C] unless stated.
 *
 * GroupNorm(8) (+SiLU) (+Dropout3d scale) backward over the channel concat of src0 [.][c0] and src1 [.][c1] (c1 = 0:
 * one source; C = c0 + c1 a multiple of 32, c0 of 4): stats [B][8][2] = the forward's (mean, rstd) per group; dnorm
 * [B][pixels][C] = gradient of the (scaled) output; draw: optional gradient added to dx unchanged; drop_scale:
 * optional [B][drop_ld] scale per (sample, channel).  dsrc0 / dsrc1 (=) when init0 / init1, else (+=).  dgamma /
 * dbeta [C] (=): params_all = 0 through the per-GroupNorm kernel, 1 through the table kernel the model uses. */
CM_API int cm_op_gn_backward(const float* src0, int c0, const float* src1, int c1, const float* gamma, const float* beta,
                             const float* stats, const float* dnorm, const float* draw, const float* drop_scale,
                             int drop_ld, int B, int pixels, int silu, float* dsrc0, int init0, float* dsrc1, int init1,
                             float* dgamma, float* dbeta, int params_all, void* stream);
/* dOut preparation of a conv: src fp32 [B][pixels][C] -> dst16 fp16 [B][pixels][C] (dup 1) or the hi|lo pair
 * [B][pixels][2C] (dup 2; NULL: no cast); acc_dst (=) src when acc_init, else (+=) (NULL: none); colsum[b * colsum_ld
 * + c] += per-sample channel sums (NULL: none).  A value beyond the fp16 range is clamped and sets device error 301. */
CM_API int cm_op_cast_colsum(const float* src, void* dst16, int dup, float* acc_dst, int acc_init, float* colsum,
                             int colsum_ld, int B, int pixels, int C, void* stream);
/* Bias gradients of n convs in one launch: tab (HOST) [n][4] = {source offset (floats from base), row stride,
 * channels, output offset (floats into grads)}; grads[out + c] = sum_b base[src + b * ld + c]. */
CM_API int cm_op_rowsum_all(const float* base, const int64_t* tab, int n, int B, float* grads, void* stream);
/* Final conv backward (unet.py:121,165-167): deps fp32 [B][cout][H][W][L-P] (API layout, future frames) times the
 * loss scale `scale`; act16 fp16 [B][L][H][W][act_ld] (act_ld 0 -> cin; act_lo > 0: hi|lo pair rows, lo at +act_lo);
 * w [cout][cin][27].  dact fp32 [B][L][H][W][cin], dw [cout][cin][27], db [cout], all (=) and scaled by `scale`.
 * dout16 NULL: the SIMT weight gradient (cin 32 or 64); else a caller-owned fp16 [B][L][H][W][32] buffer that
 * receives the packed d_eps * scale, and dw comes from the conv weight gradient over it, as in the training backward. */
CM_API int cm_op_final_conv_backward(const float* deps, float scale, const void* act16, int act_ld, int act_lo,
                                     const float* w, float* dact, float* dw, float* db, int B, int H, int W, int L,
                                     int P, int cin, int cout, void* dout16, void* stream);
/* First conv weight / bias gradient (unet.py:32): x [B][cin][H][W][F], past [B][cin][H][W][P] (API layout), dout fp32
 * [B][L][H][W][cout]; dw [cout][cin][27], db [cout] (=). */
CM_API int cm_op_first_conv_wgrad(const float* x, const float* past, const float* dout, float* dw, float* db, int B,
                                  int H, int W, int P, int F, int cin, int cout, void* stream);
/* Time-embedding MLP backward as the training backward runs it (embeddings.py:22-34, layers.py:35,62): e [B][base],
 * h1 / h2 [B][E] the pre-activations, dtemb [B][ld] the gradient of every block's dense_1 output (block k: columns
 * offs[k] .. + couts[k], weight wd[k] [couts[k]][E]); wd / couts / offs / goff_w / goff_b are HOST arrays [nblocks]
 * (wd: device pointers).  Outputs (=): dense_1 weight / bias gradients into dense_grads at goff_w / goff_b, dw1
 * [E][base], db1 [E], dw2 [E][E], db2 [E], and ds1 / ds2 [B][E], the gradients w.r.t. SiLU(h1) and SiLU(h2). */
CM_API int cm_op_temb_backward(const float* e, const float* h1, const float* h2, const float* dtemb, int ld, int B,
                               int base, int E, const float* w2, const void* const* wd, const int32_t* couts,
                               const int32_t* offs, int nblocks, float* dense_grads, const int64_t* goff_w,
                               const int64_t* goff_b, float* dw1, float* db1, float* dw2, float* db2, float* ds1,
                               float* ds2, void* stream);
/* Loss scale of the training backward: scale_out[0] = S = 2^e with e = floor(log2(target / max|x|)) clamped to
 * [-60, 60] (1 when max|x| is 0 or not finite), scale_out[1] = 1/S (device float[2]). */
CM_API int cm_op_loss_scale(const float* x, int64_t n, float target, float* scale_out, void* stream);

/* ---- second backbone: DiT4D_V4 (SURVEY.md section 8 f2) ------------------------------------------------------
 * Replaces /root/reference/models/backbones/DiT4D_V4.py:228-375 (selected by --arch DDPM-DiT at
 * models/diffusion/ddpm.py:88-104) for inference / sampling: same forward(future, t, past) contract and the same
 * reverse chain (cm_chain_args) as the UNet plan; parameters are bound by the reference's state_dict names. */
typedef struct cm_dit_config {
  int32_t in_channels, out_channels;   /* mprops_count (1..4)                                   */
  int32_t rows, cols;                  /* MACROPROPS.ROWS / COLS                                */
  int32_t past_len, future_len;        /* DATASET.PAST_LEN / FUTURE_LEN                         */
  int32_t t_patch, patch;              /* T_PATCH_SIZE / PATCH_SIZE                             */
  int32_t hidden, depth, heads;        /* HIDDEN_SIZE / DEPTH / NUM_HEADS                       */
  int32_t mlp_hidden;                  /* int(HIDDEN_SIZE * MLP_RATIO)                          */
  int32_t time_multiple;               /* TIME_EMB_MULT                                         */
  int32_t table_steps;                 /* rows of the sinusoid table (total_time_steps)         */
  int32_t t_max_slots;                 /* rows of temporal_pos_embed (T_max // t_patch)         */
} cm_dit_config;
typedef struct cm_dit cm_dit;
CM_API int cm_dit_create(const cm_dit_config* cfg, cm_dit** out);                  /* DiT4D_V4.__init__ :229-311 */
CM_API int cm_dit_destroy(cm_dit* d);
CM_API int cm_dit_param_count(const cm_dit* d);
CM_API int cm_dit_param_info(const cm_dit* d, int idx, char* name, int name_cap, int64_t* shape5, int* ndim);
CM_API int cm_dit_bind_params(cm_dit* d, const void* const* ptrs, int count);      /* state_dict order of param_info */
CM_API int cm_dit_pack(cm_dit* d, void* stream);                                   /* fp16 hi|lo caches; after load / weight change */
/* DiT4D_V4.forward(future, t, past) :348-375 (eval): future fp32 [B,C,H,W,F], t int64 [B], past fp32 [B,C,H,W,P], all device */
CM_API int cm_dit_forward(cm_dit* d, const float* future, const int64_t* t, const float* past, float* eps_out, int batch,
                   void* stream);
/* _generate_ddpm / _generate_ddim with this backbone (ddpm.py:206-282): the update is fused into the un-patch kernel;
 * the AdaLN vectors of all timesteps come from a table built once per weight load; use_graph = 0 eager launches,
 * != 0 one captured step replayed nsteps times (seed / offset / x / past go through buffers the handle owns) */
CM_API int cm_dit_sample(cm_dit* d, const cm_chain_args* args, void* stream);
CM_API double cm_dit_flops_per_sample(const cm_dit* d);
CM_API int64_t cm_dit_last_launches(const cm_dit* d);

/* ---- callers either side of the hot path (SURVEY.md section 8 f3 / f4) -------------------------------------- */

/* Data feed: one batch of (past, future) windows gathered ON the device from HBM-resident raw sequences.
 * Replaces MacropropsDataset.__getitem__ + DataLoader collate + the per-step host->device copy
 * (/root/reference/utils/dataset.py:46-53, models/diffusion/ddpm.py:136-137).
 * seq: fp32 [n_seq][channels][rows][cols][raw_len]; seq_idx / t0: int32 device tables of the dataset's windows
 * (sequence and first frame, the (seq_idx, t) pairs of dataset.py:33-37); ids: int64 [batch] device, the windows of
 * this batch (NULL: windows 0..batch-1); past: fp32 [batch][channels][rows][cols][past_len], future: fp32
 * [batch][channels][rows][cols][future_len].  Bit-exact copy; ONE launch, stream-ordered, no allocation. */
CM_API int cm_window_gather(const float* seq, int64_t n_seq, int channels, int rows, int cols, int raw_len,
                     const int32_t* seq_idx, const int32_t* t0, const int64_t* ids, int batch, int past_len,
                     int future_len, float* past, float* future, void* stream);

/* Metrics tail: per (sample, frame) reductions from which PSNR / MASK_PSNR / RE_DENSITY / TV_OVER_TIME and the
 * macro-property ranges are closed forms (/root/reference/utils/metrics/metricsGenerator.py:43-92,120-186,293-339).
 * pred, gt: fp32 [n][channels >= 3][rows][cols][frames] on the device (rho, vx, vy first).
 * out: fp64 [n][frames][CM_METRICS_PER_FRAME] on the device:
 *   [0..2]  sum (gt - pred)^2 per property        [3..5]  the same over cells with gt rho > 1e-5   [6] number of such cells
 *   [7..9]  total variation of pred per property  [10..12] total variation of gt
 *   [13]    sum of pred rho   [14] sum of gt rho   [15 + 2c], [16 + 2c]  min / max of gt property c */
#define CM_METRICS_PER_FRAME 21
CM_API int cm_metrics_reduce(const float* pred, const float* gt, int n, int channels, int rows, int cols, int frames,
                      double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CROWDMOD_B200_H */
