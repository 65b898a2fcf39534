/* ralenet_b200.h -- C ABI of libralenet_b200.so: RA-LENet forward/backward hot path on sm_100a.
 *
 * The reference (caprilovel/ECG_Denoise) is pure Python/PyTorch and has no FFI of its own; the
 * boundary it exposes for this path is the nn.Module surface (SURVEY.md section 8b).  Each entry
 * point below replaces the body of one reference forward (and its autograd backward); the
 * reference lines are cited per function (paths relative to the reference root).  The host-side
 * mirror of the reference interface (same class names / constructor signatures / state_dict) lives
 * in ecg_denoise_b200/model/ and binds these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C: raw device pointers + sizes, no torch types.  All tensors are fp32, contiguous and
 *     16-byte aligned (activations, weights, LayerNorm vectors and positional tiles are accessed 16
 *     bytes at a time; a misaligned pointer is rejected with RL_ERR_SHAPE).
 *   - activations inside the network are token-major [B][L][C] (the reference's layout after
 *     rearrange 'b c l -> b l c', model/transformer.py:630).  One "window" = one ECG window.
 *   - the library never allocates, frees or synchronises: every buffer (incl. workspaces) is owned
 *     by the caller; `stream` is a cudaStream_t passed as void*.  Entry points are re-entrant.
 *   - return value: 0 = ok, <0 = RL_ERR_* ; ralenet_last_error() gives a thread-local message.
 *   - gradients of parameters are ACCUMULATED (+=) into the given buffers, which the caller zero-fills when it
 *     wants plain gradients.  Data gradients are overwritten.  By default the per-CTA partial sums are added with
 *     fp32 atomics, so their low bits depend on scheduling; the whole-network backward with RL_NET_DETERMINISTIC
 *     (rl_net_cfg.flags) stores them into partial slabs and adds them in a fixed order instead (bit-reproducible).
 *   - head_dim is 4 everywhere (C / H == 4), softmax scale = 4^-0.5 (model/transformer.py:277-278).
 */
#ifndef RALENET_B200_H
#define RALENET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RL_ABI_VERSION 4

enum {
  RL_OK = 0,
  RL_ERR_SHAPE = -1,      /* unsupported / inconsistent sizes                     */
  RL_ERR_NULL = -2,       /* required pointer is NULL                              */
  RL_ERR_CUDA = -3,       /* CUDA runtime error (message has the cudaError string) */
  RL_ERR_ARCH = -4        /* device is not sm_100                                  */
};

/* local-enhancement mode of Mlp (model/transformer.py:142-146) */
enum { RL_LE_NONE = 0, RL_LE_PARTIAL = 1, RL_LE_DEPTHWISE = 2 };

/* flags of the attention / feed-forward halves */
enum {
  RL_F_PRENORM = 1,   /* apply (x*sqrt(C) + PE, LayerNorm) resp. LayerNorm in front (TransformerBlock) */
  RL_F_RESIDUAL = 2,  /* add the block input to the result (TransformerBlock)                          */
  RL_F_TF32 = 4       /* forward only: single-pass TF32 projection / feed-forward GEMMs (RL_NET_TF32)  */
};
/* RL_F_TF32 is an inference precision: ralenet_attn_fwd / ralenet_ffn_fwd / ralenet_block_fwd reject it together with
 * saved-tensor pointers (q, k, v, o, lse, h) with RL_ERR_SHAPE, ralenet_block_fwd rejects halves whose RL_F_TF32 bits
 * differ, and ralenet_attn_bwd / ralenet_ffn_bwd reject the bit. */

int ralenet_abi_version(void);
const char* ralenet_last_error(void);
/* checks that device `dev` is sm_100 (B200); RL_ERR_ARCH otherwise.  No fallback exists. */
int ralenet_check_device(int dev);

/* ------------------------------------------------------------------------------------------
 * Attention half of TransformerBlock:  y = x + proj(softmax(0.5 q k^T + bias) v),
 * q,k,v = to_q/to_kv(LN1(x*sqrt(C) + P)).
 * Replaces TransformerBlock.forward_part1 + the residual (model/transformer.py:383-390, 405),
 * MSAttention.forward (:289-323), LinearProjection.forward (:226-247),
 * AbsPositionalEncoding.forward (:179-181) and the R-wave bias RelativePositionEmbedding.forward /
 * mask_fill (:534-558) -- the bias is applied from its (2W-1) x H table, never materialised.
 * Without RL_F_PRENORM / RL_F_RESIDUAL it is MSAttention.forward alone.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, L, C, H;          /* windows, tokens/window, channels, heads (C == 4*H)             */
  int32_t W, c0;               /* R-wave bias window and its offset ((L-W)/2); W == 0: no bias  */
  int32_t flags;               /* RL_F_*                                                        */
  int32_t _pad;
  const float* x;              /* [B,L,C]                                                       */
  const float* pe;             /* [L,C] positional table P[:L] (needed with RL_F_PRENORM)       */
  const float* ln_w; const float* ln_b;     /* norm1 [C]                                        */
  const float* wq;  const float* bq;        /* to_q  [C,C],[C]    (bias may be NULL)            */
  const float* wkv; const float* bkv;       /* to_kv [2C,C],[2C]                                */
  const float* wp;  const float* bp;        /* proj  [C,C],[C]                                  */
  const float* table;          /* relative_position_bias_table [(2W-1),H] or NULL              */
  float* y;                    /* [B,L,C]                                                       */
  /* saved for backward; all NULL for inference */
  float* q; float* k; float* v; float* o;   /* [B,L,C] each                                     */
  float* lse;                  /* [B,H,L] log2-domain log-sum-exp                               */
} rl_attn_fwd_args;

typedef struct {
  int32_t B, L, C, H, W, c0, flags, _pad;
  const float* g;              /* dL/dy [B,L,C]                                                 */
  const float* x; const float* pe;
  const float* ln_w; const float* ln_b;
  const float* wq; const float* wkv; const float* wp;
  const float* table;
  const float* q; const float* k; const float* v; const float* o; const float* lse;
  float* dx;                   /* [B,L,C] dL/dx (overwritten)                                   */
  /* scratch written by the kernel, consumed by the weight-gradient GEMMs of the same call */
  float* dqkv;                 /* [B,L,3C]                                                      */
  float* u;                    /* [B,L,C] LN1 output                                            */
  /* parameter gradients (+=); any may be NULL to skip (frozen core, ralenet_12leads.py:695) */
  float* d_ln_w; float* d_ln_b;
  float* d_wq; float* d_bq; float* d_wkv; float* d_bkv; float* d_wp; float* d_bp;
  float* d_table;
} rl_attn_bwd_args;

int ralenet_attn_fwd(const rl_attn_fwd_args* a, void* stream);
int ralenet_attn_bwd(const rl_attn_bwd_args* a, void* stream);
/* Forward kernels of the wide stages (C = 64, 128).  mode 2: tcgen05 tile kernels (128 tokens = 4 / 8 windows per
 * tile, heads split over a cluster; attn_umma.cu); mode 0: one-window mma.sync kernels (attn.cu); mode 1 (default):
 * the tile kernels while the launch is a single wave of CTAs (the training batch), the others beyond.  All compute
 * the same function; the switch exists for A/B measurements and the agreement test.  Initial value: environment
 * variable RALENET_ATTN_UMMA.  Returns the previous mode.  Not thread-safe against running calls. */
int ralenet_set_attn_umma(int mode);
/* Weight-gradient GEMMs (dW += dY^T X over all tokens) of the stages with C >= 32 and of the patch layers:
 * 1 (default) = tcgen05 kernels (wgrad_umma.cu), 0 = mma.sync kernels (wgrad.cu).  Same function; A/B switch,
 * initial value from RALENET_WGRAD_UMMA.  Returns the previous setting. */
int ralenet_set_wgrad_umma(int on);
/* 1 (default) = register-tile weight-gradient kernel (wgrad_reg.cu: operands streamed from global memory straight
 * into mma.sync fragments, accumulators in registers) for every group whose dimensions are multiples of 32; 0 = the
 * kernels selected by ralenet_set_wgrad_umma.  By default (1) it takes the groups whose largest dW has at most four
 * 32 x 32 tiles (the HBM-bound ones: C = 32 stages and the 32-wide patch layers), 2 = every eligible group.
 * Same function; A/B switch, initial value from RALENET_WGRAD_REG.  Returns the previous setting. */
int ralenet_set_wgrad_reg(int on);

/* ------------------------------------------------------------------------------------------
 * Feed-forward half:  y = x + fc2(GELU(leconv(GELU(fc1(LN2(x))))))  (+ extra)
 * Replaces TransformerBlock.forward_part2 + residual (model/transformer.py:392-395, 410),
 * Mlp.forward (:149-161), PartialConv_1d.forward_split_cat (:54-59) / depthwise Conv1d (:146).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, L, C, le_mode, flags, _pad;
  const float* x;              /* [B,L,C]                                                       */
  const float* extra;          /* optional [B,L,C] added to y (x_mid += x4, transformer.py:646) */
  const float* ln_w; const float* ln_b;     /* norm2 [C]                                        */
  const float* w1; const float* b1;         /* fc1 [4C,C],[4C]                                  */
  const float* w2; const float* b2;         /* fc2 [C,4C],[C]                                   */
  const float* lew;            /* partial: [3]; depthwise: [4C,3]; else NULL                   */
  float* y;                    /* [B,L,C]                                                       */
  float* h;                    /* saved fc1 output (pre-GELU) [B,L,4C] or NULL                  */
} rl_ffn_fwd_args;

typedef struct {
  int32_t B, L, C, le_mode, flags, _pad;
  const float* g;              /* dL/dy                                                         */
  const float* x; const float* ln_w; const float* ln_b;
  const float* w1; const float* w2; const float* lew;
  const float* h;              /* saved by forward                                              */
  float* dx;                   /* [B,L,C] (the gradient w.r.t. `extra` is g itself)             */
  float* dh; float* g2;        /* scratch [B,L,4C] each                                         */
  float* u;                    /* scratch [B,L,C]                                               */
  float* d_ln_w; float* d_ln_b; float* d_w1; float* d_b1; float* d_w2; float* d_b2; float* d_lew;
} rl_ffn_bwd_args;

int ralenet_ffn_fwd(const rl_ffn_fwd_args* a, void* stream);
int ralenet_ffn_bwd(const rl_ffn_bwd_args* a, void* stream);

/* TransformerBlock.forward (model/transformer.py:398-411): attention half then feed-forward half, f->x == a->y.
 * Narrow stages (C <= 32, 256-sample windows, both halves RL_F_PRENORM | RL_F_RESIDUAL) run as ONE fused launch (the
 * block's x1 is written for the backward and read back by the same CTA); every other shape runs the two halves one
 * after the other.  ralenet_set_block_fuse(0) forces the two-launch form (A/B; initial value RALENET_BLOCK_FUSE). */
int ralenet_block_fwd(const rl_attn_fwd_args* a, const rl_ffn_fwd_args* f, void* stream);
int ralenet_set_block_fuse(int on);

/* ------------------------------------------------------------------------------------------
 * PatchMerging.forward (model/transformer.py:440-460): [B,L,C] -> LN(2C) -> Linear(2C,2C) -> [B,L/2,2C]
 * PatchSeparate.forward (:418-424) + U-skip add (:650,654,658): [B,L,C] -> [B,2L,C/2]
 * mode 0 = merge, 1 = separate.  L, C are the INPUT sizes.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, L, C, mode;
  const float* x; const float* skip;        /* skip: optional [B,2L,C/2] (separate only)        */
  const float* ln_w; const float* ln_b; const float* w;
  float* y;
  float* u;                    /* saved LN output, same shape as y, or NULL                     */
} rl_patch_fwd_args;

typedef struct {
  int32_t B, L, C, mode;
  const float* g; const float* g2;          /* dL/dy, optional second gradient summed with g    */
  const float* x; const float* ln_w; const float* w;
  const float* u;              /* saved by forward                                              */
  float* dx;                   /* [B,L,C]                                                       */
  float* gsum;                 /* scratch [B,L*C] receiving g + g2 (required when g2 != NULL)   */
  float* d_ln_w; float* d_ln_b; float* d_w;
} rl_patch_bwd_args;

int ralenet_patch_fwd(const rl_patch_fwd_args* a, void* stream);
int ralenet_patch_bwd(const rl_patch_bwd_args* a, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stem  conv1 = Conv1d(2,8,3,p1) -> LeakyReLU(0.2) -> BatchNorm1d(8)  (model/transformer.py:570-574, 623)
 * output is written token-major [B,L,8] (the rearrange of :630 is fused).
 * Training takes two calls so a data-parallel host can all-reduce the 17 floats in between:
 *   ralenet_stem_stats   : stats[0:8]=sum, [8:16]=sum of squares, [16]=count  (overwritten)
 *   ralenet_stem_apply   : normalise with the (all-reduced) stats, update running stats (momentum
 *                          0.1, unbiased variance) and num_batches_tracked.
 * Eval: ralenet_stem_apply with training == 0 uses the running statistics.
 * Backward mirrors it: ralenet_stem_bwd_stats (sums[0:8]=sum dyhat, [8:16]=sum dyhat*ahat, also
 * d_bn_w/d_bn_b), all-reduce, ralenet_stem_bwd_apply (conv weight/bias/input gradients).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, L, training, _pad;
  const float* x;              /* [B,2,L] channels-first input                                  */
  const float* conv_w; const float* conv_b; /* [8,2,3],[8]                                      */
  const float* bn_w; const float* bn_b;     /* [8]                                              */
  float* running_mean; float* running_var;  /* [8] (updated in training)                        */
  int64_t* num_batches_tracked;             /* scalar, may be NULL                              */
  float* stats;                /* [17]                                                          */
  float* partials;             /* scratch [B*16]                                                */
  float* y;                    /* [B,L,8]                                                       */
  float momentum, eps;
} rl_stem_args;

typedef struct {
  int32_t B, L, training, _pad;
  const float* g; const float* g2;          /* dL/dy [B,L,8] token-major, optional 2nd addend   */
  const float* x; const float* conv_w; const float* conv_b; const float* bn_w;
  const float* running_mean; const float* running_var;   /* eval-mode backward                  */
  const float* stats;          /* forward stats [17] (all-reduced)                              */
  float* sums;                 /* [16] backward sums                                            */
  float* partials;             /* scratch [B*16]                                                */
  float* dx;                   /* [B,2,L] or NULL                                               */
  float* d_conv_w; float* d_conv_b; float* d_bn_w; float* d_bn_b;
  float eps; float _padf;
} rl_stem_bwd_args;

int ralenet_stem_stats(const rl_stem_args* a, void* stream);
int ralenet_stem_apply(const rl_stem_args* a, void* stream);
int ralenet_stem_bwd_stats(const rl_stem_bwd_args* a, void* stream);
int ralenet_stem_bwd_apply(const rl_stem_bwd_args* a, void* stream);

/* ------------------------------------------------------------------------------------------
 * Head  transconv(x_1^T + stem_out) = Conv1d(8,2,3,p1)   (model/transformer.py:664-667)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, L;
  const float* x; const float* skip;        /* [B,L,8] token-major each                          */
  const float* w; const float* b;           /* [2,8,3],[2]                                       */
  float* out;                  /* [B,2,L] channels-first                                        */
} rl_head_fwd_args;

typedef struct {
  int32_t B, L;
  const float* dout;           /* [B,2,L]                                                       */
  const float* x; const float* skip; const float* w;
  float* ds;                   /* [B,L,8] gradient w.r.t. (x + skip)                            */
  float* d_w; float* d_b;
} rl_head_bwd_args;

int ralenet_head_fwd(const rl_head_fwd_args* a, void* stream);
int ralenet_head_bwd(const rl_head_bwd_args* a, void* stream);

/* ------------------------------------------------------------------------------------------
 * Loss + metrics: F.mse_loss (denoise_train.py:53) with its gradient, and the per-window
 * RMSE / SNR of local_utils/evaluate.py:27-29, 49-51, in one pass.
 *   loss[0] += sum((pred-target)^2) * inv_count        (caller zero-fills; inv_count = 1/numel
 *   dout     = 2*(pred-target)*inv_count * gscale        of the GLOBAL batch under data parallel)
 *   weight (optional [per]): R-wave-weighted variant, loss = mean(w*(pred-target)^2); w == NULL
 *   is exactly MSE (the reference has no weighted loss, SURVEY F4).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, per;              /* windows, elements per window (C*L)                            */
  const float* pred; const float* target; const float* weight;
  float* dout;                 /* [B,per] or NULL                                               */
  float* loss;                 /* [1] (+=)                                                      */
  float* rmse; float* snr;     /* [B] each or NULL                                              */
  float inv_count, gscale;
  float* partials;             /* [B] scratch or NULL: per-window loss sums are stored here and   */
                               /* added to loss[0] in window order (deterministic); NULL: atomics */
} rl_mse_args;
int ralenet_mse(const rl_mse_args* a, void* stream);

/* ------------------------------------------------------------------------------------------
 * newrale lead-mixing convs: Conv1d(k=13, pad=6) (+ LeakyReLU(0.01))   (model/ralenet_12leads.py:684-709)
 * channels-first [B,Cin,L] -> [B,Cout,L].  act: 0 = none, 1 = LeakyReLU(slope).
 * backward: dy is the gradient w.r.t. the activated output; pre-activation sign is recomputed.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, L, Cin, Cout, K, act;
  float slope; float _padf;
  const float* x; const float* w; const float* b;
  float* y;
} rl_conv_fwd_args;
typedef struct {
  int32_t B, L, Cin, Cout, K, act;
  float slope; float _padf;
  const float* dy; const float* x; const float* w; const float* b;
  float* dx;                   /* or NULL                                                       */
  float* d_w; float* d_b;      /* (+=) or NULL                                                  */
} rl_conv_bwd_args;
int ralenet_conv1d_fwd(const rl_conv_fwd_args* a, void* stream);
int ralenet_conv1d_bwd(const rl_conv_bwd_args* a, void* stream);
/* deterministic twin of ralenet_conv1d_bwd: same kernels and the same += semantics of d_w / d_b, but every window
 * stores its weight and bias gradients into its own slot of a partial slab in `slab` (caller-owned scratch of at least
 * ralenet_conv1d_slab_bytes bytes, any content), and a reduction kernel on the same stream adds the slots in window
 * order.  The result is bit-identical from run to run for a fixed build, shape and ralenet_set_conv_mma setting,
 * whatever the scheduling.  dx is a plain store in both functions and equal between them.  Like ralenet_conv1d_bwd,
 * d_b is only written when d_w is given.  RL_ERR_NULL for a NULL slab, RL_ERR_SHAPE for a short one.
 * ralenet_conv1d_slab_bytes = 4 * (B*Cout*Cin*K + B*Cout) floats, each of the two regions rounded up to 16 bytes
 * (0 for a non-positive size). */
uint64_t ralenet_conv1d_slab_bytes(int32_t B, int32_t Cin, int32_t Cout, int32_t K);
int ralenet_conv1d_bwd_det(const rl_conv_bwd_args* a, float* slab, uint64_t slab_bytes, void* stream);
/* k = 13 layers: 1 (default) = implicit-GEMM tensor-core kernels (conv_mma.cu), 0 = scalar FMA kernels (stem_head.cu).
 * Same function; A/B switch, initial value from RALENET_CONV_MMA.  Returns the previous setting. */
int ralenet_set_conv_mma(int on);

/* ------------------------------------------------------------------------------------------
 * Flat multi-tensor Adam: torch.optim.Adam(lr=1e-3) defaults (denoise_train.py:24, 57) over one
 * contiguous fp32 buffer.  g is multiplied by gscale first (1/world_size after a sum all-reduce).
 * ------------------------------------------------------------------------------------------ */
int ralenet_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                 float beta2, float eps, int32_t step, float gscale, void* stream);
/* same, but the 1-based step count lives in device memory and is incremented by the call itself
 * (so the whole train step can be replayed from a CUDA graph). */
int ralenet_adam_dev(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                     float beta2, float eps, int32_t* step_dev, float gscale, void* stream);

/* ------------------------------------------------------------------------------------------
 * Whole network (ralenet.forward, model/transformer.py:621-667; raletransformer.py:640-680):
 * one host call enqueues every kernel of the forward (resp. backward) on `stream`.
 * ------------------------------------------------------------------------------------------ */
enum { RL_BLK_WQ = 0, RL_BLK_BQ, RL_BLK_WKV, RL_BLK_BKV, RL_BLK_WP, RL_BLK_BP, RL_BLK_LN1W, RL_BLK_LN1B,
       RL_BLK_LN2W, RL_BLK_LN2B, RL_BLK_W1, RL_BLK_B1, RL_BLK_W2, RL_BLK_B2, RL_BLK_LEW, RL_BLK_NPTR };
#define RL_NBLOCKS 18

/* pointer table, used once for parameters and once for their gradients (NULL grads = frozen).
 * blocks are in forward order: dtransformer1.{0,1}, dtransformer2.*, dtransformer3.*,
 * dtransformer34.*, transformer.*, utransformer4.*, utranformer3.*, utransformer2.*, utransformer1.* */
typedef struct {
  float* stem[4];              /* conv1.0.weight, conv1.0.bias, conv1.2.weight, conv1.2.bias     */
  float* table[4];             /* rwattn1..4 tables, NULL for the no-R-wave variant              */
  float* blk[RL_NBLOCKS][RL_BLK_NPTR];
  float* pm[4][3];             /* pm1..4: reduction.weight, norm.weight, norm.bias               */
  float* ps[4][3];             /* ps1..4                                                         */
  float* head[2];              /* transconv.0.weight, bias                                       */
} rl_net_ptrs;

typedef struct {
  int32_t B, L0;               /* windows, samples per window (256; 512 for the nra variant)     */
  int32_t le_mode;             /* RL_LE_*                                                        */
  int32_t training;            /* BatchNorm batch statistics + running-stat update               */
  int32_t save;                /* keep activations for ralenet_net_bwd                           */
  int32_t flags;               /* RL_NET_* (0: default)                                          */
  const float* pe[5];          /* P[:L_s] per stage, [L_s, C_s]                                  */
  float* running_mean; float* running_var; int64_t* num_batches_tracked;
  float* bn_stats;             /* [64]: [0:17] forward stats, [32:48] backward sums              */
  void* ws; uint64_t ws_bytes; /* workspace of >= ralenet_net_workspace_bytes_ex(B, L0, save, flags) */
} rl_net_cfg;

/* RL_NET_DETERMINISTIC: the backward pass (ralenet_net_bwd / ralenet_net_bwd_stem) gives bit-identical parameter
 * gradients, BatchNorm sums and dx from run to run for a fixed build, batch shape and kernel-selection switches,
 * whatever the scheduling of CTAs and streams: every cross-CTA accumulation into a parameter gradient is a plain store
 * into its own slot of a partial slab in the workspace, and a reduction kernel adds the slots in slot order with one
 * read-modify-write per gradient element.  The forward pass is deterministic in either mode. */
/* RL_NET_TF32: inference precision of ralenet_net_fwd with save == 0 (RL_ERR_SHAPE with save != 0: no backward may
 * consume such a forward).  The q|k|v, output-projection, fc1 and fc2 GEMMs of every block run ONE tf32 tensor-core pass
 * on operands rounded to nearest (ties away) to a 10-bit mantissa, instead of the 3-pass split that keeps the default
 * fp32-grade.  The attention core (softmax logits), LayerNorm, GELU, positional encoding, R-wave bias, patch layers,
 * stem and head are computed exactly as in the default mode.  Precision contract: the output is held to the reduced-
 * precision gate |out - ref| <= 1e-2 * (|ref| + rms(ref)) against the fp64 reference, and per-window SNR / RMSE within
 * 0.01 dB of the default mode.  Deterministic (bit-identical from run to run) like the default forward; combining it
 * with RL_NET_DETERMINISTIC is legal (that bit has no effect on a forward without save).  The workspace size does not
 * depend on it. */
enum { RL_NET_DETERMINISTIC = 1, RL_NET_TF32 = 2 };

uint64_t ralenet_net_workspace_bytes(int32_t B, int32_t L0, int32_t save);      /* == _ex(B, L0, save, 0) */
/* the deterministic mode needs the partial slabs on top (a function of B and L0 only) */
uint64_t ralenet_net_workspace_bytes_ex(int32_t B, int32_t L0, int32_t save, int32_t flags);
/* forward: phase 1 (training only) computes BN partial stats into cfg->bn_stats[0:17];
 * the host may all-reduce them; phase 2 runs the rest.  Eval mode: call phase 2 only. */
int ralenet_net_fwd_stats(const rl_net_cfg* cfg, const rl_net_ptrs* P, const float* x, void* stream);
int ralenet_net_fwd(const rl_net_cfg* cfg, const rl_net_ptrs* P, const float* x, float* out, void* stream);
/* backward: phase 1 runs everything down to the BN backward sums (cfg->bn_stats[32:48]); the host
 * may all-reduce them; phase 2 finishes the stem (conv grads, dx). */
int ralenet_net_bwd(const rl_net_cfg* cfg, const rl_net_ptrs* P, const rl_net_ptrs* G,
                    const float* x, const float* dout, void* stream);
int ralenet_net_bwd_stem(const rl_net_cfg* cfg, const rl_net_ptrs* P, const rl_net_ptrs* G,
                         const float* x, float* dx, void* stream);

/* ------------------------------------------------------------------------------------------
 * Record <-> window pipeline for long recordings (inference).  The reference cuts records into 256-sample
 * windows on the host (local_utils/local_utils.py:47-65, 116-130) after per-lead z-normalisation (np_norm,
 * :261-266) and never stitches them back.  x, y: [R][C][T] channels-first records; win: [R*nper][C][W] with
 * nper = (T - W)/stride + 1 full windows per record; stats: [R*C][2] = (mean, 1/std) or NULL (no normalisation).
 * scatter averages overlapping windows (deterministic gather form), undoes the normalisation, and passes
 * samples not covered by a full window through from x.
 * ------------------------------------------------------------------------------------------ */
int ralenet_record_stats(const float* x, int32_t RC, int64_t T, float* stats, void* stream);
int32_t ralenet_windows_per_record(int64_t T, int32_t W, int32_t stride);
int ralenet_window_gather(const float* x, const float* stats, float* win, int32_t R, int32_t C, int64_t T,
                          int32_t W, int32_t stride, void* stream);
int ralenet_window_scatter(const float* win, const float* x, const float* stats, float* y, int32_t R, int32_t C,
                           int64_t T, int32_t W, int32_t stride, void* stream);

/* ------------------------------------------------------------------------------------------
 * Efficient channel attention on the feed-forward output (eca_layer_1d, model/transformer.py:100-113, used by
 * Mlp.forward :158 when use_eca=True):   s[b,c] = sigmoid( sum_k w[k] * mean_t x[b,t,c+k-(K-1)/2] )  (zero padded
 * over the channel axis),  y = x * s  (+ res: the block residual, fused).  x, y, res: [B,L,C]; w: [K] (K odd <= 15,
 * Conv1d(1,1,K,bias=False)); s: [B,C] saved for backward (may be NULL in forward-only use).  256 % C == 0.
 * backward: dx = g*s + dm/L with dm the adjoint of the channel convolution; d_w (+=) may be NULL;
 * the gradient w.r.t. res is g itself (caller's business).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, L, C, K;
  const float* x; const float* res; const float* w;
  float* y; float* s;
} rl_eca_fwd_args;
typedef struct {
  int32_t B, L, C, K;
  const float* g; const float* x; const float* w; const float* s;
  float* dx; float* d_w;
} rl_eca_bwd_args;
int ralenet_eca_fwd(const rl_eca_fwd_args* a, void* stream);
int ralenet_eca_bwd(const rl_eca_bwd_args* a, void* stream);

/* SNR-targeted noise mixing (single_snr_noise_add, local_utils/local_utils.py:176-192), one window per CTA:
 *   out[b] = data[b] + noise[b] * sqrt( mean(data[b]^2) / 10^(snr_db[b]/10) / mean(noise[b]^2) )
 * with the means over all `per` elements (leads x samples) of window b.  data, noise, out: [B][per]; snr_db: [B]. */
int ralenet_snr_mix(const float* data, const float* noise, const float* snr_db, float* out, int32_t B, int32_t per,
                    void* stream);

/* Device-side training-batch synthesiser (synth.cu; SURVEY.md section 8 f3): MIT-BIH-style windows generated on
 * the GPU -- beat trains of P-QRS-T Gaussians (R peak of the middle beat at L/2 +- 8), per-lead z-normalisation
 * (np_norm, local_utils/local_utils.py:261-266), and bw / ma / em style noise (kind 0 / 1 / 2, 3 = all three, the
 * reference's `emb`) with zero mean; mix with ralenet_snr_mix for the reference's SNR-targeted pairs
 * (local_utils.py:176-192).  clean, noise: [B][leads][L], L <= 1024.  The random stream is a pure function of
 * (seed, *counter_dev, window, lead, sample); counter_dev (device int32, e.g. the Adam step counter) may be NULL. */
int ralenet_synth_windows(float* clean, float* noise, int32_t B, int32_t leads, int32_t L, uint64_t seed,
                          const int32_t* counter_dev, int32_t kind, void* stream);

/* Device-side record sampler (records.cu; SURVEY.md section 8 f3 on real data): training windows cut from a bank of
 * clean records and paired with windows of a bank of noise records, one CTA per window; mix with ralenet_snr_mix.
 *   records [R][leads][T] (leads <= 12), stats [R*leads][2] from ralenet_record_stats or NULL (no z-normalisation),
 *   noise [N][noise_leads][Tn] (noise_leads = 1 or leads; clean lead l reads noise lead l % noise_leads),
 *   snr_levels [n_snr] dB.  Outputs clean_out / noise_out [B][leads][W] (clean_out z-normalised exactly like
 *   ralenet_window_gather), snr_out [B] dB, meta [B][4] = (record, offset, noise record, noise offset) or NULL.
 * The grid of a bank is item = record * nper + k, offset k * stride, nper = (T - W)/stride + 1, n = R * nper items;
 * spe = n / (world * B) steps per epoch (drop-last).  With c = *counter (0 when NULL), rank r, slot i takes item
 * perm_e((c % spe) * world * B + r * B + i) of epoch e = c / spe, perm_e a keyed bijection of [0, n) (4-round Feistel
 * network with cycle walking).  Noise record, noise offset (uniform in [0, Tn - W]) and SNR level are hashed from
 * (seed, c, r * B + i).  Every draw is a pure function of (seed, c, global slot), so the slices of `world` ranks
 * concatenate to the batch of world * B windows that one rank would draw.  meta needs T, Tn <= INT32_MAX. */
typedef struct {
  const float* records; const float* stats; const float* noise; const float* snr_levels;
  const int32_t* counter;
  float* clean_out; float* noise_out; float* snr_out;
  int32_t* meta;
  int64_t T, Tn;
  uint64_t seed;
  int32_t R, leads, N, noise_leads, n_snr, W, stride, B, rank, world;
} rl_sample_args;
int ralenet_record_sample(const rl_sample_args* a, void* stream);

/* Ordered evaluation draw over held-out banks (records.cu), the device side of the per-epoch test loop
 * (denoise_train.py:66-81 over the test loader; the reference's test sets are one noisy copy per intensity,
 * dict_data/{m4,m2,0,p2,p4}).  Same banks, statistics, outputs and layouts as rl_sample_args; one CTA per slot.
 * The evaluation set is every grid window at every level: item e = g * n_snr + lvl, g = record * nper + k the grid
 * window in record-major order (the order of ralenet_window_gather), n_eval = R * nper * n_snr items.  With
 * c = *counter (0 when NULL), slot i of rank r takes e = c * world * B + r * B + i: no shuffle, no drop-last, and the
 * ranks together cover the set exactly once.  Noise record and noise offset are hashed from (seed, g, lvl) alone, so
 * every run, epoch and rank split sees the same noisy test set.  A slot with e >= n_eval writes zeroed clean and noise
 * windows, snr_out = 0, meta = (-1, -1, -1, -1) and level = -1.  level [B]: level index of the slot (valid = level >= 0).
 * Mix with ralenet_snr_mix.  Offsets must fit int32 (T, Tn <= INT32_MAX), like meta. */
typedef struct {
  const float* records; const float* stats; const float* noise; const float* snr_levels;
  const int32_t* counter;
  float* clean_out; float* noise_out; float* snr_out;
  int32_t* meta; int32_t* level;
  int64_t T, Tn;
  uint64_t seed;
  int32_t R, leads, N, noise_leads, n_snr, W, stride, B, rank, world;
} rl_enum_args;
int ralenet_record_enumerate(const rl_enum_args* a, void* stream);

/* Evaluation metrics of one batch (local_utils/evaluate.py:27-29, 49-51 per window, summed per level as
 * denoise_train.py:100-101 reports them).  For window b with level[b] >= 0, over all `per` elements (leads x samples),
 * in fp64:  snr_out = 10 log10(sum y^2 / sum (y - pred)^2),  snr_in = the same with noisy in place of pred,
 * rmse = sqrt(mean((y - pred)^2)), y = clean.  Optional per-window outputs snr_in / snr_out / rmse [B] (float; 0 for
 * windows with level < 0).  acc [n_snr][4] += (count, sum snr_in, sum snr_out, sum rmse) per level: the windows'
 * values go through partials [B][4] (fp64 scratch) and one CTA adds them in a fixed order, so the whole evaluation
 * is bit-reproducible (no floating-point atomics).  Windows with level < 0 or >= n_snr add nothing.  counter (device
 * int32, may be NULL) is incremented after the sums, so a captured draw + forward + metrics step advances by itself
 * (as ralenet_adam_dev does with the step count). */
typedef struct {
  const float* clean; const float* noisy; const float* pred;   /* [B][per] each                            */
  const int32_t* level;                                        /* [B]                                      */
  float* snr_in; float* snr_out; float* rmse;                  /* [B] each or NULL                         */
  double* partials;                                            /* [B][4] scratch                           */
  double* acc;                                                 /* [n_snr][4] (+=)                          */
  int32_t* counter;                                            /* or NULL                                  */
  int32_t B, per, n_snr, _pad;
} rl_eval_args;
int ralenet_eval_metrics(const rl_eval_args* a, void* stream);

/* Weight-gradient GEMM over the token dimension (used by every *_bwd above; exported for benchmarks):
 *   dW[n*K + k] += sum_m dY[m*ldy + n] * X[m*ldx + k],   db[n] += sum_m dY[m*ldy + n]   (db may be NULL) */
int ralenet_wgrad(const float* dY, int32_t ldy, const float* X, int32_t ldx, int32_t M, int32_t N, int32_t K,
                  float* dW, float* db, void* stream);

/* ------------------------------------------------------------------------------------------
 * Data-parallel exchange steps over NVLink / NVSwitch peer memory (comm.cu).  Net-new: the reference is
 * single-GPU (main.py:1-3); the contract is "N ranks on a sharded batch == one process on the global batch"
 * (SURVEY.md section 8e): BatchNorm statistics of the stem (model/transformer.py:570-574) summed over the ranks in
 * forward and backward, and ONE sum of the flat gradient buffer fused in front of Adam (denoise_train.py:57).
 * Every rank owns one symmetric buffer of ralenet_comm_bytes(n) bytes, allocated and peer-mapped by the HOST
 * (e.g. torch.distributed._symmetric_memory; the library never allocates): its first n floats are the flat gradient
 * buffer the backward kernels accumulate into, the rest (exchange slots, barrier flags) must start zeroed.
 * peer[i] = address of rank i's buffer in THIS process (peer[rank] = the local buffer), mc = multicast (NVLS) mapping
 * of the same buffers or NULL, epoch = 2 + RL_COMM_MAXG zero-initialised uint32 counters in local device memory.
 * All ranks must issue the same sequence of comm calls.  Pure kernel launches: capturable in CUDA graphs.
 * ------------------------------------------------------------------------------------------ */
#define RL_COMM_MAXW 8
#define RL_COMM_MAXG 128
typedef struct {
  int32_t world, rank;
  void* peer[RL_COMM_MAXW];
  void* mc;
  uint64_t n;                  /* floats of the gradient region (multiple of 4)                  */
  uint32_t* epoch;
} rl_comm;
uint64_t ralenet_comm_bytes(uint64_t n);
/* vals[0:n] (local device memory, n <= 32) <- sum over the ranks, added in rank order (bit-identical on every rank).
 * set 0 / 1 = two independent slot sets (forward statistics / backward sums). */
int ralenet_comm_exchange(const rl_comm* c, int32_t set, float* vals, int32_t n, void* stream);
/* gradient all-reduce (sum) fused with flat Adam: reduce-scatter + broadcast through multimem.ld_reduce / multimem.st
 * (peer loads / stores when mc == NULL), then p, m, v updated from the local copy of the sum * gscale; *step_dev is
 * incremented first (as ralenet_adam_dev).  grid = CTAs (<= RL_COMM_MAXG, the same on every rank; 0 = default). */
int ralenet_comm_allreduce_adam(const rl_comm* c, float* p, float* m, float* v, float lr, float beta1, float beta2,
                                float eps, int32_t* step_dev, float gscale, int32_t grid, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stand-alone forwards of helper modules that ralenet.forward fuses away (small_ops.cu; NOT on the hot path):
 *   ralenet_linear_fwd       y[M,N] = x[M,K] w[N,K]^T (+ b[N])     nn.Linear inside LinearProjection.forward
 *                            (model/transformer.py:226-247: to_q, to_kv) called on its own
 *   ralenet_linear_bwd_data  dx[M,K] = dy[M,N] w[N,K]              (weight gradient: ralenet_wgrad)
 *   ralenet_pe_add           y = x + P[:L]  broadcast over the batch, per = L*C   AbsPositionalEncoding.forward (:179-181)
 *   ralenet_pconv1           PartialConv_1d.forward_split_cat (:54-59) with one convolved channel: channels-first
 *                            [B,C,L], channel 0 <- Conv1d(1,1,3,pad 1,no bias), channels 1.. copied; transpose = 1
 *                            gives the data gradient;  ralenet_pconv1_wgrad: dw[3] += the weight gradient
 * ------------------------------------------------------------------------------------------ */
int ralenet_linear_fwd(const float* x, const float* w, const float* b, float* y, int32_t M, int32_t K, int32_t N,
                       void* stream);
int ralenet_linear_bwd_data(const float* dy, const float* w, float* dx, int32_t M, int32_t K, int32_t N, void* stream);
int ralenet_pe_add(const float* x, const float* pe, float* y, int32_t B, int32_t per, void* stream);
int ralenet_pconv1(const float* x, const float* w, float* y, int32_t B, int32_t C, int32_t L, int32_t transpose,
                   void* stream);
int ralenet_pconv1_wgrad(const float* dy, const float* x, float* dw, int32_t B, int32_t C, int32_t L, void* stream);

/* Per-launch timing for bench.py's roofline pass: after ralenet_profile_begin(stream) every kernel this
 * library launches is followed by a CUDA event on `stream`; ralenet_profile_end() waits for the last one and
 * returns the number of launches, their labels ("kernel<C>", label_stride bytes each) and durations in ms.
 * Not thread-safe; do not use while capturing a CUDA graph. */
int ralenet_profile_begin(void* stream);
int ralenet_profile_end(char* labels, int32_t label_stride, float* ms, int32_t max_n);

/* number of kernels launched by this library on the calling thread since the last reset
 * (bench.py's gpu_launches). */
int64_t ralenet_launch_count(int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* RALENET_B200_H */
