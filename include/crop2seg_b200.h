/*
 * crop2seg_b200 -- C ABI of the B200-native L-TAE + TemporalAggregator hot path.
 *
 * Drop-in boundary for the temporal-attention bottleneck of Many98/Crop2Seg.  The
 * reference has no native layer: its interface for this path is the Python
 * nn.Module API (SURVEY.md section 8b).  Each entry point below names the reference
 * call it replaces (paths relative to the reference checkout).  The Python modules
 * in crop2seg_b200/ bind these symbols with ctypes and keep the reference's
 * constructor / forward / state_dict contract; see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - tensors are dense, row-major ("contiguous") in the shapes given;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every function returns 0 on success, a C2S_ERR_* code otherwise, never aborts;
 *     c2s_last_error() returns a thread-local, human readable message;
 *   - nothing here synchronises the host with the device.
 */
#ifndef CROP2SEG_B200_H_
#define CROP2SEG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C2S_ABI_VERSION 12

enum c2s_status {
  C2S_OK = 0,
  C2S_ERR_BAD_ARGUMENT = 1,  /* NULL pointer, non-positive size, inconsistent descriptor      */
  C2S_ERR_UNSUPPORTED = 2,   /* valid but not implemented by the kernels (message says which) */
  C2S_ERR_CUDA = 3,          /* a CUDA runtime call or kernel launch failed                   */
  C2S_ERR_NO_DEVICE = 4      /* no sm_100 device / wrong architecture                         */
};

enum c2s_dtype { C2S_F32 = 0, C2S_BF16 = 1 };

/* TemporalAggregator(mode) -- temporal_aggregator.py:10 */
enum c2s_agg_mode { C2S_AGG_ATT_GROUP = 0, C2S_AGG_ATT_MEAN = 1, C2S_AGG_MEAN = 2 };

/* positional encoder variant chosen by LTAE.__init__ -- tae.py:406-426 */
enum c2s_pe_mode {
  C2S_PE_NONE = 0,            /* positional_encoding=False                              */
  C2S_PE_SINUSOID = 1,        /* PositionalEncoder                positional_encoding.py:7  */
  C2S_PE_SINUSOID_LINEAR = 2, /* PositionalEncoder(add_linear)    positional_encoding.py:39 */
  C2S_PE_DOY_TABLE = 3        /* AbsolutePositionalEncoder        positional_encoding.py:46 */
};

enum c2s_ltae_flags {
  C2S_LTAE_ATTN_ONLY = 1 << 0,       /* LTAE4WTAE: return the attention masks only (tae.py:589-635) */
  C2S_LTAE_SKIP_ATTN_STORE = 1 << 1, /* caller does not consume attn (model-level return_att=False)  */
  C2S_LTAE_ZERO_PADDED = 1 << 2,     /* caller guarantees x == 0 on padded frames (temp_shared_block.py:30-40):
                                        padded frames are then never read                             */
  C2S_LTAE_BN_BATCH_STATS = 1 << 3,  /* training: BatchNorm1d uses batch statistics (tae.py:445)     */
  C2S_LTAE_REUSE_FOLDED = 1 << 4     /* the workspace is the one of the previous call with the same descriptor and
                                        UNCHANGED parameters: the weight-only preparation (folded score / projection
                                        weights, fragment orders) is not rebuilt; positions and masks still are */
};

/* ------------------------------------------------------------------------------------------
 * TemporalAggregator.forward(x, pad_mask, attn_mask)          temporal_aggregator.py:14-77
 * ---------------------------------------------------------------------------------------- */
typedef struct c2s_agg_desc {
  int32_t B, T, C, H, W; /* x[B,T,C,H,W]                                                      */
  int32_t n_heads;       /* attn[n_heads,B,T,ha,wa]  (ignored for C2S_AGG_MEAN)               */
  int32_t ha, wa;        /* attention resolution                                              */
  int32_t mode;          /* enum c2s_agg_mode                                                 */
  int32_t dtype;         /* enum c2s_dtype of x and out; attn is always float32               */
} c2s_agg_desc;

/* Scratch bytes c2s_agg_forward can use for this descriptor: the reduced attention map of att_mean / the AvgPool2d
 * branch (required there) followed by B int32 for the sample order of the pipelined kernel (longest series first;
 * optional: with a smaller or NULL workspace the samples are walked in index order, same results). */
size_t c2s_agg_workspace_bytes(const c2s_agg_desc* desc);

/* out[B,C,H,W] = sum_t resize(attn)[c // (C/n_heads), b, t] * (pad ? 0 : 1) * x[b,t,c]
 * pad_mask: uint8 [B,T] (non-zero = padded frame) or NULL.  Padded frames of x are not read. */
int c2s_agg_forward(const c2s_agg_desc* desc, const void* x, const float* attn,
                    const uint8_t* pad_mask, void* out, void* workspace, size_t workspace_bytes,
                    void* stream);

/* TemporalAggregator(att_group) fused with the decoder's skip convolution (SURVEY.md section 8f, rank 1):
 *   out[B,C,H,W] = relu( BatchNorm2d_eval( Conv2d_1x1( aggregate(x, attn, pad) ) ) )
 * = UpConvBlock.skip_conv (conv.py:378-382, applied at conv.py:408) on the skip map of utae.py:225-229, without the
 * skip map being written to and re-read from HBM.  Running statistics (c2s_agg_skipconv_backward below).  Serves what
 * the shipped models use: att_group, bfloat16, C = 64, 16 heads, x2/x4/x8 up-sampling, H*W % 128 == 0; anything else returns
 * C2S_ERR_UNSUPPORTED (run c2s_agg_forward and the convolution separately). */
typedef struct c2s_skipconv_params {
  const float* conv_weight;      /* skip_conv.0.weight [C,C,1,1]                               */
  const float* conv_bias;        /* skip_conv.0.bias   [C] or NULL                             */
  const float* bn_weight;        /* skip_conv.1.weight [C] or NULL (affine=False)              */
  const float* bn_bias;          /* skip_conv.1.bias   [C] or NULL                             */
  const float* bn_running_mean;  /* skip_conv.1.running_mean [C]                               */
  const float* bn_running_var;   /* skip_conv.1.running_var  [C]                               */
  float bn_eps;                  /* 1e-5 (nn.BatchNorm2d default)                              */
} c2s_skipconv_params;
size_t c2s_agg_skipconv_workspace_bytes(const c2s_agg_desc* desc);
int c2s_agg_skipconv_forward(const c2s_agg_desc* desc, const void* x, const float* attn, const uint8_t* pad_mask,
                             const c2s_skipconv_params* params, void* out, void* workspace, size_t workspace_bytes,
                             void* stream);

/* Backward of c2s_agg_skipconv_forward with the BatchNorm frozen (eval mode: running statistics), i.e. what autograd
 * derives from relu(BatchNorm2d_eval(Conv2d_1x1(aggregate(x, attn, pad)))) with the skip map rounded to bf16 as the
 * forward rounds it.  `out` is the forward's output (its ReLU decision), grad_out [B,C,H,W] bf16.  x is read once; the
 * skip map is recomputed on chip and never written.  Same shapes as the forward; anything else returns
 * C2S_ERR_BAD_ARGUMENT.  Every output pointer may be NULL (that gradient is skipped). */
typedef struct c2s_skipconv_bwd_io {
  void* grad_x;             /* out [B,T,C,H,W] bf16, exactly 0 on padded frames                                         */
  float* grad_attn;         /* acc [16,B,T,ha,wa], ZERO-FILLED by the caller; float atomics as in c2s_agg_backward      */
  float* grad_conv_weight;  /* out [C,C] (skip_conv.0.weight)        deterministic: fixed-order reduction, no atomics   */
  float* grad_conv_bias;    /* out [C]   (skip_conv.0.bias)                                                              */
  float* grad_bn_weight;    /* out [C]   (skip_conv.1.weight)                                                            */
  float* grad_bn_bias;      /* out [C]   (skip_conv.1.bias)                                                              */
} c2s_skipconv_bwd_io;
/* Scratch bytes: prepared weights plus one partial of the parameter gradients per (sample, 128-pixel block). */
size_t c2s_agg_skipconv_backward_workspace_bytes(const c2s_agg_desc* desc);
int c2s_agg_skipconv_backward(const c2s_agg_desc* desc, const void* x, const float* attn, const uint8_t* pad_mask,
                              const c2s_skipconv_params* params, const void* out, const void* grad_out,
                              const c2s_skipconv_bwd_io* io, void* workspace, size_t workspace_bytes, void* stream);

/* The same block with its BatchNorm normalising by batch statistics (training mode, or track_running_stats=False):
 *   z = Conv2d_1x1(aggregate(x, attn, pad))  (bf16, [B,C,H,W]),  out = relu( BatchNorm2d_train(z) )
 * over N = B*H*W pixels per channel (an all-padded sample counts: its skip map is 0, its z the conv bias).  z crosses HBM
 * once; the statistics are merged from per-tile (mean, M2) partials in a fixed order (bit-identical from run to run).
 * bn_batch_mean/var: float32 [C] (biased variance); the caller updates the running statistics (as c2s_ltae_forward).
 * params->bn_running_mean/var are ignored and may be NULL.  out may be z (when z is not needed afterwards).  Same shapes
 * as c2s_agg_skipconv_forward; anything else returns C2S_ERR_UNSUPPORTED. */
size_t c2s_agg_skipconv_bstats_workspace_bytes(const c2s_agg_desc* desc);
int c2s_agg_skipconv_bstats_forward(const c2s_agg_desc* desc, const void* x, const float* attn, const uint8_t* pad_mask,
                                    const c2s_skipconv_params* params, void* z, void* out, float* bn_batch_mean,
                                    float* bn_batch_var, void* workspace, size_t workspace_bytes, void* stream);
/* Backward of c2s_agg_skipconv_bstats_forward from its z, batch statistics and out (distinct from z).  io as in
 * c2s_agg_skipconv_backward; grad_conv_bias is written as zeros (batch statistics cancel a per-channel constant of z).
 * grad_bn_weight / grad_bn_bias / grad_conv_weight are deterministic.  Unsupported shapes return C2S_ERR_BAD_ARGUMENT. */
size_t c2s_agg_skipconv_bstats_backward_workspace_bytes(const c2s_agg_desc* desc);
int c2s_agg_skipconv_bstats_backward(const c2s_agg_desc* desc, const void* x, const float* attn, const uint8_t* pad_mask,
                                     const c2s_skipconv_params* params, const void* z, const float* bn_batch_mean,
                                     const float* bn_batch_var, const void* out, const void* grad_out,
                                     const c2s_skipconv_bwd_io* io, void* workspace, size_t workspace_bytes, void* stream);

/* Backward of TemporalAggregator.forward (what autograd derives from temporal_aggregator.py:14-77):
 *   grad_x[b,t,c]        = resize(attn)[c // (C/n_heads), b, t] * (pad ? 0 : 1) * grad_out[b,c]      (x's dtype)
 *   grad_attn[h,b,t,:,:] = resize^T( sum_{c in head h} x[b,t,c] * grad_out[b,c] )                  (float32)
 * grad_x / grad_attn may be NULL when not needed; grad_attn must be ZERO-FILLED by the caller (it is
 * accumulated with float atomics, so its low bits depend on the execution order -- the reference's own
 * backward is non-deterministic too, train.py:623-626).  x is only read when grad_attn is requested.
 * The AvgPool2d branch (attention not coarser than x, temporal_aggregator.py:28-29) pools the attention into the
 * workspace, differentiates against the pooled maps and spreads their gradient over the k x k windows. */
size_t c2s_agg_backward_workspace_bytes(const c2s_agg_desc* desc);
int c2s_agg_backward(const c2s_agg_desc* desc, const void* x, const float* attn, const uint8_t* pad_mask,
                     const void* grad_out, void* grad_x, float* grad_attn, void* workspace,
                     size_t workspace_bytes, void* stream);

/* pad_mask[b,t] = (input[b,t,:,:,:] == pad_value).all()   utae.py:201-203, wtae.py:221-223, timeunet.py:170-172
 * (SURVEY.md section 8a row a9).  x: n_frames contiguous frames of frame_elems elements; mask: uint8 [n_frames],
 * 1 = padded.  A frame is left at the first value that differs, so only padded frames are read to the end. */
int c2s_pad_mask(const void* x, int32_t dtype, int64_t n_frames, int64_t frame_elems, float pad_value,
                 uint8_t* mask, void* stream);

/* Lengths-aware frame packing for blocks shared across the sequence -- TemporallySharedBlock.smart_forward,
 * temp_shared_block.py:18-47 (SURVEY.md section 8f rank 2): `out[~pad_mask]` / `temp[~pad_mask] = ...` without the
 * nonzero() host synchronisation of boolean indexing.
 *   c2s_frame_index   : slot[f] = number of valid frames before f (pad_mask[f] == 0), -1 for padded frames;
 *                       *n_valid = number of valid frames (device scalar).  pad_mask: uint8 [n_frames].
 *   c2s_frames_gather : packed[slot[f]] = frames[f] for every valid frame; frames: [n_frames][frame_elems],
 *                       packed: [>= n_valid][frame_elems].  Padded frames are not read.
 *   c2s_frames_scatter: out[f] = slot[f] >= 0 ? packed[slot[f]] : pad_value; out: [n_frames][frame_elems].
 * dtype: enum c2s_dtype of frames / packed / out.  At most 65535 frames per gather / scatter call. */
int c2s_frame_index(const uint8_t* pad_mask, int64_t n_frames, int32_t* slot, int32_t* n_valid, void* stream);
int c2s_frames_gather(const void* frames, const int32_t* slot, void* packed, int64_t n_frames, int64_t frame_elems,
                      int32_t dtype, void* stream);
int c2s_frames_scatter(const void* packed, const int32_t* slot, void* out, int64_t n_frames, int64_t frame_elems,
                       int32_t dtype, float pad_value, void* stream);

/* ------------------------------------------------------------------------------------------
 * LTAE / LTAE4WTAE                                             tae.py:349-635
 * ---------------------------------------------------------------------------------------- */
typedef struct c2s_ltae_desc {
  int32_t B, T, C, H, W; /* x[B,T,C,H,W], C = in_channels                                     */
  int32_t n_head;        /* tae.py:358                                                        */
  int32_t d_k;           /* tae.py:359                                                        */
  int32_t d_model;       /* width after inconv; == C when has_inconv == 0 (tae.py:398-403)    */
  int32_t c_out;         /* mlp[-1]; ignored with C2S_LTAE_ATTN_ONLY                          */
  int32_t has_inconv;    /* d_model is not None                                               */
  int32_t pe_mode;       /* enum c2s_pe_mode                                                  */
  int32_t pe_abs;        /* use_abs_rel_enc: add AbsolutePositionalEncoder(positions[...,1])  */
  int32_t pos_dtype;     /* 0: int64 positions, 1: float32 positions                          */
  int32_t dtype;         /* enum c2s_dtype of x and out; attn is always float32               */
  int32_t flags;         /* enum c2s_ltae_flags                                               */
  float gn_eps;          /* 1e-5 (nn.GroupNorm default)                                       */
  float bn_eps;          /* 1e-5 (nn.BatchNorm1d default)                                     */
  float attn_keep_scale; /* 1/(1-p) of ScaledDotProductAttention.dropout (tae.py:819), used with attn_keep */
  float mlp_keep_scale;  /* 1/(1-p) of the MLP dropout (tae.py:448), used with mlp_keep        */
} c2s_ltae_desc;

/* state_dict tensors, float32, reference shapes (SURVEY.md section 8b). NULL where absent. */
typedef struct c2s_ltae_params {
  const float* in_norm_weight;   /* [C]                                                        */
  const float* in_norm_bias;     /* [C]                                                        */
  const float* inconv_weight;    /* [d_model, C]  (Conv1d weight [d_model,C,1])                */
  const float* inconv_bias;      /* [d_model]                                                  */
  const float* query;            /* attention_head.Q [n_head, 1, d_k]                          */
  const float* key_weight;       /* attention_head.fc1_k.weight [n_head*d_k, d_model]          */
  const float* key_bias;         /* attention_head.fc1_k.bias   [n_head*d_k]                   */
  const float* mlp_weight;       /* mlp.0.weight [c_out, d_model]                              */
  const float* mlp_bias;         /* mlp.0.bias   [c_out]                                       */
  const float* bn_weight;        /* mlp.2.weight [c_out]                                       */
  const float* bn_bias;          /* mlp.2.bias   [c_out]                                       */
  const float* bn_running_mean;  /* mlp.2.running_mean [c_out]                                 */
  const float* bn_running_var;   /* mlp.2.running_var  [c_out]                                 */
  const float* out_norm_weight;  /* [c_out]                                                    */
  const float* out_norm_bias;    /* [c_out]                                                    */
  const float* pe_denom;         /* PositionalEncoder.denom [d_model/n_head] (plain attribute) */
  const float* pe_fc_weight;     /* positional_encoder.fc.weight: [d_model,d_model] (add_linear)
                                    or [d_model/n_head, 365] (C2S_PE_DOY_TABLE)                */
  const float* pe_fc_bias;
  const float* pe_abs_fc_weight; /* positional_encoder_abs.fc.weight [d_model/n_head, 365]     */
  const float* pe_abs_fc_bias;
  /* training-mode dropout, drawn by the caller (torch's Philox stream cannot be reproduced in a kernel):
   * uint8 keep masks, NULL = no dropout.  The attention is masked BEFORE it is returned (tae.py:836-837). */
  const uint8_t* attn_keep;      /* [n_head, B, T, H, W]                                        */
  const uint8_t* mlp_keep;       /* [B, c_out, H, W], applied after the ReLU (tae.py:447-448)   */
  /* training: if not NULL, c2s_ltae_forward also writes the rows o[B*H*W][d_model] that enter the MLP
   * (tae.py:479-486, the concatenated heads); c2s_ltae_backward's caller needs them for the MLP gradients */
  float* save_o;
  /* training (C2S_LTAE_BN_BATCH_STATS): if not NULL, the pre-BatchNorm MLP rows y[B*H*W][c_out] are written here instead
   * of into the workspace, so that c2s_ltae_mlp_backward (c2s_ltae_mlp_bwd_io.y_rows) need not recompute them */
  float* save_y;
} c2s_ltae_params;

/* Scratch bytes for c2s_ltae_forward (folded weights + per-sample positional tables). */
size_t c2s_ltae_workspace_bytes(const c2s_ltae_desc* desc);

/* LTAE.forward(x, batch_positions, pad_mask) -> (out, attn)            tae.py:451-504
 * LTAE4WTAE.forward(...) -> attn   (flags & C2S_LTAE_ATTN_ONLY)         tae.py:589-635
 *   positions : int64 or float32 [B,T] ([B,T,2] when pe_abs), NULL iff pe_mode == NONE
 *   pad_mask  : uint8 [B,T] or NULL
 *   out       : [B,c_out,H,W] in desc->dtype (NULL with ATTN_ONLY)
 *   attn      : float32 [n_head,B,T,H,W] (may be NULL with SKIP_ATTN_STORE)
 *   bn_batch_mean/var : float32 [c_out], written only with BN_BATCH_STATS (biased variance);
 *                       the caller updates the running statistics (tae.py:445 semantics)
 * Day-of-year positions outside [0,364] make the call fail with C2S_ERR_BAD_ARGUMENT only
 * when they can be checked on the host; on the device they are clamped -- the Python
 * wrapper validates the range like F.one_hot does (positional_encoding.py:63). */
int c2s_ltae_forward(const c2s_ltae_desc* desc, const c2s_ltae_params* params, const void* x,
                     const void* positions, const uint8_t* pad_mask, void* out, float* attn,
                     float* bn_batch_mean, float* bn_batch_var, void* workspace,
                     size_t workspace_bytes, void* stream);

/* Encoders with several learned queries (num_queries = n > 1, eval mode)                    tae.py:486-499
 * The attention head returns n rows per pixel; mlp.0 / BatchNorm1d (running statistics) / ReLU act row by row, but
 * out_norm is applied to the transposed tensor [B*H*W, c_out, n] (tae.py:488): the statistics of a group run over its
 * channels AND the n queries.  The caller runs c2s_ltae_forward once per query (params->query = the rows of that
 * query, params->save_o = its rows o) and hands the stacked rows over:
 *   o_rows : float32 [n_queries][B*H*W][d_model]
 *   out    : [B][n_queries][c_out][H][W] in desc->dtype
 * desc: B, H, W, d_model, c_out, n_head, dtype, gn_eps, bn_eps are read. */
int c2s_ltae_rows_forward(const c2s_ltae_desc* desc, const c2s_ltae_params* params, const float* o_rows,
                          int32_t n_queries, void* out, void* stream);

/* Backward of LTAE.forward / LTAE4WTAE.forward through everything that touches the [B*H*W, T, C] features
 * (autograd of tae.py:451-504 in the reference).  The rows after the attention (MLP, BatchNorm, ReLU, output
 * GroupNorm on [B*H*W, d_model] / [B*H*W, c_out]) are differentiated by the caller, who passes grad_o; the kernel
 * returns grad_x and the gradients of the FOLDED quantities of c2s_ltae_prep.cuh, from which the caller derives the
 * state_dict gradients on [16, C] / [B, T, 16] sized tensors:
 *     U[c][h]      = gamma_c sum_d qk[h][d] Wc[d][c]           (score weights; qk = q_h^T Wk_h / sqrt(d_k))
 *     cpos[b][t][h] = qk[h] . (bc + Wc beta + PE[b][t]) + q_h . bk_h / sqrt(d_k)
 * Buffers marked acc are accumulated with float atomics and must be zeroed by the caller. */
typedef struct c2s_ltae_bwd_io {
  const float* grad_o;    /* in  [B*H*W][d_model] d loss / d o (NULL with C2S_LTAE_ATTN_ONLY)              */
  const float* grad_attn; /* in  [n_head][B][T][H][W] d loss / d attn (as returned, after dropout) or NULL */
  void* grad_x;           /* out [B][T][C][H][W] in desc->dtype                                            */
  float* grad_u;          /* acc [C][16]                                                                   */
  float* grad_cpos;       /* acc [B][T][16]                                                                */
  float* grad_gamma;      /* acc [C]  direct term of in_norm.weight (zn = gamma zr + beta sa)              */
  float* grad_beta;       /* acc [C]  direct term of in_norm.bias                                          */
  float* zn_rows;         /* out [B*H*W][n_head][C]: grad_Wc[d][c] (direct) = sum_n grad_o[n][d] zn[n][h(d)][c] */
  float* sa_rows;         /* out [B*H*W][16]:        grad_bc[d]   (direct) = sum_n grad_o[n][d] sa[n][h(d)]   */
  float* grad_pe;         /* acc [B][T][d_model] direct term of the positional table, or NULL              */
} c2s_ltae_bwd_io;

/* Backward of the rows behind the attention: mlp.0 (Linear), mlp.2 (BatchNorm1d, batch statistics with
 * C2S_LTAE_BN_BATCH_STATS, running statistics otherwise), ReLU, dropout mask (params->mlp_keep), out_norm
 * (autograd through tae.py:442-449, 486-488).  Produces grad_o for c2s_ltae_backward.  acc buffers must be zeroed. */
typedef struct c2s_ltae_mlp_bwd_io {
  const float* o_rows;          /* in  [B*H*W][d_model] rows saved by c2s_ltae_forward (params->save_o)   */
  const float* y_rows;          /* in  [B*H*W][c_out] y = o Wm^T + bm saved by c2s_ltae_forward (params->save_y), or
                                       NULL: recomputed from o_rows                                        */
  const void* grad_out;         /* in  [B][c_out][H][W] in desc->dtype                                     */
  const float* bn_mean;         /* in  [c_out] batch mean of the forward (training) or running_mean        */
  const float* bn_var;          /* in  [c_out] biased batch variance (training) or running_var             */
  float* grad_o;                /* out [B*H*W][d_model]                                                    */
  float* grad_mlp_weight;       /* acc [c_out][d_model]                                                    */
  float* grad_mlp_bias;         /* acc [c_out]                                                             */
  float* grad_bn_weight;        /* acc [c_out]                                                             */
  float* grad_bn_bias;          /* acc [c_out]                                                             */
  float* grad_out_norm_weight;  /* acc [c_out]                                                             */
  float* grad_out_norm_bias;    /* acc [c_out]                                                             */
} c2s_ltae_mlp_bwd_io;

size_t c2s_ltae_mlp_backward_workspace_bytes(const c2s_ltae_desc* desc);
int c2s_ltae_mlp_backward(const c2s_ltae_desc* desc, const c2s_ltae_params* params, const c2s_ltae_mlp_bwd_io* io,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Direct term of the in-projection gradient from the two stages above (what autograd derives from tae.py:478-480):
 *   grad_inconv_weight[h*dh+i][c] += sum_rows grad_o[row][h*dh+i] * zn_rows[row][h][c]      (acc [d_model][C])
 *   grad_inconv_bias[h*dh+i]      += sum_rows grad_o[row][h*dh+i] * sa_rows[row][h]         (acc [d_model] or NULL)
 * grad_o from c2s_ltae_mlp_backward, zn_rows / sa_rows from c2s_ltae_backward. */
int c2s_ltae_inconv_grad(const float* grad_o, const float* zn_rows, const float* sa_rows, float* grad_inconv_weight,
                         float* grad_inconv_bias, int64_t n_rows, int32_t n_head, int32_t d_model, int32_t C, void* stream);

/* Adjoint of the weight folding: grad_u / grad_cpos (and the direct in_norm terms) of c2s_ltae_backward -> gradients of
 * in_norm, inconv, attention_head.Q and attention_head.fc1_k (what autograd derives from tae.py:463-479, 760-778).  Must be
 * called with the SAME desc, params and workspace right after c2s_ltae_backward (its folded tensors and positional table
 * are read from the workspace).  Output pointers may be NULL.  grad_inconv_weight / bias receive the folded part only:
 * c2s_ltae_inconv_grad adds the direct term.  grad_pe (acc [B][T][d_model], may be NULL) receives += grad_cpos . qk, the
 * path of a learnable positional table through the scores.  Deterministic (no atomics). */
typedef struct c2s_ltae_fold_bwd_io {
  const float* grad_u;            /* in  [C][16]      from c2s_ltae_backward                      */
  const float* grad_cpos;         /* in  [B][T][16]                                               */
  const float* grad_gamma_direct; /* in  [C] or NULL  (c2s_ltae_bwd_io.grad_gamma)                */
  const float* grad_beta_direct;  /* in  [C] or NULL  (c2s_ltae_bwd_io.grad_beta)                 */
  float* grad_in_norm_weight;     /* out [C]                                                      */
  float* grad_in_norm_bias;       /* out [C]                                                      */
  float* grad_inconv_weight;      /* out [d_model][C]                                             */
  float* grad_inconv_bias;        /* out [d_model]                                                */
  float* grad_query;              /* out [n_head][d_k]                                            */
  float* grad_key_weight;         /* out [n_head*d_k][d_model]                                    */
  float* grad_key_bias;           /* out [n_head*d_k]                                             */
  float* grad_pe;                 /* acc [B][T][d_model] or NULL                                  */
} c2s_ltae_fold_bwd_io;
int c2s_ltae_fold_backward(const c2s_ltae_desc* desc, const c2s_ltae_params* params, const c2s_ltae_fold_bwd_io* io,
                           void* workspace, size_t workspace_bytes, void* stream);

size_t c2s_ltae_backward_workspace_bytes(const c2s_ltae_desc* desc);
int c2s_ltae_backward(const c2s_ltae_desc* desc, const c2s_ltae_params* params, const void* x, const void* positions,
                      const uint8_t* pad_mask, const c2s_ltae_bwd_io* io, void* workspace, size_t workspace_bytes,
                      void* stream);

/* ------------------------------------------------------------------------------------------
 * Edges of the tile inference pipeline (SURVEY.md section 8f, rank 3)
 *   before the model: DatasetCreator._patchify          src/helpers/dataset_creator.py:347-388
 *                     S2TSCZCropDataset.__getitem__     src/datasets/s2_ts_cz_crop.py:374, 393-398
 *                     pad_collate                       src/utils.py:14-66
 *   after the model:  generate_prediction               src/webapp/prediction.py:316-333
 * ---------------------------------------------------------------------------------------- */
enum c2s_raw_dtype { C2S_RAW_I16 = 0, C2S_RAW_U16 = 1, C2S_RAW_F32 = 2 };

typedef struct c2s_tile_desc {
  int32_t T, T_pad;      /* frames of the tile / frames of a model input (>= T; the rest is pad_value)       */
  int32_t C;             /* channels (10 Sentinel-2 bands)                                                   */
  int32_t H, W;          /* tile size in pixels (10980 x 10980; the webapp's sub-tiles are 1098 x 1098)      */
  int32_t patch;         /* patch edge (128), a multiple of 8                                                */
  int32_t grid_h, grid_w;/* patch rows / columns of the zero-padded tile; 0 = ceil(H / patch), ceil(W / patch)
                            (the webapp pads by a fixed 182 pixels: 10 x 10 for 1098, dataset_creator.py:386) */
  int32_t patch_begin;   /* first patch of this call in the row-major patch list (shard / batch offset)      */
  int32_t patch_count;   /* patches of this call                                                             */
  int32_t src_dtype;     /* enum c2s_raw_dtype of the raw tile (c2s_tile_patchify)                           */
  int32_t dst_dtype;     /* enum c2s_dtype of the patches (c2s_tile_patchify) / of the logits (c2s_tile_classmap) */
  float pad_value;       /* value of the frames T .. T_pad-1 (0, src/utils.py:14)                            */
} c2s_tile_desc;

/* patches[p, t, c, y, x] = (pad0(tile)[t, channels_order[c], Y, X] - mean[c]) / std[c]   (t < T, fp32 arithmetic)
 *                        = pad_value                                                    (T <= t < T_pad)
 * with (Y, X) the pixel of patch patch_begin + p in the tile zero-padded (RAW zeros, so padding normalises to
 * -mean/std) to grid_h x grid_w patches.  tile: [T, C, H, W] raw; channels_order: int32 [C]; mean, std: float32 [C]
 * in the REORDERED channel order (prediction.py:244-249); patches: [patch_count, T_pad, C, patch, patch]. */
int c2s_tile_patchify(const c2s_tile_desc* desc, const void* tile, const int32_t* channels_order, const float* mean,
                      const float* std, void* patches, void* stream);

/* classmap[Y, X] = first argmax_k softmax_k(logits[p, :, y, x]); proba[k, Y, X] = softmax (float32, may be NULL):
 * the patches patch_begin .. patch_begin + patch_count - 1 put back row-major and cropped to H x W
 * (prediction.py:318-320, 326-333, which moves every patch to the host first).  logits: [patch_count, K, patch, patch];
 * classmap: uint8 [H, W]; proba: float32 [K, H, W].  Calls for different patch ranges fill disjoint parts of the same
 * maps.  K <= 32. */
int c2s_tile_classmap(const c2s_tile_desc* desc, const void* logits, int32_t n_classes, uint8_t* classmap, float* proba,
                      void* stream);

/* ------------------------------------------------------------------------------------------
 * Loss side of the training step (SURVEY.md section 8f, rank 4)
 *   get_dilated + boundary labels        src/learning/utils.py:198-222, 283-285
 *   nn.CrossEntropyLoss(weight, label_smoothing) on [B,K,H,W] scores   train.py:462-467, learning/utils.py:322
 *   FocalCELoss(gamma=2.0)               src/learning/focal_loss.py:7-44, learning/utils.py:269, 318
 * ---------------------------------------------------------------------------------------- */
enum c2s_loss_kind { C2S_LOSS_CROSS_ENTROPY = 0, C2S_LOSS_FOCAL = 1 };

typedef struct c2s_loss_desc {
  int32_t B, K, H, W;    /* scores[B,K,H,W], target[B,H,W] int64                                              */
  int32_t dtype;         /* enum c2s_dtype of the scores and of their gradient                                */
  int32_t kind;          /* enum c2s_loss_kind                                                                */
  int32_t ignore_index;  /* FocalCELoss.ignore_index (-100); nn.CrossEntropyLoss always ignores -100           */
  int32_t size_average;  /* FocalCELoss.size_average: mean over the kept pixels (1) or sum (0)                 */
  float gamma;           /* FocalCELoss.gamma                                                                  */
  float label_smoothing; /* nn.CrossEntropyLoss(label_smoothing=...)                                           */
} c2s_loss_desc;

/* boundary[b,y,x] = 1 where more than one class occurs in the 4- (or 8-) neighbourhood of (y,x) including itself, the
 * image border adding no class (zero padding of the one-hot planes), else 0 -- `torch.where(get_dilated(y, K, dev,
 * connectivity).sum(1) > 1, 1, 0)` without the B x K x H x W one-hot tensor and its grouped convolution.
 * target, boundary: int64 [B,H,W]. */
int c2s_boundary_target(const int64_t* target, int32_t B, int32_t H, int32_t W, int32_t connectivity, int64_t* boundary,
                        void* stream);

/* loss (device float scalar):
 *   kind CROSS_ENTROPY: sum_i [(1-eps) w[y_i] nll_i + eps/K sum_k w[k] (-log p_ik)] / sum_i w[y_i]   over y_i != -100
 *   kind FOCAL        : mean (or sum) over y_i != ignore_index of -(1 - p_i)^gamma log p_i,  p_i = softmax(scores_i)[y_i];
 *                       with a class weight the reference's [N,1] x [N] broadcast (focal_loss.py:34-36) is kept: the loss
 *                       is (sum_i w[y_i]) (sum_j focal_j), divided by N^2 for the mean
 * weight: float32 [K] or NULL.  Labels outside [0, K) that are not the ignore value are dropped like ignored ones (torch
 * raises a device assertion for them).  The workspace (c2s_seg_loss_workspace_bytes, 8-byte aligned) carries the
 * normalisation from the forward to c2s_seg_loss_backward, which writes grad_scores = grad_loss * d loss / d scores
 * (grad_loss: device float scalar). Deterministic: fixed-order two-stage reduction, no atomics. */
size_t c2s_seg_loss_workspace_bytes(void);
int c2s_seg_loss_forward(const c2s_loss_desc* desc, const void* scores, const int64_t* target, const float* weight,
                         float* loss, void* workspace, size_t workspace_bytes, void* stream);
int c2s_seg_loss_backward(const c2s_loss_desc* desc, const void* scores, const int64_t* target, const float* weight,
                          const void* workspace, const float* grad_loss, void* grad_scores, void* stream);

/* ------------------------------------------------------------------------------------------
 * library services
 * ---------------------------------------------------------------------------------------- */
/* ------------------------------------------------------------------------------------------
 * Shared convolutional encoder over the B*T frames (SURVEY.md section 8f, rank 4)
 *   ConvLayer = Conv2d(reflect padding) -> GroupNorm -> ReLU      src/backbones/conv.py:29-96
 *   ConvBlock / DownConvBlock                                      conv.py:164-200, 238-296
 *   smart_forward over the valid frames                            temp_shared_block.py:18-47
 * Forward only.  Frames are packed (c2s_frame_index / c2s_frames_gather): [frames][C][H][W].
 * ---------------------------------------------------------------------------------------- */
typedef struct c2s_conv_desc {
  int32_t frames;                  /* packed frames                                              */
  int32_t c_in, c_out;
  int32_t H, W;                    /* input resolution                                           */
  int32_t kernel, stride, padding; /* nn.Conv2d(k, stride, padding, padding_mode='reflect')      */
  int32_t dtype;                   /* enum c2s_dtype of x and y                                  */
} c2s_conv_desc;

/* 1 when c2s_conv2d_forward serves the layer on the tensor cores (bf16):
 *   3x3, stride 1, padding 1, W = 128 / 64 / 32, c_in <= 16 or c_in = 64, c_out = 64   (in_conv, conv1 / conv2 of the down blocks)
 *   3x3, stride 1, padding 1, W = 16, 2 <= H <= 16, c_in and c_out 64 or 128           (conv1 / conv2 of U-TAE's last down block)
 *   4x4, stride 2, padding 1, W = 128 / 64 / 32, even H, 64 -> 64 channels             (the strided layer of DownConvBlock, conv.py:252-263)
 * Other layers are the caller's business. */
int c2s_conv2d_supported(const c2s_conv_desc* desc);
size_t c2s_conv2d_workspace_bytes(const c2s_conv_desc* desc); /* prepared bf16 weights */

/* Optional normalisation of the convolution's INPUT on the fly: x is then the RAW output of the previous ConvLayer stage
 * and the kernel reads relu(GroupNorm(x)) -- the previous stage's normalisation pass never touches memory. */
typedef struct c2s_conv_input_norm {
  const float* stats;   /* [frames][n_sub][2] sums of the previous stage (c2s_conv2d_forward: n_sub = 4)       */
  const float* gamma;   /* nn.GroupNorm.weight [c_in]                                                          */
  const float* beta;    /* nn.GroupNorm.bias   [c_in]                                                          */
  int32_t n_groups, n_sub, relu;
  float eps;
} c2s_conv_input_norm;

/* y[f, o, y, x] = bias[o] + sum_{c, ky, kx} weight[o, c, ky, kx] * x'[f, c, reflect(s y + ky - 1), reflect(s x + kx - 1)]
 *   x      : [frames, c_in, H, W] bf16;  x' = x, or relu(GroupNorm(x)) rounded to bf16 when in_norm is given (3x3 only)
 *   weight : float32 [c_out, c_in, k, k] (nn.Conv2d.weight), bias float32 [c_out] | NULL
 *   y      : [frames, c_out, H / s, W / s] bf16, the RAW convolution output (GroupNorm needs the whole frame first)
 *   stats  : float32 [frames][4][2] = (sum, sum of squares) of the fp32 outputs per frame and quarter of the c_out channels
 *            (16 or 32 channels; written, not accumulated), for c2s_group_norm_relu / c2s_conv_input_norm with n_sub = 4;
 *            or NULL
 *   workspace: c2s_conv2d_workspace_bytes, 16-byte aligned */
int c2s_conv2d_forward(const c2s_conv_desc* desc, const void* x, const c2s_conv_input_norm* in_norm, const float* weight,
                       const float* bias, void* y, float* stats, void* workspace, size_t workspace_bytes, void* stream);

/* stats[f][g] = (sum, sum of squares) over the channels of group g and the hw pixels of frame f of x[frames, C, hw]. */
int c2s_group_stats(const void* x, int32_t dtype, int64_t frames, int32_t channels, int64_t hw, int32_t n_groups,
                    float* stats, void* stream);

/* out = act(GroupNorm(x)) [+ residual]: nn.GroupNorm(n_groups, C) with the statistics of c2s_conv2d_forward (n_sub = 4)
 * or c2s_group_stats (n_sub = n_groups), then ReLU when `relu` (conv.py:83-86), then the residual of DownConvBlock
 * (`out + conv2(out)`, conv.py:291).  x, residual, out : [frames, C, hw] in `dtype`; out may alias x. */
int c2s_group_norm_relu(const void* x, const float* stats, int32_t n_sub, const float* gamma, const float* beta,
                        const void* residual, void* out, int32_t dtype, int64_t frames, int32_t channels, int64_t hw,
                        int32_t n_groups, float eps, int32_t relu, void* stream);

int c2s_abi_version(void);
const char* c2s_last_error(void);
/* Number of kernels this library launched (all threads of the process) since the last reset
 * (bench.py reports it as gpu_launches). */
int64_t c2s_launch_count(void);
void c2s_reset_launch_count(void);
/* Kernel-selection switches for parity tests and A/B measurements (process-wide, value 0 = what production runs).
 * They replace environment variables: nothing on the call path reads the environment. */
enum c2s_option {
  C2S_OPT_LTAE_KERNEL = 0, /* enum c2s_ltae_kernel: which kernel serves c2s_ltae_forward                       */
  C2S_OPT_AGG_KERNEL = 1,  /* 0 = automatic, 1 = register-streaming aggregator kernels (no bulk-copy pipeline) */
  C2S_OPT_AGG_TAPS = 2,    /* 0 = automatic, 1 = bilinear taps read from global memory (no staged rows)        */
  C2S_OPT_LTAE_BWD_KERNEL = 3 /* 0 = automatic (tensor-core kernel where eligible), 1 = fp32 CUDA-core kernel     */
};
enum c2s_ltae_kernel {
  C2S_LTAE_KERNEL_AUTO = 0,
  C2S_LTAE_KERNEL_GENERAL = 1, /* fp32 CUDA-core kernel (c2s_ltae.cu), any shape                                   */
  C2S_LTAE_KERNEL_SLAB = 2,    /* whole-slab kernel with CTA-wide phases (c2s_ltae_fa.cu) where eligible, else general */
  C2S_LTAE_KERNEL_TEAM = 3    /* team-pipelined slab kernel (c2s_ltae_team.cu) where eligible, else slab / general */
};
int c2s_set_option(int option, int value); /* C2S_ERR_BAD_ARGUMENT for an unknown option / value */
int c2s_get_option(int option);            /* current value, -1 for an unknown option            */
/* Name of the kernel the library launched last (diagnostics). */
const char* c2s_last_kernel(void);
/* Name of the last L-TAE attention kernel ("ltae_forward<...>") the library launched (diagnostics: which of the
 * kernels behind c2s_ltae_forward served the call). */
const char* c2s_last_ltae_kernel(void);

#ifdef __cplusplus
}
#endif
#endif /* CROP2SEG_B200_H_ */
