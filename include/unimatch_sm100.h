/* unimatch_sm100.h -- C ABI of libunimatch_sm100.so (B200 / sm_100a kernels for the UniMatch matching path).
 *
 * The reference (autonomousvision/unimatch) is pure Python/PyTorch and has no FFI of its own; these entry
 * points are what a binding for its hot-path functions would call.  Each declaration cites the reference
 * function it replaces (paths relative to the reference checkout).
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer to fp32 data unless stated otherwise; the caller owns all memory
 *    (outputs pre-allocated); nothing is allocated, freed or retained.
 *  - Feature maps are channel-last: a "token matrix" [N, L, C] with L = h*w (row-major y, x) and C = 128.
 *    Two-view tensors stack view 0 of all B pairs, then view 1: N = 2B, stream n = view*B + b.
 *  - Flow-like maps are channel-last too: [B, h, w, F] with F = 2 (flow: x, y) or 1 (disparity, inverse depth).
 *  - `stream` is a cudaStream_t passed as void*.  Work is enqueued, never synchronised.
 *  - Return value: 0 on success, a negative UM_E* code otherwise; um_last_error() gives the message
 *    (thread-local).  There is no CPU fallback: without a usable device every launcher fails.
 */
#ifndef UNIMATCH_SM100_H_
#define UNIMATCH_SM100_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UM_OK 0
#define UM_EINVAL (-22)   /* bad argument (shape, alignment, unsupported mode) */
#define UM_ECUDA (-5)     /* CUDA runtime error at launch */

#define UM_FEATURE_DIM 128

/* ABI version and build info. */
int um_abi_version(void);
const char* um_build_info(void);
const char* um_last_error(void);
/* Number of kernel launches issued through this library by the calling process (for bench `gpu_launches`). */
int64_t um_launch_count(void);

/* ---- window attention ------------------------------------------------------------------------------------
 * mask_mode */
#define UM_MASK_NONE 0
#define UM_MASK_SWIN 1     /* additive -100 between different shift regions (utils.py:84-108, :199-216)   */
#define UM_MASK_CAUSAL 2   /* keys with x_k > x_q get logit -1e9 (matching.py:138-142)                    */

/* Geometry of one windowed-attention problem over an h x w token grid.
 *   kh, kw : number of windows along y and x (window = (h/kh) x (w/kw) tokens)
 *   sh, sw : cyclic roll applied before splitting (attention.py:72-79, :132-138), 0 = unshifted
 * 2-D Swin: kh = kw = K, (sh, sw) = (wh/2, ww/2) on shifted layers.  1-D (per image row): kh = h.
 * Full attention: kh = kw = 1. */
typedef struct um_attn_geom {
  int32_t h, w;
  int32_t kh, kw;
  int32_t sh, sw;
  int32_t mask_mode;
} um_attn_geom;

/* out[n, t, :] = softmax_k( q[n,t,:] . k[m,k,:] / sqrt(128) + mask ) v[m,k,:],  m = (n + kv_shift) mod N,
 * keys k ranging over the window of token t.
 * Replaces single_head_full_attention (attention.py:8-16), single_head_full_attention_1d (:19-42),
 * single_head_split_window_attention (:45-104) and single_head_split_window_attention_1d (:107-163).
 * q, k, v, out: [N, L, *] with row strides ldq, ldk, ldv, ldo (floats, multiples of 4) and batch stride L*ld. */
int um_window_attention(const float* q, const float* k, const float* v, float* out,
                        int32_t n_streams, int32_t kv_shift,
                        int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo,
                        const um_attn_geom* geom, void* workspace, int64_t workspace_bytes, int32_t flags,
                        void* stream);
/* Dense 2-D windows of >= 128 tokens run on the tcgen05 tensor cores (fp16 hi/lo split operands, fp32
 * accumulation, fp32-faithful); they need a device scratch buffer of um_window_attention_workspace() bytes for the
 * window-major operand planes (0 = this geometry runs on CUDA cores and needs none).  flags: */
#define UM_ATTN_FORCE_CUDA_CORES 1   /* diagnostic: use the exact-fp32 CUDA-core kernel for every shape */
int64_t um_window_attention_workspace(const um_attn_geom* geom, int32_t n_streams);
/* Diagnostic: device buffer (>= 128*64 + 128*128 floats) that receives the raw S tile and the un-normalised O tile
 * of CTA (0,0,0) of the next tensor-core attention launches; NULL disables. */
void um_debug_set_dump(float* device_buffer);

/* The same attention on operands that are ALREADY window-major fp16 (hi, lo) planes [2][n_streams][kh*kw][lp][128]
 * (lp = um_attention_planes_lp(geom): the window length rounded up to 128; rows [lw, lp) of every window must be zero):
 * the projection GEMM writes them directly (um_conv_desc.win_dst), so the fp32 q/k/v rows never exist.
 * Output: fp32 rows (out, row stride ldo) and/or fp16 (hi, lo) planes [2][>= n_streams*h*w rows][128] in token order
 * (out_split, planes split_plane_stride halves apart) = the operand planes of the merge Linear layer.
 * um_attention_planes_lp() == 0: geometry runs on the CUDA-core kernel (um_window_attention) instead.
 * Replaces single_head_split_window_attention / single_head_full_attention (attention.py:8-16, :45-104). */
int32_t um_attention_planes_lp(const um_attn_geom* geom);
int um_window_attention_planes(const void* q_planes, const void* k_planes, const void* v_planes, float* out, int64_t ldo,
                               void* out_split, int64_t split_plane_stride, int32_t n_streams, int32_t kv_shift,
                               const um_attn_geom* geom, void* stream);

/* value_mode for um_softmax_expectation */
#define UM_VALUE_TENSOR 0   /* values[m, k, 0..vdim)                                                        */
#define UM_VALUE_COORDS 1   /* analytic pixel coordinates of key k: (x_k, y_k), vdim = 2                    */
#define UM_VALUE_XCOORD 2   /* analytic x_k only, vdim = 1                                                   */
/* post_op */
#define UM_POST_NONE 0
#define UM_POST_MINUS_OWN 1   /* out = E[value] - (x_t, y_t)   (matching.py:31-34)                          */
#define UM_POST_OWN_MINUS 2   /* out = x_t - E[value]          (matching.py:146-149)                        */

/* out[n, t, 0..vdim) = post( sum_k softmax_k( q[n,t,:] . k[m,k,:] / sqrt(128) + mask ) value_k ).
 * The L x L score matrix never leaves the SM.
 * Replaces global_correlation_softmax (matching.py:7-36), global_correlation_softmax_stereo (:126-151)
 * and the global branch of SelfAttnPropagation.forward (attention.py:194-215).
 * n_streams queries streams are processed (n = 0..n_streams-1), keys taken from stream (n + kv_shift) mod
 * n_total.  values (UM_VALUE_TENSOR): [n_total, L, vdim] contiguous, indexed by the KEY stream. */
int um_softmax_expectation(const float* q, const float* k, const float* values, float* out,
                           int32_t n_streams, int32_t n_total, int32_t kv_shift,
                           int64_t ldq, int64_t ldk, int32_t vdim, int32_t value_mode, int32_t post_op,
                           const um_attn_geom* geom, void* workspace, int64_t workspace_bytes, int32_t flags,
                           void* stream);
/* Global (one window = the whole map) problems of >= 128 tokens run on the tcgen05 tensor cores: S = Q K^T tiles in
 * TMEM, softmax and sum_k p_k value_k in registers.  Scratch bytes (0 = CUDA-core path, none needed); flags as above. */
int64_t um_softmax_expectation_workspace(const um_attn_geom* geom, int32_t n_total, int32_t value_mode);

/* ---- local (windowed, HBM/L2-bound) matching --------------------------------------------------------------
 * flow[b, y, x, :] = sum_k softmax_k( f0[b,y,x,:] . f1[b, y+dy_k, x+dx_k, :] / sqrt(128) ) (dx_k, dy_k),
 * (2ry+1) x (2rx+1) integer window, out-of-image taps get logit -1e9.
 * stereo != 0: returns -flow_x only ([B,h,w,1]).
 * Replaces local_correlation_softmax (matching.py:39-83) and local_correlation_softmax_stereo (:154-200). */
int um_local_corr_softmax(const float* f0, const float* f1, float* flow,
                          int32_t batch, int32_t h, int32_t w, int32_t ry, int32_t rx, int32_t stereo,
                          void* stream);

/* corr[b, y, x, k] = f0[b,y,x,:] . bilinear(f1[b], x + dx_k + u, y + dy_k + v) / sqrt(128), k = iy*(2r+1)+ix,
 * zero padding, align_corners=True; (u, v) = flow[b,y,x,:] (flow_dim 2) or (-flow[b,y,x,0], 0) when
 * flow_dim == 1 (disparity, unimatch.py:277-287).  corr is channel-last [B, h, w, (2r+1)^2].
 * Replaces local_correlation_with_flow (matching.py:86-123). */
int um_local_corr_volume(const float* f0, const float* f1, const float* flow, float* corr,
                         int32_t batch, int32_t h, int32_t w, int32_t radius, int32_t flow_dim, void* stream);
/* The same volume from fp16 (hi, lo) feature planes f0_planes / f1_planes [2][B][h][w][128] (um_split_planes), on the
 * tcgen05 tensor cores: one GEMM per 16 x 8 pixel tile against f1 over the bounding box of the tile's windows, with
 * fp32-faithful 3xFP16 dot products.  Tiles whose box is too large (a rough flow) are computed on CUDA cores instead;
 * fallback_tiles (device int32 or NULL) receives their number.  Outputs: corr (fp32 [B,h,w,81], or NULL) and/or out_split
 * (fp16 (hi, lo) planes [2][B][h][w][cp_split], channels [off_split, off_split + 81) written, the others untouched; or
 * NULL), the split being that of um_split_planes. */
int um_local_corr_volume_planes(const void* f0_planes, const void* f1_planes, const float* flow, float* corr,
                                void* out_split, int32_t cp_split, int32_t off_split, int32_t batch, int32_t h, int32_t w,
                                int32_t radius, int32_t flow_dim, int32_t* fallback_tiles, void* stream);

/* out[b,y,x,:] = bilinear(f[b], x + u, y + v), zeros outside, align_corners=True; (u,v) as above.
 * Replaces flow_warp (geometry.py:65-72, bilinear_sample :41-62). */
int um_flow_warp(const float* f, const float* flow, float* out,
                 int32_t batch, int32_t h, int32_t w, int32_t flow_dim, void* stream);

/* Occlusion masks from a forward / backward flow pair, both PLANAR [B,2,H,W] (what UniMatch.forward returns):
 * fwd_occ[b,y,x] = | fwd + warp(bwd, fwd) | > alpha (|fwd| + |bwd|) + beta, bwd_occ likewise with the roles swapped;
 * 1.0 = occluded.  Replaces forward_backward_consistency_check (geometry.py:75-96; called at evaluate_flow.py:792). */
int um_fb_consistency(const float* fwd_flow, const float* bwd_flow, float alpha, float beta, float* fwd_occ,
                      float* bwd_occ, int32_t batch, int32_t h, int32_t w, void* stream);

/* out[b,y,x,:] = sum_{3x3 nb} softmax( q[b,y,x,:] . k[b,nb,:] / sqrt(128) ) flow[b,nb,:]; out-of-image
 * neighbours take part with logit 0 and value 0 (zero-padded unfold).
 * Replaces SelfAttnPropagation.forward_local_window_attn (attention.py:217-253). */
int um_propagate_local(const float* q, const float* k, const float* flow, float* out,
                       int32_t batch, int32_t h, int32_t w, int32_t radius, int32_t flow_dim,
                       int64_t ldq, int64_t ldk, void* stream);

/* Plane-sweep matching: out[b,y,x,0] = sum_d softmax_d( f0 . bilinear(f1, proj_d(x,y)) / sqrt(128) ) cand_d
 * (or cand_argmax when from_argmax), proj_d = K (R K^-1 [x,y,1]^T / cand_d + t), uv = xy / max(z, 1e-3).
 * Kmat [B,9] (already scaled to the feature resolution), Kinv [B,9], pose [B,16] row-major (host computes the
 * 3x3 inverse).  cand: [D] inverse-depth candidates.
 * Replaces correlation_softmax_depth (matching.py:203-236) + warp_with_pose_depth_candidates (:239-282). */
int um_depth_corr_softmax(const float* f0, const float* f1, const float* Kmat, const float* Kinv,
                          const float* pose, const float* cand, float* out,
                          int32_t batch, int32_t h, int32_t w, int32_t num_cand, int32_t from_argmax,
                          void* stream);

/* ---- glue on the path ---------------------------------------------------------------------------------------
 * x[n, y, x, :] += table[(y mod wh), (x mod ww), :], table [wh, ww, 128] = PositionEmbeddingSine on the window.
 * Replaces feature_add_position (utils.py:111-131). */
int um_add_position(const float* x, const float* table, float* out,
                    int32_t n_streams, int32_t h, int32_t w, int32_t wh, int32_t ww, void* stream);

/* out = residual + LayerNorm(x) * gamma + beta over the last dim (128), eps 1e-5; residual may be NULL.
 * Replaces norm1/norm2 + the residual add of TransformerLayer.forward (transformer.py:137-144). */
int um_layernorm_residual(const float* x, const float* residual, const float* gamma, const float* beta,
                          float* out, int64_t rows, int64_t ldx, int64_t ldr, int64_t ldo, void* stream);

/* Convex upsampling: up[b, c, y*F+ky, x*F+kx] = sum_t softmax_t(mask[b,y,x, t*F*F + ky*F + kx]) * mult*flow[b, nb_t, c],
 * 3x3 zero-padded neighbourhood.  mask channel-last [B,h,w,9*F*F]; flow [B,h,w,fd]; up is PLANAR [B, fd, h*F, w*F]
 * (the layout the reference returns).  Replaces upsample_flow_with_mask (utils.py:134-152). */
int um_convex_upsample(const float* flow, const float* mask, float* up,
                       int32_t batch, int32_t h, int32_t w, int32_t flow_dim, int32_t factor, float mult,
                       void* stream);

/* Bilinear x2 upsampling (align_corners=True) of a channel-last flow map, values multiplied by `mult`.
 * Replaces F.interpolate(flow, scale_factor=2, mode='bilinear', align_corners=True) * 2 (unimatch.py:154). */
int um_upsample2x(const float* flow, float* out, int32_t batch, int32_t h, int32_t w, int32_t flow_dim,
                  float mult, void* stream);

/* Planar bilinear resize with align_corners=True: out[b,c] = scale[c] * resize(in[b,c]) for [B, C <= 3, H, W] fp32 tensors;
 * `scale` = HOST array of C floats or NULL; flip_x != 0 mirrors the output horizontally.  The callers' side of the boundary:
 * F.interpolate(..., mode='bilinear', align_corners=True) before the model and on its output, with the flow-component /
 * disparity rescale and the hflip of the bidirectional-disparity trick folded in (evaluate_flow.py:733-755,
 * evaluate_stereo.py:776-813, evaluate_depth.py:372-400). */
int um_resize_bilinear(const float* in, float* out, int32_t batch, int32_t channels, int32_t h_in, int32_t w_in,
                       int32_t h_out, int32_t w_out, const float* scale, int32_t flip_x, void* stream);

/* GRU gate fusions of SepConvGRU (reg_refine.py:37-52): rows of 128 hidden channels, independent row strides
 * (floats, multiples of 4) so the z|r pre-activations may live side by side in one fused conv output.
 *   um_gru_rh:     rh = sigmoid(r_pre) * h
 *   um_gru_update: h_out = (1 - sigmoid(z_pre)) * h + sigmoid(z_pre) * tanh(q_pre)                          */
int um_gru_rh(const float* r_pre, int64_t ldr, const float* h, int64_t ldh, float* rh, int64_t ldo, int64_t rows,
              void* stream);
int um_gru_update(const float* z_pre, int64_t ldz, const float* q_pre, int64_t ldq, const float* h, int64_t ldh,
                  float* h_out, int64_t ldo, int64_t rows, void* stream);

/* ---- tensor-core implicit-GEMM convolution / Linear layer (fp16 hi/lo split operands, fp32 accumulate) ----------
 * Replaces the nn.Conv2d calls of BasicUpdateBlock (reg_refine.py:6-119), refine_proj (unimatch.py:315) and, as a
 * 1x1 convolution over a [rows/16, 16] grid, nn.Linear (transformer.py:58-60,137,141).
 * Activations: channel-last fp16 planes [2 (hi,lo)][B][H][W][cin_p], cin_p % 64 == 0, padding channels zero.
 * Weights: fp16 planes [2][cout_p][ktot], K ordered (source, tap = ky*kw+kx, ci), ktot = sum_s kh*kw*cin_p[s].
 * Stride 1, 2, 4 or 8 (TMA element strides), zero padding (pad_h, pad_w).  Up to two sources are accumulated (= convolution of their concatenation). */
#define UM_ACT_NONE 0
#define UM_ACT_RELU 1
#define UM_ACT_TANH 2
#define UM_ACT_SIGMOID 3
#define UM_ACT_GELU 4      /* exact erf form (nn.GELU default, transformer.py:34) */
#define UM_CONV_LINEAR 0   /* y = act(acc + bias) -> out_f32 and/or out_split                                          */
#define UM_CONV_GRU_ZR 1   /* cout 256: z = sigmoid(y[0:128]) -> out_f32; sigmoid(y[128:256]) * aux0 -> out_split       */
#define UM_CONV_GRU_Q 2    /* cout 128: (1 - aux1) * aux0 + aux1 * tanh(y) -> out_f32 and/or out_split (reg_refine.py:41-42) */
#define UM_CONV_LN 3       /* cout 128, no bias: aux0 (optional residual) + LayerNorm(acc) * gamma + beta, eps 1e-5
                              (transformer.py:137-144) -> out_f32 and/or out_split                                       */
typedef struct um_conv_desc {
  const void* src[2];
  int32_t cin_p[2];
  int32_t nsrc;
  int32_t batch, h, w;
  const void* weights;
  const float* bias;          /* [cout] or NULL */
  int32_t kh, kw, pad_h, pad_w;
  int32_t cout, cout_p, bn;   /* bn = output-channel tile (16, 64, 96, 128, 192 or 256); cout_p % bn == 0.  Long-K launches
                               * (K >= 192, bn >= 64) over an even number of 16 x 8 pixel tiles run on CTA pairs
                               * (cta_group::2: two SMs share every MMA and each stages half of the weight tile);
                               * bn = 96 exists only as such a launch (Linear + ReLU).  UM_CONV_PAIR=0 disables pairs. */
  int32_t mode, act;
  float* out_f32;             /* [B,H,W,*] row stride ld_f32 floats, written at channel offset off_f32; or NULL */
  int64_t ld_f32;
  int32_t off_f32;
  int32_t cp_split;           /* channels of the split destination buffer */
  void* out_split;            /* fp16 planes [2][B][H][W][cp_split], written at channel offset off_split; or NULL */
  int32_t off_split;
  int32_t stride;             /* 1, 2, 4 or 8; output is [B, (h+2*pad_h-kh)/stride+1, (w+2*pad_w-kw)/stride+1, cout] */
  const float* aux0;          /* GRU: h   [B,H,W,128] row stride ld_aux0;  LN: residual or NULL */
  int64_t ld_aux0;
  const float* aux1;          /* GRU_Q: z [B,H,W,128] row stride ld_aux1 */
  int64_t ld_aux1;
  const float* gamma;         /* LN: [128] */
  const float* beta;          /* LN: [128] */
  /* batch == 1 only: distance in halves between the hi and the lo plane of the sources / of out_split when the planes are
   * row ranges of larger buffers (0 = densely stacked planes) */
  int64_t src_plane_stride, split_plane_stride;
  /* Window-major operand planes for um_window_attention_planes (a 128 -> cout Linear layer, bn 128, batch 1, pixels =
   * token rows): output channels [win_c0, win_c1) (128-aligned; operand o = (c - win_c0) / 128) are written as fp16
   * (hi, lo) rows of win_dst[o][2][win_streams][kh*kw][win_lp][128] at the row the window split / cyclic shift of
   * win_geom assigns to the token (attention.py:72-83 as address arithmetic); rows >= win_streams*h*w are skipped and
   * the padding rows [lw, win_lp) of every window are never written.  NULL = off. */
  void* win_dst;
  int32_t win_c0, win_c1, win_lp, win_streams;
  um_attn_geom win_geom;
  /* Optional fp32 tensor [B,H,W,>= cout] (row stride ld_pre floats) added to the accumulator before the post-operation: the
   * part of a convolution whose input channels do not change between calls (SepConvGRU over cat[h, inp, motion]: `inp`, and
   * in the first half `h`, are the same in every refinement iteration, unimatch.py:315-333) is computed once by the caller
   * and only the channels that changed are convolved per call.  Not for UM_CONV_LN; bn >= 32; cout % 32 == 0. */
  const float* pre;
  int64_t ld_pre;
} um_conv_desc;
int um_conv2d_tc(const um_conv_desc* desc, void* stream);

/* Fused transformer FFN (transformer.py:137-144, TransformerLayer.mlp + norm2 + residual) on token rows:
 *   out = residual + LayerNorm( GELU( [src0 | src1] W1^T ) W2^T ) * gamma + beta        (no biases, eps 1e-5)
 * src0 / src1: fp16 (hi, lo) planes [2][>= rows][128] (source, message), planes src_plane_stride halves apart;
 * w1: prepared planes [2][hidden][256] (K ordered source | message), w2: [2][128][hidden] (um_conv2d_tc weight layout);
 * residual: fp32 rows (row stride ld_res) or NULL; out_f32 (row stride ld_f32) and/or out_split planes [2][>= rows][128].
 * The hidden activation (4 KB per row as split planes) never leaves the SM: one CTA-pair kernel, hidden channels produced
 * 128 at a time into TMEM, GELU'd in place and consumed as the A operand of the second GEMM.
 * rows must be a multiple of 256 (pairs of 128-row tiles; callers with other row counts use two um_conv2d_tc launches),
 * hidden a multiple of 128. */
typedef struct um_ffn_desc {
  const void* src[2];
  int64_t src_plane_stride;
  int64_t rows;
  const void* w1;
  const void* w2;
  int32_t hidden;
  const float* residual;
  int64_t ld_res;
  const float* gamma;
  const float* beta;
  float* out_f32;
  int64_t ld_f32;
  void* out_split;
  int64_t split_plane_stride;
} um_ffn_desc;
int um_ffn_tc(const um_ffn_desc* desc, void* stream);

/* Direct 7x7 convolution (padding 3, stride 1 or 2) for inputs with 1-3 channels, exact fp32: the image stem
 * (backbone.py:55, with normalize_img of utils.py:23-31 folded in as x*scale[c]+shift[c]; scale/shift are HOST arrays of 3
 * floats or NULL) and refine.encoder.convf1 (reg_refine.py:62,70).  nchw != 0: planar sources in0 (images [0, n_half)) and
 * in1 (the rest), i.e. the two views without a concatenation copy; else one channel-last source [n,h,w,cin].
 * Output channel-last fp32 (row stride ld_out) and/or fp16 (hi, lo) planes of width cp; cout a multiple of 16, <= 128. */
int um_conv7x7_small(const float* in0, const float* in1, int32_t nchw, int32_t n_half, int32_t n, int32_t h, int32_t w,
                     int32_t cin, int32_t stride, const float* weight, const float* bias, int32_t cout, int32_t relu,
                     const float* scale, const float* shift, float* out_f32, int64_t ld_out, void* out_split, int32_t cp,
                     void* stream);

/* InstanceNorm2d (eps 1e-5, no affine, biased variance; backbone.py:7,41) on channel-last fp32 [n, hw, c] maps.
 * stats: [n][2][c] = mean, 1/sqrt(var+eps); scratch: um_instance_norm_scratch_floats(n, c) floats.
 * apply: y = IN(a) (stats_a may be NULL = identity), optional ReLU, optional + res (itself optionally normalised by
 * stats_res), optional ReLU; written as fp32 and/or fp16 (hi, lo) planes [2][n*hw][cp] at channel offset off. */
int64_t um_instance_norm_scratch_floats(int32_t n, int32_t c);
int um_instance_norm_stats(const float* x, int64_t ld, int32_t n, int32_t hw, int32_t c, float* scratch, float* stats,
                           void* stream);
int um_instance_norm_apply(const float* a, int64_t ld_a, const float* stats_a, int32_t relu_a, const float* res,
                           int64_t ld_res, const float* stats_res, int32_t relu_out, float* out_f32, int64_t ld_o,
                           void* out_split, int32_t cp, int32_t off, int32_t n, int32_t hw, int32_t c, void* stream);

/* fp32 rows [rows, channels] (row stride ld) -> fp16 (hi, lo) planes of a [>= rows, cp] buffer at channel offset off;
 * the lo plane starts dst_plane_stride halves after the hi plane (0 = rows * cp, densely stacked). */
int um_split_planes(const float* src, int64_t rows, int32_t channels, int64_t ld, void* dst, int32_t cp, int32_t off,
                    int64_t dst_plane_stride, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNIMATCH_SM100_H_ */
