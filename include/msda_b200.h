/*
 * msda_b200.h -- C ABI of the B200-native multi-scale deformable attention library
 * (libmsda_b200.so, built from weed_instance_segmentation_b200/csrc/).
 *
 * This is the drop-in boundary for the one hot path this repository accelerates:
 * the pixel-decoder multi-scale deformable attention of the Mask2Former model that
 * marco-conciatori-public/weed_instance_segmentation fine-tunes.  The reference has no
 * FFI of its own; the interface each entry point replaces is the Python function
 *
 *   transformers/models/mask2former/modeling_mask2former.py:798-837   (M2F:798)
 *     multi_scale_deformable_attention(value, value_spatial_shapes,
 *                                      sampling_locations, attention_weights)
 *
 * called from M2F:980 by every pixel-decoder encoder layer and reached from the
 * reference at models/mask2former/train.py:196 (train), train.py:28 (validation),
 * models/metrics.py:56 and models/mask2former/inference.py:27.  The five-tensor
 * argument order (value, value_spatial_shapes, level_start_index, sampling_locations,
 * attention_weights) is the original Deformable-DETR operator order that
 * transformers/models/deformable_detr/modeling_deformable_detr.py:171-181 keeps.
 *
 * Conventions
 *   - Plain pointers and sizes only; no torch types.  Every `dev` pointer is CUDA device
 *     memory on the current device, every `host` pointer is ordinary host memory.
 *   - All tensors are contiguous, C order:
 *       value  (B, S, H, D)         dtype = value_dtype
 *       loc    (B, Q, H, L, P, 2)   float32 always, last dim (x, y), normalised to [0,1]
 *       attn   (B, Q, H, L, P)      dtype = attn_dtype (post-softmax weights)
 *       out    (B, Q, H*D)          dtype = value_dtype, channel index h*D + d
 *     Level l occupies rows [level_start_index[l], + H_l*W_l) of S, row-major y*W_l + x.
 *   - The library borrows the pointers for the duration of the call's enqueued work,
 *     allocates nothing persistent on the device, holds no global mutable state besides
 *     a thread-local error string and optional profiling events, and launches on the
 *     stream given (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - Return value: 0 on success, otherwise one of MSDA_B200_ERR_*; the message is
 *     available from msda_b200_last_error() on the calling thread.  Nothing throws.
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef MSDA_B200_H_
#define MSDA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_B200_ABI_VERSION 14
#define MSDA_B200_MAX_LEVELS 8

/* dtype codes */
#define MSDA_B200_F32 0
#define MSDA_B200_BF16 1
#define MSDA_B200_U8 2 /* planes of msda_b200_point_sample_forward only (binary target masks stay 1 byte/pixel) */

/* error codes */
#define MSDA_B200_OK 0
#define MSDA_B200_ERR_INVALID 1     /* null pointer, negative size, level table outside S ...   */
#define MSDA_B200_ERR_UNSUPPORTED 2 /* head dim / dtype combination without a kernel            */
#define MSDA_B200_ERR_CUDA 3        /* a CUDA runtime call or launch failed                      */
#define MSDA_B200_ERR_WORKSPACE 4   /* workspace missing or smaller than ..._workspace_bytes()   */

/* flags (msda_b200_desc.flags) */
/* Bits 2, 8 and 32 are retired (in-place bf16 atomics, no-window forward, pixel-sorted backward) and are not reused;
 * every entry point that takes a descriptor returns MSDA_B200_ERR_INVALID for a bit not defined here. */
#define MSDA_B200_FLAG_PROFILE 1u        /* record CUDA events around each kernel (see below)    */
#define MSDA_B200_FLAG_BWD_V1 4u         /* backward: per-corner reduction kernel (v1) instead of */
                                         /* the group-sorted tensor-core kernel (v3, bf16,        */
                                         /* D=32 & P=4)                                           */
#define MSDA_B200_FLAG_STRICT_PADDING 16u /* forward: skip the FMA of every zero-weight corner, so a non-finite  */
                                         /* value in a pixel grid_sample's zeros padding never reads (M2F:823)  */
                                         /* cannot become 0 * Inf = NaN; 25-30 % slower (the backward kernels    */
                                         /* always treat out-of-level corners as unread)                         */
#define MSDA_B200_FLAG_DETERMINISTIC 64u /* backward: bit-identical grad_value, grad_loc / grad_offsets and         */
                                         /* grad_attn / grad_logits for bit-identical inputs, whatever the stream,  */
                                         /* query_order or host-pipeline chunking; takes precedence over BWD_V1. No */
                                         /* float atomics: the per-corner kernel writes grad_loc / grad_attn and    */
                                         /* four (grad_value row, query, weight) records per sample, a stable radix */
                                         /* sort groups them by row in sample order, and LPP lanes per (batch, row, */
                                         /* head) sum their records in fp32 in that order and write grad_value once */
                                         /* (every element, rows no sample reads get 0).  Same dtypes and           */
                                         /* geometries as the default backward.                                     */
                                         /* Needs a workspace (fp32 values too) of 24 bytes per record (4 per       */
                                         /* sample: uint32 key + uint64 payload, double-buffered for the sort),     */
                                         /* 8 bytes per (batch, row, head) bucket and the sort's scratch; problems  */
                                         /* over 2^31 - 1 records or 2^32 - 1 buckets are MSDA_B200_ERR_UNSUPPORTED */

/* Problem description: plain old data, filled by the caller on the host. */
typedef struct msda_b200_desc {
  int32_t B;           /* batch                                                                  */
  int32_t S;           /* value rows = sum_l H_l*W_l (may be larger than the sum)                */
  int32_t Q;           /* queries                                                                */
  int32_t H;           /* heads                                                                  */
  int32_t D;           /* channels per head: 8, 16, 32, 64, 128                                  */
  int32_t L;           /* levels, 1..MSDA_B200_MAX_LEVELS                                        */
  int32_t P;           /* points per level; L*P <= 64 (backward: see below)                      */
  int32_t value_dtype; /* MSDA_B200_F32 | MSDA_B200_BF16: value, out, grad_out, grad_value       */
  int32_t attn_dtype;  /* MSDA_B200_F32 | MSDA_B200_BF16: attn, grad_attn                        */
  uint32_t flags;      /* MSDA_B200_FLAG_*                                                       */
  const int32_t* spatial_shapes_hw;  /* host, L x 2 = (H_l, W_l); M2F:1312 spatial_shapes_list   */
  const int64_t* level_start_index;  /* host, L; M2F:1321                                        */
} msda_b200_desc;

/* ABI version of the loaded library (== MSDA_B200_ABI_VERSION it was built with). */
int msda_b200_abi_version(void);

/* Message of the last failure on this thread ("" if none). Never NULL. */
const char* msda_b200_last_error(void);

/*
 * Forward.  Replaces M2F:798-837.
 *   out[b,q,h*D+d] = sum_{l,p} attn[b,q,h,l,p] * bilinear(value_l[b,:,h,d]; x = loc_x*W_l - 0.5,
 *                                                         y = loc_y*H_l - 0.5), zeros outside.
 * query_order (dev, optional, Q int32): a permutation of 0..Q-1 giving the order in which
 * queries are assigned to thread blocks (scheduling only; results do not depend on it).
 */
int msda_b200_forward(const msda_b200_desc* desc, const void* value /*dev*/, const float* loc /*dev*/,
                      const void* attn /*dev*/, void* out /*dev*/, const int32_t* query_order /*dev|NULL*/,
                      void* stream);

/* Bytes of device scratch msda_b200_backward needs for this problem (0 if none).  bf16 values: B*S*H*D float32
 * accumulators.  MSDA_B200_FLAG_DETERMINISTIC: the layout its comment describes, whatever the dtypes (0 for an
 * invalid or unsupported descriptor). */
size_t msda_b200_backward_workspace_bytes(const msda_b200_desc* desc);

/*
 * Backward.  Replaces autograd through M2F:798-837 (grid_sampler_2d_backward x L, etc.).
 * Writes every element of grad_value (B,S,H,D; the library zero-fills it first),
 * grad_loc (B,Q,H,L,P,2) float32 and grad_attn (B,Q,H,L,P).
 * grad_value is summed with unordered float atomics, so its last bits vary from run to run; set
 * MSDA_B200_FLAG_DETERMINISTIC for run-to-run identical gradients.
 * Geometry: the forward takes every L*P <= 64.  The backward's per-corner kernel holds the L*P samples of 128 / LPP
 * queries (LPP = D * sizeof(value) / 16) in shared memory, at most 227 KB per block, so small head dims allow less:
 *   fp32 D = 8: L*P <= 50 (fused backward: 45);  bf16 D = 8: L*P <= 32 (28);  bf16 D = 16: L*P <= 50 (45);
 *   every other (dtype, D): L*P <= 64.
 * Past its limit msda_b200_backward and msda_b200_backward_fused return MSDA_B200_ERR_UNSUPPORTED before any CUDA
 * call, as does msda_b200_host_pipeline_create with a backward; msda_b200_backward_workspace_bytes returns 0.
 */
int msda_b200_backward(const msda_b200_desc* desc, const void* value /*dev*/, const float* loc /*dev*/,
                       const void* attn /*dev*/, const void* grad_out /*dev*/, void* grad_value /*dev*/,
                       float* grad_loc /*dev*/, void* grad_attn /*dev*/, void* workspace /*dev|NULL*/,
                       size_t workspace_bytes, const int32_t* query_order /*dev|NULL*/, void* stream);

/*
 * Fused-prologue variants.  Replace M2F:952-971 + M2F:798-837 in one launch: the kernel takes the raw outputs
 * of the module's `sampling_offsets` and `attention_weights` projections and computes
 *   attn = softmax(logits over the L*P entries of each (query, head))                 (M2F:955-960)
 *   loc  = ref_points[b,q,l,:] + offsets[b,q,h,l,p,:] / (W_l, H_l)                     (M2F:962-971)
 * on the fly, so sampling_locations and attention_weights never round-trip through HBM.
 *   offsets (B,Q,H,L,P,2) and logits (B,Q,H,L*P): dtype = attn_dtype;  ref_points (B,Q,L,2) float32.
 *   attn_out (optional, float32, (B,Q,H,L,P)): the softmax output, for callers that return it (M2F:983).
 * The backward writes grad_offsets / grad_logits (dtype = attn_dtype); reference points get no gradient
 * (they are constants of the geometry, M2F:1095-1125).
 * ref_points may be NULL when Q == S and the levels are packed as level_start_index says (the pixel decoder's
 * self-attention: query i sits on pixel i): the kernels then compute the reference point of a query from its index --
 * the centre of its own pixel, (x + 0.5) / W_q, (y + 0.5) / H_q, for every level -- which is what
 * Mask2FormerPixelDecoderEncoderOnly.get_reference_points (M2F:1095-1125) returns for valid_ratios == 1 (no padding).
 */
int msda_b200_forward_fused(const msda_b200_desc* desc, const void* value /*dev*/, const void* offsets /*dev*/,
                            const void* logits /*dev*/, const float* ref_points /*dev|NULL*/, void* out /*dev*/,
                            float* attn_out /*dev|NULL*/, const int32_t* query_order /*dev|NULL*/, void* stream);

int msda_b200_backward_fused(const msda_b200_desc* desc, const void* value /*dev*/, const void* offsets /*dev*/,
                             const void* logits /*dev*/, const float* ref_points /*dev|NULL*/, const void* grad_out /*dev*/,
                             void* grad_value /*dev*/, void* grad_offsets /*dev*/, void* grad_logits /*dev*/,
                             void* workspace /*dev|NULL*/, size_t workspace_bytes,
                             const int32_t* query_order /*dev|NULL*/, void* stream);

/*
 * Encoder-layer epilogue (SURVEY.md section 8(f) rank 2): fused residual add + LayerNorm over rows of `channels`
 * (a multiple of 128, at most 512; 256 in Mask2Former).  Replaces M2F:1049-1050 and M2F:1058-1059,
 *   y = LayerNorm(x + residual) * gamma + beta,
 * and their autograd nodes.  x / residual may be float32 or bfloat16 (dtype codes as above); y, mean, rstd,
 * gamma, beta and every gradient are float32.  grad_sum is d loss / d (x + residual), i.e. the gradient of both
 * inputs; grad_sum_lowp (optional) receives the same values in bfloat16 for a bfloat16 x.  The library zero-fills
 * grad_gamma / grad_beta before accumulating.
 * y_lowp (optional): the same y rounded to bfloat16 -- the operand of the projection that follows under autocast
 * (fc1 after the first LayerNorm, M2F:1052), so no separate cast kernel runs; grad_y_lowp (optional) is the gradient
 * that came back through that copy and is added to grad_y inside the backward kernel.
 */
int msda_b200_add_layernorm_forward(const void* x /*dev*/, int x_dtype, const void* residual /*dev*/, int residual_dtype,
                                    const float* gamma /*dev*/, const float* beta /*dev*/, float eps, float* y /*dev*/,
                                    void* y_lowp /*dev|NULL, bfloat16*/, float* mean /*dev, rows*/, float* rstd /*dev, rows*/,
                                    int64_t rows, int32_t channels, void* stream);

int msda_b200_add_layernorm_backward(const float* grad_y /*dev*/, const void* grad_y_lowp /*dev|NULL, bfloat16*/,
                                     const void* x /*dev*/, int x_dtype, const void* residual /*dev*/, int residual_dtype,
                                     const float* gamma /*dev*/, const float* mean /*dev*/, const float* rstd /*dev*/,
                                     float* grad_sum /*dev*/, void* grad_sum_lowp /*dev|NULL*/, float* grad_gamma /*dev*/,
                                     float* grad_beta /*dev*/, int64_t rows, int32_t channels, void* stream);

/*
 * The same with the encoder layer's closing clamp folded in (M2F:1062-1065, torch.clamp(y, -clamp, clamp) on the output
 * of the final LayerNorm while training): y is clamped before it is written (NaN stays NaN, as torch.clamp), and the
 * backward rebuilds y from x, residual, mean, rstd, gamma and beta and passes the incoming gradient only where
 * -clamp <= y <= clamp (torch.clamp's backward; false for NaN).  The reference clamps only after a host-side
 * isfinite().all() check; for finite activations the clamp is the identity, so folding it in removes the clamp, two
 * compare, one logical-and and one multiply kernel per layer and step without changing a value.  clamp > 0.
 */
int msda_b200_add_layernorm_clamp_forward(const void* x /*dev*/, int x_dtype, const void* residual /*dev*/,
                                          int residual_dtype, const float* gamma /*dev*/, const float* beta /*dev*/,
                                          float eps, float clamp, float* y /*dev*/, void* y_lowp /*dev|NULL, bfloat16*/,
                                          float* mean /*dev, rows*/, float* rstd /*dev, rows*/, int64_t rows,
                                          int32_t channels, void* stream);

int msda_b200_add_layernorm_clamp_backward(const float* grad_y /*dev*/, const void* grad_y_lowp /*dev|NULL, bfloat16*/,
                                           const void* x /*dev*/, int x_dtype, const void* residual /*dev*/,
                                           int residual_dtype, const float* gamma /*dev*/, const float* beta /*dev*/,
                                           float clamp, const float* mean /*dev*/, const float* rstd /*dev*/,
                                           float* grad_sum /*dev*/, void* grad_sum_lowp /*dev|NULL*/,
                                           float* grad_gamma /*dev*/, float* grad_beta /*dev*/, int64_t rows,
                                           int32_t channels, void* stream);

/*
 * Operands of the attention module under bfloat16 autocast (M2F:936-937, 947, 952-956) in one pass:
 *   query_bf16 = bfloat16(hidden + pos)  (read by the sampling_offsets / attention_weights projections),
 *   value_bf16 = bfloat16(hidden)        (read by value_proj),
 * with the roundings of the stock sequence (fp32 add, one round-to-nearest-even).  hidden / pos: float32, `elements`
 * each (a multiple of 8), contiguous.  Backward: grad_hidden = f32(grad_query) + f32(grad_value), grad_pos (optional) =
 * f32(grad_query); either incoming gradient may be NULL (= zero).
 */
int msda_b200_query_value_cast_forward(const float* hidden /*dev*/, const float* pos /*dev*/, void* query_bf16 /*dev*/,
                                       void* value_bf16 /*dev*/, int64_t elements, void* stream);

int msda_b200_query_value_cast_backward(const void* grad_query_bf16 /*dev|NULL*/, const void* grad_value_bf16 /*dev|NULL*/,
                                        float* grad_hidden /*dev*/, float* grad_pos /*dev|NULL*/, int64_t elements,
                                        void* stream);

/*
 * float32 projections on the bf16 tensor cores (csrc/gemm_f32.cu): the row-major products of F.linear and its backward,
 *   y[rows, out] = x[rows, in] . weight[out, in]^T (+ bias[out]) (+ ReLU when `relu` != 0; needs a bias),
 *   grad_x[rows, in] = grad_y[rows, out] . weight[out, in],     grad_weight[out, in] = grad_y^T . x,
 * as cuBLASLt GEMMs with CUBLAS_COMPUTE_32F_EMULATED_16BFX9 (every float32 operand split into three bfloat16 terms, nine
 * products accumulated in float32: at least SGEMM's accuracy, ~2x its speed on B200).  The CUDA toolkit's cuBLASLt
 * (>= 12.9) is opened at first use; msda_b200_linear_f32_available() returns 1 when it is there and accepts the compute
 * type, else 0 (the calls then return MSDA_B200_ERR_UNSUPPORTED).  `workspace` (device, caller-owned, may be NULL with
 * 0 bytes) bounds what cuBLASLt may use for split-K; 32-64 MB is plenty.  All tensors contiguous float32 on the device.
 */
int msda_b200_linear_f32_available(void);
int msda_b200_linear_f32_forward(const float* x /*dev*/, const float* weight /*dev*/, const float* bias /*dev|NULL*/,
                                 int relu, float* y /*dev*/, int64_t rows, int32_t out_features, int32_t in_features,
                                 void* workspace /*dev|NULL*/, size_t workspace_bytes, void* stream);
int msda_b200_linear_f32_grad_input(const float* grad_y /*dev*/, const float* weight /*dev*/, float* grad_x /*dev*/,
                                    int64_t rows, int32_t out_features, int32_t in_features, void* workspace /*dev|NULL*/,
                                    size_t workspace_bytes, void* stream);
int msda_b200_linear_f32_grad_weight(const float* grad_y /*dev*/, const float* x /*dev*/, float* grad_weight /*dev*/,
                                     int64_t rows, int32_t out_features, int32_t in_features,
                                     void* workspace /*dev|NULL*/, size_t workspace_bytes, void* stream);

/*
 * Column sum of a contiguous (rows x cols) matrix into float32 -- the bias gradient of a projection
 * (grad_bias = sum over rows of grad_out).  cols a multiple of 8 (bf16) / 4 (f32), at most 2048 / 1024.
 * The library zero-fills `out` first.
 */
int msda_b200_column_sum(const void* matrix /*dev*/, int dtype, float* out /*dev, cols*/, int64_t rows, int32_t cols,
                         void* stream);

/*
 * The FFN's ReLU backward and fc1's bias gradient (M2F:1052-1053) in one pass: grad_masked = grad_y where y > 0 else 0
 * (aten threshold_backward with the saved activation y = relu(z)), column_sum = sum over rows of grad_masked (float32,
 * zero-filled by the library first).  grad_y, y, grad_masked: contiguous (rows x cols), all of `dtype`; cols as above.
 */
int msda_b200_relu_backward_column_sum(const void* grad_y /*dev*/, const void* y /*dev*/, int dtype,
                                       void* grad_masked /*dev*/, float* column_sum /*dev, cols*/, int64_t rows,
                                       int32_t cols, void* stream);

/*
 * Batched bilinear point sampling -- the `sample_point` primitive of the loss / matcher path
 * (transformers/models/mask2former/modeling_mask2former.py:245-274: grid_sample, bilinear, zeros padding,
 * align_corners=False, coordinates normalised to [0,1] as (x, y)).  One call samples R rows of K points:
 *   planes[r]          device pointer to a contiguous (h, w) plane of rows[r].dtype (MSDA_B200_F32 / _BF16 / _U8)
 *   rows[r].coord_row  which row of `coords` (C, K, 2) the plane is sampled at (planes may share a point set)
 *   out                (R, K) float32
 * Planes are read in place: no gather of matched masks, no padding, no upcast.  The backward adds
 * grad_out[r, k] * bilinear weight into grad_planes[r] (float32 planes, accumulated with atomics -- the caller
 * zero-fills them; NULL entries are skipped).  Coordinates carry no gradient (the reference samples them under
 * no_grad, M2F:721-729).
 */
typedef struct msda_b200_ps_row {
  int32_t h, w;       /* plane extent                              */
  int32_t coord_row;  /* row of the coordinate table               */
  int32_t dtype;      /* MSDA_B200_F32, MSDA_B200_BF16 or MSDA_B200_U8 */
} msda_b200_ps_row;

int msda_b200_point_sample_forward(const void* const* planes /*dev, R*/, const msda_b200_ps_row* rows /*dev, R*/,
                                   const float* coords /*dev, (C,K,2)*/, float* out /*dev, (R,K)*/, int64_t R,
                                   int32_t K, void* stream);
int msda_b200_point_sample_backward(float* const* grad_planes /*dev, R*/, const msda_b200_ps_row* rows /*dev, R*/,
                                    const float* coords /*dev*/, const float* grad_out /*dev, (R,K)*/, int64_t R,
                                    int32_t K, void* stream);

/*
 * Deterministic form of msda_b200_point_sample_backward: bit-identical grad_planes for bit-identical inputs, whatever
 * the stream or the order of the rows among different planes.  Same contract otherwise: it adds into zero-filled float32
 * planes, NULL entries of grad_planes are skipped, corners outside the plane or with a NaN coordinate add nothing.
 *   key_base[r] (dev, R int64)  destination keys of row r's plane: pixel y*w + x of it has the key key_base[r] + y*w + x.
 *                               The caller numbers every pixel of every distinct gradient plane with one key in
 *                               [0, keys): rows that write into the same plane have the same key_base, distinct planes
 *                               have disjoint ranges [key_base, key_base + h*w).  A key outside [0, keys) adds nothing.
 *   keys                        the number of keys.
 * Each (row, point) writes four records, one per bilinear corner, at index 4*(r*K + k) + corner: a uint32 key and a
 * uint64 payload (r << 32 | float32 bits of grad_out[r, k] * wx * wy -- the value the atomic form adds).  A stable
 * radix sort over ceil(log2(keys + 1)) bits groups them by pixel in (row, point, corner) order; the thread at the start
 * of each run sums it in fp32 in that order and adds the sum to its pixel once.  No float atomics.
 * Workspace (device, at least ..._workspace_bytes(R, K, keys), 256-byte aligned): 24 bytes per record (key + payload,
 * double-buffered for the sort) and the sort's scratch.  More than 2^31 - 1 records (4*R*K) or keys >= 2^32 - 1 is
 * MSDA_B200_ERR_UNSUPPORTED.  The workspace size is 0 for invalid or unsupported arguments.
 */
size_t msda_b200_point_sample_backward_det_workspace_bytes(int64_t R, int32_t K, int64_t keys);
int msda_b200_point_sample_backward_det(float* const* grad_planes /*dev, R*/, const msda_b200_ps_row* rows /*dev, R*/,
                                        const int64_t* key_base /*dev, R*/, int64_t keys, const float* coords /*dev*/,
                                        const float* grad_out /*dev, (R,K)*/, int64_t R, int32_t K,
                                        void* workspace /*dev*/, size_t workspace_bytes, void* stream);

/*
 * Backward of bilinear resizing, F.interpolate(x, size=(Ho, Wo), mode="bilinear", align_corners=False) without a scale
 * factor (the pixel decoder's FPN upsampling, M2F:1360-1371), for NC contiguous float32 planes:
 *   grad_in (NC, Hi, Wi) = adjoint of the resize applied to grad_out (NC, Ho, Wo),
 * with ATen's index arithmetic (scale = (float)in / out, src = max(scale * (dst + 0.5) - 0.5, 0), i0 = (int)src,
 * i1 = i0 + (i0 < in - 1)).  A gather: every grad_in element is written once (no zero-fill needed) with the sum of the
 * output pixels that read it, in a fixed order, in fp32 -- bit-identical results for bit-identical inputs.
 */
int msda_b200_resize_bilinear_backward(const float* grad_out /*dev*/, float* grad_in /*dev*/, int64_t NC, int32_t Hi,
                                       int32_t Wi, int32_t Ho, int32_t Wo, void* stream);

/*
 * Instance post-processing (csrc/postprocess.cu): the mask side of Mask2FormerImageProcessor.
 * post_process_instance_segmentation (transformers 5.5.0, image_processing_mask2former.py:605-724) for a whole batch,
 * with no host round trip.  The caller keeps the class side in torch (softmax, per-image topk(Q, sorted=False) over the
 * Q*C (query, class) scores, the label gather, pred_score = topk score * mask_score).
 *   mask_logits (dev)  (B, Q, h, w) of `dtype` (MSDA_B200_F32 | MSDA_B200_BF16), contiguous
 *   topk_index  (dev)  (B, Q) int64: selection j of image b picks query topk_index[b, j] / C (an index outside
 *                      [0, Q*C) selects an empty mask)
 *   target_hw   (dev)  (B, 2) int32 (H_i, W_i) > 0; (384, 384) for every image reproduces target_sizes=None
 *   maps        (dev)  sum_i H_i*W_i float32: image i's (H_i, W_i) map follows image i-1's
 *   table       (dev)  (B, Q, 3) int32: float32 bits of pred_score, label, segment id (-1 = not kept)
 * scores: upsamples each selected plane to 384 x 384 with ATen's bilinear arithmetic (bf16: rounded to bf16), masks
 *   it at logit > 0, writes mask_score (dev, (B, Q) float32) = sum(sigmoid * mask) / (sum(mask) + 1e-6), both sums in
 *   fp32 in a fixed order (bf16: sigmoid rounded to bf16 first), and keeps in the workspace the mask bit-packed (18 KB
 *   per selection) and whether it is non-empty after ATen's nearest resize to (H_i, W_i).
 * paint: a selection is kept when it is non-empty there and (double)pred_score >= threshold; kept selections get ids
 *   0, 1, ... in selection order; each target pixel gets the id of the last kept selection whose resized mask covers
 *   it, else -1.  pred_score (dev, (B, Q) float32) and labels (dev, (B, Q) int64) are copied into the table.  max_h
 *   (host) >= every H_i.  Run it after scores, on the same workspace.
 * binary_maps: (n_inst, H, W) float32 0/1 maps of image `image`'s kept selections, in id order, from the table paint
 *   wrote (n_inst = its kept count, H, W = its target size).
 * Workspace (dev, at least _workspace_bytes(B, Q, C)): B*Q*(18432 + 4) bytes.  B <= 65535, Q <= 1024 and Q*C <= 2^31-1,
 * else MSDA_B200_ERR_UNSUPPORTED; the workspace size is 0 for invalid or unsupported arguments.  No float atomics:
 * bit-identical results for bit-identical inputs, whatever the stream.
 */
size_t msda_b200_postprocess_workspace_bytes(int32_t B, int32_t Q, int32_t C);
int msda_b200_postprocess_scores(const void* mask_logits /*dev*/, int32_t dtype, const int64_t* topk_index /*dev*/,
                                 int32_t C, const int32_t* target_hw /*dev*/, int32_t B, int32_t Q, int32_t h, int32_t w,
                                 float* mask_score /*dev*/, void* workspace /*dev*/, size_t workspace_bytes, void* stream);
int msda_b200_postprocess_paint(const void* workspace /*dev*/, size_t workspace_bytes, const float* pred_score /*dev*/,
                                const int64_t* labels /*dev*/, double threshold, const int32_t* target_hw /*dev*/,
                                int32_t B, int32_t Q, int32_t max_h, float* maps /*dev*/, int32_t* table /*dev*/,
                                void* stream);
int msda_b200_postprocess_binary_maps(const void* workspace /*dev*/, size_t workspace_bytes, const int32_t* table /*dev*/,
                                      int32_t B, int32_t Q, int32_t image, int32_t H, int32_t W, int32_t n_inst,
                                      float* out /*dev*/, void* stream);

/*
 * Pixel-decoder input assembly (SURVEY.md section 8(f) rank 3; M2F:1301-1313): GroupNorm of a 1x1-conv output
 * x (B, C, HW; NCHW with the spatial dims flattened; float32 or bfloat16) fused with the flatten / transpose / concat
 * that feeds the encoder:   out[b, p, c] = (x[b, c, p] - mean[b, g]) * rstd[b, g] * gamma[c] + beta[c],   g = c / (C/G),
 * float32, written into rows of a (B, S, C) tensor: `out` points at the first row of this level and consecutive batch
 * items are `out_batch_stride` ELEMENTS apart (S * C), so the three levels land side by side without a concat copy.
 * stats (B * G * 2 float32) receives (mean, rstd) for the backward.  C / G <= 8 (GroupNorm(32, 256)).
 * Backward: grad_x (dtype of x, NCHW) from grad_out (the same rows, float32); grad_gamma / grad_beta (C float32) are
 * ACCUMULATED (the caller zero-fills them once for all levels); scratch: B * G * 2 float32.
 */
int msda_b200_groupnorm_to_rows_forward(const void* x /*dev*/, int x_dtype, const float* gamma /*dev*/,
                                        const float* beta /*dev*/, float eps, float* out /*dev*/, int64_t out_batch_stride,
                                        float* stats /*dev*/, int64_t B, int32_t C, int64_t HW, int32_t G, void* stream);
int msda_b200_groupnorm_to_rows_backward(const float* grad_out /*dev*/, int64_t grad_out_batch_stride, const void* x /*dev*/,
                                         int x_dtype, const float* gamma /*dev*/, const float* stats /*dev*/,
                                         void* grad_x /*dev*/, float* grad_gamma /*dev*/, float* grad_beta /*dev*/,
                                         float* scratch /*dev*/, int64_t B, int32_t C, int64_t HW, int32_t G, void* stream);

/*
 * Host-buffer pipeline: the op with every tensor in HOST memory (the boundary a caller without device
 * buffers binds; bench.py's `e2e` leg).  The batch is cut into chunks of `chunk_images` images; each chunk
 * is copied to a device staging slot, run through msda_b200_forward (+ msda_b200_backward) and its results
 * copied back, on three streams (H2D, compute, D2H) over a ring of `slots` staging slots, so the two copy
 * directions and the kernels overlap -- within a step and across consecutive steps.  All host pointers use
 * the layouts of msda_b200_forward / msda_b200_backward; page-locked (pinned) memory is needed for the
 * copies to overlap.  The pipeline owns its device staging memory (cudaMalloc at create, on the current
 * device) and copies the descriptor's host arrays; `query_order` (device pointer or NULL) stays caller-owned.
 *
 *   create : desc->B is the batch of one step; with_backward = 0 builds a forward-only pipeline
 *            (grad_out and the grad_* pointers of step are then ignored).
 *   step   : enqueue one whole batch; returns without waiting.  Work starts after everything already
 *            enqueued on `stream` (fork).  Host buffers must stay untouched until join + synchronise.
 *   join   : make `stream` wait for everything enqueued so far (join) -- CUDA events recorded on `stream`
 *            before the first step and after join bracket the device time of the steps in between.
 *   sync   : block the host until everything enqueued so far has finished.
 */
typedef struct msda_b200_host_pipeline msda_b200_host_pipeline;

int msda_b200_host_pipeline_create(const msda_b200_desc* desc, int32_t chunk_images, int32_t slots,
                                   int32_t with_backward, const int32_t* query_order /*dev|NULL*/,
                                   msda_b200_host_pipeline** pipeline);
int msda_b200_host_pipeline_step(msda_b200_host_pipeline* pipeline, const void* value /*host*/,
                                 const float* sampling_loc /*host*/, const void* attn_weight /*host*/,
                                 const void* grad_output /*host*/, void* output /*host*/, void* grad_value /*host*/,
                                 float* grad_sampling_loc /*host*/, void* grad_attn_weight /*host*/, void* stream);
int msda_b200_host_pipeline_join(msda_b200_host_pipeline* pipeline, void* stream);
int msda_b200_host_pipeline_sync(msda_b200_host_pipeline* pipeline);
int msda_b200_host_pipeline_destroy(msda_b200_host_pipeline* pipeline);

/*
 * Profiling aid for bench.py: when desc->flags has MSDA_B200_FLAG_PROFILE the library records
 * CUDA events on `stream` around each kernel it launches.  After the stream has been
 * synchronised, msda_b200_profile_ms(which, &ms) returns the device time of the last such launch
 * on this thread.  `which`: one of MSDA_B200_PROF_*.
 */
#define MSDA_B200_PROF_FWD 0          /* forward gather kernel                                    */
#define MSDA_B200_PROF_BWD_ZERO 1     /* zero-fill of grad_value / workspace                      */
#define MSDA_B200_PROF_BWD_MAIN 2     /* backward gather + scatter kernel                         */
#define MSDA_B200_PROF_BWD_CONVERT 3  /* fp32 workspace -> bf16 grad_value                        */
#define MSDA_B200_PROF_COUNT 4
int msda_b200_profile_ms(int which, float* ms);

/* Number of kernels the library launched in this process since the last reset. Memsets are not counted, nor are
 * the cuBLASLt GEMMs of msda_b200_linear_f32_*; the radix sort of a deterministic backward counts as one. */
int64_t msda_b200_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_H_ */
