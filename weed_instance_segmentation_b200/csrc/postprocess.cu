// Instance post-processing of Mask2Former outputs: the mask side of
//   Mask2FormerImageProcessor.post_process_instance_segmentation   (transformers 5.5.0,
//   image_processing_mask2former.py:605-724, "M2FIP" below)
// as batched kernels.  M2FIP resizes every mask-logit plane bilinearly to 384 x 384, thresholds it at 0, scores each of
// the Q top-k (query, class) selections of an image by the mean sigmoid over its mask, nearest-resizes the selected
// masks to the target size and, one selection at a time on the host, paints every kept one (score >= threshold, not
// empty after the nearest resize) into a -1-filled map; later selections overwrite earlier ones and segment ids count
// up in selection order.  Here two passes do the same for the whole batch without a host round trip:
//
//   score pass  one block per (image, selection): the selected query's plane is upsampled to 384 x 384 with ATen's
//               upsample_bilinear2d arithmetic and expression order (bf16 logits: the value rounded to bf16 as
//               F.interpolate stores it), thresholded at 0, and reduced to sum(sigmoid * mask) and sum(mask) in fp32
//               in a fixed order (per-thread sums, then a fixed shuffle tree; bf16: the sigmoid rounded to bf16 first,
//               as torch computes it).  It writes mask_score = sum(sigmoid * mask) / (sum(mask) + 1e-6), the 384^2
//               mask bit-packed to the workspace, and whether the mask survives the nearest resize to the image's
//               target size: ATen's nearest map src = min((int)floorf(dst * ((float)384 / out)), 383) samples a set
//               of rows and columns of the 384-grid, and the mask is non-empty there iff a set bit lies on one of
//               those rows and one of those columns.
//   paint pass  one block per (target row, image): warp 0 turns (non-empty, score >= threshold) into the kept list
//               and segment ids in selection order with ballots; the block then finds, for the 384-grid row that the
//               target row samples, the last kept selection whose bit is set in each of the 384 columns, and writes
//               the float id (or -1) of every target pixel from that row of owners.  The first row's block also
//               writes the image's (score, label, id) table.
//
// No float atomics anywhere: results do not depend on the stream or on repetition.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "bilinear_index.cuh"
#include "msda_b200.h"
#include "internal.h"

namespace {

constexpr int kS = 384;                               // M2FIP's fixed resampling size (M2FIP:665-667)
constexpr int kWordsPerRow = kS / 32;                 // one 32-bit word per 32 columns
constexpr int kWordsPerMask = kS * kWordsPerRow;      // 4608 words = 18 KB per selection
constexpr int kMaxQ = 1024;                           // kept lists live in shared memory
constexpr int kMaxB = 65535;                          // paint grid.y
constexpr int kScoreThreads = 512;
constexpr int kScoreWarps = kScoreThreads / 32;
constexpr int kPaintThreads = 256;
constexpr int kMapThreads = 256;

size_t bits_bytes(int32_t B, int32_t Q) { return (size_t)B * Q * kWordsPerMask * sizeof(uint32_t); }
size_t workspace_size(int32_t B, int32_t Q) { return bits_bytes(B, Q) + (size_t)B * Q * sizeof(int32_t); }

// ATen's upsample_nearest2d source index (nearest_neighbor_compute_source_index, no scale factor).
__device__ __forceinline__ int nearest_src(int dst, float scale, int in) {
  return min((int)floorf(dst * scale), in - 1);
}

__device__ __forceinline__ float load_f(const float* p) { return __ldg(p); }
__device__ __forceinline__ float load_f(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
// Storage rounding of a value computed in fp32 (identity for fp32).
__device__ __forceinline__ float round_as(float v, const float*) { return v; }
__device__ __forceinline__ float round_as(float v, const __nv_bfloat16*) {
  return __bfloat162float(__float2bfloat16_rn(v));
}

template <typename T>
__global__ void __launch_bounds__(kScoreThreads)
pp_score_kernel(const T* __restrict__ logits, const int64_t* __restrict__ topk_index,
                const int32_t* __restrict__ target_hw, int Q, int C, int h, int w, float scale_h, float scale_w,
                float* __restrict__ mask_score, uint32_t* __restrict__ bits, int32_t* __restrict__ nonempty) {
  __shared__ BilinearSrc s_y[kS], s_x[kS];
  __shared__ unsigned char s_row[kS], s_col[kS];  // 384-grid rows / columns the nearest resize samples
  __shared__ float s_sum[kScoreWarps];
  __shared__ int s_cnt[kScoreWarps];
  const int sel = blockIdx.x;  // image * Q + selection
  const int b = sel / Q;
  const int64_t k = topk_index[sel];
  const bool valid = k >= 0 && k < (int64_t)Q * C;  // anything else selects an empty mask
  const int q = valid ? (int)(k / C) : 0;
  const int H = target_hw[2 * b], W = target_hw[2 * b + 1];
  for (int i = threadIdx.x; i < kS; i += kScoreThreads) {
    s_y[i] = bilinear_source_index(scale_h, i, h);
    s_x[i] = bilinear_source_index(scale_w, i, w);
    s_row[i] = 0;
    s_col[i] = 0;
  }
  __syncthreads();
  // Racing stores of the same value 1: the flags are exact whatever the order.
  for (int y = threadIdx.x; y < H; y += kScoreThreads) s_row[nearest_src(y, (float)kS / H, kS)] = 1;
  for (int x = threadIdx.x; x < W; x += kScoreThreads) s_col[nearest_src(x, (float)kS / W, kS)] = 1;
  __syncthreads();

  const T* plane = logits + ((int64_t)b * Q + q) * h * w;
  uint32_t* out_bits = bits + (size_t)sel * kWordsPerMask;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float acc = 0.f;
  int cnt = 0;
  bool hit = false;
  // Warp `warp` owns words warp, warp + kScoreWarps, ...; lane l of a word is column 32 * (word % 12) + l.
  for (int wi = warp; wi < kWordsPerMask; wi += kScoreWarps) {
    const int r = wi / kWordsPerRow, c = (wi - r * kWordsPerRow) * 32 + lane;
    const BilinearSrc sy = s_y[r], sx = s_x[c];
    const T* row0 = plane + (int64_t)sy.i0 * w;
    const T* row1 = plane + (int64_t)sy.i1 * w;
    // ATen upsample_bilinear2d_out_frame, same expression order
    const float v = round_as(sy.l0 * (sx.l0 * load_f(row0 + sx.i0) + sx.l1 * load_f(row0 + sx.i1)) +
                                 sy.l1 * (sx.l0 * load_f(row1 + sx.i0) + sx.l1 * load_f(row1 + sx.i1)),
                             plane);
    const bool m = valid && v > 0.f;
    // torch's sigmoid (1 / (1 + exp(-x)) in fp32, stored in the logits' dtype), times the 0/1 mask: a NaN logit
    // makes the sum NaN as in M2FIP
    const float sig = round_as(1.f / (1.f + expf(-v)), plane);
    acc += sig * (m ? 1.f : 0.f);
    cnt += m ? 1 : 0;
    hit |= m && s_row[r] && s_col[c];
    const uint32_t word = __ballot_sync(0xffffffffu, m);
    if (lane == 0) out_bits[wi] = word;
  }
  for (int o = 16; o > 0; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
    s_sum[warp] = acc;
    s_cnt[warp] = cnt;
  }
  const int any_hit = __syncthreads_or(hit);
  if (threadIdx.x == 0) {
    float s = 0.f;
    int n = 0;
    for (int i = 0; i < kScoreWarps; ++i) {
      s += s_sum[i];
      n += s_cnt[i];
    }
    mask_score[sel] = s / ((float)n + 1e-6f);
    nonempty[sel] = any_hit ? 1 : 0;
  }
}

__device__ __forceinline__ bool mask_bit(const uint32_t* bits, int sel, int r, int c) {
  return (__ldg(bits + (size_t)sel * kWordsPerMask + r * kWordsPerRow + (c >> 5)) >> (c & 31)) & 1u;
}

__global__ void __launch_bounds__(kPaintThreads)
pp_paint_kernel(const uint32_t* __restrict__ bits, const int32_t* __restrict__ nonempty,
                const float* __restrict__ pred_score, const int64_t* __restrict__ labels, double threshold,
                const int32_t* __restrict__ target_hw, int Q, float* __restrict__ maps, int32_t* __restrict__ table) {
  __shared__ int s_sel[kMaxQ];  // kept selections in selection order; position = segment id
  __shared__ int s_n;
  __shared__ float s_owner[kS];
  const int b = blockIdx.y, y = blockIdx.x;
  const int H = target_hw[2 * b], W = target_hw[2 * b + 1];
  if (y >= H) return;
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    int n = 0;
    for (int base = 0; base < Q; base += 32) {
      const int j = base + lane;
      const int idx = b * Q + j;
      const float score = j < Q ? pred_score[idx] : 0.f;
      const bool kept = j < Q && nonempty[idx] && (double)score >= threshold;  // M2FIP compares Python floats
      const uint32_t ballot = __ballot_sync(0xffffffffu, kept);
      const int id = n + __popc(ballot & ((1u << lane) - 1u));
      if (kept) s_sel[id] = j;
      if (y == 0 && j < Q) {
        table[3 * idx] = __float_as_int(score);
        table[3 * idx + 1] = (int32_t)labels[idx];
        table[3 * idx + 2] = kept ? id : -1;
      }
      n += __popc(ballot);
    }
    if (lane == 0) s_n = n;
  }
  __syncthreads();
  const int n = s_n;
  const int r = nearest_src(y, (float)kS / H, kS);
  for (int c = threadIdx.x; c < kS; c += kPaintThreads) {
    float owner = -1.f;
    for (int i = n - 1; i >= 0; --i) {
      if (mask_bit(bits, b * Q + s_sel[i], r, c)) {
        owner = (float)i;
        break;
      }
    }
    s_owner[c] = owner;
  }
  __syncthreads();
  int64_t off = 0;  // images' maps lie back to back
  for (int i = 0; i < b; ++i) off += (int64_t)target_hw[2 * i] * target_hw[2 * i + 1];
  float* out = maps + off + (int64_t)y * W;
  const float scale_w = (float)kS / W;
  for (int x = threadIdx.x; x < W; x += kPaintThreads) out[x] = s_owner[nearest_src(x, scale_w, kS)];
}

__global__ void __launch_bounds__(kMapThreads)
pp_binary_maps_kernel(const uint32_t* __restrict__ bits, const int32_t* __restrict__ table, int b, int Q, int H, int W,
                      int n_inst, float* __restrict__ out) {
  __shared__ int s_sel[kMaxQ];
  for (int i = threadIdx.x; i < n_inst; i += kMapThreads) s_sel[i] = -1;
  __syncthreads();
  for (int j = threadIdx.x; j < Q; j += kMapThreads) {
    const int id = table[3 * (b * Q + j) + 2];
    if (id >= 0 && id < n_inst) s_sel[id] = j;  // ids are distinct
  }
  __syncthreads();
  const int64_t plane = (int64_t)H * W;
  const int64_t p = blockIdx.x * (int64_t)kMapThreads + threadIdx.x;
  if (p >= plane) return;
  const int y = (int)(p / W), x = (int)(p - (int64_t)y * W);
  const int r = nearest_src(y, (float)kS / H, kS), c = nearest_src(x, (float)kS / W, kS);
  for (int i = 0; i < n_inst; ++i)
    out[i * plane + p] = s_sel[i] >= 0 && mask_bit(bits, b * Q + s_sel[i], r, c) ? 1.f : 0.f;
}

// 0 when (B, Q) is valid, else the failure code (message set).
int check_bq(int32_t B, int32_t Q) {
  if (B <= 0 || Q <= 0) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "postprocess: B and Q must be positive");
  if (B > kMaxB || Q > kMaxQ)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "postprocess: B > 65535 or Q > 1024");
  return 0;
}

}  // namespace

extern "C" size_t msda_b200_postprocess_workspace_bytes(int32_t B, int32_t Q, int32_t C) {
  if (B <= 0 || Q <= 0 || C <= 0 || B > kMaxB || Q > kMaxQ || (int64_t)Q * C > INT32_MAX) return 0;
  return workspace_size(B, Q);
}

extern "C" int msda_b200_postprocess_scores(const void* mask_logits, int32_t dtype, const int64_t* topk_index, int32_t C,
                                            const int32_t* target_hw, int32_t B, int32_t Q, int32_t h, int32_t w,
                                            float* mask_score, void* workspace, size_t workspace_bytes, void* stream) {
  if (const int rc = check_bq(B, Q)) return rc;
  if (C <= 0 || h <= 0 || w <= 0)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "postprocess_scores: C, h and w must be positive");
  if ((int64_t)Q * C > INT32_MAX)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "postprocess_scores: Q * C > 2^31 - 1");
  if (dtype != MSDA_B200_F32 && dtype != MSDA_B200_BF16)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "postprocess_scores: mask logits must be F32 or BF16");
  if (!mask_logits || !topk_index || !target_hw || !mask_score || !workspace)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "postprocess_scores: NULL pointer");
  if (workspace_bytes < workspace_size(B, Q))
    return msda_b200_internal_fail(MSDA_B200_ERR_WORKSPACE, "postprocess_scores: workspace too small");
  uint32_t* bits = static_cast<uint32_t*>(workspace);
  int32_t* nonempty = reinterpret_cast<int32_t*>(static_cast<char*>(workspace) + bits_bytes(B, Q));
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const float sh = (float)h / kS, sw = (float)w / kS;
  const unsigned blocks = (unsigned)B * Q;
  if (dtype == MSDA_B200_F32)
    pp_score_kernel<float><<<blocks, kScoreThreads, 0, s>>>(static_cast<const float*>(mask_logits), topk_index,
                                                             target_hw, Q, C, h, w, sh, sw, mask_score, bits, nonempty);
  else
    pp_score_kernel<__nv_bfloat16><<<blocks, kScoreThreads, 0, s>>>(static_cast<const __nv_bfloat16*>(mask_logits),
                                                                     topk_index, target_hw, Q, C, h, w, sh, sw,
                                                                     mask_score, bits, nonempty);
  return launched("postprocess_scores");
}

extern "C" int msda_b200_postprocess_paint(const void* workspace, size_t workspace_bytes, const float* pred_score,
                                           const int64_t* labels, double threshold, const int32_t* target_hw,
                                           int32_t B, int32_t Q, int32_t max_h, float* maps, int32_t* table,
                                           void* stream) {
  if (const int rc = check_bq(B, Q)) return rc;
  if (max_h <= 0) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "postprocess_paint: max_h must be positive");
  if (!workspace || !pred_score || !labels || !target_hw || !maps || !table)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "postprocess_paint: NULL pointer");
  if (workspace_bytes < workspace_size(B, Q))
    return msda_b200_internal_fail(MSDA_B200_ERR_WORKSPACE, "postprocess_paint: workspace too small");
  const uint32_t* bits = static_cast<const uint32_t*>(workspace);
  const int32_t* nonempty = reinterpret_cast<const int32_t*>(static_cast<const char*>(workspace) + bits_bytes(B, Q));
  pp_paint_kernel<<<dim3((unsigned)max_h, (unsigned)B), kPaintThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      bits, nonempty, pred_score, labels, threshold, target_hw, Q, maps, table);
  return launched("postprocess_paint");
}

extern "C" int msda_b200_postprocess_binary_maps(const void* workspace, size_t workspace_bytes, const int32_t* table,
                                                 int32_t B, int32_t Q, int32_t image, int32_t H, int32_t W,
                                                 int32_t n_inst, float* out, void* stream) {
  if (const int rc = check_bq(B, Q)) return rc;
  if (image < 0 || image >= B || H <= 0 || W <= 0 || n_inst < 0 || n_inst > Q)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID,
                                   "postprocess_binary_maps: image outside [0, B), H or W not positive, or n_inst "
                                   "outside [0, Q]");
  if (n_inst == 0) return MSDA_B200_OK;
  if (!workspace || !table || !out)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "postprocess_binary_maps: NULL pointer");
  if (workspace_bytes < workspace_size(B, Q))
    return msda_b200_internal_fail(MSDA_B200_ERR_WORKSPACE, "postprocess_binary_maps: workspace too small");
  const int64_t blocks = ((int64_t)H * W + kMapThreads - 1) / kMapThreads;
  if (blocks > INT32_MAX)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "postprocess_binary_maps: map too large");
  pp_binary_maps_kernel<<<(unsigned)blocks, kMapThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint32_t*>(workspace), table, image, Q, H, W, n_inst, out);
  return launched("postprocess_binary_maps");
}
