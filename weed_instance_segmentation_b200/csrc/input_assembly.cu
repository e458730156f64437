// input_assembly.cu -- pixel-decoder input assembly (SURVEY.md section 8(f) rank 3).
//
// Replaces, per feature level, the tail of `input_projections[level]` and the flatten / transpose / concat that
// follows it in Mask2FormerPixelDecoder.forward (M2F:1301-1313):
//     x = Conv2d(C_in, 256, 1)(feature)            (stays a library GEMM)
//     x = GroupNorm(32, 256)(x)                    (B, 256, H, W)
//     x = x.flatten(2).transpose(1, 2)             (B, H*W, 256) view
//     input_embeds_flat = cat(levels, dim=1)       (B, S, 256) copy
// The reference runs a GroupNorm kernel (read + write the NCHW tensor) and then a strided concat copy (read + write
// again). Here: one statistics pass over the conv output and ONE normalise-and-transpose pass that writes each level
// straight into its row range of the (B, S, 256) encoder input. Backward: one reduction pass and one transposing
// pass. Everything is HBM-bound streaming; tiles go through a 32 x 33 shared-memory transpose so both the NCHW side
// (contiguous along pixels) and the row side (contiguous along channels) are accessed in full 128-byte lines.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "msda_b200.h"
#include "internal.h"

namespace {

template <typename T> __device__ __forceinline__ float ld(const T* p);
template <> __device__ __forceinline__ float ld<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ld<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ void st(T* p, float v);
template <> __device__ __forceinline__ void st<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void st<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

__device__ __forceinline__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
  return t;
}

// one block per (batch, group): the group's cpg channels are cpg * HW CONTIGUOUS elements of the NCHW tensor.
// One pass of shifted sums in fp64: with K = the group's first element, s = sum(x - K) and ss = sum((x - K)^2), then
// mean = K + s/n and var = ss/n - (s/n)^2. In fp32, E[x^2] - mean^2 cancels catastrophically when |mean| >> std (at
// mean 100 and std 1 the rounding of sums of x^2 ~ 1e4 swamps a variance of 1), and fp32 shifted sums still carry
// ~1e-7 of the variance plus (K - mean)^2 / var times that. In fp64 (x - K is exact) the statistics are accurate to
// far below their fp32 rounding. Measured on a B200 (1000 W) at config 2: 117 / 109 us per call (fp32 / bf16 input)
// against 113 / 106 us with fp32 sums. Measured and dropped: eight loads deep per thread (fp32 79 us, bf16 124 us);
// pairwise fp32 terms into the fp64 sums (188 / 182 us).
template <typename T>
__global__ void __launch_bounds__(256) gn_stats_kernel(const T* __restrict__ x, float2* __restrict__ stats, int C, int HW,
                                                       int G, float eps) {
  __shared__ double red[8];
  const int b = blockIdx.x / G, g = blockIdx.x % G;
  const int cpg = C / G;
  const long long n = (long long)cpg * HW;
  const T* base = x + ((long long)b * C + (long long)g * cpg) * HW;
  const double k = ld<T>(base);
  double s = 0.0, ss = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = (double)ld<T>(base + i) - k;
    s += v;
    ss = fma(v, v, ss);
  }
  const double sum = block_sum(s, red), sumsq = block_sum(ss, red);
  if (threadIdx.x == 0) {
    const double ms = sum / (double)n;
    const double mean = k + ms;
    const double var = fmax(sumsq / (double)n - ms * ms, 0.0);  // biased variance, as nn.GroupNorm
    stats[blockIdx.x] = make_float2((float)mean, (float)(1.0 / sqrt(var + (double)eps)));
  }
}

// tile = 32 channels x 32 pixels; out rows are (pixel, channel) with `out_batch_stride` elements between batch items
template <typename T>
__global__ void __launch_bounds__(256) gn_apply_transpose_kernel(const T* __restrict__ x, const float2* __restrict__ stats,
                                                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                 float* __restrict__ out, long long out_batch_stride, int C,
                                                                 int HW, int G) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int cpg = C / G;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = c0 + ty + 8 * j, p = p0 + tx;
    float v = 0.f;
    if (c < C && p < HW) {
      const float2 ms = stats[b * G + c / cpg];
      v = (ld<T>(x + ((long long)b * C + c) * HW + p) - ms.x) * ms.y * gamma[c] + beta[c];
    }
    tile[ty + 8 * j][tx] = v;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int p = p0 + ty + 8 * j, c = c0 + tx;
    if (c < C && p < HW) out[(long long)b * out_batch_stride + (long long)p * C + c] = tile[tx][ty + 8 * j];
  }
}

// backward reduction, one block per (batch, group): m1 = mean(dy * gamma), m2 = mean(dy * gamma * xhat) over the group,
// and the per-channel sums for grad_gamma / grad_beta (atomically added over the batch; the caller zero-fills them).
// A thread owns pixels: it reads the group's cpg <= 8 adjacent channels of dy (one 32-byte sector of the row) and the
// same pixel of the cpg NCHW channel planes (each plane coalesced across the threads).
template <typename T>
__global__ void __launch_bounds__(256) gn_bwd_reduce_kernel(const float* __restrict__ grad_out, long long go_batch_stride,
                                                            const T* __restrict__ x, const float2* __restrict__ stats,
                                                            const float* __restrict__ gamma, float2* __restrict__ m12,
                                                            float* __restrict__ grad_gamma, float* __restrict__ grad_beta,
                                                            int C, int HW, int G) {
  constexpr int MAXC = 8;
  __shared__ double red[8];
  const int b = blockIdx.x / G, g = blockIdx.x % G;
  const int cpg = C / G;
  const float2 ms = stats[blockIdx.x];
  float dg[MAXC], db[MAXC];
#pragma unroll
  for (int cc = 0; cc < MAXC; ++cc) dg[cc] = db[cc] = 0.f;
  const T* xg = x + ((long long)b * C + (long long)g * cpg) * HW;
  const float* gg = grad_out + (long long)b * go_batch_stride + g * cpg;
  for (int p = threadIdx.x; p < HW; p += blockDim.x) {
#pragma unroll
    for (int cc = 0; cc < MAXC; ++cc)
      if (cc < cpg) {
        const float dy = gg[(long long)p * C + cc];
        const float xh = (ld<T>(xg + (long long)cc * HW + p) - ms.x) * ms.y;
        dg[cc] = fmaf(dy, xh, dg[cc]);
        db[cc] += dy;
      }
  }
  double s1 = 0.0, s2 = 0.0;
#pragma unroll
  for (int cc = 0; cc < MAXC; ++cc)
    if (cc < cpg) {
      const double sdg = block_sum((double)dg[cc], red), sdb = block_sum((double)db[cc], red);
      const int c = g * cpg + cc;
      if (threadIdx.x == 0) {
        atomicAdd(grad_gamma + c, (float)sdg);
        atomicAdd(grad_beta + c, (float)sdb);
      }
      s1 += sdb * (double)gamma[c];
      s2 += sdg * (double)gamma[c];
    }
  if (threadIdx.x == 0) {
    const double n = (double)cpg * HW;
    m12[blockIdx.x] = make_float2((float)(s1 / n), (float)(s2 / n));
  }
}

// dx = rstd * (dy * gamma - m1 - xhat * m2), read dy from the (pixel, channel) rows, write dx in NCHW
template <typename T>
__global__ void __launch_bounds__(256) gn_bwd_apply_transpose_kernel(const float* __restrict__ grad_out, long long go_batch_stride,
                                                                     const T* __restrict__ x, const float2* __restrict__ stats,
                                                                     const float2* __restrict__ m12, const float* __restrict__ gamma,
                                                                     T* __restrict__ grad_x, int C, int HW, int G) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int cpg = C / G;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int p = p0 + ty + 8 * j, c = c0 + tx;
    tile[ty + 8 * j][tx] = (c < C && p < HW) ? grad_out[(long long)b * go_batch_stride + (long long)p * C + c] : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = c0 + ty + 8 * j, p = p0 + tx;
    if (c < C && p < HW) {
      const int gi = b * G + c / cpg;
      const float2 ms = stats[gi], m = m12[gi];
      const long long i = ((long long)b * C + c) * HW + p;
      const float xh = (ld<T>(x + i) - ms.x) * ms.y;
      st<T>(grad_x + i, ms.y * (tile[tx][ty + 8 * j] * gamma[c] - m.x - xh * m.y));
    }
  }
}

int validate(int64_t B, int32_t C, int64_t HW, int32_t G, int dtype, const char* who) {
  if (B < 0 || HW < 0 || C <= 0 || G <= 0 || C % G != 0) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, who);
  if (C / G > 8) return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, who);  // at most 8 channels per group (256 / 32)
  if (dtype != MSDA_B200_F32 && dtype != MSDA_B200_BF16) return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, who);
  if (HW > 0x7fffffffll || B * G > 0x7fffffffll || B > 65535) return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, who);
  return MSDA_B200_OK;
}

}  // namespace

extern "C" {

int msda_b200_groupnorm_to_rows_forward(const void* x, int x_dtype, const float* gamma, const float* beta, float eps,
                                        float* out, int64_t out_batch_stride, float* stats, int64_t B, int32_t C, int64_t HW,
                                        int32_t G, void* stream) {
  if (int rc = validate(B, C, HW, G, x_dtype, "groupnorm_to_rows_forward: bad shape or dtype")) return rc;
  if (B == 0 || HW == 0) return MSDA_B200_OK;
  if (!x || !gamma || !beta || !out || !stats)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "groupnorm_to_rows_forward: NULL pointer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  float2* s2 = reinterpret_cast<float2*>(stats);
  const dim3 grid((unsigned)((HW + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B);
  if (x_dtype == MSDA_B200_F32) {
    gn_stats_kernel<float><<<(unsigned)(B * G), 256, 0, st>>>(static_cast<const float*>(x), s2, C, (int)HW, G, eps);
    if (int rc = launched("groupnorm_to_rows_forward: statistics")) return rc;
    gn_apply_transpose_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(x), s2, gamma, beta, out,
                                                          out_batch_stride, C, (int)HW, G);
  } else {
    gn_stats_kernel<__nv_bfloat16><<<(unsigned)(B * G), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), s2, C, (int)HW, G, eps);
    if (int rc = launched("groupnorm_to_rows_forward: statistics")) return rc;
    gn_apply_transpose_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), s2, gamma, beta, out,
                                                                  out_batch_stride, C, (int)HW, G);
  }
  return launched("groupnorm_to_rows_forward: normalise");
}

int msda_b200_groupnorm_to_rows_backward(const float* grad_out, int64_t grad_out_batch_stride, const void* x, int x_dtype,
                                         const float* gamma, const float* stats, void* grad_x, float* grad_gamma,
                                         float* grad_beta, float* scratch, int64_t B, int32_t C, int64_t HW, int32_t G,
                                         void* stream) {
  if (int rc = validate(B, C, HW, G, x_dtype, "groupnorm_to_rows_backward: bad shape or dtype")) return rc;
  if (B == 0 || HW == 0) return MSDA_B200_OK;
  if (!grad_out || !x || !gamma || !stats || !grad_x || !grad_gamma || !grad_beta || !scratch)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "groupnorm_to_rows_backward: NULL pointer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const float2* s2 = reinterpret_cast<const float2*>(stats);
  float2* m12 = reinterpret_cast<float2*>(scratch);
  const dim3 grid((unsigned)((HW + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B);
  if (x_dtype == MSDA_B200_F32) {
    gn_bwd_reduce_kernel<float><<<(unsigned)(B * G), 256, 0, st>>>(grad_out, grad_out_batch_stride, static_cast<const float*>(x),
                                                                  s2, gamma, m12, grad_gamma, grad_beta, C, (int)HW, G);
    if (int rc = launched("groupnorm_to_rows_backward: reduction")) return rc;
    gn_bwd_apply_transpose_kernel<float><<<grid, 256, 0, st>>>(grad_out, grad_out_batch_stride, static_cast<const float*>(x), s2,
                                                              m12, gamma, static_cast<float*>(grad_x), C, (int)HW, G);
  } else {
    gn_bwd_reduce_kernel<__nv_bfloat16><<<(unsigned)(B * G), 256, 0, st>>>(
        grad_out, grad_out_batch_stride, static_cast<const __nv_bfloat16*>(x), s2, gamma, m12, grad_gamma, grad_beta, C, (int)HW, G);
    if (int rc = launched("groupnorm_to_rows_backward: reduction")) return rc;
    gn_bwd_apply_transpose_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(
        grad_out, grad_out_batch_stride, static_cast<const __nv_bfloat16*>(x), s2, m12, gamma,
        static_cast<__nv_bfloat16*>(grad_x), C, (int)HW, G);
  }
  return launched("groupnorm_to_rows_backward: transpose");
}

}  // extern "C"
