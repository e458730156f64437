// layer_epilogue.cu -- fused residual-add + LayerNorm for the pixel-decoder encoder layer (SURVEY.md section 8(f) rank 2).
//
// Replaces, on both sides of the MSDeformAttn op,
//     hidden_states = residual + hidden_states                      (M2F:1049, M2F:1058)
//     hidden_states = self.{self_attn,final}_layer_norm(hidden_states)   (M2F:1050, M2F:1059)
// and their autograd nodes by one kernel per direction. Rows are d_model wide (256 in Mask2Former); one warp owns
// one row, statistics in fp32 registers, 16-byte accesses. Under autocast the branch input is bf16 (GEMM output)
// and the residual fp32; the output is fp32, as torch's autocast LayerNorm produces.
//
//   forward : y = (s - mean(s)) * rstd(s) * gamma + beta,  s = x + r        (saves mean, rstd)
//   backward: ds = rstd * (g - mean_c(g) - xhat * mean_c(g * xhat)),  g = dy * gamma,  xhat = (s - mean) * rstd
//             dgamma = sum_rows dy * xhat,  dbeta = sum_rows dy             (block partials -> fp32 atomics)
//             ds is the gradient of both x and r; it is written in fp32 and, if asked, also in x's dtype.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "msda_b200.h"
#include "internal.h"

namespace {

constexpr int kMaxC = 512;             // up to 4 float4 chunks per lane (backward keeps 32 KB of block partials)
constexpr int kRowsPerBlock = 8;       // 8 warps
constexpr int kThreads = kRowsPerBlock * 32;

template <typename T>
__device__ __forceinline__ float4 load4(const void* base, long long idx4);
template <>
__device__ __forceinline__ float4 load4<float>(const void* base, long long idx4) {
  return __ldg(reinterpret_cast<const float4*>(base) + idx4);
}
template <>
__device__ __forceinline__ float4 load4<__nv_bfloat16>(const void* base, long long idx4) {
  const uint2 v = __ldg(reinterpret_cast<const uint2*>(base) + idx4);
  return make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u), __uint_as_float(v.y << 16),
                     __uint_as_float(v.y & 0xffff0000u));
}
__device__ __forceinline__ void store4_bf16(void* base, long long idx4, float4 v) {
  const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 o;
  o.x = *reinterpret_cast<const unsigned*>(&lo);
  o.y = *reinterpret_cast<const unsigned*>(&hi);
  reinterpret_cast<uint2*>(base)[idx4] = o;
}

__device__ __forceinline__ float clamp_keep_nan(float v, float c) { return v < -c ? -c : (v > c ? c : v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// CH = C / 128 float4 chunks per lane (lane owns elements (k*32 + lane)*4 .. +3)
template <typename XT, typename RT, int CH>
__global__ void __launch_bounds__(kThreads) add_layernorm_fwd_kernel(const void* __restrict__ x, const void* __restrict__ r,
                                                                     const float* __restrict__ gamma,
                                                                     const float* __restrict__ beta, float eps,
                                                                     float* __restrict__ y, void* __restrict__ y_lowp,
                                                                     float* __restrict__ mean_out,
                                                                     float* __restrict__ rstd_out, long long N,
                                                                     float clamp) {
  constexpr int C = CH * 128;
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
  if (row >= N) return;
  float4 s[CH];
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < CH; ++k) {
    const long long i4 = row * (C / 4) + k * 32 + lane;
    const float4 a = load4<XT>(x, i4), b = load4<RT>(r, i4);
    s[k] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    sum += (s[k].x + s[k].y) + (s[k].z + s[k].w);
  }
  const float mean = warp_sum(sum) * (1.f / C);
  float var = 0.f;
#pragma unroll
  for (int k = 0; k < CH; ++k) {
    const float dx = s[k].x - mean, dy = s[k].y - mean, dz = s[k].z - mean, dw = s[k].w - mean;
    var += (dx * dx + dy * dy) + (dz * dz + dw * dw);
  }
  const float rstd = rsqrtf(warp_sum(var) * (1.f / C) + eps);
#pragma unroll
  for (int k = 0; k < CH; ++k) {
    const int c4 = k * 32 + lane;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + c4), bt = __ldg(reinterpret_cast<const float4*>(beta) + c4);
    float4 o;
    o.x = (s[k].x - mean) * rstd * g.x + bt.x;
    o.y = (s[k].y - mean) * rstd * g.y + bt.y;
    o.z = (s[k].z - mean) * rstd * g.z + bt.z;
    o.w = (s[k].w - mean) * rstd * g.w + bt.w;
    // torch.clamp(y, -clamp, clamp) (M2F:1062-1065; +inf = off): comparisons, not fminf / fmaxf, so that NaN stays NaN
    o.x = clamp_keep_nan(o.x, clamp); o.y = clamp_keep_nan(o.y, clamp);
    o.z = clamp_keep_nan(o.z, clamp); o.w = clamp_keep_nan(o.w, clamp);
    reinterpret_cast<float4*>(y)[row * (C / 4) + c4] = o;
    if (y_lowp) store4_bf16(y_lowp, row * (C / 4) + c4, o);  // the next projection's bf16 operand, no separate cast
  }
  if (lane == 0) {
    mean_out[row] = mean;
    rstd_out[row] = rstd;
  }
}

template <typename XT, typename RT, int CH, bool LOWP>
__global__ void __launch_bounds__(kThreads) add_layernorm_bwd_kernel(const float* __restrict__ dy,
                                                                     const void* __restrict__ dy_lowp,
                                                                     const void* __restrict__ x,
                                                                     const void* __restrict__ r,
                                                                     const float* __restrict__ gamma,
                                                                     const float* __restrict__ mean_in,
                                                                     const float* __restrict__ rstd_in,
                                                                     float* __restrict__ ds, void* __restrict__ ds_lowp,
                                                                     float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                                     long long N, int rows_per_block,
                                                                     const float* __restrict__ beta, float clamp) {
  constexpr int C = CH * 128;
  __shared__ float4 sg[kRowsPerBlock][CH * 32], sb[kRowsPerBlock][CH * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 accg[CH], accb[CH];
#pragma unroll
  for (int k = 0; k < CH; ++k) accg[k] = accb[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  const long long row0 = (long long)blockIdx.x * rows_per_block;
  const long long row1 = row0 + rows_per_block < N ? row0 + rows_per_block : N;
  for (long long row = row0 + warp; row < row1; row += kRowsPerBlock) {
    const float mean = mean_in[row], rstd = rstd_in[row];
    float4 xh[CH], g[CH];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < CH; ++k) {
      const int c4 = k * 32 + lane;
      const long long i4 = row * (C / 4) + c4;
      const float4 a = load4<XT>(x, i4), b = load4<RT>(r, i4);
      float4 d = __ldg(reinterpret_cast<const float4*>(dy) + i4);
      if (dy_lowp) {  // gradient that arrived through the bf16 copy of y (the projection fed from it)
        const float4 e = load4<__nv_bfloat16>(dy_lowp, i4);
        d.x += e.x; d.y += e.y; d.z += e.z; d.w += e.w;
      }
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + c4);
      xh[k] = make_float4((a.x + b.x - mean) * rstd, (a.y + b.y - mean) * rstd, (a.z + b.z - mean) * rstd,
                          (a.w + b.w - mean) * rstd);
      if (beta) {  // clamped forward: torch.clamp's backward passes the gradient where -clamp <= y <= clamp (false for NaN)
        const float4 bt = __ldg(reinterpret_cast<const float4*>(beta) + c4);
        const float y0 = xh[k].x * gm.x + bt.x, y1 = xh[k].y * gm.y + bt.y, y2 = xh[k].z * gm.z + bt.z, y3 = xh[k].w * gm.w + bt.w;
        d.x = (y0 >= -clamp && y0 <= clamp) ? d.x : 0.f;
        d.y = (y1 >= -clamp && y1 <= clamp) ? d.y : 0.f;
        d.z = (y2 >= -clamp && y2 <= clamp) ? d.z : 0.f;
        d.w = (y3 >= -clamp && y3 <= clamp) ? d.w : 0.f;
      }
      g[k] = make_float4(d.x * gm.x, d.y * gm.y, d.z * gm.z, d.w * gm.w);
      s1 += (g[k].x + g[k].y) + (g[k].z + g[k].w);
      s2 += (g[k].x * xh[k].x + g[k].y * xh[k].y) + (g[k].z * xh[k].z + g[k].w * xh[k].w);
      accg[k].x += d.x * xh[k].x; accg[k].y += d.y * xh[k].y; accg[k].z += d.z * xh[k].z; accg[k].w += d.w * xh[k].w;
      accb[k].x += d.x; accb[k].y += d.y; accb[k].z += d.z; accb[k].w += d.w;
    }
    const float m1 = warp_sum(s1) * (1.f / C), m2 = warp_sum(s2) * (1.f / C);
#pragma unroll
    for (int k = 0; k < CH; ++k) {
      const long long i4 = row * (C / 4) + k * 32 + lane;
      float4 o;
      o.x = rstd * (g[k].x - m1 - xh[k].x * m2);
      o.y = rstd * (g[k].y - m1 - xh[k].y * m2);
      o.z = rstd * (g[k].z - m1 - xh[k].z * m2);
      o.w = rstd * (g[k].w - m1 - xh[k].w * m2);
      reinterpret_cast<float4*>(ds)[i4] = o;
      if (LOWP) store4_bf16(ds_lowp, i4, o);
    }
  }
  // block-level reduction of the gamma / beta partials, then one fp32 atomic per channel and block
#pragma unroll
  for (int k = 0; k < CH; ++k) {
    sg[warp][k * 32 + lane] = accg[k];
    sb[warp][k * 32 + lane] = accb[k];
  }
  __syncthreads();
  for (int c4 = threadIdx.x; c4 < CH * 32; c4 += kThreads) {
    float4 tg = sg[0][c4], tb = sb[0][c4];
#pragma unroll
    for (int w = 1; w < kRowsPerBlock; ++w) {
      const float4 a = sg[w][c4], b = sb[w][c4];
      tg.x += a.x; tg.y += a.y; tg.z += a.z; tg.w += a.w;
      tb.x += b.x; tb.y += b.y; tb.z += b.z; tb.w += b.w;
    }
    atomicAdd(dgamma + c4 * 4 + 0, tg.x); atomicAdd(dgamma + c4 * 4 + 1, tg.y);
    atomicAdd(dgamma + c4 * 4 + 2, tg.z); atomicAdd(dgamma + c4 * 4 + 3, tg.w);
    atomicAdd(dbeta + c4 * 4 + 0, tb.x); atomicAdd(dbeta + c4 * 4 + 1, tb.y);
    atomicAdd(dbeta + c4 * 4 + 2, tb.z); atomicAdd(dbeta + c4 * 4 + 3, tb.w);
  }
}

template <int CH>
int launch_fwd_ch(int xd, int rd, const void* x, const void* r, const float* gamma, const float* beta, float eps, float* y,
                  void* y_lowp, float* mean, float* rstd, long long N, float clamp, cudaStream_t st) {
  const unsigned blocks = (unsigned)((N + kRowsPerBlock - 1) / kRowsPerBlock);
  using bf = __nv_bfloat16;
  if (xd == MSDA_B200_BF16 && rd == MSDA_B200_F32)
    add_layernorm_fwd_kernel<bf, float, CH><<<blocks, kThreads, 0, st>>>(x, r, gamma, beta, eps, y, y_lowp, mean, rstd, N, clamp);
  else if (xd == MSDA_B200_F32 && rd == MSDA_B200_F32)
    add_layernorm_fwd_kernel<float, float, CH><<<blocks, kThreads, 0, st>>>(x, r, gamma, beta, eps, y, y_lowp, mean, rstd, N, clamp);
  else if (xd == MSDA_B200_BF16 && rd == MSDA_B200_BF16)
    add_layernorm_fwd_kernel<bf, bf, CH><<<blocks, kThreads, 0, st>>>(x, r, gamma, beta, eps, y, y_lowp, mean, rstd, N, clamp);
  else
    add_layernorm_fwd_kernel<float, bf, CH><<<blocks, kThreads, 0, st>>>(x, r, gamma, beta, eps, y, y_lowp, mean, rstd, N, clamp);
  return launched("add_layernorm_forward");
}

template <int CH>
int launch_bwd_ch(int xd, int rd, const float* dy, const void* dy_lowp, const void* x, const void* r, const float* gamma,
                  const float* mean,
                  const float* rstd, float* ds, void* ds_lowp, float* dgamma, float* dbeta, long long N,
                  const float* beta, float clamp, cudaStream_t st) {
  // Exactly ONE wave of resident blocks: 148 SMs x what the kernel's register count lets an SM hold (3 at 80 registers).
  // The former fixed 148 x 4 ran as 1.33 waves -- a third of the time on a quarter-full GPU (ncu r02: dram 50 %).
  // Each block walks a contiguous range of rows so the gamma / beta partials stay in registers.
  using bf = __nv_bfloat16;
#define MSDA_LN_BWD_LAUNCH(KERN)                                                                                  \
  do {                                                                                                            \
    int occ = 0;                                                                                                  \
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, KERN, kThreads, 0) != cudaSuccess || occ < 1) occ = 3; \
    long long blocks = 148LL * occ;                                                                               \
    if (blocks > (N + kRowsPerBlock - 1) / kRowsPerBlock) blocks = (N + kRowsPerBlock - 1) / kRowsPerBlock;       \
    const int rows_per_block = (int)((N + blocks - 1) / blocks);                                                  \
    blocks = (N + rows_per_block - 1) / rows_per_block;                                                           \
    KERN<<<(unsigned)blocks, kThreads, 0, st>>>(dy, dy_lowp, x, r, gamma, mean, rstd, ds, ds_lowp, dgamma, dbeta, N, \
                                                rows_per_block, beta, clamp);                                     \
  } while (0)
#define MSDA_LN_BWD(XT, RT)                                                              \
  do {                                                                                   \
    if (ds_lowp) MSDA_LN_BWD_LAUNCH((add_layernorm_bwd_kernel<XT, RT, CH, true>));       \
    else MSDA_LN_BWD_LAUNCH((add_layernorm_bwd_kernel<XT, RT, CH, false>));              \
  } while (0)
  if (xd == MSDA_B200_BF16 && rd == MSDA_B200_F32) MSDA_LN_BWD(bf, float);
  else if (xd == MSDA_B200_F32 && rd == MSDA_B200_F32) MSDA_LN_BWD(float, float);
  else if (xd == MSDA_B200_BF16 && rd == MSDA_B200_BF16) MSDA_LN_BWD(bf, bf);
  else MSDA_LN_BWD(float, bf);
#undef MSDA_LN_BWD
#undef MSDA_LN_BWD_LAUNCH
  return launched("add_layernorm_backward");
}

bool bad_dtype(int d) { return d != MSDA_B200_F32 && d != MSDA_B200_BF16; }

}  // namespace

extern "C" {

// clamp: +inf = plain LayerNorm; finite = torch.clamp(y, -clamp, clamp) applied to the output (M2F:1062-1065)
static int add_layernorm_forward_impl(const void* x, int x_dtype, const void* residual, int residual_dtype,
                                      const float* gamma, const float* beta, float eps, float* y, void* y_lowp, float* mean,
                                      float* rstd, int64_t rows, int32_t channels, float clamp, void* stream) {
  if (rows < 0 || channels <= 0 || channels % 128 != 0 || channels > kMaxC)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "add_layernorm: channels must be a multiple of 128, at most 512");
  if (bad_dtype(x_dtype) || bad_dtype(residual_dtype))
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "add_layernorm: dtype must be 0 (f32) or 1 (bf16)");
  if (!(clamp > 0.f)) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "add_layernorm: clamp must be positive");
  if (rows == 0) return MSDA_B200_OK;
  if (!x || !residual || !gamma || !beta || !y || !mean || !rstd)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "add_layernorm_forward: NULL tensor pointer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (channels / 128) {
    case 1: return launch_fwd_ch<1>(x_dtype, residual_dtype, x, residual, gamma, beta, eps, y, y_lowp, mean, rstd, rows, clamp, st);
    case 2: return launch_fwd_ch<2>(x_dtype, residual_dtype, x, residual, gamma, beta, eps, y, y_lowp, mean, rstd, rows, clamp, st);
    case 4: return launch_fwd_ch<4>(x_dtype, residual_dtype, x, residual, gamma, beta, eps, y, y_lowp, mean, rstd, rows, clamp, st);
  }
  return MSDA_B200_ERR_UNSUPPORTED;
}

// beta == NULL: plain LayerNorm backward; else the backward of the clamped forward (needs beta to rebuild y)
static int add_layernorm_backward_impl(const float* grad_y, const void* grad_y_lowp, const void* x, int x_dtype,
                                       const void* residual, int residual_dtype, const float* gamma, const float* beta,
                                       float clamp, const float* mean, const float* rstd, float* grad_sum,
                                       void* grad_sum_lowp, float* grad_gamma, float* grad_beta, int64_t rows,
                                       int32_t channels, void* stream) {
  if (rows < 0 || channels <= 0 || channels % 128 != 0 || channels > kMaxC)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "add_layernorm: channels must be a multiple of 128, at most 512");
  if (bad_dtype(x_dtype) || bad_dtype(residual_dtype))
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "add_layernorm: dtype must be 0 (f32) or 1 (bf16)");
  if (!grad_gamma || !grad_beta)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "add_layernorm_backward: NULL gamma/beta gradient");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (cudaMemsetAsync(grad_gamma, 0, sizeof(float) * channels, st) != cudaSuccess) return MSDA_B200_ERR_CUDA;
  if (cudaMemsetAsync(grad_beta, 0, sizeof(float) * channels, st) != cudaSuccess) return MSDA_B200_ERR_CUDA;
  if (rows == 0) return MSDA_B200_OK;
  if (!grad_y || !x || !residual || !gamma || !mean || !rstd || !grad_sum)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "add_layernorm_backward: NULL tensor pointer");
  switch (channels / 128) {
    case 1: return launch_bwd_ch<1>(x_dtype, residual_dtype, grad_y, grad_y_lowp, x, residual, gamma, mean, rstd, grad_sum, grad_sum_lowp, grad_gamma, grad_beta, rows, beta, clamp, st);
    case 2: return launch_bwd_ch<2>(x_dtype, residual_dtype, grad_y, grad_y_lowp, x, residual, gamma, mean, rstd, grad_sum, grad_sum_lowp, grad_gamma, grad_beta, rows, beta, clamp, st);
    case 4: return launch_bwd_ch<4>(x_dtype, residual_dtype, grad_y, grad_y_lowp, x, residual, gamma, mean, rstd, grad_sum, grad_sum_lowp, grad_gamma, grad_beta, rows, beta, clamp, st);
  }
  return MSDA_B200_ERR_UNSUPPORTED;
}

int msda_b200_add_layernorm_forward(const void* x, int x_dtype, const void* residual, int residual_dtype,
                                    const float* gamma, const float* beta, float eps, float* y, void* y_lowp, float* mean,
                                    float* rstd, int64_t rows, int32_t channels, void* stream) {
  return add_layernorm_forward_impl(x, x_dtype, residual, residual_dtype, gamma, beta, eps, y, y_lowp, mean, rstd, rows,
                                    channels, INFINITY, stream);
}

int msda_b200_add_layernorm_backward(const float* grad_y, const void* grad_y_lowp, const void* x, int x_dtype, const void* residual,
                                     int residual_dtype, const float* gamma, const float* mean, const float* rstd,
                                     float* grad_sum, void* grad_sum_lowp, float* grad_gamma, float* grad_beta,
                                     int64_t rows, int32_t channels, void* stream) {
  return add_layernorm_backward_impl(grad_y, grad_y_lowp, x, x_dtype, residual, residual_dtype, gamma, nullptr, INFINITY,
                                     mean, rstd, grad_sum, grad_sum_lowp, grad_gamma, grad_beta, rows, channels, stream);
}

int msda_b200_add_layernorm_clamp_forward(const void* x, int x_dtype, const void* residual, int residual_dtype,
                                          const float* gamma, const float* beta, float eps, float clamp, float* y,
                                          void* y_lowp, float* mean, float* rstd, int64_t rows, int32_t channels,
                                          void* stream) {
  return add_layernorm_forward_impl(x, x_dtype, residual, residual_dtype, gamma, beta, eps, y, y_lowp, mean, rstd, rows,
                                    channels, clamp, stream);
}

int msda_b200_add_layernorm_clamp_backward(const float* grad_y, const void* grad_y_lowp, const void* x, int x_dtype,
                                           const void* residual, int residual_dtype, const float* gamma, const float* beta,
                                           float clamp, const float* mean, const float* rstd, float* grad_sum,
                                           void* grad_sum_lowp, float* grad_gamma, float* grad_beta, int64_t rows,
                                           int32_t channels, void* stream) {
  if (!beta) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "add_layernorm_clamp_backward: beta is NULL");
  if (!(clamp > 0.f)) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "add_layernorm: clamp must be positive");
  return add_layernorm_backward_impl(grad_y, grad_y_lowp, x, x_dtype, residual, residual_dtype, gamma, beta, clamp, mean,
                                     rstd, grad_sum, grad_sum_lowp, grad_gamma, grad_beta, rows, channels, stream);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// Column sum of a (rows x cols) matrix into fp32: the bias gradient of a projection (grad_bias = sum_rows grad_out).
// torch's generic reduce kernel needs ~110 us per projection at config 2 (172 032 rows); this one streams the
// matrix once with 16-byte loads. cols must be a multiple of 8 (bf16) / 4 (fp32) and at most 2048.
// ---------------------------------------------------------------------------------------------------------------
namespace {

template <typename T>
struct ColVec;
template <>
struct ColVec<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void load(const void* base, long long idx, float (&f)[4]) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(base) + idx);
    f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
  }
  static __device__ __forceinline__ void store(void* base, long long idx, const float (&f)[4]) {
    reinterpret_cast<float4*>(base)[idx] = make_float4(f[0], f[1], f[2], f[3]);
  }
};
template <>
struct ColVec<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void load(const void* base, long long idx, float (&f)[8]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(base) + idx);
    f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
    f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
    f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xffff0000u);
    f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xffff0000u);
  }
  // exact for values that came out of load() (bfloat16-representable): the low 16 bits are zero
  static __device__ __forceinline__ void store(void* base, long long idx, const float (&f)[8]) {
    uint4 v;
    v.x = (__float_as_uint(f[0]) >> 16) | (__float_as_uint(f[1]) & 0xffff0000u);
    v.y = (__float_as_uint(f[2]) >> 16) | (__float_as_uint(f[3]) & 0xffff0000u);
    v.z = (__float_as_uint(f[4]) >> 16) | (__float_as_uint(f[5]) & 0xffff0000u);
    v.w = (__float_as_uint(f[6]) >> 16) | (__float_as_uint(f[7]) & 0xffff0000u);
    reinterpret_cast<uint4*>(base)[idx] = v;
  }
};

// block = (cv column vectors) x (rl row lanes); every thread walks rows r0 + ry, r0 + ry + rl, ...
// RELU: m is the gradient that arrived at relu(z), y = relu(z) the saved activation; the kernel also writes the masked
// gradient (aten threshold_backward: grad where y > 0, else 0) to gm -- the FFN's ReLU backward and the bias gradient of
// fc1 (M2F:1052-1053) in one pass over the (rows x 1024) matrix instead of a mask kernel and a second read.
template <typename T, bool RELU>
__global__ void __launch_bounds__(256) colsum_kernel(const void* __restrict__ m, float* __restrict__ out, long long rows,
                                                     int cv /* cols / N */, int rl, int rows_per_block,
                                                     const void* __restrict__ y = nullptr, void* __restrict__ gm = nullptr) {
  constexpr int N = ColVec<T>::N;
  extern __shared__ float s_part[];  // [rl][cv * N]
  const int cx = threadIdx.x % cv, ry = threadIdx.x / cv;
  float acc[N];
#pragma unroll
  for (int j = 0; j < N; ++j) acc[j] = 0.f;
  if (ry < rl) {
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    const long long r1 = r0 + rows_per_block < rows ? r0 + rows_per_block : rows;
    for (long long r = r0 + ry; r < r1; r += rl) {
      float f[N];
      ColVec<T>::load(m, r * cv + cx, f);
      if (RELU) {
        float a[N];
        ColVec<T>::load(y, r * cv + cx, a);
#pragma unroll
        for (int j = 0; j < N; ++j) f[j] = a[j] > 0.f ? f[j] : 0.f;
        ColVec<T>::store(gm, r * cv + cx, f);
      }
#pragma unroll
      for (int j = 0; j < N; ++j) acc[j] += f[j];
    }
#pragma unroll
    for (int j = 0; j < N; ++j) s_part[(ry * cv + cx) * N + j] = acc[j];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < cv * N; c += blockDim.x) {
    float t = 0.f;
    for (int y = 0; y < rl; ++y) t += s_part[y * cv * N + c];
    atomicAdd(out + c, t);
  }
}

}  // namespace

static int column_sum_impl(const void* matrix, int dtype, float* out, int64_t rows, int32_t cols, const void* y, void* gm,
                           void* stream);

extern "C" int msda_b200_column_sum(const void* matrix, int dtype, float* out, int64_t rows, int32_t cols, void* stream) {
  return column_sum_impl(matrix, dtype, out, rows, cols, nullptr, nullptr, stream);
}

extern "C" int msda_b200_relu_backward_column_sum(const void* grad_y, const void* y, int dtype, void* grad_masked,
                                                  float* column_sum, int64_t rows, int32_t cols, void* stream) {
  if (rows > 0 && (!y || !grad_masked))
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "relu_backward_column_sum: NULL tensor pointer");
  return column_sum_impl(grad_y, dtype, column_sum, rows, cols, y ? y : grad_y, grad_masked ? grad_masked : (void*)1, stream);
}

static int column_sum_impl(const void* matrix, int dtype, float* out, int64_t rows, int32_t cols, const void* y, void* gm,
                           void* stream) {
  if (bad_dtype(dtype)) return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "column_sum: dtype must be 0 (f32) or 1 (bf16)");
  const int n = dtype == MSDA_B200_BF16 ? 8 : 4;
  if (rows < 0 || cols <= 0 || cols % n != 0 || cols > 2048)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "column_sum: cols must be a multiple of 8 (bf16) / 4 (f32), at most 2048");
  if (!out) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "column_sum: NULL output");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (cudaMemsetAsync(out, 0, sizeof(float) * cols, st) != cudaSuccess)
    return msda_b200_internal_fail(MSDA_B200_ERR_CUDA, "column_sum: memset failed");
  if (rows == 0) return MSDA_B200_OK;
  if (!matrix) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "column_sum: NULL matrix");
  const int cv = cols / n;  // 16-byte column vectors per row
  if (cv > 256) return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "column_sum: too many columns");
  const int rl = 256 / cv;  // rows walked in parallel by one block
  const int threads = 256;
  long long blocks = 148 * 8;
  const long long min_rows = (long long)rl * 4;
  if (blocks * min_rows > rows) blocks = (rows + min_rows - 1) / min_rows;
  if (blocks < 1) blocks = 1;
  const int rows_per_block = (int)((rows + blocks - 1) / blocks);
  blocks = (rows + rows_per_block - 1) / rows_per_block;
  const size_t smem = sizeof(float) * (size_t)rl * cols;
  if (gm) {
    if (dtype == MSDA_B200_BF16)
      colsum_kernel<__nv_bfloat16, true><<<(unsigned)blocks, threads, smem, st>>>(matrix, out, rows, cv, rl, rows_per_block, y, gm);
    else
      colsum_kernel<float, true><<<(unsigned)blocks, threads, smem, st>>>(matrix, out, rows, cv, rl, rows_per_block, y, gm);
  } else if (dtype == MSDA_B200_BF16)
    colsum_kernel<__nv_bfloat16, false><<<(unsigned)blocks, threads, smem, st>>>(matrix, out, rows, cv, rl, rows_per_block);
  else
    colsum_kernel<float, false><<<(unsigned)blocks, threads, smem, st>>>(matrix, out, rows, cv, rl, rows_per_block);
  return launched("column_sum");
}

// ---------------------------------------------------------------------------------------------------------------
// Query / value operands of the attention module under bf16 autocast (M2F:936-937, 947, 952-956):
//   query = bfloat16(hidden + pos)   -- what the sampling_offsets / attention_weights projections read
//   value = bfloat16(hidden)         -- what value_proj reads
// Stock PyTorch runs an fp32 add (read 2, write 1 tensor) and two cast kernels (read 1, write 1/2 each); one pass here
// reads hidden and pos once and writes the two bf16 operands. Backward: grad_hidden = f32(grad_query) + f32(grad_value),
// grad_pos = f32(grad_query), again one pass instead of two casts and an add. Same roundings as the stock sequence
// (fp32 add, one round-to-nearest-even to bfloat16; bfloat16 -> fp32 is exact).
// ---------------------------------------------------------------------------------------------------------------
namespace {

__device__ __forceinline__ uint4 pack8_bf16(const float4& a, const float4& b) {
  const __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
  const __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y), p3 = __floats2bfloat162_rn(b.z, b.w);
  uint4 o;
  o.x = *reinterpret_cast<const unsigned*>(&p0); o.y = *reinterpret_cast<const unsigned*>(&p1);
  o.z = *reinterpret_cast<const unsigned*>(&p2); o.w = *reinterpret_cast<const unsigned*>(&p3);
  return o;
}
__device__ __forceinline__ void unpack8_bf16(const uint4& v, float4& a, float4& b) {
  a = make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u), __uint_as_float(v.y << 16),
                  __uint_as_float(v.y & 0xffff0000u));
  b = make_float4(__uint_as_float(v.z << 16), __uint_as_float(v.z & 0xffff0000u), __uint_as_float(v.w << 16),
                  __uint_as_float(v.w & 0xffff0000u));
}

__global__ void __launch_bounds__(256) qv_cast_fwd_kernel(const float4* __restrict__ hidden, const float4* __restrict__ pos,
                                                          uint4* __restrict__ query, uint4* __restrict__ value,
                                                          long long n8) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const float4 h0 = __ldg(hidden + 2 * i), h1 = __ldg(hidden + 2 * i + 1);
    const float4 p0 = __ldg(pos + 2 * i), p1 = __ldg(pos + 2 * i + 1);
    value[i] = pack8_bf16(h0, h1);
    query[i] = pack8_bf16(make_float4(h0.x + p0.x, h0.y + p0.y, h0.z + p0.z, h0.w + p0.w),
                          make_float4(h1.x + p1.x, h1.y + p1.y, h1.z + p1.z, h1.w + p1.w));
  }
}

// grad_query / grad_value may be NULL (no gradient arrived through that operand): treated as zero
__global__ void __launch_bounds__(256) qv_cast_bwd_kernel(const uint4* __restrict__ grad_query,
                                                          const uint4* __restrict__ grad_value,
                                                          float4* __restrict__ grad_hidden, float4* __restrict__ grad_pos,
                                                          long long n8) {
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float4 q0 = z, q1 = z, v0 = z, v1 = z;
    if (grad_query) unpack8_bf16(__ldg(grad_query + i), q0, q1);
    if (grad_value) unpack8_bf16(__ldg(grad_value + i), v0, v1);
    grad_hidden[2 * i] = make_float4(q0.x + v0.x, q0.y + v0.y, q0.z + v0.z, q0.w + v0.w);
    grad_hidden[2 * i + 1] = make_float4(q1.x + v1.x, q1.y + v1.y, q1.z + v1.z, q1.w + v1.w);
    if (grad_pos) {
      grad_pos[2 * i] = q0;
      grad_pos[2 * i + 1] = q1;
    }
  }
}

int qv_blocks(long long n8) {
  const long long want = (n8 + 255) / 256;
  return (int)(want < 148 * 16 ? (want < 1 ? 1 : want) : 148 * 16);
}

}  // namespace

extern "C" int msda_b200_query_value_cast_forward(const float* hidden, const float* pos, void* query_bf16, void* value_bf16,
                                                  int64_t elements, void* stream) {
  if (elements < 0 || elements % 8 != 0)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "query_value_cast: element count must be a multiple of 8");
  if (elements == 0) return MSDA_B200_OK;
  if (!hidden || !pos || !query_bf16 || !value_bf16)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "query_value_cast_forward: NULL tensor pointer");
  const long long n8 = elements / 8;
  qv_cast_fwd_kernel<<<qv_blocks(n8), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(hidden), reinterpret_cast<const float4*>(pos), reinterpret_cast<uint4*>(query_bf16),
      reinterpret_cast<uint4*>(value_bf16), n8);
  return launched("query_value_cast_forward");
}

extern "C" int msda_b200_query_value_cast_backward(const void* grad_query_bf16, const void* grad_value_bf16,
                                                   float* grad_hidden, float* grad_pos, int64_t elements, void* stream) {
  if (elements < 0 || elements % 8 != 0)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "query_value_cast: element count must be a multiple of 8");
  if (elements == 0) return MSDA_B200_OK;
  if (!grad_hidden) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "query_value_cast_backward: grad_hidden is NULL");
  const long long n8 = elements / 8;
  qv_cast_bwd_kernel<<<qv_blocks(n8), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const uint4*>(grad_query_bf16), reinterpret_cast<const uint4*>(grad_value_bf16),
      reinterpret_cast<float4*>(grad_hidden), reinterpret_cast<float4*>(grad_pos), n8);
  return launched("query_value_cast_backward");
}
