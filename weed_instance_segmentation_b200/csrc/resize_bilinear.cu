// Deterministic backward of bilinear resizing: the adjoint of
//   F.interpolate(x, size=(Ho, Wo), mode="bilinear", align_corners=False)       (no scale factor)
// which the pixel decoder's FPN tail uses to upsample the finest encoder level (M2F:1360-1371). torch's CUDA backward
// scatters with float atomics and raises under torch.use_deterministic_algorithms; this one gathers instead: one
// thread per grad_in element sums every output pixel that read it, in a fixed order (rows, then columns), in fp32,
// and writes the element once -- no zero-fill, no atomics. Zero weights are not skipped, so a non-finite grad_out
// value reaches the same grad_in elements as in torch.
//
// Index arithmetic of ATen's upsample_bilinear2d (area_pixel_compute_scale / area_pixel_compute_source_index):
//   scale = (float)in / out,  src = max(scale * (dst + 0.5) - 0.5, 0),  i0 = (int)src,  i1 = i0 + (i0 < in - 1),
//   l1 = src - i0,  l0 = 1 - l1.
// i0 is non-decreasing in dst, so the outputs that read input index i (i0 == i or i1 == i, i.e. i0 in {i - 1, i}) are
// one contiguous range; it is estimated from the inverse map with a margin and then settled with the formula above.
#include <cuda_runtime.h>

#include <cstdint>

#include "msda_b200.h"

extern "C" int msda_b200_internal_fail(int code, const char* msg);  // msda_b200.cu: sets msda_b200_last_error()
extern "C" void msda_b200_internal_count_launch(void);               // msda_b200.cu: launch counter

namespace {

constexpr int kRbThreads = 256;

struct Src {
  int i0, i1;
  float l0, l1;
};

__device__ __forceinline__ Src source_index(float scale, int dst, int in) {
  const float s = fmaxf(scale * (dst + 0.5f) - 0.5f, 0.f);
  Src r;
  r.i0 = (int)s;
  r.i1 = r.i0 + (r.i0 < in - 1 ? 1 : 0);
  r.l1 = s - r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}

// Weight with which output index `dst` reads input index i (both taps when i0 == i1 at the last index).
__device__ __forceinline__ float tap_weight(const Src& s, int i) {
  return (s.i0 == i ? s.l0 : 0.f) + (s.i1 == i ? s.l1 : 0.f);
}

// [lo, hi] of the output indices that read input index i.
__device__ __forceinline__ int2 output_range(float scale, int i, int in, int out) {
  const float inv = 1.f / scale;
  int lo = max((int)floorf((i - 0.5f) * inv - 0.5f) - 2, 0);
  int hi = min((int)ceilf((i + 1.5f) * inv - 0.5f) + 2, out - 1);
  while (lo > 0 && source_index(scale, lo - 1, in).i0 >= i - 1) --lo;
  while (lo <= hi && source_index(scale, lo, in).i0 < i - 1) ++lo;
  while (hi + 1 < out && source_index(scale, hi + 1, in).i0 <= i) ++hi;
  while (hi >= lo && source_index(scale, hi, in).i0 > i) --hi;
  return make_int2(lo, hi);
}

__global__ void __launch_bounds__(kRbThreads)
resize_bilinear_bwd_kernel(const float* __restrict__ grad_out, float* __restrict__ grad_in, long long total, int Hi,
                           int Wi, int Ho, int Wo, float scale_h, float scale_w) {
  const long long t = blockIdx.x * (long long)kRbThreads + threadIdx.x;
  if (t >= total) return;
  const int x = (int)(t % Wi);
  const int y = (int)((t / Wi) % Hi);
  const long long nc = t / ((long long)Wi * Hi);
  const int2 ry = output_range(scale_h, y, Hi, Ho), rx = output_range(scale_w, x, Wi, Wo);
  const float* go = grad_out + nc * Ho * Wo;
  float acc = 0.f;
  for (int oy = ry.x; oy <= ry.y; ++oy) {
    const float wy = tap_weight(source_index(scale_h, oy, Hi), y);
    for (int ox = rx.x; ox <= rx.y; ++ox) {
      const float wx = tap_weight(source_index(scale_w, ox, Wi), x);
      acc = fmaf(__ldg(go + (long long)oy * Wo + ox), wy * wx, acc);
    }
  }
  grad_in[t] = acc;
}

}  // namespace

extern "C" int msda_b200_resize_bilinear_backward(const float* grad_out, float* grad_in, int64_t NC, int32_t Hi,
                                                  int32_t Wi, int32_t Ho, int32_t Wo, void* stream) {
  if (NC < 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "resize_bilinear: negative count or empty extent");
  if (NC == 0) return MSDA_B200_OK;
  if (!grad_out || !grad_in) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "resize_bilinear: NULL pointer");
  const long long plane = (long long)Hi * Wi;
  if (NC > 0x7fffffffll * kRbThreads / plane)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "resize_bilinear: grid too large");
  const long long total = NC * plane;
  const long long blocks = (total + kRbThreads - 1) / kRbThreads;
  resize_bilinear_bwd_kernel<<<(unsigned)blocks, kRbThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      grad_out, grad_in, total, Hi, Wi, Ho, Wo, (float)Hi / Ho, (float)Wi / Wo);
  msda_b200_internal_count_launch();
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MSDA_B200_OK : msda_b200_internal_fail(MSDA_B200_ERR_CUDA, cudaGetErrorString(e));
}
