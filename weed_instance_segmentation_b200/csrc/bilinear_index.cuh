// Index arithmetic of ATen's upsample_bilinear2d (area_pixel_compute_scale / area_pixel_compute_source_index) for
// F.interpolate(x, size=..., mode="bilinear", align_corners=False) without a scale factor:
//   scale = (float)in / out,  src = max(scale * (dst + 0.5) - 0.5, 0),  i0 = (int)src,  i1 = i0 + (i0 < in - 1),
//   l1 = src - i0,  l0 = 1 - l1.
// Shared by the resize backward (resize_bilinear.cu) and the instance post-processing (postprocess.cu).
#pragma once

struct BilinearSrc {
  int i0, i1;
  float l0, l1;
};

__device__ __forceinline__ BilinearSrc bilinear_source_index(float scale, int dst, int in) {
  const float s = fmaxf(scale * (dst + 0.5f) - 0.5f, 0.f);
  BilinearSrc r;
  r.i0 = (int)s;
  r.i1 = r.i0 + (r.i0 < in - 1 ? 1 : 0);
  r.l1 = s - r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}
