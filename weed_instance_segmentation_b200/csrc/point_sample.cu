// Batched bilinear point sampling for the loss / matcher path (SURVEY.md section 8(f) rank 4).
//
// The reference samples masks at random points through `sample_point` (M2F:245-274: grid_sample, bilinear,
// zeros padding, align_corners=False) once per image in the Hungarian matcher (M2F:455-474) and three times per
// decoder layer in the mask loss (M2F:619-631, :718-737), each call on freshly gathered / padded copies of the masks.
// Here one launch samples any number of ROWS: a row is one 2-D plane (a pointer, so planes stay where they are --
// no gather, no padding, no dtype upcast), its extent, and the row of the coordinate table it reads (several planes
// may share one point set, as in the matcher).  The backward scatters into fp32 planes with atomics; its deterministic
// form (msda_b200_point_sample_backward_det) sorts the contributions by destination pixel and sums each pixel in a
// fixed order instead.
//
// Same bilinear primitive as the MSDeformAttn kernels: pix = ((2c - 1 + 1) * n - 1) / 2 evaluated in ATen's order
// without FMA contraction, corners outside the plane contribute zero, NaN coordinates contribute zero.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <climits>
#include <cstdint>

#include "msda_b200.h"
#include "msda_bwd_det.cuh"

extern "C" int msda_b200_internal_fail(int code, const char* msg);  // msda_b200.cu: sets msda_b200_last_error()
extern "C" void msda_b200_internal_count_launch(void);               // msda_b200.cu: launch counter

namespace {

constexpr int kPsThreads = 256;

struct Corner {
  int i0;        // floor(pix)
  float w0, w1;  // weights of i0 and i0 + 1 (zero when outside [0, n))
};

__device__ __forceinline__ Corner corner_setup(float c, int n) {
  const float g = __fadd_rn(__fmul_rn(2.f, c), -1.f);
  const float pix = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(g, 1.f), (float)n), -1.f), 0.5f);
  Corner r;
  const bool ok = (pix > -2.f) && (pix < (float)(n + 1));  // false for NaN
  const float fl = floorf(pix);
  r.i0 = ok ? __float2int_rd(pix) : -4;
  const float l = pix - fl;
  r.w0 = (r.i0 >= 0 && r.i0 < n) ? 1.f - l : 0.f;
  r.w1 = (r.i0 + 1 >= 0 && r.i0 + 1 < n) ? l : 0.f;
  return r;
}

__device__ __forceinline__ float load_plane(const void* plane, int dtype, long long idx) {
  if (dtype == MSDA_B200_U8) return (float)__ldg(reinterpret_cast<const unsigned char*>(plane) + idx);
  return dtype == MSDA_B200_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(plane)[idx])
                                 : __ldg(reinterpret_cast<const float*>(plane) + idx);
}

__global__ void __launch_bounds__(kPsThreads)
point_sample_fwd_kernel(const void* const* __restrict__ planes, const msda_b200_ps_row* __restrict__ rows,
                        const float2* __restrict__ coords, float* __restrict__ out, int K, unsigned chunks) {
  // 1-D grid, row-major: the blocks of one row are scheduled together, so its plane is fetched from DRAM once and
  // then served by L2 (with the row on the fast grid axis every resident block reads a different plane: measured
  // 24.9 GB of DRAM reads and 14 % L2 hits for the 8 700-row matcher launch, profiles/r01_notes.md)
  const long long r = blockIdx.x / chunks;
  const int k = (int)(blockIdx.x % chunks) * kPsThreads + threadIdx.x;
  if (k >= K) return;
  const msda_b200_ps_row row = rows[r];
  const void* plane = planes[r];
  const float2 c = __ldg(coords + (long long)row.coord_row * K + k);
  const Corner cx = corner_setup(c.x, row.w), cy = corner_setup(c.y, row.h);
  float acc = 0.f;
  // order of accumulation as in ATen's kernel: nw, ne, sw, se
  const long long base = (long long)cy.i0 * row.w + cx.i0;
  if (cy.w0 != 0.f) {
    if (cx.w0 != 0.f) acc = fmaf(load_plane(plane, row.dtype, base), cx.w0 * cy.w0, acc);
    if (cx.w1 != 0.f) acc = fmaf(load_plane(plane, row.dtype, base + 1), cx.w1 * cy.w0, acc);
  }
  if (cy.w1 != 0.f) {
    if (cx.w0 != 0.f) acc = fmaf(load_plane(plane, row.dtype, base + row.w), cx.w0 * cy.w1, acc);
    if (cx.w1 != 0.f) acc = fmaf(load_plane(plane, row.dtype, base + row.w + 1), cx.w1 * cy.w1, acc);
  }
  out[r * K + k] = acc;
}

__global__ void __launch_bounds__(kPsThreads)
point_sample_bwd_kernel(float* const* __restrict__ grad_planes, const msda_b200_ps_row* __restrict__ rows,
                        const float2* __restrict__ coords, const float* __restrict__ grad_out, int K, unsigned chunks) {
  const long long r = blockIdx.x / chunks;
  const int k = (int)(blockIdx.x % chunks) * kPsThreads + threadIdx.x;
  if (k >= K) return;
  float* gp = grad_planes[r];
  if (gp == nullptr) return;
  const msda_b200_ps_row row = rows[r];
  const float2 c = __ldg(coords + (long long)row.coord_row * K + k);
  const float g = grad_out[r * K + k];
  const Corner cx = corner_setup(c.x, row.w), cy = corner_setup(c.y, row.h);
  const long long base = (long long)cy.i0 * row.w + cx.i0;
  if (cy.w0 != 0.f) {
    if (cx.w0 != 0.f) atomicAdd(gp + base, g * (cx.w0 * cy.w0));
    if (cx.w1 != 0.f) atomicAdd(gp + base + 1, g * (cx.w1 * cy.w0));
  }
  if (cy.w1 != 0.f) {
    if (cx.w0 != 0.f) atomicAdd(gp + base + row.w, g * (cx.w0 * cy.w1));
    if (cx.w1 != 0.f) atomicAdd(gp + base + row.w + 1, g * (cx.w1 * cy.w1));
  }
}

// Deterministic backward, step 1: the contributions point_sample_bwd_kernel adds, as records (msda_bwd_det.cuh) at
// index 4 * (r*K + k) + corner (corners nw, ne, sw, se):
//   key     key_base[r] + pixel, or `keys` for a corner with zero weight, outside the plane or with a NaN coordinate
//           (and for a row without a gradient plane, or a key outside [0, keys))
//   payload r << 32 | bits of the contribution g * (wx * wy) (float32)
__global__ void __launch_bounds__(kPsThreads)
point_sample_bwd_det_records_kernel(float* const* __restrict__ grad_planes, const msda_b200_ps_row* __restrict__ rows,
                                    const int64_t* __restrict__ key_base, long long keys,
                                    const float2* __restrict__ coords, const float* __restrict__ grad_out, int K,
                                    unsigned chunks, unsigned* __restrict__ rec_keys,
                                    unsigned long long* __restrict__ rec_vals) {
  const long long r = blockIdx.x / chunks;
  const int k = (int)(blockIdx.x % chunks) * kPsThreads + threadIdx.x;
  if (k >= K) return;
  const msda_b200_ps_row row = rows[r];
  const float2 c = __ldg(coords + (long long)row.coord_row * K + k);
  const float g = grad_out[r * K + k];
  const Corner cx = corner_setup(c.x, row.w), cy = corner_setup(c.y, row.h);
  const long long base = (long long)cy.i0 * row.w + cx.i0;
  const long long kb = grad_planes[r] != nullptr ? key_base[r] : -1;
  const float w[4] = {cx.w0 * cy.w0, cx.w1 * cy.w0, cx.w0 * cy.w1, cx.w1 * cy.w1};
  const long long pix[4] = {base, base + 1, base + row.w, base + row.w + 1};
  const long long out = 4 * (r * K + k);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const long long key = kb + pix[j];
    const bool live = kb >= 0 && w[j] != 0.f && key >= 0 && key < keys;
    rec_keys[out + j] = live ? (unsigned)key : (unsigned)keys;
    rec_vals[out + j] = (unsigned long long)r << 32 | __float_as_uint(live ? g * w[j] : 0.f);
  }
}

// Step 3, after the sort: the thread at the start of each run of equal keys sums the run in sorted order in fp32 and
// adds the sum to its pixel with one read-modify-write. A run holds every contribution to one pixel, so each pixel has
// one writer; a long run (many points on a tiny plane) is walked by its one thread.
__global__ void __launch_bounds__(kPsThreads)
point_sample_bwd_det_sum_kernel(float* const* __restrict__ grad_planes, const int64_t* __restrict__ key_base,
                                const unsigned* __restrict__ rec_keys, const unsigned long long* __restrict__ rec_vals,
                                int n, unsigned sentinel) {
  const int i = blockIdx.x * kPsThreads + threadIdx.x;
  if (i >= n) return;
  const unsigned key = rec_keys[i];
  if (key == sentinel || (i > 0 && rec_keys[i - 1] == key)) return;
  const unsigned long long first = rec_vals[i];
  float acc = __uint_as_float((unsigned)first);
  for (int j = i + 1; j < n && rec_keys[j] == key; ++j) acc += __uint_as_float((unsigned)rec_vals[j]);
  const long long r = (long long)(first >> 32);
  grad_planes[r][key - key_base[r]] += acc;
}

int check(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return MSDA_B200_OK;
  msda_b200_internal_fail(MSDA_B200_ERR_CUDA, cudaGetErrorString(e));
  (void)what;
  return MSDA_B200_ERR_CUDA;
}

int check_args(const void* a, const void* b, const void* c, const void* d, int64_t R, int32_t K) {
  if (R < 0 || K < 0) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "point_sample: negative row / point count");
  if (R > 0x7fffffffll) return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "point_sample: more than 2^31-1 rows");
  if (R != 0 && K != 0 && (!a || !b || !c || !d))
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "point_sample: NULL pointer");
  return MSDA_B200_OK;
}

// The deterministic backward's arguments, checked before anything touches the device; *lay is its workspace layout.
int check_det_args(const void* a, const void* b, const void* c, const void* d, const void* e, int64_t keys, int64_t R,
                   int32_t K, DetLayout* lay) {
  if (int rc = check_args(a, b, c, d, R, K)) return rc;
  if (keys < 0) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "point_sample: negative key count");
  if (R != 0 && K != 0 && !e) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "point_sample: NULL pointer");
  if (R * (long long)K > INT_MAX / 4)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED,
                                   "point_sample: deterministic backward of more than 2^31 - 1 records (4 per point)");
  if (keys >= 0xffffffffll)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED,
                                   "point_sample: deterministic backward of 2^32 - 1 or more destination pixels");
  *lay = det_sort_layout(4 * R * (long long)K, keys, false);
  return MSDA_B200_OK;
}

}  // namespace

extern "C" int msda_b200_point_sample_forward(const void* const* planes, const msda_b200_ps_row* rows, const float* coords,
                                              float* out, int64_t R, int32_t K, void* stream) {
  if (int rc = check_args(planes, rows, coords, out, R, K)) return rc;
  if (R == 0 || K == 0) return MSDA_B200_OK;
  const unsigned chunks = (unsigned)((K + kPsThreads - 1) / kPsThreads);
  if (R * (long long)chunks > 0x7fffffffll)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "point_sample: rows x points exceeds the grid limit");
  point_sample_fwd_kernel<<<(unsigned)(R * chunks), kPsThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      planes, rows, reinterpret_cast<const float2*>(coords), out, K, chunks);
  msda_b200_internal_count_launch();
  return check("point_sample_forward");
}

extern "C" int msda_b200_point_sample_backward(float* const* grad_planes, const msda_b200_ps_row* rows,
                                               const float* coords, const float* grad_out, int64_t R, int32_t K,
                                               void* stream) {
  if (int rc = check_args(grad_planes, rows, coords, grad_out, R, K)) return rc;
  if (R == 0 || K == 0) return MSDA_B200_OK;
  const unsigned chunks = (unsigned)((K + kPsThreads - 1) / kPsThreads);
  if (R * (long long)chunks > 0x7fffffffll)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "point_sample: rows x points exceeds the grid limit");
  point_sample_bwd_kernel<<<(unsigned)(R * chunks), kPsThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      grad_planes, rows, reinterpret_cast<const float2*>(coords), grad_out, K, chunks);
  msda_b200_internal_count_launch();
  return check("point_sample_backward");
}

extern "C" size_t msda_b200_point_sample_backward_det_workspace_bytes(int64_t R, int32_t K, int64_t keys) {
  const int p = 1;  // any non-NULL pointer: only the sizes are checked here
  DetLayout lay;
  size_t sort = 0;
  if (check_det_args(&p, &p, &p, &p, &p, keys, R, K, &lay) || msda_b200_internal_det_sort_bytes(&lay, &sort)) return 0;
  return lay.sort_off + sort;
}

extern "C" int msda_b200_point_sample_backward_det(float* const* grad_planes, const msda_b200_ps_row* rows,
                                                   const int64_t* key_base, int64_t keys, const float* coords,
                                                   const float* grad_out, int64_t R, int32_t K, void* workspace,
                                                   size_t workspace_bytes, void* stream) {
  DetLayout lay;
  if (int rc = check_det_args(grad_planes, rows, coords, grad_out, key_base, keys, R, K, &lay)) return rc;
  if (R == 0 || K == 0) return MSDA_B200_OK;
  const unsigned chunks = (unsigned)((K + kPsThreads - 1) / kPsThreads);
  if (R * (long long)chunks > 0x7fffffffll)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "point_sample: rows x points exceeds the grid limit");
  size_t sort = 0;
  if (int rc = msda_b200_internal_det_sort_bytes(&lay, &sort)) return rc;
  if (!workspace || workspace_bytes < lay.sort_off + sort)
    return msda_b200_internal_fail(MSDA_B200_ERR_WORKSPACE, "point_sample: deterministic backward workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  point_sample_bwd_det_records_kernel<<<(unsigned)(R * chunks), kPsThreads, 0, st>>>(
      grad_planes, rows, key_base, keys, reinterpret_cast<const float2*>(coords),
      grad_out, K, chunks, reinterpret_cast<unsigned*>(ws + lay.keys_off[0]),
      reinterpret_cast<unsigned long long*>(ws + lay.vals_off[0]));
  msda_b200_internal_count_launch();
  if (int rc = check("point_sample_backward_det")) return rc;
  const unsigned* sorted_keys = nullptr;
  const unsigned long long* sorted_vals = nullptr;
  if (int rc = msda_b200_internal_det_sort(&lay, workspace, &sorted_keys, &sorted_vals, st)) return rc;
  const int n = (int)lay.records;
  point_sample_bwd_det_sum_kernel<<<(n + kPsThreads - 1) / kPsThreads, kPsThreads, 0, st>>>(
      grad_planes, key_base, sorted_keys, sorted_vals, n, (unsigned)keys);
  msda_b200_internal_count_launch();
  return check("point_sample_backward_det");
}
