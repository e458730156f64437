// msda_bwd_det.cu -- grad_value of the deterministic backward (MSDA_B200_FLAG_DETERMINISTIC).
//
// msda_bwd_kernel<ACC = 2> (msda_b200.cu) has written four records per sample in sample order (layout:
// msda_bwd_det.cuh). Here they are
//   1. sorted by key with CUB's stable radix sort over the key's bits: each (b, row, h) bucket is then a contiguous
//      run of records in sample order -- an order fixed by the inputs, not by scheduling;
//   2. turned into [begin, end) per bucket: the thread on each run boundary writes it (one writer per word);
//   3. pulled: LPP lanes per bucket walk its run and sum weight * grad_out[b, q, h, :] in fp32 registers, then write
//      the grad_value row once in its dtype. Empty buckets (and rows outside every level) get 0.
// Every floating-point sum is done by one thread in a fixed order, so equal inputs give equal bits.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <climits>
#include <cub/device/device_radix_sort.cuh>

#include "msda_b200.h"
#include "internal.h"
#include "msda_bwd_det.cuh"

namespace {

#include "msda_common.cuh"

constexpr int kDetNT = 256;

__global__ void __launch_bounds__(kDetNT) msda_bwd_det_ranges_kernel(const unsigned* __restrict__ keys, int n,
                                                                    unsigned sentinel, uint2* __restrict__ ranges) {
  const int i = blockIdx.x * kDetNT + threadIdx.x;
  if (i >= n) return;
  const unsigned k = keys[i];
  if (k == sentinel) return;
  if (i == 0 || keys[i - 1] != k) ranges[k].x = (unsigned)i;
  if (i == n - 1 || keys[i + 1] != k) ranges[k].y = (unsigned)i + 1;
}

template <typename VT, int D>
__global__ void __launch_bounds__(kDetNT) msda_bwd_det_pull_kernel(const uint2* __restrict__ ranges,
                                                                  const unsigned long long* __restrict__ vals,
                                                                  const uint4* __restrict__ grad_out,
                                                                  uint4* __restrict__ grad_value, long long buckets,
                                                                  int S, int Q, int H) {
  constexpr int VEC = Vec16<VT>::N;
  constexpr int LPP = D / VEC;
  const long long t = blockIdx.x * (long long)kDetNT + threadIdx.x;
  const long long k = t / LPP;
  const int c = (int)(t - k * LPP);
  if (k >= buckets) return;
  const int h = (int)(k % H);
  const long long b = k / ((long long)S * H);
  const uint2 r = ranges[k];
  const uint4* go = grad_out + (b * Q * H + h) * LPP + c;
  const long long q_stride = (long long)H * LPP;
  float acc[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
#pragma unroll 4
  for (unsigned i = r.x; i < r.y; ++i) {
    const unsigned long long rec = __ldg(vals + i);
    const float w = __uint_as_float((unsigned)rec);
    float g[VEC];
    Vec16<VT>::unpack(ldg16(go + (long long)(rec >> 32) * q_stride), g);
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] = fmaf(w, g[j], acc[j]);
  }
  grad_value[k * LPP + c] = Vec16<VT>::pack(acc);
}

int check_supported(const DetLayout& lay) {
  if (lay.records > INT_MAX)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED,
                                   "deterministic backward: more than 2^31 - 1 records (4 per sample)");
  if (lay.keys > 0xffffffffll)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED,
                                   "deterministic backward: B*S*H does not fit a 32-bit sort key");
  return MSDA_B200_OK;
}

template <typename VT, int D>
int launch_pull(const DetLayout& lay, const msda_b200_desc* d, const uint2* ranges, const unsigned long long* vals,
                const void* grad_out, void* grad_value, cudaStream_t st) {
  constexpr int LPP = D / Vec16<VT>::N;
  const long long blocks = (lay.keys * LPP + kDetNT - 1) / kDetNT;
  if (blocks > 0x7fffffffll)
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "deterministic backward: grid too large");
  msda_bwd_det_pull_kernel<VT, D><<<(unsigned)blocks, kDetNT, 0, st>>>(
      ranges, vals, static_cast<const uint4*>(grad_out), static_cast<uint4*>(grad_value), lay.keys, d->S, d->Q, d->H);
  return launched("deterministic backward: grad_value");
}

template <typename VT>
int dispatch_pull(const DetLayout& lay, const msda_b200_desc* d, const uint2* ranges, const unsigned long long* vals,
                  const void* grad_out, void* grad_value, cudaStream_t st) {
  switch (d->D) {
    case 8: return launch_pull<VT, 8>(lay, d, ranges, vals, grad_out, grad_value, st);
    case 16: return launch_pull<VT, 16>(lay, d, ranges, vals, grad_out, grad_value, st);
    case 32: return launch_pull<VT, 32>(lay, d, ranges, vals, grad_out, grad_value, st);
    case 64: return launch_pull<VT, 64>(lay, d, ranges, vals, grad_out, grad_value, st);
    case 128: return launch_pull<VT, 128>(lay, d, ranges, vals, grad_out, grad_value, st);
  }
  return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "deterministic backward: head dim");
}

}  // namespace

extern "C" int msda_b200_internal_det_sort_bytes(const DetLayout* lay, size_t* bytes) {
  *bytes = 0;
  if (lay->records == 0) return MSDA_B200_OK;
  cub::DoubleBuffer<unsigned> kb(nullptr, nullptr);
  cub::DoubleBuffer<unsigned long long> vb(nullptr, nullptr);
  const cudaError_t e =
      cub::DeviceRadixSort::SortPairs(nullptr, *bytes, kb, vb, (int)lay->records, 0, lay->key_bits, (cudaStream_t)0);
  return e == cudaSuccess ? MSDA_B200_OK : cuda_error("deterministic sort: scratch size", e);
}

extern "C" int msda_b200_internal_det_sort(const DetLayout* lay, void* workspace, const unsigned** keys,
                                           const unsigned long long** vals, cudaStream_t st) {
  char* ws = static_cast<char*>(workspace);
  cub::DoubleBuffer<unsigned> kb(reinterpret_cast<unsigned*>(ws + lay->keys_off[0]),
                                 reinterpret_cast<unsigned*>(ws + lay->keys_off[1]));
  cub::DoubleBuffer<unsigned long long> vb(reinterpret_cast<unsigned long long*>(ws + lay->vals_off[0]),
                                           reinterpret_cast<unsigned long long*>(ws + lay->vals_off[1]));
  size_t sort = 0;
  if (int rc = msda_b200_internal_det_sort_bytes(lay, &sort)) return rc;
  const cudaError_t e =
      cub::DeviceRadixSort::SortPairs(ws + lay->sort_off, sort, kb, vb, (int)lay->records, 0, lay->key_bits, st);
  if (e != cudaSuccess) return cuda_error("deterministic sort", e);
  msda_b200_internal_count_launch();  // the sort's kernels count as one launch
  *keys = kb.Current();
  *vals = vb.Current();
  return MSDA_B200_OK;
}

// Workspace of the deterministic backward for a validated descriptor: the records, the bucket ranges and the sort's
// scratch as CUB reports it (which reads the current device's attributes).
extern "C" int msda_b200_internal_det_workspace_bytes(const msda_b200_desc* desc, size_t* bytes) {
  const DetLayout lay = det_layout(desc);
  if (int rc = check_supported(lay)) return rc;
  size_t sort = 0;
  if (int rc = msda_b200_internal_det_sort_bytes(&lay, &sort)) return rc;
  *bytes = lay.sort_off + sort;
  return MSDA_B200_OK;
}

// Steps 1-3 above, after msda_bwd_kernel<ACC = 2> wrote the records into the first key / payload buffers. The
// workspace holds at least msda_b200_internal_det_workspace_bytes(desc).
extern "C" int msda_b200_internal_det_grad_value(const msda_b200_desc* desc, const void* grad_out, void* grad_value,
                                                 void* workspace, cudaStream_t st) {
  const DetLayout lay = det_layout(desc);
  if (int rc = check_supported(lay)) return rc;
  char* ws = static_cast<char*>(workspace);
  uint2* ranges = reinterpret_cast<uint2*>(ws + lay.ranges_off);
  const unsigned long long* vals = reinterpret_cast<const unsigned long long*>(ws + lay.vals_off[0]);
  const cudaError_t e = cudaMemsetAsync(ranges, 0, (size_t)lay.keys * sizeof(uint2), st);
  if (e != cudaSuccess) return cuda_error("deterministic backward: memset", e);
  if (lay.records) {
    const unsigned* keys = nullptr;
    if (int rc = msda_b200_internal_det_sort(&lay, workspace, &keys, &vals, st)) return rc;
    const int n = (int)lay.records;
    msda_bwd_det_ranges_kernel<<<(n + kDetNT - 1) / kDetNT, kDetNT, 0, st>>>(keys, n, (unsigned)lay.keys, ranges);
    if (int rc = launched("deterministic backward: ranges")) return rc;
  }
  if (desc->value_dtype == MSDA_B200_BF16)
    return dispatch_pull<__nv_bfloat16>(lay, desc, ranges, vals, grad_out, grad_value, st);
  return dispatch_pull<float>(lay, desc, ranges, vals, grad_out, grad_value, st);
}
