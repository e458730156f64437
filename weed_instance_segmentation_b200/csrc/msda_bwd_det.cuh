// msda_bwd_det.cuh -- workspace layout and sort of the deterministic backwards: the one of multi-scale deformable
// attention (MSDA_B200_FLAG_DETERMINISTIC; msda_b200.cu's msda_bwd_kernel<ACC = 2> writes the records, msda_bwd_det.cu
// sorts them and pulls grad_value from them) and the one of point sampling (point_sample.cu). Included after
// msda_b200.h and cuda_runtime.h.
//
// Both write (uint32 key, uint64 payload) records into the first key / payload buffers of the layout; a stable CUB
// radix sort over the key's bits (msda_b200_internal_det_sort, internal.h) then groups them by key, each group in record order,
// which depends on the inputs alone. The key `keys` (one past the last destination) marks a record that adds nothing
// and sorts last.
//
// Multi-scale deformable attention: every sample contributes four records, one per slot of its clamped 2x2 bilinear
// footprint, at index 4 * si + slot (si = ((b*Q + q)*H + h)*L*P + s, the sample's own index):
//   key     (b*S + row)*H + h   -- grad_value's row order; `keys` (= B*S*H, one past the last row) for a dead or
//                                  zero-weight slot, so those sort last
//   payload q << 32 | bits of the slot weight attn * wy * wx (float32)
#pragma once

#include <stddef.h>

struct DetLayout {
  long long records;  // 4 per sample (4 * B*Q*H*L*P) or per sampled point
  long long keys;     // destinations: the number of buckets, and the sentinel key
  int key_bits;       // bits of the sort key (enough for the sentinel)
  size_t keys_off[2], vals_off[2];  // double buffers of the sort: uint32 keys, uint64 payloads
  size_t ranges_off;  // keys x uint2 [begin, end) of each bucket in the sorted records
  size_t sort_off;    // the radix sort's scratch
};

inline size_t det_align(size_t n) { return (n + 255) & ~size_t(255); }

// `records` records sorted over the keys [0, keys] (`keys` is the sentinel); `ranges`: room for a [begin, end) pair
// per key after the payloads.
inline DetLayout det_sort_layout(long long records, long long keys, bool ranges) {
  DetLayout t;
  t.records = records;
  t.keys = keys;
  t.key_bits = 0;
  while (t.key_bits < 63 && (t.keys >> t.key_bits) != 0) ++t.key_bits;
  const size_t kb = det_align((size_t)t.records * 4), vb = det_align((size_t)t.records * 8);
  t.keys_off[0] = 0;
  t.keys_off[1] = kb;
  t.vals_off[0] = 2 * kb;
  t.vals_off[1] = 2 * kb + vb;
  t.ranges_off = 2 * kb + 2 * vb;
  t.sort_off = t.ranges_off + (ranges ? det_align((size_t)t.keys * 8) : 0);
  return t;
}

inline DetLayout det_layout(const msda_b200_desc* d) {
  return det_sort_layout(4ll * d->B * d->Q * d->H * d->L * d->P, (long long)d->B * d->S * d->H, true);
}
