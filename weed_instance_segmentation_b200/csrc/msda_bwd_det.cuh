// msda_bwd_det.cuh -- workspace layout of the deterministic backward (MSDA_B200_FLAG_DETERMINISTIC), shared by
// msda_b200.cu (whose msda_bwd_kernel<ACC = 2> writes the records) and msda_bwd_det.cu (which sorts them and pulls
// grad_value from them). Included after msda_b200.h.
//
// Every sample contributes four records, one per slot of its clamped 2x2 bilinear footprint, at index 4 * si + slot
// (si = ((b*Q + q)*H + h)*L*P + s, the sample's own index):
//   key     (b*S + row)*H + h   -- grad_value's row order; `keys` (= B*S*H, one past the last row) for a dead or
//                                  zero-weight slot, so those sort last
//   payload q << 32 | bits of the slot weight attn * wy * wx (float32)
// A stable radix sort over the key's bits then puts each (b, row, h) bucket in sample order, which depends on the
// inputs alone.
#pragma once

#include <stddef.h>

struct DetLayout {
  long long records;  // 4 * B*Q*H*L*P
  long long keys;     // B*S*H: the number of buckets, and the sentinel key
  int key_bits;       // bits of the sort key (enough for the sentinel)
  size_t keys_off[2], vals_off[2];  // double buffers of the sort: uint32 keys, uint64 payloads
  size_t ranges_off;  // keys x uint2 [begin, end) of each bucket in the sorted records
  size_t sort_off;    // the radix sort's scratch
};

inline size_t det_align(size_t n) { return (n + 255) & ~size_t(255); }

inline DetLayout det_layout(const msda_b200_desc* d) {
  DetLayout t;
  t.records = 4ll * d->B * d->Q * d->H * d->L * d->P;
  t.keys = (long long)d->B * d->S * d->H;
  t.key_bits = 0;
  while (t.key_bits < 63 && (t.keys >> t.key_bits) != 0) ++t.key_bits;
  const size_t kb = det_align((size_t)t.records * 4), vb = det_align((size_t)t.records * 8);
  t.keys_off[0] = 0;
  t.keys_off[1] = kb;
  t.vals_off[0] = 2 * kb;
  t.vals_off[1] = 2 * kb + vb;
  t.ranges_off = 2 * kb + 2 * vb;
  t.sort_off = t.ranges_off + det_align((size_t)t.keys * 8);
  return t;
}
