// msda_bwd_mma.cuh -- backward v3: pixel-GROUP-sorted accumulation with warp-level tensor-core products.
// Included by msda_b200.cu inside its anonymous namespace (uses KParams, Level, Axis, Vec16, red_add_f32x4).
//
// Why: v1 issues one fp32 reduction per bilinear corner and is bound by L2 reduction throughput.  v2 (a pixel-sorted
// CUDA-core pull, in git at commit 71afd7d) sorted the 4 corner contributions of every sample by pixel and was bound by
// instruction issue (~9-13 warp instructions per contribution, half of them the divergent run-boundary code).  Once
// contributions are grouped by target pixels the work IS two small matrix products, so v3 groups SAMPLES by aligned
// 4x2-pixel groups (8 "slots") and lets mma.sync.m16n8k16 (bf16 in, fp32 accumulate) do both products for 16 list
// rows at a time:
//
//   dots   D2[row, slot]   = sum_ch  GO[row, ch] * V[slot, ch]        (-> grad_attn / grad_loc, exact bf16 products)
//   scatter GV[ch, slot]  += sum_row GO[row, ch] * Wt[row, slot]      (-> grad_value; Wt = attn * bilinear weight of
//                                                                      the sample's corner that falls on the slot)
//
//   per thread block = (batch, head, tile of TQ queries), per level:
//     a  sample descriptors (slot weights, derivative codes, clamped base pixel) + bounding box of the touched pixels
//     b  window of 4x2 pixel groups (<= GCAP groups, around the mean position if the box is larger; samples outside
//        take the v1 route)
//     c  histogram of (sample, group) rows: a sample's 2x2 footprint meets 1, 2 or 4 groups (1.9 on average,
//        against 4 corner entries in v2)
//     d  one-counter-per-thread scan -> segment starts + a table of work items (group, <= 64 rows)
//     e  fill: row = {sample id, 8 bf16 slot weights}
//     f  pull: a warp takes an item, loads the group's 8 value rows once (one LDG.128 per lane), and per 16 rows
//        issues 4 ldmatrix.x4 (the staged grad_out rows, plain and transposed), 1 ldmatrix.x2 (weights), 4 HMMA;
//        the 16x8 dots go to shared memory per (sample, corner); one red.global.add.v4.f32 per lane and slot at the
//        end of the item
//     g  fallback contributions: direct reductions (v1 route)
//     h  one thread per sample folds its four dots into grad_attn / grad_loc
//
// grad_out rows are staged ONCE per block with their 32 channels permuted so that (i) the m16n8k16 fragments of both
// products come straight out of ldmatrix and (ii) every lane ends up holding 4 consecutive channels of a slot, i.e.
// one 16-byte reduction.  Stored row = 4 chunks of 8 bf16; chunk j, element i holds channel 4*i + j; the chunk index
// is XOR-swizzled (go_swizzle) so the eight 16-byte pieces of one ldmatrix tile spread over the banks.
//
// Numerics: the dots are exact bf16 x bf16 products accumulated in fp32; the scatter uses slot weights rounded to
// bf16 (relative 2^-9 per contribution, the same size as the bf16 rounding of grad_value itself).

__device__ __forceinline__ void ldsm_x4(unsigned (&r)[4], unsigned addr) {
  asm("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(unsigned (&r)[4], unsigned addr) {
  asm("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2_trans(unsigned (&r)[2], unsigned addr) {
  asm("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
// 8x8 b16 tile held one row per quad of lanes -> its transpose in the same layout (what ldmatrix.trans of the same
// tile returns), without going back to shared memory
__device__ __forceinline__ unsigned movm_trans(unsigned x) {
  unsigned y;
  asm("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
// D (16x8, fp32) += A (16x16, bf16, row) * B (16x8, bf16, col)
__device__ __forceinline__ void mma_bf16(float (&d)[4], unsigned a0, unsigned a1, unsigned a2, unsigned a3, unsigned b0,
                                         unsigned b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// XOR swizzle of the 16-byte chunk index of staged grad_out row `row`.  Eight list rows of one ldmatrix tile are mostly
// queries of a small 2-D patch (row = 16*y + x inside the 8 x 16 query tile): bit 0 of x selects the upper / lower half
// of the 128-byte bank line (64-byte rows), bit 1 of x and bit 0 of y go into the swizzle, so a 4 x 2 patch of queries
// hits eight different 16-byte bank groups.
__device__ __forceinline__ int go_swizzle(int row) { return ((row >> 1) & 1) | ((row >> 3) & 2); }

#ifndef MSDA_MMA_MOVM
#define MSDA_MMA_MOVM 1
#endif

struct MmaSmem {
  size_t w, go, wrow, dot, a, xy, cnt, item, id, fb, misc, stat, total;
};

constexpr int kMmaItemRows = 64;  // rows per work item (4 HMMA row blocks)

template <int NT, int TQ, int P, int GCAP, int RCAP, bool FUSED>
__host__ __device__ inline MmaSmem mma_smem_layout() {
  constexpr int NS = TQ * P;
  MmaSmem s;
  size_t o = 0;
  s.w = o;    o += sizeof(float4) * NS;
  s.go = o;   o += 64 * (TQ + 1);            // + one all-zero row (padding rows of the last row block of an item)
  s.wrow = o; o += 16 * RCAP;
  s.dot = o;  o += sizeof(float4) * NS;
  s.a = o;    o += sizeof(float) * NS;
  s.xy = o;   o += sizeof(int) * NS;          // x | y << 12 | derivative codes << 24
  s.cnt = o;  o += sizeof(int) * GCAP;        // histogram, then fill cursors
  s.item = o; o += sizeof(uint2) * (GCAP + RCAP / kMmaItemRows + 8);  // (rows | n | slot mask, pixel offset)
  s.id = o;   o += sizeof(unsigned) * RCAP;      // row code: staged grad_out row offset | sample | footprint position
  s.fb = o;   o += sizeof(unsigned short) * NS * 4;
  o = (o + 15) & ~size_t(15);
  s.misc = o; o += sizeof(int) * 64;
  s.stat = o;  // (fused prologue: the softmax statistics live in registers, see f_lse / f_dsum)
  s.total = o;
  return s;
}

template <int P>
struct Log2P;
template <> struct Log2P<1> { static constexpr int v = 0; };
template <> struct Log2P<2> { static constexpr int v = 1; };
template <> struct Log2P<4> { static constexpr int v = 2; };
template <> struct Log2P<8> { static constexpr int v = 3; };

// misc slots; MI_WSUM = 16 holds the per-warp scan totals
enum { MI_MINX = 0, MI_MAXX, MI_MINY, MI_MAXY, MI_SUMX, MI_SUMY, MI_NACT, MI_FBN, MI_TOTAL, MI_NITEMS, MI_WSUM = 16 };

// derivative code k of a sample's packed codes (2 bits each, value + 1) -> d(slot weight)/d(pixel coord)
__device__ __forceinline__ float gdec(int code, int k) { return (float)(((code >> (2 * k)) & 3) - 1); }

template <typename AT, int NT, int TQ, int P, int GCAP, int RCAP, bool FUSED>
__global__ void __launch_bounds__(NT, 4) msda_bwd_mma_kernel(const __grid_constant__ KParams p) {
  using VT = __nv_bfloat16;
  constexpr int LPP = 4;             // 16-byte pieces per 32-channel bf16 row
  constexpr int G = NT / LPP;
  constexpr int NS = TQ * P;
  constexpr int LP2 = Log2P<P>::v;
  constexpr int NW = NT / 32;
  static_assert(GCAP == NT, "the scan gives every thread one group counter");
  static_assert(NS % NT == 0, "every thread owns NS/NT samples per level");
  static_assert(NS <= 512, "row code: 9 bits of sample index");
  static_assert(RCAP < 2048 && RCAP % 16 == 0, "row index is 11 bits in the item word");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const MmaSmem lay = mma_smem_layout<NT, TQ, P, GCAP, RCAP, FUSED>();
  float4* s_w = reinterpret_cast<float4*>(smem_raw + lay.w);
  unsigned* s_go32 = reinterpret_cast<unsigned*>(smem_raw + lay.go);
  uint4* s_wrow = reinterpret_cast<uint4*>(smem_raw + lay.wrow);
  float* s_dot = reinterpret_cast<float*>(smem_raw + lay.dot);
  float* s_a = reinterpret_cast<float*>(smem_raw + lay.a);
  int* s_xy = reinterpret_cast<int*>(smem_raw + lay.xy);
  int* s_cnt = reinterpret_cast<int*>(smem_raw + lay.cnt);
  uint2* s_item = reinterpret_cast<uint2*>(smem_raw + lay.item);
  unsigned* s_id = reinterpret_cast<unsigned*>(smem_raw + lay.id);
  unsigned short* s_fb = reinterpret_cast<unsigned short*>(smem_raw + lay.fb);
  int* const s_misc2 = reinterpret_cast<int*>(smem_raw + lay.misc);  // two sets of 32, alternating by level

  int b, tile, h;
  decode_block(p, b, tile, h);
  const int q0 = tile * TQ;
  const int nq = min(TQ, p.Q - q0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = tid / LPP, c = tid % LPP;
  const unsigned gmask = ((1u << LPP) - 1u) << ((lane / LPP) * LPP);
  const long long acc_base = (long long)b * p.batch_stride16;
  const uint4* const vrow = reinterpret_cast<const uint4*>(p.value) + acc_base;
  float* const acc_f = reinterpret_cast<float*>(p.grad_value_acc) + acc_base * 8;
  const unsigned go_sa = (unsigned)__cvta_generic_to_shared(s_go32);
  const unsigned wrow_sa = (unsigned)__cvta_generic_to_shared(s_wrow);

  // per-thread samples: si = r*NT + tid; their loc / attn are prefetched one level ahead
  constexpr int SPT = NS / NT;
  float2 pre_loc[SPT];
  float pre_a[SPT];
  float2 f_ref[SPT];  // fused prologue with implicit reference points: the thread's queries' own pixel centres
#pragma unroll
  for (int r = 0; r < SPT; ++r) {
    f_ref[r] = make_float2(0.f, 0.f);
    const int ql = (r * NT + tid) >> LP2;
    if (FUSED && !p.ref && ql < nq) f_ref[r] = implicit_reference_point(p, p.q_order ? p.q_order[q0 + ql] : q0 + ql);
  }
  auto fetch_level = [&](int l) {
#pragma unroll
    for (int r = 0; r < SPT; ++r) {
      const int si = r * NT + tid;
      const int ql = si >> LP2, pt = si & (P - 1);
      pre_loc[r] = make_float2(0.f, 0.f);
      pre_a[r] = 0.f;
      if (l < p.L && ql < nq) {
        const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
        const long long gi = (((long long)b * p.Q + q) * p.H + h) * p.LP + l * P + pt;
        if (FUSED) {
          // loc = ref + off / (W_l, H_l) (M2F:963-971); the implicit reference point of a query (ref == NULL) does not
          // depend on the level and was computed once in f_ref
          const float2 off = load_pair<AT>(p.offsets, gi);
          const float2 rp = p.ref ? __ldg(reinterpret_cast<const float2*>(p.ref) + ((long long)b * p.Q + q) * p.L + l)
                                  : f_ref[r];
          pre_loc[r] = make_float2(__fadd_rn(rp.x, __fdiv_rn(off.x, (float)p.lv[l].W)),
                                   __fadd_rn(rp.y, __fdiv_rn(off.y, (float)p.lv[l].H)));
          pre_a[r] = to_float<AT>(reinterpret_cast<const AT*>(p.logits)[gi]);  // raw logit; softmax applied at use
        } else {
          pre_loc[r] = __ldg(reinterpret_cast<const float2*>(p.loc) + gi);
          pre_a[r] = to_float<AT>(reinterpret_cast<const AT*>(p.attn)[gi]);
        }
      }
    }
  };
  fetch_level(0);

  // grad_out rows of the tile, staged once: channel-permuted and chunk-swizzled (see the file header)
  for (int i = tid; i < TQ * LPP; i += NT) {
    const int ql = i >> 2, cc = i & 3;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (ql < nq) {
      const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
      v = ldg16(reinterpret_cast<const uint4*>(p.grad_out) + (((long long)b * p.Q + q) * p.H + h) * LPP + cc);
    }
    // v holds channels 8cc .. 8cc+7; word cc of stored chunk j = (channel 8cc + j, channel 8cc + 4 + j)
    const int sw = go_swizzle(ql);
    unsigned* row = s_go32 + ql * 16 + cc;
    row[(0 ^ sw) << 2] = __byte_perm(v.x, v.z, 0x5410);
    row[(1 ^ sw) << 2] = __byte_perm(v.x, v.z, 0x7632);
    row[(2 ^ sw) << 2] = __byte_perm(v.y, v.w, 0x5410);
    row[(3 ^ sw) << 2] = __byte_perm(v.y, v.w, 0x7632);
  }
  if (tid < 16) s_go32[TQ * 16 + tid] = 0u;

  // Fused prologue: the P = 4 samples (r, tid) of one (query, level) sit in four adjacent lanes, and sample r of every
  // level belongs to query r * NT / P + tid / P -- so the softmax statistics of a thread's own queries never leave its
  // registers: f_lse = max + log(sum exp(x - max)) (a_j = exp(x_j - f_lse)), f_dsum = sum_k a_k * d(loss)/d(a_k).
  // (In shared memory they cost 1.5 KB per block, which took the fused kernel from 4 to 3 blocks per SM.)
  static_assert(!FUSED || P == 4, "fused prologue: four lanes per (query, head) row");
  float f_lse[SPT], f_dsum[SPT];
  // d(loss)/d(a) of the thread's samples, kept in fp32 until the softmax backward after the last level: parked in a
  // bf16 grad_logits it would carry a 2^-9 rounding into ga - f_dsum, which cancels when the row's ga share a common
  // part (value rows with a non-zero mean, one dominant logit). Local memory, indexed by the runtime level.
  float ga_park[SPT][MSDA_B200_MAX_LEVELS];
#pragma unroll
  for (int r = 0; r < SPT; ++r) { f_lse[r] = 0.f; f_dsum[r] = 0.f; }
  if (FUSED) {
#pragma unroll
    for (int r = 0; r < SPT; ++r) {
      const int ql = (r * NT + tid) >> LP2;
      const bool valid = ql < nq;
      const int q = valid ? (p.q_order ? p.q_order[q0 + ql] : q0 + ql) : 0;
      float mx, inv;
      softmax_stats_x4<AT>(reinterpret_cast<const AT*>(p.logits) + (((long long)b * p.Q + q) * p.H + h) * p.LP, p.LP,
                           tid & 3, valid, mx, inv);
      f_lse[r] = valid ? mx - logf(inv) : 0.f;
    }
  }

  auto init_misc = [&](int* m) {  // called by threads 0..15
    int init = 0;
    if (tid == MI_MINX || tid == MI_MINY) init = 0x7fffffff;
    if (tid == MI_MAXX || tid == MI_MAXY) init = -1;
    m[tid] = init;
  };
  if (tid < 16) init_misc(s_misc2);
  s_cnt[tid] = 0;
  __syncthreads();

  // Barriers per level: after a, in d (2), after e, after f/g.  Phase h and the next level's phase a touch only the
  // thread's own samples (same sample <-> thread mapping), the counters are re-armed for the next level while the
  // current one is still running (other s_misc set after a, s_cnt after e).
  for (int l = 0; l < p.L; ++l) {
    const Level lv = p.lv[l];
    const int dxs = lv.W > 1 ? 1 : 0, dys = lv.H > 1 ? 1 : 0;
    int* const s_misc = s_misc2 + (l & 1) * 32;

    // ---- a: descriptors + bounding box (thread-local first, then one set of warp reductions)
    int t_mnx = 0x7fffffff, t_mxx = -1, t_mny = 0x7fffffff, t_mxy = -1;
#pragma unroll
    for (int r = 0; r < SPT; ++r) {
      const int si = r * NT + tid;
      const int ql = si >> LP2;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      int gcode = 0x55;  // code 1 == derivative 0 == slot not read
      float a = 0.f;
      int xb = 0, yb = 0;
      if (ql < nq) {
        a = FUSED ? expf(pre_a[r] - f_lse[r]) : pre_a[r];
        const Axis ax = axis_setup(pre_loc[r].x, lv.W), ay = axis_setup(pre_loc[r].y, lv.H);
        xb = ax.base; yb = ay.base;
        if (ax.ok && ay.ok) {
          w = make_float4(ax.s0, ax.s1, ay.s0, ay.s1);
          gcode = ((int)ax.g0 + 1) | (((int)ax.g1 + 1) << 2) | (((int)ay.g0 + 1) << 4) | (((int)ay.g1 + 1) << 6);
          if ((ax.g0 != 0.f || ax.g1 != 0.f) && (ay.g0 != 0.f || ay.g1 != 0.f)) {
            t_mnx = min(t_mnx, xb); t_mxx = max(t_mxx, xb + dxs);
            t_mny = min(t_mny, yb); t_mxy = max(t_mxy, yb + dys);
          }
        }
      }
      s_w[si] = w; s_a[si] = a; s_xy[si] = xb | (yb << 12) | (gcode << 24);
    }
    {
      const int mnx = __reduce_min_sync(0xffffffffu, t_mnx), mxx = __reduce_max_sync(0xffffffffu, t_mxx);
      const int mny = __reduce_min_sync(0xffffffffu, t_mny), mxy = __reduce_max_sync(0xffffffffu, t_mxy);
      if (lane == 0 && mxx >= 0) {
        atomicMin(&s_misc[MI_MINX], mnx); atomicMax(&s_misc[MI_MAXX], mxx);
        atomicMin(&s_misc[MI_MINY], mny); atomicMax(&s_misc[MI_MAXY], mxy);
      }
    }
    __syncthreads();
    if (tid < 16) init_misc(s_misc2 + ((l + 1) & 1) * 32);

    // ---- b: window of pixel groups (every thread computes the same rectangle); group (i, j) = pixels
    // [4*(gx_lo+i), +4) x [2*(gy_lo+j), +2)
    int gx_lo = 0, gy_lo = 0, gw = 0, gh = 0;
    if (s_misc[MI_MAXX] >= 0) {  // block-uniform
      const int a0 = s_misc[MI_MINX] >> 2, a1 = s_misc[MI_MAXX] >> 2, b0 = s_misc[MI_MINY] >> 1, b1 = s_misc[MI_MAXY] >> 1;
      const int bw = a1 - a0 + 1, bh = b1 - b0 + 1;
      if (bw <= 64 && bw * bh <= GCAP) {
        gx_lo = a0; gy_lo = b0; gw = bw; gh = bh;
      } else {
        // bounding box too large (scattered samples): a GCAP-group rectangle around the mean position; the rest of the
        // samples take the fallback route.  Rare, so the sums are only formed here.
        int sx = 0, sy = 0, na = 0;
#pragma unroll
        for (int r = 0; r < SPT; ++r) {
          const int xy = s_xy[r * NT + tid];
          const int gc = xy >> 24;
          if (((gc & 15) != 5) && ((gc >> 4) != 5)) { sx += xy & 0xfff; sy += (xy >> 12) & 0xfff; ++na; }
        }
        sx = __reduce_add_sync(0xffffffffu, sx); sy = __reduce_add_sync(0xffffffffu, sy); na = __reduce_add_sync(0xffffffffu, na);
        if (lane == 0) { atomicAdd(&s_misc[MI_SUMX], sx); atomicAdd(&s_misc[MI_SUMY], sy); atomicAdd(&s_misc[MI_NACT], na); }
        __syncthreads();
        const int nact = max(s_misc[MI_NACT], 1);
        gw = min(bw, 16);
        gh = min(bh, GCAP / gw);
        const int cx = (s_misc[MI_SUMX] / nact) >> 2, cy = (s_misc[MI_SUMY] / nact) >> 1;
        gx_lo = min(max(cx - gw / 2, a0), a1 - gw + 1);
        gy_lo = min(max(cy - gh / 2, b0), b1 - gh + 1);
      }
    }

    // ---- c: histogram of (sample, group) rows.  Combination k = cj*2 + ci: ci / cj = 0 is the group of the
    // footprint's first column / row, 1 the next group (only when the footprint straddles a group boundary).
    // code = group index in the window, or -1 (no active corner there / handed to the fallback list).
    int code[SPT][4];
#pragma unroll
    for (int r = 0; r < SPT; ++r) {
      const int si = r * NT + tid;
      const int xy = s_xy[si];
      const int x = xy & 0xfff, y = (xy >> 12) & 0xfff, gcode = xy >> 24;
      const bool ax0 = (gcode & 3) != 1, ax1 = ((gcode >> 2) & 3) != 1;
      const bool ay0 = ((gcode >> 4) & 3) != 1, ay1 = ((gcode >> 6) & 3) != 1;
      const bool xsplit = (x & 3) == 3, ysplit = (y & 1) == 1;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int ci = k & 1, cj = k >> 1;
        const bool cx0 = (ci == 0) && ax0, cx1 = ax1 && (ci == 0 ? !xsplit : xsplit);
        const bool cy0 = (cj == 0) && ay0, cy1 = ay1 && (cj == 0 ? !ysplit : ysplit);
        int cd = -1;
        if ((cx0 || cx1) && (cy0 || cy1)) {
          const int gxl = ((x + ci) >> 2) - gx_lo, gyl = ((y + cj) >> 1) - gy_lo;
          if ((unsigned)gxl < (unsigned)gw && (unsigned)gyl < (unsigned)gh) {
            cd = gyl * gw + gxl;
            atomicAdd(&s_cnt[cd], 1);
          } else {
#pragma unroll
            for (int cn = 0; cn < 4; ++cn)
              if (((cn & 1) ? cx1 : cx0) && ((cn & 2) ? cy1 : cy0))
                s_fb[atomicAdd(&s_misc[MI_FBN], 1)] = (unsigned short)(si * 4 + cn);
          }
        }
        code[r][k] = cd;
      }
    }
    __syncthreads();

    // ---- d: exclusive scan, one group per thread; rows in the low half, work items in the high half
    {
      const int cnt = s_cnt[tid];
      const int v = cnt | (((cnt + kMmaItemRows - 1) / kMmaItemRows) << 16);
      int incl = v;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += t;
      }
      if (lane == 31) s_misc[MI_WSUM + warp] = incl;
      __syncthreads();
      int base = 0;
#pragma unroll
      for (int w2 = 0; w2 < NW; ++w2)
        if (w2 < warp) base += s_misc[MI_WSUM + w2];
      const int excl = base + incl - v;
      const int row_start = excl & 0xffff, item_start = excl >> 16;
      s_cnt[tid] = row_start;
      if (tid == NT - 1) {
        s_misc[MI_TOTAL] = (excl + v) & 0xffff;
        s_misc[MI_NITEMS] = (excl + v) >> 16;
      }
      if (cnt > 0) {
        // item = (first row [0,11) | rows [11,18) | in-level mask of the group's 8 slots [18,26),
        //         16-byte-unit offset of the group's first pixel inside the level)
        const int gyl = tid / gw, gxl = tid - gyl * gw;
        const int px0 = (gx_lo + gxl) << 2, py0 = (gy_lo + gyl) << 1;
        const unsigned xbits = (1u << min(lv.W - px0, 4)) - 1u;
        const unsigned mask = xbits | (py0 + 1 < lv.H ? xbits << 4 : 0u);
        const unsigned pixoff = (unsigned)((py0 * lv.W + px0) * (p.H * LPP));
        for (int j = 0; j * kMmaItemRows < cnt; ++j) {
          const int rb = row_start + j * kMmaItemRows;
          const int n = rb < RCAP ? min(min(kMmaItemRows, cnt - j * kMmaItemRows), RCAP - rb) : 0;
          s_item[item_start + j] = make_uint2((unsigned)(n ? rb : 0) | ((unsigned)n << 11) | (mask << 18), pixoff);
        }
      }
    }
    __syncthreads();

    // ---- e: fill
#pragma unroll
    for (int r = 0; r < SPT; ++r) {
      const int si = r * NT + tid;
      const int xy = s_xy[si];
      const int x = xy & 0xfff, y = (xy >> 12) & 0xfff;
      const float4 w = s_w[si];
      const float a = s_a[si];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int cd = code[r][k];
        if (cd >= 0) {
          const int ci = k & 1, cj = k >> 1;
          // Measured and dropped: warp-aggregated ranks from __match_any_sync in the histogram pass (MATCH.ANY costs far
          // more than the serialised same-address atomics it removes, 0.87 -> 1.00 ms); dealing the query slots out so
          // that one instruction's eight queries lie >= 4 pixels apart (fewer same-address lanes, 0.87 -> 0.90 ms).
          // (also measured and dropped: keeping the rank the histogram pass's atomic returned, packed into `code`, and
          // replacing this second round of atomics by a broadcast LDS of the group's start -- 0.877 vs 0.867 ms)
          const int slot = atomicAdd(&s_cnt[cd], 1);
          if (slot < RCAP) {
            // first column / row of the footprint relative to the group: -1 = only the second one lies in it
            const int bx = ci ? -1 : (x & 3), by = cj ? -1 : (y & 1);
            // row code: [0,14) byte offset of the staged grad_out row incl. its swizzle, [14,23) sample, [23,26) bx + 1,
            // [26,28) by + 1
            const int ql = si >> LP2;
            s_id[slot] = (unsigned)(ql * 64 + (go_swizzle(ql) << 4)) | ((unsigned)(si | ((bx + 1) << 9) | ((by + 1) << 12)) << 14);
            const float y0w = by == 0 ? a * w.z : (by == -1 ? a * w.w : 0.f);
            const float y1w = by == 1 ? a * w.z : (by == 0 ? a * w.w : 0.f);
            const unsigned p0 = Vec16<VT>::pack2(y0w * w.x, y0w * w.y), p1 = Vec16<VT>::pack2(y1w * w.x, y1w * w.y);
            const unsigned long long r0 = bx >= 0 ? ((unsigned long long)p0 << (16 * bx)) : (unsigned long long)(p0 >> 16);
            const unsigned long long r1 = bx >= 0 ? ((unsigned long long)p1 << (16 * bx)) : (unsigned long long)(p1 >> 16);
            s_wrow[slot] = make_uint4((unsigned)r0, (unsigned)(r0 >> 32), (unsigned)r1, (unsigned)(r1 >> 32));
          } else {
            // row list full: this group's corners of the sample take the fallback route
            const int gcode = xy >> 24;
            const bool ax0 = (gcode & 3) != 1, ax1 = ((gcode >> 2) & 3) != 1;
            const bool ay0 = ((gcode >> 4) & 3) != 1, ay1 = ((gcode >> 6) & 3) != 1;
            const bool xsplit = (x & 3) == 3, ysplit = (y & 1) == 1;
            const bool cx0 = (ci == 0) && ax0, cx1 = ax1 && (ci == 0 ? !xsplit : xsplit);
            const bool cy0 = (cj == 0) && ay0, cy1 = ay1 && (cj == 0 ? !ysplit : ysplit);
#pragma unroll
            for (int cn = 0; cn < 4; ++cn)
              if (((cn & 1) ? cx1 : cx0) && ((cn & 2) ? cy1 : cy0))
                s_fb[atomicAdd(&s_misc[MI_FBN], 1)] = (unsigned short)(si * 4 + cn);
          }
        }
      }
    }
    __syncthreads();
    s_cnt[tid] = 0;  // for the next level's histogram

    // ---- f: pull.  Warp-level: item -> 8 value rows -> row blocks of 16.  The value rows of the next item are
    // requested before the current one is processed.
    {
      const int g8 = lane >> 2, t4 = lane & 3;
      const int n_items = s_misc[MI_NITEMS];
      const int pix16 = p.H * LPP;  // 16-byte units per pixel
      // lane (g8, t4): value row of slot g8 (x = g8 % 4, y = g8 / 4), channels 8*t4 .. +7; accumulator channels
      // 4*g8 .. +3 of slots 2*t4 and 2*t4 + 1 (x = 2*(t4 % 2) (+1), y = t4 / 2)
      const uint4* const v_lane = vrow + (lv.start * p.H + h) * LPP + ((g8 >> 2) * lv.W + (g8 & 3)) * pix16 + t4;
      float* const acc_lane = acc_f + (long long)((lv.start * p.H + h) * LPP + ((t4 >> 1) * lv.W + 2 * (t4 & 1)) * pix16) * 8 + 4 * g8;
      const int kx = 2 * (t4 & 1) + 1, ky = (t4 >> 1) + 1;
      const unsigned vbit = 1u << (18 + g8), fbit = 1u << (18 + 2 * t4);
      const unsigned lsel = ((unsigned)lane >> 4) << 4;  // chunk select of the ldmatrix row addresses
      auto load_v = [&](uint2 item) -> uint4 {
        if (item.x & vbit) return ldg16(v_lane + (int)item.y);
        return make_uint4(0u, 0u, 0u, 0u);
      };
      int it = warp;
      uint2 item = it < n_items ? s_item[it] : make_uint2(0u, 0u);
      uint4 vv = load_v(item);
      while (it < n_items) {
        const int it_n = it + NW;  // (items handed out on demand through an atomic counter were measured slower: 0.885 vs 0.867 ms)
        const uint2 item_n = it_n < n_items ? s_item[it_n] : make_uint2(0u, 0u);
        const uint4 vv_n = load_v(item_n);
        const int n = (int)((item.x >> 11) & 127u);
        if (n != 0) {
          const int rbeg = (int)(item.x & 0x7ffu), rend = rbeg + n;
          const unsigned bv00 = __byte_perm(vv.x, vv.z, 0x5410);  // channels 8t, 8t+4   <-> k = 2t, 2t+1 of chunk 0
          const unsigned bv01 = __byte_perm(vv.x, vv.z, 0x7632);  // channels 8t+1, 8t+5 <-> chunk 1
          const unsigned bv10 = __byte_perm(vv.y, vv.w, 0x5410);  // channels 8t+2, 8t+6 <-> chunk 2
          const unsigned bv11 = __byte_perm(vv.y, vv.w, 0x7632);  // channels 8t+3, 8t+7 <-> chunk 3
          float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};
          // row codes are fetched one row block ahead
          const unsigned kNoRow = 0x0fffc000u | (unsigned)(TQ * 64);  // all-zero grad_out row, matches no (sample, corner)
          int r0 = rbeg;
          unsigned code_l = r0 + (lane & 15) < rend ? s_id[r0 + (lane & 15)] : kNoRow;
          while (true) {
            const int rn = r0 + 16;
            const unsigned code_ln = rn + (lane & 15) < rend ? s_id[rn + (lane & 15)] : kNoRow;
            const int idx = r0 + (lane & 15);
            const unsigned ga = go_sa + ((code_l & 0x3fffu) ^ lsel);
            unsigned a[4], a2[4], tA[4], tB[4], bw[2];
            ldsm_x4(a, ga);
            ldsm_x4(a2, ga ^ 32u);
#if MSDA_MMA_MOVM
#pragma unroll
            for (int j = 0; j < 4; ++j) { tA[j] = movm_trans(a[j]); tB[j] = movm_trans(a2[j]); }
#else
            ldsm_x4_trans(tA, ga);
            ldsm_x4_trans(tB, ga ^ 32u);
#endif
            ldsm_x2_trans(bw, idx < rend ? wrow_sa + idx * 16 : go_sa + TQ * 64);
            float d[4] = {0.f, 0.f, 0.f, 0.f};
            mma_bf16(d, a[0], a[1], a[2], a[3], bv00, bv01);
            mma_bf16(d, a2[0], a2[1], a2[2], a2[3], bv10, bv11);
            mma_bf16(acc0, tA[0], tA[2], tA[1], tA[3], bw[0], bw[1]);
            mma_bf16(acc1, tB[0], tB[2], tB[1], tB[3], bw[0], bw[1]);
            // dots of rows g8 and g8 + 8 at slots 2*t4, 2*t4 + 1 -> the (sample, corner) they belong to
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const unsigned code = __shfl_sync(0xffffffffu, code_l, g8 + 8 * e);
              const int cxa = kx - (int)((code >> 23) & 7u), cy = ky - (int)((code >> 26) & 3u);
              float* dst = s_dot + ((code >> 14) & 511u) * 4 + cy * 2 + cxa;
              if ((unsigned)cy < 2u && (unsigned)cxa < 2u) dst[0] = d[2 * e];
              if ((unsigned)cy < 2u && (unsigned)(cxa + 1) < 2u) dst[1] = d[2 * e + 1];
            }
            if (rn >= rend) break;
            r0 = rn; code_l = code_ln;
          }
          // flush: lane (g8, t4) holds channels 4*g8 .. +3 of slots 2*t4 (acc*[0], acc*[2]) and 2*t4 + 1 (acc*[1], acc*[3])
          float* const dst = acc_lane + (long long)(int)item.y * 8;
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const float v0 = acc0[s], v1 = acc0[2 + s], v2 = acc1[s], v3 = acc1[2 + s];
            const unsigned nz = (__float_as_uint(v0) | __float_as_uint(v1) | __float_as_uint(v2) | __float_as_uint(v3)) << 1;
            if ((item.x & (fbit << s)) && nz != 0u) red_add_f32x4(dst + s * pix16 * 8, v0, v1, v2, v3);
          }
        }
        it = it_n; item = item_n; vv = vv_n;
      }
    }

    // in flight during the fallback pass and the per-sample gradients of this level (issued before the pull it would
    // hide its latency better, but its six registers push the pull over the 64-register budget of 4 blocks / SM:
    // spills, 0.887 vs 0.867 ms)
    fetch_level(l + 1);

    // ---- g: fallback contributions (outside the window / row list full): direct reduction, four lanes per corner
    {
      const int nfb = s_misc[MI_FBN];
      for (int k = g; k < nfb; k += G) {
        const int id = s_fb[k];
        const int si = id >> 2, cn = id & 3;
        const float4 w = s_w[si];
        const float wgt = s_a[si] * ((cn & 2) ? w.w : w.z) * ((cn & 1) ? w.y : w.x);
        const int xy = s_xy[si];
        const int x = (xy & 0xfff) + (cn & 1), y = ((xy >> 12) & 0xfff) + ((cn >> 1) & 1);
        const long long off = (long long)((lv.start + y * lv.W + x) * p.H + h) * LPP;
        float vf[8], gf[8];
        Vec16<VT>::unpack(ldg16(vrow + off + c), vf);
        {
          // lane c needs channels 8c .. 8c+7: word c of stored chunk j = (channel 8c + j, channel 8c + 4 + j)
          const int ql = si >> LP2, sw = go_swizzle(ql);
          const unsigned* row = s_go32 + ql * 16 + c;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const unsigned u = row[(j ^ sw) << 2];
            gf[j] = __uint_as_float(u << 16);
            gf[j + 4] = __uint_as_float(u & 0xffff0000u);
          }
        }
        float d = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) d = fmaf(gf[j], vf[j], d);
#pragma unroll
        for (int o = 1; o < LPP; o <<= 1) d += __shfl_xor_sync(gmask, d, o);
        if (c == 0) s_dot[id] = d;
        if (wgt != 0.f) {
          float* dst = acc_f + (off + c) * 8;
          red_add_f32x4(dst, wgt * gf[0], wgt * gf[1], wgt * gf[2], wgt * gf[3]);
          red_add_f32x4(dst + 4, wgt * gf[4], wgt * gf[5], wgt * gf[6], wgt * gf[7]);
        }
      }
    }
    __syncthreads();

    // ---- h: per-sample gradients; a corner that is not read (derivative code 1) has no dot
#pragma unroll
    for (int r = 0; r < SPT; ++r) {
      const int si = r * NT + tid;
      const int ql = si >> LP2, pt = si & (P - 1);
      const bool valid = ql < nq;
      const int q = valid ? (p.q_order ? p.q_order[q0 + ql] : q0 + ql) : 0;
      const long long gi = (((long long)b * p.Q + q) * p.H + h) * p.LP + l * P + pt;
      float4 d = *reinterpret_cast<const float4*>(&s_dot[si * 4]);
      const float4 w = s_w[si];
      const int gcode = s_xy[si] >> 24;
      const float a = s_a[si];
      const float gl = gdec(gcode, 0), gr = gdec(gcode, 1), gt = gdec(gcode, 2), gb = gdec(gcode, 3);
      d.x = (gl != 0.f && gt != 0.f) ? d.x : 0.f;
      d.y = (gr != 0.f && gt != 0.f) ? d.y : 0.f;
      d.z = (gl != 0.f && gb != 0.f) ? d.z : 0.f;
      d.w = (gr != 0.f && gb != 0.f) ? d.w : 0.f;
      const float top_s = w.x * d.x + w.y * d.y, bot_s = w.x * d.z + w.y * d.w;
      const float top_g = gl * d.x + gr * d.y, bot_g = gl * d.z + gr * d.w;
      const float g_attn = w.z * top_s + w.w * bot_s;
      const float g_px = w.z * top_g + w.w * bot_g, g_py = gt * top_s + gb * bot_s;
      if (!FUSED) {
        if (valid) {
          reinterpret_cast<AT*>(p.grad_attn)[gi] = from_float<AT>(g_attn);
          reinterpret_cast<float2*>(p.grad_loc)[gi] = make_float2((float)lv.W * a * g_px, (float)lv.H * a * g_py);
        }
      } else {
        if (valid) store_pair<AT>(p.grad_offsets, gi, a * g_px, a * g_py);
        ga_park[r][l] = g_attn;  // finished after the last level
        float t = valid ? a * g_attn : 0.f;  // the P samples of one (query, level) sit in P adjacent lanes
#pragma unroll
        for (int o = 1; o < P; o <<= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        f_dsum[r] += t;  // every one of the four lanes keeps the row's sum
      }
    }
  }

  if (FUSED) {
    // softmax backward over the L*P logits of each (query, head): g_j = a_j * (ga_j - sum_k a_k ga_k).  Lane pt of the
    // row's four lanes finishes the logits (l, pt) of every level l -- exactly the ones it parked itself in phase h.
#pragma unroll
    for (int r = 0; r < SPT; ++r) {
      const int ql = (r * NT + tid) >> LP2, pt = tid & (P - 1);
      if (ql < nq) {
        const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
        const long long row = (((long long)b * p.Q + q) * p.H + h) * p.LP;
        for (int l = 0; l < p.L; ++l) {
          const long long gi = row + l * P + pt;
          const float a = expf(to_float<AT>(reinterpret_cast<const AT*>(p.logits)[gi]) - f_lse[r]);
          reinterpret_cast<AT*>(p.grad_logits)[gi] = from_float<AT>(a * (ga_park[r][l] - f_dsum[r]));
        }
      }
    }
  }
}
