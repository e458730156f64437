// msda_b200.cu -- multi-scale deformable attention, forward + backward, for sm_100a (B200).
//
// Replaces transformers/models/mask2former/modeling_mask2former.py:798-837 (M2F:798) and the
// autograd graph behind it; C ABI in include/msda_b200.h.  See DESIGN.md for the data layout,
// the roofline of each kernel and the scheduling rationale.
//
// Kernel plan (one thread block = one (batch, head, tile of TQ queries)):
//   phase 1  every thread turns (loc, attn) of one sample into a *descriptor* in shared memory:
//            four slot weights, the 16-byte-unit offset of the top-left slot, done once per sample
//            instead of once per lane that touches the sample;
//   phase 2  LPP = D*sizeof(T)/16 lanes own one (query, head) pair and stream the L*P samples:
//            one broadcast LDS.128 for the weights, four 128-bit value loads (the 2x2 bilinear
//            footprint; each corner is one contiguous D*sizeof(T)-byte run), fp32 FMAs;
//   phase 3  (backward only) one thread per sample folds the per-lane partial dot products into
//            grad_attn / grad_loc.
//
// Out-of-range corners: the 2x2 footprint is clamped into the level and the bilinear weights are
// re-slotted (a corner that falls outside gets weight 0, the surviving one moves to the slot that
// is actually loaded), so phase 2 has no bounds checks and never forms an out-of-bounds address.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <type_traits>

#include "msda_b200.h"
#include "msda_bwd_det.cuh"

// msda_bwd_det.cu: the deterministic backward's sort and grad_value pull (CUB stays out of this file)
extern "C" int msda_b200_internal_det_workspace_bytes(const msda_b200_desc* desc, size_t* bytes);
extern "C" int msda_b200_internal_det_grad_value(const msda_b200_desc* desc, const void* grad_out, void* grad_value,
                                                 void* workspace, cudaStream_t stream);

namespace {

#include "msda_common.cuh"

template <int NT, int LPP, int QPG>
struct Tile {
  static constexpr int NG = NT / LPP;   // (query, head) pairs in flight per block
  static constexpr int TQ = NG * QPG;   // queries per block
  static constexpr int ROW = TQ + 1;    // padded row of the [sample][query] descriptor arrays
};

__device__ __forceinline__ void decode_block(const KParams& p, int& b, int& tile, int& h) {
  int bid = blockIdx.x;
  h = bid % p.H;
  bid /= p.H;
  tile = bid % p.num_tiles;
  b = bid / p.num_tiles;
}

// ---------------------------------------------------------------------------------------------
// Fused prologue helpers (M2F:952-971): attn = softmax(logits over L*P), loc = ref + off / (W_l, H_l)
// ---------------------------------------------------------------------------------------------
template <typename AT>
__device__ __forceinline__ float2 load_pair(const void* base, long long idx);
template <>
__device__ __forceinline__ float2 load_pair<float>(const void* base, long long idx) {
  return __ldg(reinterpret_cast<const float2*>(base) + idx);
}
template <>
__device__ __forceinline__ float2 load_pair<__nv_bfloat16>(const void* base, long long idx) {
  const __nv_bfloat162 v = reinterpret_cast<const __nv_bfloat162*>(base)[idx];
  return make_float2(__low2float(v), __high2float(v));
}
template <typename AT>
__device__ __forceinline__ void store_pair(void* base, long long idx, float x, float y);
template <>
__device__ __forceinline__ void store_pair<float>(void* base, long long idx, float x, float y) {
  reinterpret_cast<float2*>(base)[idx] = make_float2(x, y);
}
template <>
__device__ __forceinline__ void store_pair<__nv_bfloat16>(void* base, long long idx, float x, float y) {
  reinterpret_cast<__nv_bfloat162*>(base)[idx] = __floats2bfloat162_rn(x, y);
}

// Reference point of query q when the caller passes none (ref == NULL; requires Q == S): the query IS pixel q of its
// level and its reference point is the centre of that pixel, the same for every level -- what
// Mask2FormerPixelDecoderEncoderOnly.get_reference_points (M2F:1095-1125) computes with valid_ratios == 1:
// linspace(0.5, n - 0.5, n)[i] / n = (i + 0.5) / n in fp32, bit for bit.
__device__ __forceinline__ float2 implicit_reference_point(const KParams& p, int q) {
  int lq = 0;
  for (int l = 1; l < p.L; ++l)
    if (q >= p.lv[l].start) lq = l;  // levels are stored in increasing row order
  const int r = q - p.lv[lq].start, W = p.lv[lq].W, H = p.lv[lq].H;
  const int y = r / W, x = r - y * W;
  return make_float2(__fdiv_rn((float)x + 0.5f, (float)W), __fdiv_rn((float)y + 0.5f, (float)H));
}

// si: global sample index ((b*Q+q)*H+h)*LP + s; ri: reference-point index (b*Q+q)*L + l
template <typename AT>
__device__ __forceinline__ float2 fused_loc(const KParams& p, long long si, long long ri, int q, const Level& lv) {
  const float2 off = load_pair<AT>(p.offsets, si);
  const float2 r = p.ref ? __ldg(reinterpret_cast<const float2*>(p.ref) + ri) : implicit_reference_point(p, q);
  return make_float2(__fadd_rn(r.x, __fdiv_rn(off.x, (float)lv.W)), __fadd_rn(r.y, __fdiv_rn(off.y, (float)lv.H)));
}

// max and 1 / sum(exp(x - max)) of the LP logits of one (query, head)
template <typename AT>
__device__ __forceinline__ void softmax_stats(const AT* lg, int LP, float& mx, float& inv) {
  mx = -INFINITY;
  for (int s = 0; s < LP; ++s) mx = fmaxf(mx, to_float<AT>(lg[s]));
  float sum = 0.f;
  for (int s = 0; s < LP; ++s) sum += expf(to_float<AT>(lg[s]) - mx);
  inv = 1.f / sum;
}

// max and 1/sum(exp(x - max)) of one (query, head) row, computed by four adjacent lanes (lane & 3 = sub) that each
// take every fourth logit; every lane of the warp must call it (full-mask shuffles), `valid` masks idle rows
template <typename AT>
__device__ __forceinline__ void softmax_stats_x4(const AT* lg, int LP, int sub, bool valid, float& mx, float& inv) {
  mx = -INFINITY;
  if (valid)
    for (int s = sub; s < LP; s += 4) mx = fmaxf(mx, to_float<AT>(lg[s]));
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
  float sum = 0.f;
  if (valid)
    for (int s = sub; s < LP; s += 4) sum += expf(to_float<AT>(lg[s]) - mx);
  sum += __shfl_xor_sync(0xffffffffu, sum, 1);
  sum += __shfl_xor_sync(0xffffffffu, sum, 2);
  inv = valid ? 1.f / sum : 0.f;
}

// softmax of the tile's (query, head) rows into shared memory, four lanes per row; row v = ql * HPB + hl is query
// q0 + ql, head h0 + hl. Each lane keeps its (up to four) logits in registers: ONE expf per logit (rows longer than
// 16 logits take the three-pass form).
template <typename AT, int NT, int HPB>
__device__ __forceinline__ void tile_softmax(const KParams& p, int b, int h0, int q0, int nq, float* s_att, bool write_out) {
  const int LP = p.LP;
  const int sub = threadIdx.x & 3;
  const int nv = nq * HPB;
  for (int vb0 = 0; vb0 < nv; vb0 += NT / 4) {
    const int v = vb0 + (threadIdx.x >> 2);
    const bool valid = v < nv;
    const int ql = v / HPB, h = h0 + v % HPB;
    const int q = valid ? (p.q_order ? p.q_order[q0 + ql] : q0 + ql) : 0;
    const long long row = (((long long)b * p.Q + q) * p.H + h) * LP;
    const AT* lg = reinterpret_cast<const AT*>(p.logits) + row;
    if (LP <= 16) {
      float e[4];
      float mx = -INFINITY;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int s = sub + 4 * r;
        e[r] = (valid && s < LP) ? to_float<AT>(lg[s]) : -INFINITY;
        mx = fmaxf(mx, e[r]);
      }
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      float sum = 0.f;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        e[r] = (valid && sub + 4 * r < LP) ? expf(e[r] - mx) : 0.f;
        sum += e[r];
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      const float inv = 1.f / sum;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int s = sub + 4 * r;
        if (valid && s < LP) {
          const float a = e[r] * inv;
          s_att[v * LP + s] = a;
          if (write_out && p.attn_out) p.attn_out[row + s] = a;
        }
      }
    } else {
      float mx, inv;
      softmax_stats_x4<AT>(lg, LP, sub, valid, mx, inv);
      if (valid)
        for (int s = sub; s < LP; s += 4) {
          const float a = expf(to_float<AT>(lg[s]) - mx) * inv;
          s_att[v * LP + s] = a;
          if (write_out && p.attn_out) p.attn_out[row + s] = a;
        }
    }
  }
}

// One sample for one lane: four 16-byte corner loads and the weighted accumulation.
// STRICT = false (default): a slot outside the level has weight exactly 0 but is still loaded from the clamped pixel
//   next to it and multiplied. With finite activations that is grid_sample's zeros padding (M2F:823) exactly.
// STRICT = true (MSDA_B200_FLAG_STRICT_PADDING): the FMA of a zero-weight corner is skipped, so a non-finite value in
//   a pixel the reference never reads cannot turn into 0 * Inf = NaN. Measured on B200 (profiles/r02_notes.md): every
//   way of guarding the corner costs 25-30 % of the forward (0.29 -> 0.38 ms): a branch per corner stops the compiler
//   from overlapping the loads of neighbouring samples, and ptxas lowers a predicated FFMA2 to FFMA2 + two SELs.
//   Hence a flag, not the default. (An in-bounds corner whose weight is exactly 0 is skipped too; the reference
//   multiplies it, which differs only if that pixel is itself non-finite.)
template <typename VT, int VEC, bool STRICT>
__device__ __forceinline__ void gather_sample(const uint4* ptr, int dx, int dy, const float4& w, float (&acc)[VEC]) {
  const uint4 v00 = ldg16(ptr), v01 = ldg16(ptr + dx), v10 = ldg16(ptr + dy), v11 = ldg16(ptr + dy + dx);
  float f[VEC];
  Vec16<VT>::unpack(v00, f);
  if (!STRICT || w.x != 0.f) {
#pragma unroll
    for (int j = 0; j < VEC; j += 2) fma2_scalar(acc[j], acc[j + 1], w.x, f[j], f[j + 1]);
  }
  Vec16<VT>::unpack(v01, f);
  if (!STRICT || w.y != 0.f) {
#pragma unroll
    for (int j = 0; j < VEC; j += 2) fma2_scalar(acc[j], acc[j + 1], w.y, f[j], f[j + 1]);
  }
  Vec16<VT>::unpack(v10, f);
  if (!STRICT || w.z != 0.f) {
#pragma unroll
    for (int j = 0; j < VEC; j += 2) fma2_scalar(acc[j], acc[j + 1], w.z, f[j], f[j + 1]);
  }
  Vec16<VT>::unpack(v11, f);
  if (!STRICT || w.w != 0.f) {
#pragma unroll
    for (int j = 0; j < VEC; j += 2) fma2_scalar(acc[j], acc[j + 1], w.w, f[j], f[j + 1]);
  }
}

// ---------------------------------------------------------------------------------------------
// Forward
// ---------------------------------------------------------------------------------------------
template <typename VT, typename AT, int D, int NT, int QPG, bool FUSED, bool STRICT>
__global__ void __launch_bounds__(NT) msda_fwd_kernel(const __grid_constant__ KParams p) {
  constexpr int VEC = Vec16<VT>::N;
  constexpr int LPP = D / VEC;
  using T = Tile<NT, LPP, QPG>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* sw = reinterpret_cast<float4*>(smem_raw);                    // [LP][ROW] slot weights * attn
  int* soff = reinterpret_cast<int*>(smem_raw + (size_t)p.LP * T::ROW * sizeof(float4));  // [LP][ROW]
  float* s_att = reinterpret_cast<float*>(soff + (size_t)p.LP * T::ROW);                  // FUSED: [TQ][LP] softmax

  int b, tile, h;
  decode_block(p, b, tile, h);
  const int q0 = tile * T::TQ;
  const int nq = min(T::TQ, p.Q - q0);
  const int LP = p.LP;

  if (FUSED) {
    tile_softmax<AT, NT, 1>(p, b, h, q0, nq, s_att, true);
    __syncthreads();
  }

  // ---- phase 1: descriptors
  for (int i = threadIdx.x; i < nq * LP; i += NT) {
    const int ql = i / LP, s = i - ql * LP;
    const int l = s / p.P;
    const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
    const long long si = (((long long)b * p.Q + q) * p.H + h) * LP + s;
    const Level lv = p.lv[l];
    const float2 xy = FUSED ? fused_loc<AT>(p, si, ((long long)b * p.Q + q) * p.L + l, q, lv)
                            : __ldg(reinterpret_cast<const float2*>(p.loc) + si);
    const float a = FUSED ? s_att[i] : to_float<AT>(reinterpret_cast<const AT*>(p.attn)[si]);
    const Axis ax = axis_setup(xy.x, lv.W), ay = axis_setup(xy.y, lv.H);
    const bool ok = ax.ok && ay.ok;
    const float wt = ok ? a * ay.s0 : 0.f, wb = ok ? a * ay.s1 : 0.f;
    sw[s * T::ROW + ql] = make_float4(wt * ax.s0, wt * ax.s1, wb * ax.s0, wb * ax.s1);
    soff[s * T::ROW + ql] = ((lv.start + ay.base * lv.W + ax.base) * p.H + h) * LPP;
  }
  __syncthreads();

  // ---- phase 2: gather
  const int g = threadIdx.x / LPP, c = threadIdx.x % LPP;
  const uint4* vb = reinterpret_cast<const uint4*>(p.value) + (long long)b * p.batch_stride16 + c;
#pragma unroll
  for (int it = 0; it < QPG; ++it) {
    const int ql = g + it * T::NG;
    if (ql >= nq) break;
    float acc[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
    for (int l = 0; l < p.L; ++l) {
      const int dx = p.lv[l].dx16, dy = p.lv[l].dy16;
#pragma unroll 4
      for (int pt = 0; pt < p.P; ++pt) {
        const int s = l * p.P + pt;
        gather_sample<VT, VEC, STRICT>(vb + soff[s * T::ROW + ql], dx, dy, sw[s * T::ROW + ql], acc);
      }
    }
    const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
    uint4* o = reinterpret_cast<uint4*>(p.out) + (((long long)b * p.Q + q) * p.H + h) * LPP + c;
    *o = Vec16<VT>::pack(acc);
  }
}

// ---------------------------------------------------------------------------------------------
// Forward, HPB heads per block (round 2)
// ---------------------------------------------------------------------------------------------
// Measured (profiles/r02_micro2.log): the L1 data array is banked like shared memory, and a warp-wide 128-bit load is
// served a quarter-warp (8 lanes) at a time. One head's D*sizeof(T) = 64-byte run always lies in the SAME half of its
// 128-byte line (offset h*64 inside the 512-byte pixel row), so two lane groups of one head always collide: 2
// wavefronts per quarter-warp, a 64 B/clk/SM ceiling -- msda_fwd_kernel runs at 73 % of exactly that. Here the lane
// groups of a block alternate between an even and an odd head, so the two 64-byte runs of every quarter-warp fall into
// different halves and the request is conflict-free (127 B/clk/SM measured). It also makes every fetched 128-byte line
// fully useful. Virtual query v = ql * HPB + hl  <->  query q0 + ql, head h0 + hl.
// LC: compile-time level count with P == 4 (0 = generic L / P from the descriptor).  With LC != 0 one thread builds the
// four descriptors of one (query, head, level): its locations are one 32-byte run, its attention weights one 8- or
// 16-byte run, and the index arithmetic (runtime divisions by L*P and P in the generic loop) is paid once per four
// samples -- the descriptor phase was 42 % of the forward (ncu r02_fwd_pair).
template <typename VT, typename AT, int D, int NT, int QPG, int HPB, bool FUSED, int LC>
__global__ void __launch_bounds__(NT) msda_fwd_pair_kernel(const __grid_constant__ KParams p) {
  constexpr int VEC = Vec16<VT>::N;
  constexpr int LPP = D / VEC;
  constexpr int NG = NT / LPP, TV = NG * QPG, TQ = TV / HPB, ROW = TV + 1;
  static_assert(NG % HPB == 0 && TV % HPB == 0, "lane groups must split evenly over the heads");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* sw = reinterpret_cast<float4*>(smem_raw);                                         // [LP][ROW] slot weights * attn
  int* soff = reinterpret_cast<int*>(smem_raw + (size_t)p.LP * ROW * sizeof(float4));       // [LP][ROW]
  float* s_att = reinterpret_cast<float*>(soff + (size_t)p.LP * ROW);                       // FUSED: [TV][LP] softmax
  float* s_ref = s_att + (size_t)TV * p.LP;                                                 // FUSED: [TQ][2] implicit ref points
  static_assert(TQ <= NT, "one thread per query computes its reference point");

  int bid = blockIdx.x;
  const int hgroups = p.H / HPB;
  const int h0 = (bid % hgroups) * HPB;
  bid /= hgroups;
  const int tile = bid % p.num_tiles;
  const int b = bid / p.num_tiles;
  const int q0 = tile * TQ;
  const int nq = min(TQ, p.Q - q0);
  const int nv = nq * HPB;
  const int LP = LC ? LC * 4 : p.LP;
  // (Measured and dropped: one block walking 2 / 4 / 8 consecutive strips of a patch so that later strips find the
  // value rows in L1 -- 0.291 / 0.301 / 0.325 ms against 0.291 for one strip per block, profiles/r02_notes.md.)

  if (FUSED) {
    // implicit reference points: once per query of the tile (they depend on neither head nor level)
    if (!p.ref && threadIdx.x < nq) {
      const float2 r = implicit_reference_point(p, p.q_order ? p.q_order[q0 + threadIdx.x] : q0 + threadIdx.x);
      s_ref[2 * threadIdx.x] = r.x;
      s_ref[2 * threadIdx.x + 1] = r.y;
    }
    tile_softmax<AT, NT, HPB>(p, b, h0, q0, nq, s_att, true);
    __syncthreads();
  }

  // ---- phase 1: descriptors (the LP samples of the HPB heads of one query are adjacent in memory)
  if (LC) {
    constexpr int PC = 4;
    // thread <-> (level, virtual query) with the virtual query on the fast axis: the float4 descriptor stores of a
    // quarter-warp then fall into eight different 16-byte bank groups (level-fastest, rows 4 * ROW * 16 = 64 (mod 128)
    // bytes apart, made them collide two ways: 3.4 M of the kernel's 6.0 M shared-store wavefronts, ncu r02)
    for (int i = threadIdx.x; i < TV * LC; i += NT) {
      const int l = i / TV, v = i - l * TV;
      if (v >= nv) continue;
      const int ql = v / HPB, h = h0 + v % HPB;
      const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
      const long long si = (((long long)b * p.Q + q) * p.H + h) * (LC * PC) + l * PC;
      const Level lv = p.lv[l];
      float2 xy[PC];
      float a[PC];
      if (FUSED) {
        const float2 r = p.ref ? __ldg(reinterpret_cast<const float2*>(p.ref) + ((long long)b * p.Q + q) * LC + l) : make_float2(s_ref[2 * ql], s_ref[2 * ql + 1]);
        float2 off[PC];
        if (std::is_same<AT, float>::value) {
          const float4 o0 = __ldg(reinterpret_cast<const float4*>(p.offsets) + si / 2);
          const float4 o1 = __ldg(reinterpret_cast<const float4*>(p.offsets) + si / 2 + 1);
          off[0] = make_float2(o0.x, o0.y); off[1] = make_float2(o0.z, o0.w);
          off[2] = make_float2(o1.x, o1.y); off[3] = make_float2(o1.z, o1.w);
        } else {
          const uint4 o = ldg16(reinterpret_cast<const uint4*>(p.offsets) + si / 4);
          float f[8];
          Vec16<__nv_bfloat16>::unpack(o, f);
#pragma unroll
          for (int pt = 0; pt < PC; ++pt) off[pt] = make_float2(f[2 * pt], f[2 * pt + 1]);
        }
#pragma unroll
        for (int pt = 0; pt < PC; ++pt) {
          xy[pt] = make_float2(__fadd_rn(r.x, __fdiv_rn(off[pt].x, (float)lv.W)), __fadd_rn(r.y, __fdiv_rn(off[pt].y, (float)lv.H)));
          a[pt] = s_att[v * (LC * PC) + l * PC + pt];
        }
      } else {
        const float4 l0 = __ldg(reinterpret_cast<const float4*>(p.loc) + si / 2);
        const float4 l1 = __ldg(reinterpret_cast<const float4*>(p.loc) + si / 2 + 1);
        xy[0] = make_float2(l0.x, l0.y); xy[1] = make_float2(l0.z, l0.w);
        xy[2] = make_float2(l1.x, l1.y); xy[3] = make_float2(l1.z, l1.w);
        if (std::is_same<AT, float>::value) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(p.attn) + si / 4);
          a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
        } else {
          const uint2 t = __ldg(reinterpret_cast<const uint2*>(p.attn) + si / 4);
          a[0] = __uint_as_float(t.x << 16); a[1] = __uint_as_float(t.x & 0xffff0000u);
          a[2] = __uint_as_float(t.y << 16); a[3] = __uint_as_float(t.y & 0xffff0000u);
        }
      }
      const int pix0 = lv.start * p.H + h;
#pragma unroll
      for (int pt = 0; pt < PC; ++pt) {
        const Axis ax = axis_setup(xy[pt].x, lv.W), ay = axis_setup(xy[pt].y, lv.H);
        const bool ok = ax.ok && ay.ok;
        const float wt = ok ? a[pt] * ay.s0 : 0.f, wb = ok ? a[pt] * ay.s1 : 0.f;
        const int s = l * PC + pt;
        sw[s * ROW + v] = make_float4(wt * ax.s0, wt * ax.s1, wb * ax.s0, wb * ax.s1);
        soff[s * ROW + v] = (pix0 + (ay.base * lv.W + ax.base) * p.H) * LPP;
      }
    }
  } else {
    for (int i = threadIdx.x; i < nv * LP; i += NT) {
      const int v = i / LP, s = i - v * LP;
      const int ql = v / HPB, h = h0 + v % HPB;
      const int l = s / p.P;
      const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
      const long long si = (((long long)b * p.Q + q) * p.H + h) * LP + s;
      const Level lv = p.lv[l];
      const float2 xy = FUSED ? fused_loc<AT>(p, si, ((long long)b * p.Q + q) * p.L + l, q, lv)
                              : __ldg(reinterpret_cast<const float2*>(p.loc) + si);
      const float a = FUSED ? s_att[i] : to_float<AT>(reinterpret_cast<const AT*>(p.attn)[si]);
      const Axis ax = axis_setup(xy.x, lv.W), ay = axis_setup(xy.y, lv.H);
      const bool ok = ax.ok && ay.ok;
      const float wt = ok ? a * ay.s0 : 0.f, wb = ok ? a * ay.s1 : 0.f;
      sw[s * ROW + v] = make_float4(wt * ax.s0, wt * ax.s1, wb * ax.s0, wb * ax.s1);
      soff[s * ROW + v] = ((lv.start + ay.base * lv.W + ax.base) * p.H + h) * LPP;
    }
  }
  __syncthreads();

  // ---- phase 2: gather
  const int g = threadIdx.x / LPP, c = threadIdx.x % LPP;
  const uint4* vb = reinterpret_cast<const uint4*>(p.value) + (long long)b * p.batch_stride16 + c;
#pragma unroll
  for (int it = 0; it < QPG; ++it) {
    const int v = g + it * NG;
    if (v >= nv) break;
    float acc[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
    const int nl = LC ? LC : p.L, np = LC ? 4 : p.P;
    for (int l = 0; l < nl; ++l) {
      const int dx = p.lv[l].dx16, dy = p.lv[l].dy16;
#pragma unroll 4
      for (int pt = 0; pt < np; ++pt) {
        const int s = l * np + pt;
        gather_sample<VT, VEC, false>(vb + soff[s * ROW + v], dx, dy, sw[s * ROW + v], acc);
      }
    }
    const int ql = v / HPB, h = h0 + v % HPB;
    const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
    uint4* o = reinterpret_cast<uint4*>(p.out) + (((long long)b * p.Q + q) * p.H + h) * LPP + c;
    *o = Vec16<VT>::pack(acc);
  }
}

// ---------------------------------------------------------------------------------------------
// Backward
// ---------------------------------------------------------------------------------------------
// ACC: 0 = fp32 accumulator with red.v4.f32 (grad_value itself for fp32 values, workspace for bf16)
//      1 = bf16 grad_value accumulated in place with red.v4.bf16x2 (MSDA_B200_FLAG_BF16_ATOMICS)
//      2 = no grad_value scatter: phase 1 writes each sample's grad_value records for msda_bwd_det.cu
//          (MSDA_B200_FLAG_DETERMINISTIC); grad_loc / grad_attn as in the other modes
template <typename VT, typename AT, int D, int NT, int QPG, int ACC, bool FUSED>
__global__ void __launch_bounds__(NT) msda_bwd_kernel(const __grid_constant__ KParams p) {
  constexpr int VEC = Vec16<VT>::N;
  constexpr int LPP = D / VEC;
  using T = Tile<NT, LPP, QPG>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int LP = p.LP;
  const size_t n = (size_t)LP * T::ROW;
  float4* ss = reinterpret_cast<float4*>(smem_raw);     // [LP][ROW] (sL, sR, sT, sB)
  float4* sg = ss + n;                                  // [LP][ROW] (gL, gR, gT, gB)
  float4* sd = sg + n;                                  // [LP][TQ][LPP] per-lane partial dots
  float* sa = reinterpret_cast<float*>(sd + (size_t)LP * T::TQ * LPP);  // [LP][ROW] attn
  int* soff = reinterpret_cast<int*>(sa + n);           // [LP][ROW]
  float* s_att = reinterpret_cast<float*>(soff + n);    // FUSED: [TQ][LP] softmax
  float* s_ga = s_att + (size_t)T::TQ * LP;             // FUSED: [TQ][LP] d loss / d attn

  int b, tile, h;
  decode_block(p, b, tile, h);
  const int q0 = tile * T::TQ;
  const int nq = min(T::TQ, p.Q - q0);

  if (FUSED) {
    tile_softmax<AT, NT, 1>(p, b, h, q0, nq, s_att, false);
    __syncthreads();
  }

  // ---- phase 1: descriptors
  for (int i = threadIdx.x; i < nq * LP; i += NT) {
    const int ql = i / LP, s = i - ql * LP;
    const int l = s / p.P;
    const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
    const long long si = (((long long)b * p.Q + q) * p.H + h) * LP + s;
    const Level lv = p.lv[l];
    const float2 xy = FUSED ? fused_loc<AT>(p, si, ((long long)b * p.Q + q) * p.L + l, q, lv)
                            : __ldg(reinterpret_cast<const float2*>(p.loc) + si);
    const float a = FUSED ? s_att[i] : to_float<AT>(reinterpret_cast<const AT*>(p.attn)[si]);
    const Axis ax = axis_setup(xy.x, lv.W), ay = axis_setup(xy.y, lv.H);
    const bool ok = ax.ok && ay.ok;
    const int k = s * T::ROW + ql;
    ss[k] = ok ? make_float4(ax.s0, ax.s1, ay.s0, ay.s1) : make_float4(0.f, 0.f, 0.f, 0.f);
    sg[k] = ok ? make_float4(ax.g0, ax.g1, ay.g0, ay.g1) : make_float4(0.f, 0.f, 0.f, 0.f);
    sa[k] = a;
    // a slot outside the level ("dead": derivative code 0) must not be read at all (zeros padding, M2F:823): samples
    // that have one are flagged in the sign bit and take predicated loads in phase 2
    const bool all_alive = ok && ax.g0 != 0.f && ax.g1 != 0.f && ay.g0 != 0.f && ay.g1 != 0.f;
    soff[k] = (((lv.start + ay.base * lv.W + ax.base) * p.H + h) * LPP) | (all_alive ? 0 : (int)0x80000000);
    if (ACC == 2) {
      // grad_value records of the four slots (msda_bwd_det.cuh), with phase 2's liveness rule and weight expression
      const float sx[2] = {ax.s0, ax.s1}, sy[2] = {ay.s0, ay.s1};
      const bool gx[2] = {ax.g0 != 0.f, ax.g1 != 0.f}, gy[2] = {ay.g0 != 0.f, ay.g1 != 0.f};
      const long long row0 = (long long)b * p.S + lv.start + ay.base * lv.W + ax.base;
      unsigned key[4];
      unsigned long long val[4];
#pragma unroll
      for (int cn = 0; cn < 4; ++cn) {
        const int cy = cn >> 1, cx = cn & 1;
        const float wc = a * sy[cy] * sx[cx];
        const bool live = ok && gx[cx] && gy[cy] && wc != 0.f;
        key[cn] = live ? (unsigned)((row0 + cy * lv.W + cx) * p.H + h) : p.det_sentinel;
        val[cn] = ((unsigned long long)q << 32) | __float_as_uint(wc);
      }
      uint4* kd = reinterpret_cast<uint4*>(p.det_keys) + si;
      *kd = make_uint4(key[0], key[1], key[2], key[3]);
      ulonglong2* vd = reinterpret_cast<ulonglong2*>(p.det_vals) + 2 * si;
      vd[0] = make_ulonglong2(val[0], val[1]);
      vd[1] = make_ulonglong2(val[2], val[3]);
    }
  }
  __syncthreads();

  // ---- phase 2: gather value corners, scatter grad_value, per-lane partial dots
  const int g = threadIdx.x / LPP, c = threadIdx.x % LPP;
  const uint4* vb = reinterpret_cast<const uint4*>(p.value) + (long long)b * p.batch_stride16 + c;
#pragma unroll
  for (int it = 0; it < QPG; ++it) {
    const int ql = g + it * T::NG;
    if (ql >= nq) break;
    const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
    float go[VEC];
    {
      const uint4 gv = ldg16(reinterpret_cast<const uint4*>(p.grad_out) + (((long long)b * p.Q + q) * p.H + h) * LPP + c);
      Vec16<VT>::unpack(gv, go);
    }
    for (int l = 0; l < p.L; ++l) {
      const int dx = p.lv[l].dx16, dy = p.lv[l].dy16;
#pragma unroll 2
      for (int pt = 0; pt < p.P; ++pt) {
        const int s = l * p.P + pt;
        const int k = s * T::ROW + ql;
        const float4 w = ss[k];
        const float a = sa[k];
        const int off_flag = soff[k];
        const int off = off_flag & 0x7fffffff;
        const uint4* ptr = vb + off;
        const int coff[4] = {0, dx, dy, dy + dx};
        bool alive[4] = {true, true, true, true};
        if (off_flag < 0) {
          const float4 gw = sg[k];
          alive[0] = gw.x != 0.f && gw.z != 0.f; alive[1] = gw.y != 0.f && gw.z != 0.f;
          alive[2] = gw.x != 0.f && gw.w != 0.f; alive[3] = gw.y != 0.f && gw.w != 0.f;
        }
        uint4 v[4];
#pragma unroll
        for (int cn = 0; cn < 4; ++cn) v[cn] = alive[cn] ? ldg16(ptr + coff[cn]) : make_uint4(0u, 0u, 0u, 0u);
        const float wc[4] = {a * w.z * w.x, a * w.z * w.y, a * w.w * w.x, a * w.w * w.y};
        float dot[4];
#pragma unroll
        for (int cn = 0; cn < 4; ++cn) {
          float f[VEC];
          Vec16<VT>::unpack(v[cn], f);
          float d = 0.f;
#pragma unroll
          for (int j = 0; j < VEC; ++j) d = fmaf(go[j], f[j], d);
          dot[cn] = d;
          if (ACC != 2 && alive[cn] && wc[cn] != 0.f) {
            // element offset of this lane's 16 bytes inside grad_value
            const long long e = ((long long)b * p.batch_stride16 + off + coff[cn] + c) * VEC;
            if (ACC == 0) {
              float* dst = reinterpret_cast<float*>(p.grad_value_acc) + e;
#pragma unroll
              for (int j = 0; j < VEC; j += 4)
                red_add_f32x4(dst + j, wc[cn] * go[j], wc[cn] * go[j + 1], wc[cn] * go[j + 2], wc[cn] * go[j + 3]);
            } else {
              float t[VEC];
#pragma unroll
              for (int j = 0; j < VEC; ++j) t[j] = wc[cn] * go[j];
              const uint4 pk = Vec16<VT>::pack(t);
              red_add_bf16x8(reinterpret_cast<VT*>(p.grad_value_acc) + e, pk.x, pk.y, pk.z, pk.w);
            }
          }
        }
        sd[((size_t)s * T::TQ + ql) * LPP + c] = make_float4(dot[0], dot[1], dot[2], dot[3]);
      }
    }
  }
  __syncthreads();

  // ---- phase 3: per-sample gradients of attention weights and sampling locations
  for (int i = threadIdx.x; i < nq * LP; i += NT) {
    const int ql = i / LP, s = i - ql * LP;
    const int l = s / p.P;
    const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
    const long long si = (((long long)b * p.Q + q) * p.H + h) * LP + s;
    float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* part = sd + ((size_t)s * T::TQ + ql) * LPP;
#pragma unroll
    for (int j = 0; j < LPP; ++j) {
      const float4 t = part[j];
      d.x += t.x; d.y += t.y; d.z += t.z; d.w += t.w;
    }
    const int k = s * T::ROW + ql;
    const float4 w = ss[k], gw = sg[k];
    const float a = sa[k];
    // d.x=(top,left) d.y=(top,right) d.z=(bottom,left) d.w=(bottom,right)
    const float top_s = w.x * d.x + w.y * d.y, bot_s = w.x * d.z + w.y * d.w;
    const float top_g = gw.x * d.x + gw.y * d.y, bot_g = gw.x * d.z + gw.y * d.w;
    const float g_attn = w.z * top_s + w.w * bot_s;
    const float g_px = w.z * top_g + w.w * bot_g;
    const float g_py = gw.z * top_s + gw.w * bot_s;
    if (FUSED) {
      // loc = ref + off / (W, H)  =>  d/d off = (d/d loc) / (W, H) = attn * d sample / d pixel
      store_pair<AT>(p.grad_offsets, si, a * g_px, a * g_py);
      s_ga[i] = g_attn;
    } else {
      reinterpret_cast<AT*>(p.grad_attn)[si] = from_float<AT>(g_attn);
      reinterpret_cast<float2*>(p.grad_loc)[si] = make_float2((float)p.lv[l].W * a * g_px, (float)p.lv[l].H * a * g_py);
    }
  }
  if (FUSED) {
    // softmax backward over the L*P logits of each (query, head): g_j = a_j * (ga_j - sum_k a_k ga_k)
    __syncthreads();
    for (int ql = threadIdx.x; ql < nq; ql += NT) {
      const int q = p.q_order ? p.q_order[q0 + ql] : q0 + ql;
      const long long row = (((long long)b * p.Q + q) * p.H + h) * LP;
      float dotsum = 0.f;
      for (int s = 0; s < LP; ++s) dotsum = fmaf(s_att[ql * LP + s], s_ga[ql * LP + s], dotsum);
      for (int s = 0; s < LP; ++s)
        reinterpret_cast<AT*>(p.grad_logits)[row + s] = from_float<AT>(s_att[ql * LP + s] * (s_ga[ql * LP + s] - dotsum));
    }
  }
}

#include "msda_bwd_sorted.cuh"
#include "msda_bwd_mma.cuh"

// fp32 accumulator -> bf16 grad_value, 8 elements per thread
__global__ void __launch_bounds__(256) msda_cvt_f32_bf16_kernel(const float4* __restrict__ src, uint4* __restrict__ dst,
                                                               long long n8) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const float4 a = __ldcs(src + 2 * i), b2 = __ldcs(src + 2 * i + 1);
    const float f[8] = {a.x, a.y, a.z, a.w, b2.x, b2.y, b2.z, b2.w};
    __stcs(dst + i, Vec16<__nv_bfloat16>::pack(f));
  }
}

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};  // process-wide: autograd runs backward on its own thread

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

struct Prof {
  int device = -1;
  cudaEvent_t ev[MSDA_B200_PROF_COUNT][2];
  bool valid[MSDA_B200_PROF_COUNT] = {};
};
thread_local Prof g_prof;

bool prof_prepare() {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return false;
  if (g_prof.device == dev) return true;
  if (g_prof.device >= 0) {
    // the old events belong to another device: release them there, then come back
    if (cudaSetDevice(g_prof.device) == cudaSuccess)
      for (int i = 0; i < MSDA_B200_PROF_COUNT; ++i) {
        cudaEventDestroy(g_prof.ev[i][0]);
        cudaEventDestroy(g_prof.ev[i][1]);
      }
    g_prof.device = -1;
    if (cudaSetDevice(dev) != cudaSuccess) return false;
  }
  for (int i = 0; i < MSDA_B200_PROF_COUNT; ++i) {
    if (cudaEventCreate(&g_prof.ev[i][0]) != cudaSuccess) return false;
    if (cudaEventCreate(&g_prof.ev[i][1]) != cudaSuccess) return false;
    g_prof.valid[i] = false;
  }
  g_prof.device = dev;
  return true;
}

struct ProfScope {
  int which;
  cudaStream_t st;
  bool on;
  ProfScope(bool enabled, int w, cudaStream_t s) : which(w), st(s), on(enabled && prof_prepare()) {
    if (on) cudaEventRecord(g_prof.ev[which][0], st);
  }
  ~ProfScope() {
    if (on) {
      cudaEventRecord(g_prof.ev[which][1], st);
      g_prof.valid[which] = true;
    }
  }
};

size_t dtype_size(int dt) { return dt == MSDA_B200_BF16 ? 2 : 4; }

int validate(const msda_b200_desc* d) {
  if (!d) return fail(MSDA_B200_ERR_INVALID, "desc is NULL");
  if (d->B < 0 || d->S < 0 || d->Q < 0) return fail(MSDA_B200_ERR_INVALID, "negative B/S/Q (%d, %d, %d)", d->B, d->S, d->Q);
  if (d->H <= 0 || d->D <= 0 || d->L <= 0 || d->P <= 0)
    return fail(MSDA_B200_ERR_INVALID, "H, D, L, P must be positive (%d, %d, %d, %d)", d->H, d->D, d->L, d->P);
  if (d->L > kMaxL) return fail(MSDA_B200_ERR_UNSUPPORTED, "L=%d exceeds MSDA_B200_MAX_LEVELS=%d", d->L, kMaxL);
  if (d->value_dtype != MSDA_B200_F32 && d->value_dtype != MSDA_B200_BF16)
    return fail(MSDA_B200_ERR_UNSUPPORTED, "value_dtype %d (want 0=f32 or 1=bf16)", d->value_dtype);
  if (d->attn_dtype != MSDA_B200_F32 && d->attn_dtype != MSDA_B200_BF16)
    return fail(MSDA_B200_ERR_UNSUPPORTED, "attn_dtype %d (want 0=f32 or 1=bf16)", d->attn_dtype);
  if (d->value_dtype == MSDA_B200_F32 && d->attn_dtype != MSDA_B200_F32)
    return fail(MSDA_B200_ERR_UNSUPPORTED, "fp32 values need fp32 attention weights");
  if (d->D != 8 && d->D != 16 && d->D != 32 && d->D != 64 && d->D != 128)
    return fail(MSDA_B200_ERR_UNSUPPORTED, "head dim D=%d (kernels exist for 8, 16, 32, 64, 128)", d->D);
  if (!d->spatial_shapes_hw || !d->level_start_index)
    return fail(MSDA_B200_ERR_INVALID, "spatial_shapes_hw / level_start_index is NULL");
  for (int l = 0; l < d->L; ++l) {
    const long long hh = d->spatial_shapes_hw[2 * l], ww = d->spatial_shapes_hw[2 * l + 1];
    const long long st = d->level_start_index[l];
    if (hh <= 0 || ww <= 0) return fail(MSDA_B200_ERR_INVALID, "level %d has non-positive shape (%lld, %lld)", l, hh, ww);
    if (st < 0 || st + hh * ww > d->S)
      return fail(MSDA_B200_ERR_INVALID, "level %d rows [%lld, %lld) fall outside S=%d", l, st, st + hh * ww, d->S);
  }
  const long long per_batch = (long long)d->S * d->H * d->D * (long long)dtype_size(d->value_dtype) / 16;
  if (per_batch >= (1ll << 31)) return fail(MSDA_B200_ERR_UNSUPPORTED, "S*H*D too large for 32-bit tile offsets");
  if ((long long)d->L * d->P > 64) return fail(MSDA_B200_ERR_UNSUPPORTED, "L*P=%d exceeds 64", d->L * d->P);
  return MSDA_B200_OK;
}

// Geometry fields of KParams; the tensor pointers are set by the caller beforehand.
void fill_geometry(const msda_b200_desc* d, KParams& p, int tq) {
  p.B = d->B; p.S = d->S; p.Q = d->Q; p.H = d->H; p.L = d->L; p.P = d->P; p.LP = d->L * d->P;
  p.num_tiles = (d->Q + tq - 1) / tq;
  const int per_pixel16 = d->H * d->D * (int)dtype_size(d->value_dtype) / 16;
  p.batch_stride16 = (long long)d->S * per_pixel16;
  for (int l = 0; l < d->L; ++l) {
    Level& lv = p.lv[l];
    lv.H = d->spatial_shapes_hw[2 * l];
    lv.W = d->spatial_shapes_hw[2 * l + 1];
    lv.start = (int)d->level_start_index[l];
    lv.dx16 = lv.W > 1 ? per_pixel16 : 0;
    lv.dy16 = lv.H > 1 ? lv.W * per_pixel16 : 0;
  }
}

int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(MSDA_B200_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return MSDA_B200_OK;
}

// Launch geometry: NT threads per block, QPG queries per lane group.
constexpr int kFwdNT = 128, kFwdQPG = 1;  // measured on config 2: 0.332 ms (256/1: 0.347, 256/2: 0.332, 512/1: 0.410)
constexpr int kBwdNT = 128, kBwdQPG = 1;

template <typename VT, typename AT, int D, bool FUSED>
int launch_fwd(const msda_b200_desc* d, KParams p, cudaStream_t st) {
  constexpr int LPP = D / Vec16<VT>::N;
  using T = Tile<kFwdNT, LPP, kFwdQPG>;
  fill_geometry(d, p, T::TQ);
  const size_t smem = (size_t)p.LP * T::ROW * (sizeof(float4) + sizeof(int)) +
                      (FUSED ? (size_t)T::TQ * p.LP * sizeof(float) : 0);
  const bool strict = (d->flags & MSDA_B200_FLAG_STRICT_PADDING) != 0;
  auto kern = strict ? msda_fwd_kernel<VT, AT, D, kFwdNT, kFwdQPG, FUSED, true>
                     : msda_fwd_kernel<VT, AT, D, kFwdNT, kFwdQPG, FUSED, false>;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return fail(MSDA_B200_ERR_CUDA, "forward: cannot reserve %zu bytes of shared memory", smem);
  const long long blocks = (long long)p.B * p.num_tiles * p.H;
  if (blocks > 0x7fffffffll) return fail(MSDA_B200_ERR_UNSUPPORTED, "forward: grid too large");
  {
    ProfScope ps((d->flags & MSDA_B200_FLAG_PROFILE) != 0, MSDA_B200_PROF_FWD, st);
    kern<<<(unsigned)blocks, kFwdNT, smem, st>>>(p);
    ++g_launches;
  }
  return check_launch("msda_b200_forward");
}

// Forward with two heads per block (see msda_fwd_pair_kernel). 128 threads, 2 (query, head) pairs per lane group
// measured best on config 2 (ms): 128/2 0.294, 128/1 0.302, 256/2 0.297, 256/1 0.307, 128/4 0.407; one head per block
// (msda_fwd_kernel) 0.313
template <typename VT, typename AT, int D, bool FUSED>
int launch_fwd_pair(const msda_b200_desc* d, KParams p, cudaStream_t st) {
  constexpr int NT = 128, QPG = 2, HPB = 2;
  constexpr int LPP = D / Vec16<VT>::N, NG = NT / LPP, TV = NG * QPG, TQ = TV / HPB, ROW = TV + 1;
  fill_geometry(d, p, TQ);
  const size_t smem = (size_t)p.LP * ROW * (sizeof(float4) + sizeof(int)) + (FUSED ? (size_t)TV * p.LP * sizeof(float) + (size_t)TQ * sizeof(float2) : 0);
  auto kern = (d->L == 3 && d->P == 4) ? msda_fwd_pair_kernel<VT, AT, D, NT, QPG, HPB, FUSED, 3>
                                       : msda_fwd_pair_kernel<VT, AT, D, NT, QPG, HPB, FUSED, 0>;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return fail(MSDA_B200_ERR_CUDA, "forward: cannot reserve %zu bytes of shared memory", smem);
  // Shared-memory carve-out: what is left of the SM's 256 KB is the L1 the gather lives in. The driver's default makes
  // room for the register limit's 9 blocks; 50 % (132 KB) holds 7 blocks of the plain kernel and leaves the gather
  // 124 KB of L1. Measured (profiles/r02_notes.md; config 2 init / trained, config 3 init / trained, ms): default
  // 0.286 / 0.306 / 0.661 / 0.717, 50 %: 0.282 / 0.301 / 0.655 / 0.696, 40 %: 0.313 / 0.337 / 0.697 / 0.747. The fused
  // prologue's blocks are 3 KB larger (softmax tile), 50 % holds only 6 of them: 0.407 vs 0.321 ms -> driver default.
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, FUSED ? -1 : 50);
  const long long blocks = (long long)p.B * p.num_tiles * (p.H / HPB);
  if (blocks > 0x7fffffffll) return fail(MSDA_B200_ERR_UNSUPPORTED, "forward: grid too large");
  {
    ProfScope ps((d->flags & MSDA_B200_FLAG_PROFILE) != 0, MSDA_B200_PROF_FWD, st);
    kern<<<(unsigned)blocks, NT, smem, st>>>(p);
    ++g_launches;
  }
  return check_launch("msda_b200_forward (head pairs)");
}

template <typename VT, typename AT, int D, int ACC, bool FUSED>
int launch_bwd(const msda_b200_desc* d, KParams p, cudaStream_t st) {
  constexpr int LPP = D / Vec16<VT>::N;
  using T = Tile<kBwdNT, LPP, kBwdQPG>;
  fill_geometry(d, p, T::TQ);
  const size_t n = (size_t)p.LP * T::ROW;
  const size_t smem = n * (2 * sizeof(float4) + sizeof(float) + sizeof(int)) +
                      (size_t)p.LP * T::TQ * LPP * sizeof(float4) +
                      (FUSED ? 2 * (size_t)T::TQ * p.LP * sizeof(float) : 0);
  auto kern = msda_bwd_kernel<VT, AT, D, kBwdNT, kBwdQPG, ACC, FUSED>;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return fail(MSDA_B200_ERR_CUDA, "backward: cannot reserve %zu bytes of shared memory", smem);
  const long long blocks = (long long)p.B * p.num_tiles * p.H;
  if (blocks > 0x7fffffffll) return fail(MSDA_B200_ERR_UNSUPPORTED, "backward: grid too large");
  {
    ProfScope ps((d->flags & MSDA_B200_FLAG_PROFILE) != 0, MSDA_B200_PROF_BWD_MAIN, st);
    kern<<<(unsigned)blocks, kBwdNT, smem, st>>>(p);
    ++g_launches;
  }
  return check_launch("msda_b200_backward");
}

template <typename VT, typename AT, bool FUSED>
int dispatch_fwd(const msda_b200_desc* d, const KParams& p, cudaStream_t st) {
  if constexpr (std::is_same<VT, __nv_bfloat16>::value) {
    // 64-byte rows (bf16, D = 32): pair an even with an odd head (bank-conflict-free quarter-warps)
    if (d->D == 32 && d->H % 2 == 0 && !(d->flags & MSDA_B200_FLAG_STRICT_PADDING))
      return launch_fwd_pair<VT, AT, 32, FUSED>(d, p, st);
  }
  switch (d->D) {
    case 8: return launch_fwd<VT, AT, 8, FUSED>(d, p, st);
    case 128: return launch_fwd<VT, AT, 128, FUSED>(d, p, st);
    case 16: return launch_fwd<VT, AT, 16, FUSED>(d, p, st);
    case 32: return launch_fwd<VT, AT, 32, FUSED>(d, p, st);
    case 64: return launch_fwd<VT, AT, 64, FUSED>(d, p, st);
  }
  return fail(MSDA_B200_ERR_UNSUPPORTED, "head dim %d", d->D);
}

// Backward v2 (msda_bwd_sorted.cuh): instantiated for the model's geometry (D = 32, P = 4).
// 128 queries / 256 threads per block measured best on config 2 (1.24 ms; 64/128: 1.35, 256/512: 1.29).
constexpr int kSortNT = 256, kSortTQ = 128, kSortCAP = 2048;

bool sorted_applicable(const msda_b200_desc* d) {
  if (d->flags & MSDA_B200_FLAG_BWD_V1) return false;
  if (d->D != 32 || d->P != 4) return false;
  // fp32 rows are 8 lanes wide: half as many entries per warp step, measured slower than v1 (2.35 vs 2.12 ms)
  if (d->value_dtype != MSDA_B200_BF16) return false;
  for (int l = 0; l < d->L; ++l)  // pixel coordinates are packed into 12 bits each
    if (d->spatial_shapes_hw[2 * l] > 4095 || d->spatial_shapes_hw[2 * l + 1] > 4095) return false;
  return true;
}

template <typename VT, typename AT, int ACC, bool FUSED, int kNT, int kTQ, int kPL>
int launch_bwd_sorted_cfg(const msda_b200_desc* d, KParams p, cudaStream_t st) {
  constexpr int D = 32, P = 4;
  constexpr int LPP = D / Vec16<VT>::N;
  fill_geometry(d, p, kTQ);
  const size_t smem = sorted_smem_layout<kNT, kTQ, P, kSortCAP, LPP>().total;
  auto kern = msda_bwd_sorted_kernel<VT, AT, D, kNT, kTQ, P, kSortCAP, ACC, FUSED, kPL>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return fail(MSDA_B200_ERR_CUDA, "backward: cannot reserve %zu bytes of shared memory", smem);
  const long long blocks = (long long)p.B * p.num_tiles * p.H;
  if (blocks > 0x7fffffffll) return fail(MSDA_B200_ERR_UNSUPPORTED, "backward: grid too large");
  {
    ProfScope ps((d->flags & MSDA_B200_FLAG_PROFILE) != 0, MSDA_B200_PROF_BWD_MAIN, st);
    kern<<<(unsigned)blocks, kNT, smem, st>>>(p);
    ++g_launches;
  }
  return check_launch("msda_b200_backward (sorted)");
}

// Backward v3 (msda_bwd_mma.cuh): group-sorted rows + mma.sync; same geometry as v2, fp32 accumulator only.
constexpr int kMmaNT = 256, kMmaTQ = 128, kMmaGCAP = 256, kMmaRCAP = 1024;

template <typename AT, bool FUSED>
int launch_bwd_mma(const msda_b200_desc* d, KParams p, cudaStream_t st) {
  constexpr int P = 4;
  fill_geometry(d, p, kMmaTQ);
  const size_t smem = mma_smem_layout<kMmaNT, kMmaTQ, P, kMmaGCAP, kMmaRCAP, FUSED>().total;
  auto kern = msda_bwd_mma_kernel<AT, kMmaNT, kMmaTQ, P, kMmaGCAP, kMmaRCAP, FUSED>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return fail(MSDA_B200_ERR_CUDA, "backward: cannot reserve %zu bytes of shared memory", smem);
  const long long blocks = (long long)p.B * p.num_tiles * p.H;
  if (blocks > 0x7fffffffll) return fail(MSDA_B200_ERR_UNSUPPORTED, "backward: grid too large");
  {
    ProfScope ps((d->flags & MSDA_B200_FLAG_PROFILE) != 0, MSDA_B200_PROF_BWD_MAIN, st);
    kern<<<(unsigned)blocks, kMmaNT, smem, st>>>(p);
    ++g_launches;
  }
  return check_launch("msda_b200_backward (group-sorted, mma)");
}

template <typename VT, typename AT, int ACC, bool FUSED>
int dispatch_bwd(const msda_b200_desc* d, const KParams& p, cudaStream_t st) {
  if constexpr (std::is_same<VT, __nv_bfloat16>::value && ACC != 2) {
    if (sorted_applicable(d)) {
      if constexpr (ACC == 0) {
        if (!(d->flags & MSDA_B200_FLAG_BWD_V2)) return launch_bwd_mma<AT, FUSED>(d, p, st);
      }
      return launch_bwd_sorted_cfg<VT, AT, ACC, FUSED, kSortNT, kSortTQ, 4>(d, p, st);
    }
  }
  switch (d->D) {
    case 8: return launch_bwd<VT, AT, 8, ACC, FUSED>(d, p, st);
    case 128: return launch_bwd<VT, AT, 128, ACC, FUSED>(d, p, st);
    case 16: return launch_bwd<VT, AT, 16, ACC, FUSED>(d, p, st);
    case 32: return launch_bwd<VT, AT, 32, ACC, FUSED>(d, p, st);
    case 64: return launch_bwd<VT, AT, 64, ACC, FUSED>(d, p, st);
  }
  return fail(MSDA_B200_ERR_UNSUPPORTED, "head dim %d", d->D);
}

template <bool FUSED>
int run_forward(const msda_b200_desc* desc, const KParams& p, cudaStream_t st) {
  const bool vbf = desc->value_dtype == MSDA_B200_BF16, abf = desc->attn_dtype == MSDA_B200_BF16;
  if (!vbf) return dispatch_fwd<float, float, FUSED>(desc, p, st);
  if (abf) return dispatch_fwd<__nv_bfloat16, __nv_bfloat16, FUSED>(desc, p, st);
  return dispatch_fwd<__nv_bfloat16, float, FUSED>(desc, p, st);
}

// Shared by the plain and the fused backward: zero-fill, main kernel, bf16 conversion.
// (Measured and dropped, round 2: running the bf16 backward as per-image chains zero-fill -> main kernel -> convert on
// internal streams forked from the caller's -- main kernels on three low-priority streams, the zero-fills and converts on
// a high-priority one, each chain in an L2-resident 22 MB slot of the workspace -- to hide the 74 us of the two small
// kernels under the main kernel. Parity-green, but 1.217 ms per step against 1.210 for the three whole-batch launches
// (3, 4 or 8 slots alike): the SMs are full of main-kernel blocks, so whatever the small kernels get they take from it.)
template <bool FUSED>
int run_backward(const msda_b200_desc* desc, KParams p, void* grad_value, void* workspace, size_t workspace_bytes,
                 bool have_tensors, cudaStream_t st) {
  const bool prof = (desc->flags & MSDA_B200_FLAG_PROFILE) != 0;
  const bool vbf = desc->value_dtype == MSDA_B200_BF16, abf = desc->attn_dtype == MSDA_B200_BF16;
  const bool bf16_atomics = vbf && (desc->flags & MSDA_B200_FLAG_BF16_ATOMICS);
  const size_t nvalue = (size_t)desc->B * desc->S * desc->H * desc->D;
  const size_t need = msda_b200_backward_workspace_bytes(desc);
  if (nvalue && !grad_value) return fail(MSDA_B200_ERR_INVALID, "backward: grad_value is NULL");
  if (need && nvalue && (!workspace || workspace_bytes < need))
    return fail(MSDA_B200_ERR_WORKSPACE, "backward: workspace of %zu bytes required, got %zu", need, workspace_bytes);
  if (nvalue && need && (reinterpret_cast<uintptr_t>(workspace) & 15))
    return fail(MSDA_B200_ERR_INVALID, "backward: workspace must be 16-byte aligned");

  // Zero-fill the accumulator (and grad_value): the scatter only touches sampled pixels.
  void* acc = need ? workspace : grad_value;
  if (nvalue) {
    ProfScope ps(prof, MSDA_B200_PROF_BWD_ZERO, st);
    const size_t acc_bytes = need ? need : nvalue * dtype_size(desc->value_dtype);
    if (cudaMemsetAsync(acc, 0, acc_bytes, st) != cudaSuccess) return check_launch("backward: memset");
  }
  if ((long long)desc->B * desc->Q != 0) {
    if (!have_tensors) return fail(MSDA_B200_ERR_INVALID, "backward: NULL tensor pointer");
    p.grad_value_acc = acc;
    int rc;
    if (!vbf) rc = dispatch_bwd<float, float, 0, FUSED>(desc, p, st);
    else if (bf16_atomics) rc = abf ? dispatch_bwd<__nv_bfloat16, __nv_bfloat16, 1, FUSED>(desc, p, st)
                                    : dispatch_bwd<__nv_bfloat16, float, 1, FUSED>(desc, p, st);
    else rc = abf ? dispatch_bwd<__nv_bfloat16, __nv_bfloat16, 0, FUSED>(desc, p, st)
                  : dispatch_bwd<__nv_bfloat16, float, 0, FUSED>(desc, p, st);
    if (rc) return rc;
  }
  if (need && nvalue) {
    ProfScope ps(prof, MSDA_B200_PROF_BWD_CONVERT, st);
    const long long n8 = (long long)(nvalue / 8);  // D is a multiple of 8, so nvalue % 8 == 0
    const int blocks = (int)((n8 + 255) / 256 < 148 * 16 ? (n8 + 255) / 256 : 148 * 16);
    msda_cvt_f32_bf16_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(workspace),
                                                     reinterpret_cast<uint4*>(grad_value), n8);
    ++g_launches;
    if (int rc = check_launch("backward: convert")) return rc;
  }
  return MSDA_B200_OK;
}

// MSDA_B200_FLAG_DETERMINISTIC: the per-corner kernel without its scatter writes grad_loc / grad_attn and the records
// of every sample; msda_bwd_det.cu orders the records and writes every element of grad_value from them. No float
// atomics, so equal inputs give equal bits.
template <bool FUSED>
int run_backward_det(const msda_b200_desc* desc, KParams p, void* grad_value, void* workspace, size_t workspace_bytes,
                     bool have_tensors, cudaStream_t st) {
  if (desc->B == 0) return MSDA_B200_OK;
  if (!grad_value) return fail(MSDA_B200_ERR_INVALID, "backward: grad_value is NULL");
  size_t need = 0;
  if (int rc = msda_b200_internal_det_workspace_bytes(desc, &need)) return rc;
  if (!workspace || workspace_bytes < need)
    return fail(MSDA_B200_ERR_WORKSPACE, "backward: workspace of %zu bytes required, got %zu", need, workspace_bytes);
  if (reinterpret_cast<uintptr_t>(workspace) & 15) return fail(MSDA_B200_ERR_INVALID, "backward: workspace must be 16-byte aligned");
  if (desc->Q != 0) {
    if (!have_tensors) return fail(MSDA_B200_ERR_INVALID, "backward: NULL tensor pointer");
    const DetLayout lay = det_layout(desc);
    p.det_keys = reinterpret_cast<unsigned*>(static_cast<char*>(workspace) + lay.keys_off[0]);
    p.det_vals = reinterpret_cast<unsigned long long*>(static_cast<char*>(workspace) + lay.vals_off[0]);
    p.det_sentinel = (unsigned)lay.keys;
    const bool vbf = desc->value_dtype == MSDA_B200_BF16, abf = desc->attn_dtype == MSDA_B200_BF16;
    int rc;
    if (!vbf) rc = dispatch_bwd<float, float, 2, FUSED>(desc, p, st);
    else rc = abf ? dispatch_bwd<__nv_bfloat16, __nv_bfloat16, 2, FUSED>(desc, p, st)
                  : dispatch_bwd<__nv_bfloat16, float, 2, FUSED>(desc, p, st);
    if (rc) return rc;
  }
  return msda_b200_internal_det_grad_value(desc, p.grad_out, grad_value, workspace, st);
}

}  // namespace

extern "C" {

// shared with layer_epilogue.cu (not part of the public header)
int msda_b200_internal_fail(int code, const char* msg) { return fail(code, "%s", msg); }
// shared with host_pipeline.cu: the descriptor checks of forward / backward
int msda_b200_internal_validate(const msda_b200_desc* desc) { return validate(desc); }
// shared with point_sample.cu: kernels launched outside this file count too
void msda_b200_internal_count_launch(void) { ++g_launches; }

int msda_b200_abi_version(void) { return MSDA_B200_ABI_VERSION; }

const char* msda_b200_last_error(void) { return g_err; }

int msda_b200_forward(const msda_b200_desc* desc, const void* value, const float* loc, const void* attn, void* out,
                      const int32_t* query_order, void* stream) {
  g_err[0] = 0;
  if (int rc = validate(desc)) return rc;
  if ((long long)desc->B * desc->Q == 0) return MSDA_B200_OK;
  if (!value || !loc || !attn || !out) return fail(MSDA_B200_ERR_INVALID, "forward: NULL tensor pointer");
  KParams p;
  memset(&p, 0, sizeof(p));
  p.value = value; p.loc = loc; p.attn = attn; p.out = out; p.q_order = query_order;
  return run_forward<false>(desc, p, reinterpret_cast<cudaStream_t>(stream));
}

int msda_b200_forward_fused(const msda_b200_desc* desc, const void* value, const void* offsets, const void* logits,
                            const float* ref_points, void* out, float* attn_out, const int32_t* query_order,
                            void* stream) {
  g_err[0] = 0;
  if (int rc = validate(desc)) return rc;
  if ((long long)desc->B * desc->Q == 0) return MSDA_B200_OK;
  if (!value || !offsets || !logits || !out) return fail(MSDA_B200_ERR_INVALID, "forward_fused: NULL tensor pointer");
  if (!ref_points && desc->Q != desc->S)
    return fail(MSDA_B200_ERR_INVALID, "forward_fused: implicit reference points (ref_points = NULL) need Q == S");
  KParams p;
  memset(&p, 0, sizeof(p));
  p.value = value; p.offsets = offsets; p.logits = logits; p.ref = ref_points; p.out = out; p.attn_out = attn_out;
  p.q_order = query_order;
  return run_forward<true>(desc, p, reinterpret_cast<cudaStream_t>(stream));
}

size_t msda_b200_backward_workspace_bytes(const msda_b200_desc* desc) {
  if (!desc) return 0;
  if (desc->flags & MSDA_B200_FLAG_DETERMINISTIC) {
    size_t bytes = 0;
    if (validate(desc) || msda_b200_internal_det_workspace_bytes(desc, &bytes)) return 0;
    return bytes;
  }
  if (desc->value_dtype == MSDA_B200_BF16 && !(desc->flags & MSDA_B200_FLAG_BF16_ATOMICS))
    return (size_t)desc->B * desc->S * desc->H * desc->D * sizeof(float);
  return 0;
}

int msda_b200_backward(const msda_b200_desc* desc, const void* value, const float* loc, const void* attn,
                       const void* grad_out, void* grad_value, float* grad_loc, void* grad_attn, void* workspace,
                       size_t workspace_bytes, const int32_t* query_order, void* stream) {
  g_err[0] = 0;
  if (int rc = validate(desc)) return rc;
  KParams p;
  memset(&p, 0, sizeof(p));
  p.value = value; p.loc = loc; p.attn = attn; p.grad_out = grad_out;
  p.grad_loc = grad_loc; p.grad_attn = grad_attn; p.q_order = query_order;
  const bool have = value && loc && attn && grad_out && grad_loc && grad_attn;
  if (desc->flags & MSDA_B200_FLAG_DETERMINISTIC)
    return run_backward_det<false>(desc, p, grad_value, workspace, workspace_bytes, have, reinterpret_cast<cudaStream_t>(stream));
  return run_backward<false>(desc, p, grad_value, workspace, workspace_bytes, have, reinterpret_cast<cudaStream_t>(stream));
}

int msda_b200_backward_fused(const msda_b200_desc* desc, const void* value, const void* offsets, const void* logits,
                             const float* ref_points, const void* grad_out, void* grad_value, void* grad_offsets,
                             void* grad_logits, void* workspace, size_t workspace_bytes, const int32_t* query_order,
                             void* stream) {
  g_err[0] = 0;
  if (int rc = validate(desc)) return rc;
  KParams p;
  memset(&p, 0, sizeof(p));
  p.value = value; p.offsets = offsets; p.logits = logits; p.ref = ref_points; p.grad_out = grad_out;
  p.grad_offsets = grad_offsets; p.grad_logits = grad_logits; p.q_order = query_order;
  if (!ref_points && desc->Q != desc->S)
    return fail(MSDA_B200_ERR_INVALID, "backward_fused: implicit reference points (ref_points = NULL) need Q == S");
  const bool have = value && offsets && logits && grad_out && grad_offsets && grad_logits;
  if (desc->flags & MSDA_B200_FLAG_DETERMINISTIC)
    return run_backward_det<true>(desc, p, grad_value, workspace, workspace_bytes, have, reinterpret_cast<cudaStream_t>(stream));
  return run_backward<true>(desc, p, grad_value, workspace, workspace_bytes, have, reinterpret_cast<cudaStream_t>(stream));
}

int msda_b200_profile_ms(int which, float* ms) {
  if (which < 0 || which >= MSDA_B200_PROF_COUNT || !ms) return fail(MSDA_B200_ERR_INVALID, "profile_ms: bad argument");
  if (g_prof.device < 0 || !g_prof.valid[which]) return fail(MSDA_B200_ERR_INVALID, "profile_ms: nothing recorded");
  const cudaError_t e = cudaEventElapsedTime(ms, g_prof.ev[which][0], g_prof.ev[which][1]);
  if (e != cudaSuccess) return fail(MSDA_B200_ERR_CUDA, "profile_ms: %s", cudaGetErrorString(e));
  return MSDA_B200_OK;
}

int64_t msda_b200_launch_count(int reset) {
  return reset ? g_launches.exchange(0) : g_launches.load();
}

}  // extern "C"
