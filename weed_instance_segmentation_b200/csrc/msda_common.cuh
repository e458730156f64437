// msda_common.cuh -- structs and device helpers shared by the kernels of msda_b200.cu and msda_bwd_mma.cuh.
// Included INSIDE msda_b200.cu's anonymous namespace (after <cuda_bf16.h>, <cuda_runtime.h> and msda_b200.h).
#pragma once

constexpr int kMaxL = MSDA_B200_MAX_LEVELS;

struct Level {
  int H, W;
  int start;  // first row of this level in S
  int dx16;   // +1 pixel in x, in 16-byte units of the value tensor (0 if W == 1)
  int dy16;   // +1 pixel in y, in 16-byte units (0 if H == 1)
};

struct KParams {
  const void* value;
  const float* loc;
  const void* attn;
  void* out;             // forward
  const void* grad_out;  // backward
  void* grad_value_acc;  // backward: fp32 accumulator (grad_value itself for fp32 values, the workspace for bf16)
  float* grad_loc;
  void* grad_attn;
  const int* q_order;
  // fused prologue (M2F:952-971): raw sampling offsets and attention logits instead of loc / attn
  const void* offsets;   // (B,Q,H,L,P,2), dtype AT
  const void* logits;    // (B,Q,H,L*P),   dtype AT
  const float* ref;      // (B,Q,L,2) reference points
  float* attn_out;       // optional (B,Q,H,L,P) softmax output
  void* grad_offsets;    // backward, dtype AT
  void* grad_logits;     // backward, dtype AT
  int B, S, Q, H, L, P, LP;
  int num_tiles;
  long long batch_stride16;  // S*H*D*sizeof(T)/16
  Level lv[kMaxL];
  // deterministic backward (msda_bwd_kernel with ACC = 2): four grad_value records per sample, see msda_bwd_det.cuh
  unsigned* det_keys;
  unsigned long long* det_vals;
  unsigned det_sentinel;
};

// ---------------------------------------------------------------------------------------------
// Sample descriptor maths (shared by forward and backward).
// ---------------------------------------------------------------------------------------------
struct Axis {
  float s0, s1;  // weights of the two loaded slots (base, base+1)
  float g0, g1;  // d(s0)/d(pixel coord), d(s1)/d(pixel coord)
  int base;      // clamped index of slot 0
  bool ok;
};

// coord: normalised location in [0,1] (may lie outside); n: level extent along this axis.
// Follows M2F:807 (grid = 2*loc - 1) and ATen grid_sampler_unnormalize(align_corners=False):
//   pix = ((grid + 1) * n - 1) / 2, evaluated in that order without FMA contraction.
__device__ __forceinline__ Axis axis_setup(float coord, int n) {
  Axis a;
  const float g = __fadd_rn(__fmul_rn(2.f, coord), -1.f);
  const float pix = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(g, 1.f), (float)n), -1.f), 0.5f);
  a.ok = (pix > -2.f) && (pix < (float)(n + 1));  // false for NaN as well
  const float fl = floorf(pix);
  const int i0 = __float2int_rd(pix);  // saturating; NaN -> 0
  const float l = pix - fl;
  const bool v0 = (i0 >= 0) && (i0 < n);
  const bool v1 = (i0 + 1 >= 0) && (i0 + 1 < n);
  const float w0 = v0 ? 1.f - l : 0.f, w1 = v1 ? l : 0.f;
  const float d0 = v0 ? -1.f : 0.f, d1 = v1 ? 1.f : 0.f;
  const int ib = min(max(i0, 0), max(n - 2, 0));
  const int shift = i0 - ib;
  a.base = ib;
  a.s0 = (shift == 0) ? w0 : ((shift == -1) ? w1 : 0.f);
  a.g0 = (shift == 0) ? d0 : ((shift == -1) ? d1 : 0.f);
  a.s1 = (shift == 0) ? w1 : ((shift == 1) ? w0 : 0.f);
  a.g1 = (shift == 0) ? d1 : ((shift == 1) ? d0 : 0.f);
  if (!a.ok) a.s0 = a.s1 = a.g0 = a.g1 = 0.f;  // NaN / far outside: contributes exactly zero (0 * NaN would not)
  return a;
}

template <typename T>
__device__ __forceinline__ float to_float(T v);
template <>
__device__ __forceinline__ float to_float<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T>
__device__ __forceinline__ T from_float(float v);
template <>
__device__ __forceinline__ float from_float<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 16 bytes of T -> VEC floats
template <typename T>
struct Vec16;
template <>
struct Vec16<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void unpack(const uint4& v, float (&f)[4]) {
    f[0] = __uint_as_float(v.x); f[1] = __uint_as_float(v.y);
    f[2] = __uint_as_float(v.z); f[3] = __uint_as_float(v.w);
  }
  static __device__ __forceinline__ uint4 pack(const float (&f)[4]) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
  }
};
template <>
struct Vec16<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void unpack(const uint4& v, float (&f)[8]) {
    // bf16 -> fp32 is a 16-bit shift: low half << 16, high half masked.
    f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
    f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
    f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xffff0000u);
    f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xffff0000u);
  }
  static __device__ __forceinline__ unsigned pack2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<unsigned*>(&h);
  }
  static __device__ __forceinline__ uint4 pack(const float (&f)[8]) {
    return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
  }
};

__device__ __forceinline__ uint4 ldg16(const uint4* p) { return __ldg(p); }

// Packed fp32 FMA (sm_100a FFMA2): (a0, a1) += w * (f0, f1), each element rounded exactly like fmaf. One instruction for two FMAs: the kernels here are bound by instruction issue, not by the FMA pipe.
__device__ __forceinline__ void fma2_scalar(float& a0, float& a1, float w, float f0, float f1) {
  asm("{ .reg .b64 ra, rw, rf;\n\t"
      "mov.b64 ra, {%0, %1};\n\t"
      "mov.b64 rw, {%2, %2};\n\t"
      "mov.b64 rf, {%3, %4};\n\t"
      "fma.rn.f32x2 ra, rw, rf, ra;\n\t"
      "mov.b64 {%0, %1}, ra; }"
      : "+f"(a0), "+f"(a1)
      : "f"(w), "f"(f0), "f"(f1));
}

// red.global.add.v4.f32 (sm_90+): one 16-byte reduction, no return value.
__device__ __forceinline__ void red_add_f32x4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}
