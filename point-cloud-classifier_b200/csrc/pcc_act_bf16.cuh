// Activation math of the bf16 paths (fused DeepSets pcc_fused*.cu, fused GraphNet pcc_gnn*.cu).  The epilogues are
// issue / MUFU bound (libm tanhf / erff cost ~30 instructions each; an exp/rcp based erf was measured 1.5x SLOWER than
// erff(): two MUFU ops per element at quarter rate), so every activation costs ONE MUFU op per element:
//   tanh: tanh.approx.f32 (abs error ~5e-4);
//   SiLU: sigmoid(z) = 0.5 (1 + tanh(z/2)) with tanh.approx;
//   GELU: 0.5 z (1 + tanh(sqrt(2/pi) (z + 0.044715 z^3))) with tanh.approx — within 5e-4 (absolute) of the
//         reference's exact-erf nn.GELU();
// all below the bf16 rounding (4e-3 relative) of the stored activation.  The fp32 parity path (pcc_common.cuh) keeps
// the exact erf / libm forms.  Forward and backward use the same functions, so act' is consistent with the act the
// forward applied, and act / act' share the tanh where both are needed.
#pragma once
#include "pcc_common.cuh"
#include "pcc_tc.cuh"

namespace pcc {
using namespace tc;

__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <int ACT>
__device__ __forceinline__ float actf(float z) {
  if (ACT == PCC_ACT_RELU) return fmaxf(z, 0.f);
  if (ACT == PCC_ACT_TANH) return tanh_approx(z);
  if (ACT == PCC_ACT_GELU) return 0.5f * z * (1.f + tanh_approx(0.7978845608028654f * z * fmaf(0.044715f, z * z, 1.f)));
  if (ACT == PCC_ACT_SILU) return z * (0.5f * (1.f + tanh_approx(0.5f * z)));
  return z;
}
// act'(z), given a = act(z) where that is cheaper
template <int ACT>
__device__ __forceinline__ float actg(float z, float a) {
  if (ACT == PCC_ACT_RELU) return z > 0.f ? 1.f : 0.f;
  if (ACT == PCC_ACT_TANH) return 1.f - a * a;
  if (ACT == PCC_ACT_GELU) {
    const float z2 = z * z;
    const float t = tanh_approx(0.7978845608028654f * z * fmaf(0.044715f, z2, 1.f));
    return 0.5f * (1.f + t) + 0.5f * z * (1.f - t * t) * (0.7978845608028654f * fmaf(0.134145f, z2, 1.f));
  }
  if (ACT == PCC_ACT_SILU) {
    const float s = 0.5f * (1.f + tanh_approx(0.5f * z));
    return s * (1.f + z * (1.f - s));
  }
  return 1.f;
}

// ---- the same activations on packed pairs (f32x2).  The gelu / silu epilogues are bound by instruction issue (a trace
// of the DeepSets backward chain: 19k of 29k cycles per tile are activation math at ~20 scalar instructions per
// element); Blackwell's packed fp32 pipe evaluates the polynomial parts of two elements per instruction, the tanh stays
// one MUFU op per element.  Same functions of z as actf / actg (identical operation order up to fma contraction).
__device__ __forceinline__ uint64_t tanh2(uint64_t x) {
  float lo, hi;
  f32x2_unpack(x, lo, hi);
  return f32x2(tanh_approx(lo), tanh_approx(hi));
}
template <int ACT>
__device__ __forceinline__ uint64_t act2(uint64_t z) {
  if (ACT == PCC_ACT_TANH) return tanh2(z);
  if (ACT == PCC_ACT_GELU) {
    constexpr float c0 = 0.7978845608028654f;
    const uint64_t t = tanh2(fmul2(z, ffma2(splat2(c0 * 0.044715f), fmul2(z, z), splat2(c0))));
    return fmul2(z, ffma2(splat2(0.5f), t, splat2(0.5f)));
  }
  if (ACT == PCC_ACT_SILU) return fmul2(z, ffma2(splat2(0.5f), tanh2(fmul2(z, splat2(0.5f))), splat2(0.5f)));
  float lo, hi;
  f32x2_unpack(z, lo, hi);
  if (ACT == PCC_ACT_RELU) return f32x2(fmaxf(lo, 0.f), fmaxf(hi, 0.f));
  return z;
}
// a = act(z), da = act'(z)
template <int ACT>
__device__ __forceinline__ void act_and_grad2(uint64_t z, uint64_t& a, uint64_t& da) {
  if (ACT == PCC_ACT_TANH) {
    a = tanh2(z);
    da = ffma2(fmul2(a, splat2(-1.f)), a, splat2(1.f));
  } else if (ACT == PCC_ACT_GELU) {
    constexpr float c0 = 0.7978845608028654f;
    const uint64_t z2 = fmul2(z, z);
    const uint64_t t = tanh2(fmul2(z, ffma2(splat2(c0 * 0.044715f), z2, splat2(c0))));
    const uint64_t h = ffma2(splat2(0.5f), t, splat2(0.5f));                       // 0.5 (1 + t)
    a = fmul2(z, h);
    // da = h + 2 z h (1 - h) u',  u' = c0 (1 + 0.134145 z^2)      (1 - t^2 = 4 h (1 - h))
    const uint64_t up2 = ffma2(splat2(2.f * c0 * 0.134145f), z2, splat2(2.f * c0));
    const uint64_t omh = ffma2(h, splat2(-1.f), splat2(1.f));
    da = ffma2(fmul2(a, omh), up2, h);
  } else if (ACT == PCC_ACT_SILU) {
    const uint64_t s = ffma2(splat2(0.5f), tanh2(fmul2(z, splat2(0.5f))), splat2(0.5f));
    a = fmul2(z, s);
    da = ffma2(a, ffma2(s, splat2(-1.f), splat2(1.f)), s);   // s + z s (1 - s)
  } else if (ACT == PCC_ACT_RELU) {
    float lo, hi;
    f32x2_unpack(z, lo, hi);
    a = f32x2(fmaxf(lo, 0.f), fmaxf(hi, 0.f));
    da = f32x2(lo > 0.f ? 1.f : 0.f, hi > 0.f ? 1.f : 0.f);
  } else {
    a = z;
    da = splat2(1.f);
  }
}

}  // namespace pcc
