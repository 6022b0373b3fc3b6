// VolumeRenderer.forward (src/nerf/modules.py:67-121) as a per-sample step function, shared by the stand-alone compositor
// (composite_kernel, nm_render.cu) and the compositor fused into the MLP kernel (nm_mlp_tc.cu), which must agree bit for
// bit.  Every floating-point operation is an explicit round-to-nearest intrinsic: the result does not depend on the
// translation unit's -fmad setting (a*b+c stays two roundings, the way torch evaluates the reference's separate ops), and
// the value returned by expf is fenced so that its last multiply cannot be contracted into the caller's arithmetic.
// Samples are visited in order, so the exclusive cumprod (nerf_helpers.py:199-223) is the sequential product torch forms.
#pragma once
#include <math_constants.h>

#include "nm_common.h"

namespace nm {

// counter-based random bits: splitmix64 of (seed, index)
__device__ __forceinline__ uint64_t hash64(uint64_t seed, uint64_t idx) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (idx + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// uniform [0,1) with 24 bits.  Used only for perturb / noise / surface sampling (distributional parity).
__device__ __forceinline__ float u01(uint64_t seed, uint64_t idx) {
  return (float)(hash64(seed, idx) >> 40) * (1.0f / 16777216.0f);
}
// uniform [0,1) with 53 bits, for draws that must resolve more than 2^24 outcomes (a face out of millions)
__device__ __forceinline__ double u01_53(uint64_t seed, uint64_t idx) {
  return (double)(hash64(seed, idx) >> 11) * (1.0 / 9007199254740992.0);
}
__device__ __forceinline__ float randn(uint64_t seed, uint64_t idx) {
  const float a = fmaxf(u01(seed, 2 * idx), 1e-7f), b = u01(seed, 2 * idx + 1);
  float l = logf(a);
  asm volatile("" : "+f"(l));
  float c = cospif(__fmul_rn(2.f, b));
  asm volatile("" : "+f"(c));
  return __fmul_rn(sqrtf(__fmul_rn(-2.f, l)), c);
}

struct CompState {
  float T, acc, depth, r, g, b;
};
__device__ __forceinline__ void comp_init(CompState& s) { s.T = 1.0f; s.acc = 0.f; s.depth = 0.f; s.r = 0.f; s.g = 0.f; s.b = 0.f; }

__device__ __forceinline__ float comp_ray_norm(const float* __restrict__ dirs, long long ray) {
  const float dx = dirs[3 * ray], dy = dirs[3 * ray + 1], dz = dirs[3 * ray + 2];
  return sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
}

// sample i of `ray`: tc = t[i], tn = t[i+1] (unused for the last sample), sigma_raw = the network's raw density.
// Returns alpha_i; *keep = 1 - alpha_i + 1e-10, the factor of the transmittance product.
__device__ __forceinline__ float comp_alpha(const CompositeArgs& a, long long ray, int i, float tc, float tn, float nrm,
                                            float sigma_raw, float* keep) {
  const int S = a.S;
  const float dist = __fmul_rn((i + 1 < S) ? __fsub_rn(tn, tc) : 1e10f, nrm);
  float sg = sigma_raw;
  if (a.noise_std > 0.f) sg = __fadd_rn(sg, __fmul_rn(randn(a.seed, (uint64_t)(ray * S + i)), a.noise_std));
  sg = fmaxf(sg, 0.f);
  float e = expf(__fmul_rn(-sg, dist));
  asm volatile("" : "+f"(e));
  const float alpha = __fsub_rn(1.0f, e);
  *keep = __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f);
  return alpha;
}

// one sample of the sequential walk: q = (sigmoid rgb, raw sigma).  Returns the weight.
__device__ __forceinline__ float comp_step(CompState& s, const CompositeArgs& a, long long ray, int i, float tc, float tn,
                                           float nrm, float4 q, float* mask_out) {
  float keep;
  const float alpha = comp_alpha(a, ray, i, tc, tn, nrm, q.w, &keep);
  const float w = __fmul_rn(alpha, s.T);
  *mask_out = (s.T > a.thr) ? 1.f : 0.f;
  s.r = __fadd_rn(s.r, __fmul_rn(w, q.x));
  s.g = __fadd_rn(s.g, __fmul_rn(w, q.y));
  s.b = __fadd_rn(s.b, __fmul_rn(w, q.z));
  s.acc = __fadd_rn(s.acc, w);
  s.depth = __fadd_rn(s.depth, __fmul_rn(w, tc));
  s.T = __fmul_rn(s.T, keep);
  return w;
}

// after the last sample of `ray`: the per-ray outputs (modules.py:99-121)
__device__ __forceinline__ void comp_finish(const CompState& s, const CompositeArgs& a, long long ray) {
  const float acc = s.acc, depth = s.depth;
  float r = s.r, g = s.g, b = s.b;
  const float ratio = __fdiv_rn(depth, acc);
  float disp = __fdiv_rn(1.0f, fmaxf(1e-10f, ratio));
  if (isnan(disp)) disp = 0.f;          // fmaxf drops a NaN operand; torch.max propagates it, then :107 zeroes it
  if (isnan(ratio)) disp = 0.f;
  if (a.depth_raw) a.depth_raw[ray] = depth;
  if (a.depth) a.depth[ray] = (!a.training && acc < 1.0f) ? 0.f : depth;
  if (a.white_bg) { const float bg = __fsub_rn(1.0f, acc); r = __fadd_rn(r, bg); g = __fadd_rn(g, bg); b = __fadd_rn(b, bg); }
  if (a.rgb) { a.rgb[3 * ray] = r; a.rgb[3 * ray + 1] = g; a.rgb[3 * ray + 2] = b; }
  if (a.acc) a.acc[ray] = acc;
  if (a.disp) a.disp[ray] = disp;
}

}  // namespace nm
