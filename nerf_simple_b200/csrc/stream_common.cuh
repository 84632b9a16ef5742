// Device helpers shared by the streaming kernels (rays_sampler.cu, composite.cu) and by the fused
// render epilogue of the MLP chain kernel (mlp_chain.cuh), so that the fused path computes exactly
// what the separate kernels compute.
#pragma once
#include <stdint.h>

#include "../../include/nerf_b200.h"

namespace nb200 {

// ------------------------------------------------------------------ device-resident step state
// What changes from one training step to the next lives on the device, so that a whole step can be
// captured once in a CUDA graph and replayed: Philox stream positions, Adam's step count, the lr.
// Read by the *_state entry points of rays_sampler.cu and hierarchical.cu.
struct TrainState {
  uint64_t select_offset;   // Philox counter of the ray selection
  uint64_t sample_offset;   // Philox counter of the stratified and the fine sampler (quads)
  int64_t step;             // optimizer steps taken so far
  float lr;                 // current learning rate
  float pad;
};
static_assert(sizeof(TrainState) == NB200_TRAIN_STATE_BYTES, "train state layout");

// ------------------------------------------------------------------------------- ray grid
// World ray r of the table [P*H*W]: pose r / (H*W), pixel (h, w) = divmod(r % (H*W), W).
// utils/xyz.py:46-49: integer centre, (gx/f, -gy/f, -1), IEEE division like torch;
// utils/rendering.py:131: transf_mats[:, :3, :3] @ rays_1_cam, origin = transf_mats[:, :3, 3].
__device__ __forceinline__ void camera_ray(const float* __restrict__ poses, int H, int W, float f, int64_t r, float (&o)[6]) {
  const int64_t hw = (int64_t)H * W;
  int64_t p;
  int h, w;
  if ((uint64_t)r < 0x80000000ull) {   // 32-bit index math (the usual case): two short divisions
    const uint32_t r32 = (uint32_t)r, hw32 = (uint32_t)hw;
    const uint32_t p32 = r32 / hw32, pix = r32 - p32 * hw32;
    const uint32_t hh = pix / (uint32_t)W;
    p = p32; h = (int)hh; w = (int)(pix - hh * (uint32_t)W);
  } else {
    p = r / hw;
    const int64_t pix = r - p * hw;
    h = (int)(pix / W); w = (int)(pix - (int64_t)h * W);
  }
  const float dx = __fdiv_rn((float)(w - W / 2), f);
  const float dy = -__fdiv_rn((float)(h - H / 2), f);
  const float dz = -1.0f;
  const float* T = poses + p * 16;
  o[0] = __ldg(T + 3);
  o[1] = __ldg(T + 7);
  o[2] = __ldg(T + 11);
#pragma unroll
  for (int a = 0; a < 3; ++a)
    o[3 + a] = fmaf(__ldg(T + 4 * a + 2), dz, fmaf(__ldg(T + 4 * a + 1), dy, __ldg(T + 4 * a) * dx));
}

// -------------------------------------------------------------------------------- sampler
__device__ __forceinline__ uint32_t mulhilo32(uint32_t a, uint32_t b, uint32_t* hi) {
  *hi = __umulhi(a, b);
  return a * b;
}

// Philox4x32-10 (Salmon et al. 2011): counter = (ctr lo, ctr hi, 0, 0), key = seed.
__device__ __forceinline__ uint4 philox4x32_10(uint64_t ctr, uint64_t seed) {
  uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0u, c3 = 0u;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, hi1;
    const uint32_t lo0 = mulhilo32(0xD2511F53u, c0, &hi0);
    const uint32_t lo1 = mulhilo32(0xCD9E8D57u, c2, &hi1);
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }

// torch.linspace(tn, tf, N+1)[i] in fp32 (symmetric two-sided fma evaluation).
__device__ __forceinline__ float tbin(int i, int N, float tn, float tf, float step) {
  return (i < (N + 1) / 2) ? fmaf(step, (float)i, tn) : fmaf(-step, (float)(N - i), tf);
}

// Philox-mode sample depth of global sample m (sample i = m % N of its ray), N % 4 == 0: the value
// stratified_ts_quad_kernel writes to ts[m] for the same (seed, offset).
__device__ __forceinline__ float philox_sample_depth(int64_t m, int i, int N, float tn, float tf, uint64_t seed, uint64_t offset) {
  const float step = __fdiv_rn(tf - tn, (float)N);
  const float bin = __fsub_rn(tbin(1, N, tn, tf, step), tbin(0, N, tn, tf, step));
  const float scale = bin * 5.9604644775390625e-08f;
  const uint4 x = philox4x32_10(offset + (uint64_t)(m >> 2), seed);
  const uint32_t k = (uint32_t)m & 3u;
  const uint32_t xs = k == 0 ? x.x : (k == 1 ? x.y : (k == 2 ? x.z : x.w));
  return __fadd_rn(__fmul_rn(scale, (float)(xs >> 8)), tbin(i, N, tn, tf, step));   // utils/rendering.py:29
}

// ---------------------------------------------------------------------------- compositing
__device__ __forceinline__ float exp2f_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2f_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// exp(-softplus(sigma) * delta) (utils/rendering.py:67) with the two natural-log constants cancelled:
//   (1 + e^sigma)^(-delta) = ex2(-delta * lg2(1 + ex2(sigma * log2 e)))
// lg2(1 + z) needs RELATIVE accuracy for tiny z (the last sample multiplies it by 1e10), so below
// 1e-2 the series log2(e) * (z - z^2/2 + z^3/3) is used; above the softplus threshold (20) the
// reference returns sigma itself.
__device__ __forceinline__ float transmit_factor(float sigma, float delta) {
  const float s2 = sigma * 1.4426950408889634f;
  const float z = exp2f_approx(s2);
  const float series = z * fmaf(z, fmaf(z, 0.4808983469629878f, -0.7213475204444817f), 1.4426950408889634f);
  const float lg = lg2f_approx(1.f + z);
  const float L = sigma > 20.f ? s2 : (z < 1e-2f ? series : lg);
  return exp2f_approx(-L * delta);
}

__device__ __forceinline__ float disparity(float depth, float acc) {
  const float q = __fdividef(depth, acc);                      // :82 depth / sum(weights)
  const float m = (q != q) ? q : fmaxf(1e-10f, q);             // torch.max propagates NaN
  return __frcp_rn(m);                                         // :83
}

// |d/|d|| of an un-normalised ray direction as the reference sees it (:37 then :62), MUFU rsqrt/sqrt.
__device__ __forceinline__ float unit_dir_norm(float ax, float ay, float az) {
  float inv;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(fmaf(az, az, fmaf(ay, ay, ax * ax))));   // :37
  const float dx = ax * inv, dy = ay * inv, dz = az * inv;
  float n;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(n) : "f"(fmaf(dz, dz, fmaf(dy, dy, dx * dx))));      // :62
  return n;
}

}  // namespace nb200
