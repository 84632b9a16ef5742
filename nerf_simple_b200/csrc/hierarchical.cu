// Hierarchical (coarse -> fine) inverse-CDF sampler.  EXTENSION: the reference has no hierarchical
// sampling ("coarse and fine is not implemented yet", configs/lego.yaml:7; utils/nets.py:45-49 are
// empty classes), so this follows the original NeRF paper (Mildenhall et al. 2020, sec. 5.2) and
// its public `sample_pdf`: pdf from the interior coarse weights over the mid-point bins, inverse
// transform sampling, then the coarse and fine depths merged in sorted order.
//
// One warp per ray.  The CDF and bins live in shared memory; every fine sample does a binary
// search; the merge is a rank count (coarse depths are sorted, fine ones need not be).
// HBM traffic: 8 B/coarse sample read (+4 B/fine sample of u) and 4 B per merged sample written.
#include "common.cuh"
#include "stream_common.cuh"

namespace nb200 {

constexpr int kHsWarps = 4;
constexpr int kHsMaxNc = 128, kHsMaxAll = 384;

__device__ __forceinline__ uint32_t hs_mulhilo(uint32_t a, uint32_t b, uint32_t* hi) { *hi = __umulhi(a, b); return a * b; }
// The fine stream's counter tag c2 = "HSP1" keeps it disjoint from philox4x32_10 (c2 = 0), the stratified sampler's
// generator: in a training step both read the same train-state position (sample_offset) with keys derived from one
// seed, and the tag is what makes their draws independent.
__device__ __forceinline__ uint4 hs_philox(uint64_t ctr, uint64_t seed) {
  uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0x48535031u /* stream tag "HSP1" */, c3 = 0u;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, hi1;
    const uint32_t lo0 = hs_mulhilo(0xD2511F53u, c0, &hi0), lo1 = hs_mulhilo(0xCD9E8D57u, c2, &hi1);
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

// mode: 0 = u supplied by the caller, 1 = deterministic linspace(0,1,Nf), 2 = Philox at offset (+ *offset_dev when
// non-null: the device-resident stream position of a CUDA-graph-replayed training step)
__global__ void __launch_bounds__(kHsWarps * 32)
sample_pdf_merge_kernel(const float* __restrict__ ts, const float* __restrict__ weights, const float* __restrict__ u_in,
                        int mode, uint64_t seed, uint64_t offset, int64_t B, int Nc, int Nf, float* __restrict__ z_all,
                        const uint64_t* __restrict__ offset_dev) {
  __shared__ float s_cdf[kHsWarps][kHsMaxNc];
  __shared__ float s_bins[kHsWarps][kHsMaxNc];
  __shared__ float s_all[kHsWarps][kHsMaxAll];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* cdf = s_cdf[warp];
  float* bins = s_bins[warp];
  float* all = s_all[warp];
  const int nb = Nc - 1;   // bins / cdf entries
  const int nw = Nc - 2;   // interior weights
  const int NA = Nc + Nf;
  if (offset_dev) offset += *offset_dev;
  for (int64_t ray = (int64_t)blockIdx.x * kHsWarps + warp; ray < B; ray += (int64_t)gridDim.x * kHsWarps) {
    const float* t = ts + ray * Nc;
    const float* w = weights + ray * Nc;
    // mid-point bins and the coarse depths themselves
    for (int i = lane; i < Nc; i += 32) {
      const float ti = __ldg(t + i);
      all[i] = ti;
      if (i < nb) bins[i] = 0.5f * (ti + __ldg(t + i + 1));
    }
    // pdf over weights[1:-1] + 1e-5, cdf = [0, cumsum(pdf)]
    float tot = 0.f;
    for (int i = lane; i < nw; i += 32) tot += __ldg(w + i + 1) + 1e-5f;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, d);
    float carry = 0.f;
    if (lane == 0) cdf[0] = 0.f;
    for (int base = 0; base < nw; base += 32) {
      const int i = base + lane;
      float p = (i < nw) ? (__ldg(w + i + 1) + 1e-5f) / tot : 0.f;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const float v = __shfl_up_sync(0xffffffffu, p, d);
        if (lane >= d) p += v;
      }
      if (i < nw) cdf[i + 1] = carry + p;
      carry += __shfl_sync(0xffffffffu, p, 31);
    }
    __syncwarp();
    // inverse transform sampling
    for (int k = lane; k < Nf; k += 32) {
      float u;
      if (mode == 0) u = __ldg(u_in + ray * Nf + k);
      else if (mode == 1) u = (Nf > 1) ? (float)k / (float)(Nf - 1) : 0.f;
      else {
        const uint64_t idx = (uint64_t)ray * (uint64_t)Nf + (uint64_t)k;
        const uint4 x = hs_philox(offset + (idx >> 2), seed);
        const uint32_t r = (idx & 3) == 0 ? x.x : ((idx & 3) == 1 ? x.y : ((idx & 3) == 2 ? x.z : x.w));
        u = (float)(r >> 8) * 5.9604644775390625e-08f;
      }
      // inds = searchsorted(cdf, u, right=True) = #entries <= u
      int lo = 0, hi = nb;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cdf[mid] <= u) lo = mid + 1; else hi = mid;
      }
      const int below = lo - 1 > 0 ? lo - 1 : 0;
      const int above = lo < nb - 1 ? lo : nb - 1;
      const float c0 = cdf[below], c1 = cdf[above];
      float denom = c1 - c0;
      denom = denom < 1e-5f ? 1.f : denom;
      const float f = (u - c0) / denom;
      all[Nc + k] = bins[below] + f * (bins[above] - bins[below]);
    }
    __syncwarp();
    // merge by rank (stable: ties keep index order); coarse depths are already sorted
    for (int e = lane; e < NA; e += 32) {
      const float v = all[e];
      int rank = 0;
      for (int j = 0; j < NA; ++j) {
        const float o = all[j];
        rank += (o < v || (o == v && j < e)) ? 1 : 0;
      }
      z_all[ray * NA + rank] = v;
    }
    __syncwarp();
  }
}

}  // namespace nb200

extern "C" int nb200_sample_pdf_merge(const float* ts, const float* weights, const float* u, int mode, uint64_t seed,
                                      uint64_t offset, int64_t B, int Nc, int Nf, float* z_all, nb200_stream_t stream) {
  using namespace nb200;
  if (B < 0 || Nc < 3 || Nf < 1 || mode < 0 || mode > 2) return NB200_ERR_ARG;
  if (Nc > kHsMaxNc || Nc + Nf > kHsMaxAll) return NB200_ERR_UNSUPPORTED;
  if (B == 0) return NB200_OK;
  if (!ts || !weights || !z_all || (mode == 0 && !u)) return NB200_ERR_ARG;
  const int64_t blocks = ceil_div64(B, kHsWarps);
  const int64_t cap = (int64_t)sm_count() * 16;
  sample_pdf_merge_kernel<<<(unsigned)(blocks < cap ? blocks : cap), kHsWarps * 32, 0, as_stream(stream)>>>(
      ts, weights, u, mode, seed, offset, B, Nc, Nf, z_all, nullptr);
  NB_LAUNCH_CHECK("sample_pdf_merge_kernel");
  return NB200_OK;
}

extern "C" int nb200_sample_pdf_merge_state(const float* ts, const float* weights, uint64_t seed, const void* state,
                                            int64_t B, int Nc, int Nf, float* z_all, nb200_stream_t stream) {
  using namespace nb200;
  if (!state || B < 0 || Nc < 3 || Nf < 1) return NB200_ERR_ARG;
  if (Nc > kHsMaxNc || Nc + Nf > kHsMaxAll) return NB200_ERR_UNSUPPORTED;
  if (B == 0) return NB200_OK;
  if (!ts || !weights || !z_all) return NB200_ERR_ARG;
  const int64_t blocks = ceil_div64(B, kHsWarps);
  const int64_t cap = (int64_t)sm_count() * 16;
  sample_pdf_merge_kernel<<<(unsigned)(blocks < cap ? blocks : cap), kHsWarps * 32, 0, as_stream(stream)>>>(
      ts, weights, nullptr, 2, seed, 0, B, Nc, Nf, z_all, &reinterpret_cast<const TrainState*>(state)->sample_offset);
  NB_LAUNCH_CHECK("sample_pdf_merge_kernel");
  return NB200_OK;
}
