// Device ray generation and stratified sampling (HBM-bound streaming kernels).
//   nb200_generate_rays  <- utils/xyz.py:38-52 + utils/rendering.py:129-134
//   nb200_stratified_ts  <- utils/rendering.py:24-30
#include <math.h>

#include "common.cuh"
#include "stream_common.cuh"

namespace nb200 {

// ---------------------------------------------------------------------------------- raygen
// One thread per ray; a ray is 24 B, so two neighbouring threads write 48 contiguous bytes and a
// warp writes 768 contiguous bytes (fully coalesced sectors).  Poses are 64 B each, L1-resident.
__global__ void __launch_bounds__(256) generate_rays_kernel(const float* __restrict__ poses, int H,
                                                            int W, float f, int64_t ray_begin,
                                                            int64_t n_rays, float* __restrict__ rays) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rays;
       i += (int64_t)gridDim.x * blockDim.x) {
    float o[6];
    camera_ray(poses, H, W, f, ray_begin + i, o);
    float2* dst = reinterpret_cast<float2*>(rays + i * 6);  // 24 B rows are 8 B aligned
    dst[0] = make_float2(o[0], o[1]);
    dst[1] = make_float2(o[2], o[3]);
    dst[2] = make_float2(o[4], o[5]);
  }
}

// --------------------------------------------------------------------------------- sampler
// Each thread produces 4 consecutive samples (one Philox call, one 16 B store when aligned).
__global__ void __launch_bounds__(256) stratified_ts_kernel(const float* __restrict__ u, uint64_t seed,
                                                            uint64_t offset, int64_t total, int N,
                                                            float tn, float tf, float* __restrict__ ts,
                                                            bool vec_ok) {
  const float step = __fdiv_rn(tf - tn, (float)N);
  const float bin = __fsub_rn(tbin(1, N, tn, tf, step), tbin(0, N, tn, tf, step));
  const int64_t nquads = (total + 3) >> 2;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nquads;
       q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t base = q << 2;
    float r[4];
    if (u != nullptr) {
      if (vec_ok && base + 3 < total) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(u + base));
        r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) r[k] = (base + k < total) ? __ldg(u + base + k) : 0.f;
      }
    } else {
      const uint4 x = philox4x32_10(offset + (uint64_t)q, seed);
      r[0] = u01(x.x); r[1] = u01(x.y); r[2] = u01(x.z); r[3] = u01(x.w);
    }
    float o[4];
    // one modulo per 4 samples (32-bit when the index allows), then wrap by compare
    int i0 = (base >> 32) == 0 ? (int)((uint32_t)base % (uint32_t)N) : (int)((uint64_t)base % (uint32_t)N);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      int i = i0 + k;
      i = i >= N ? i - N : i;
      i = i >= N ? i % N : i;                        // N < 4 only
      // utils/rendering.py:29: bin_diff*unif + t_bins[:-1]; two roundings, never an fma
      o[k] = __fadd_rn(__fmul_rn(bin, r[k]), tbin(i, N, tn, tf, step));
    }
    if (vec_ok && base + 3 < total) {
      *reinterpret_cast<float4*>(ts + base) = make_float4(o[0], o[1], o[2], o[3]);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (base + k < total) ts[base + k] = o[k];
    }
  }
}

// Fast path for N % 4 == 0 (a quad never straddles two rays).  The grid-stride is a multiple of
// the quads per ray, so a thread always lands on the same four bins: the bin edges are computed
// once per thread and a quad costs one Philox call + 4 x (shift, I2F, FMUL, FADD).  Same counter
// convention (offset + quad index) and the same two roundings as the generic kernel above:
// bin * (m * 2^-24) == m * (bin * 2^-24) exactly, the scale being a power of two.
template <bool kHasU>
__global__ void __launch_bounds__(256) stratified_ts_quad_kernel(const float* __restrict__ u, uint64_t seed,
                                                                 uint64_t offset, int64_t nquads, int N, int64_t stride,
                                                                 float tn, float tf, float* __restrict__ ts,
                                                                 const uint64_t* __restrict__ offset_dev) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= stride) return;
  if (offset_dev) offset += *offset_dev;   // device-resident stream position (CUDA-graph replays)
  const float step = __fdiv_rn(tf - tn, (float)N);
  const float bin = __fsub_rn(tbin(1, N, tn, tf, step), tbin(0, N, tn, tf, step));
  const float scale = kHasU ? bin : bin * 5.9604644775390625e-08f;
  const int i0 = (int)(tid % (N >> 2)) << 2;
  float tb[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) tb[k] = tbin(i0 + k, N, tn, tf, step);
  for (int64_t q = tid; q < nquads; q += stride) {
    float r[4];
    if constexpr (kHasU) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(u) + q);
      r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
    } else {
      const uint4 x = philox4x32_10(offset + (uint64_t)q, seed);
      r[0] = (float)(x.x >> 8); r[1] = (float)(x.y >> 8); r[2] = (float)(x.z >> 8); r[3] = (float)(x.w >> 8);
    }
    // utils/rendering.py:29: bin_diff*unif + t_bins[:-1]; two roundings, never an fma
    reinterpret_cast<float4*>(ts)[q] = make_float4(__fadd_rn(__fmul_rn(scale, r[0]), tb[0]), __fadd_rn(__fmul_rn(scale, r[1]), tb[1]),
                                                   __fadd_rn(__fmul_rn(scale, r[2]), tb[2]), __fadd_rn(__fmul_rn(scale, r[3]), tb[3]));
  }
}

// ------------------------------------------------------------------------------------ Adam
// torch.optim.Adam (no weight decay, no amsgrad) over one flat buffer: train.py:43,55.
__global__ void __launch_bounds__(256) adam_flat_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                        float* __restrict__ m, float* __restrict__ v, int64_t n, float lr,
                                                        float beta1, float beta2, float eps, float bc1, float bc2_sqrt) {
  const int64_t i4 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= n) return;
  const float step_size = lr / bc1;
  if (i4 + 3 < n) {
    float4 pp = *reinterpret_cast<float4*>(p + i4), mm = *reinterpret_cast<float4*>(m + i4), vv = *reinterpret_cast<float4*>(v + i4);
    const float4 gg = *reinterpret_cast<const float4*>(g + i4);
    float* pa = &pp.x; float* ma = &mm.x; float* va = &vv.x; const float* ga = &gg.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      ma[k] = beta1 * ma[k] + (1.f - beta1) * ga[k];
      va[k] = beta2 * va[k] + (1.f - beta2) * ga[k] * ga[k];
      pa[k] -= step_size * ma[k] / (sqrtf(va[k]) / bc2_sqrt + eps);
    }
    *reinterpret_cast<float4*>(p + i4) = pp; *reinterpret_cast<float4*>(m + i4) = mm; *reinterpret_cast<float4*>(v + i4) = vv;
  } else {
    for (int64_t i = i4; i < n; ++i) {
      m[i] = beta1 * m[i] + (1.f - beta1) * g[i];
      v[i] = beta2 * v[i] + (1.f - beta2) * g[i] * g[i];
      p[i] -= step_size * m[i] / (sqrtf(v[i]) / bc2_sqrt + eps);
    }
  }
}

// ---------------------------------------------------------------------- train-step helpers
// Ray selection on the device: rg.select('train', B) + train_imgs[ray_ids] (train.py:47-49,
// utils/dataload.py:141-153).  The reference draws a CPU randperm over the whole table (328 ms per
// step); here B indices are drawn uniformly WITH replacement from Philox (seed, offset + i) and
// the 24-byte ray row and 12-byte colour row are gathered in the same kernel.
__global__ void __launch_bounds__(256) select_rays_kernel(const float* __restrict__ rays_table,
                                                          const float* __restrict__ gt_table, int64_t n_table,
                                                          uint64_t seed, uint64_t offset, int64_t B,
                                                          float* __restrict__ rays, float* __restrict__ gt,
                                                          int64_t* __restrict__ ids, const uint64_t* __restrict__ offset_dev) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  if (offset_dev) offset += *offset_dev;
  const uint4 x = philox4x32_10(offset + (uint64_t)i, seed);
  // 64 random bits -> [0, n_table): high word of the 64x64 product (bias < n_table * 2^-64)
  const uint64_t r64 = ((uint64_t)x.y << 32) | x.x;
  const int64_t id = (int64_t)__umul64hi(r64, (uint64_t)n_table);
  const float2* src = reinterpret_cast<const float2*>(rays_table + id * 6);
  float2* dst = reinterpret_cast<float2*>(rays + i * 6);
  const float2 a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);
  dst[0] = a; dst[1] = b; dst[2] = c;
  if (gt_table != nullptr) {
    gt[i * 3] = __ldg(gt_table + id * 3);
    gt[i * 3 + 1] = __ldg(gt_table + id * 3 + 1);
    gt[i * 3 + 2] = __ldg(gt_table + id * 3 + 2);
  }
  if (ids != nullptr) ids[i] = id;
}

// MSELoss(rgb, gt) over B*3 values and its gradient (train.py:42,52): loss = mean((rgb-gt)^2),
// d_rgb = 2 (rgb - gt) / (3B).  One block, fixed summation order (deterministic loss).
__global__ void __launch_bounds__(1024) mse_loss_grad_kernel(const float* __restrict__ rgb, const float* __restrict__ gt,
                                                             int64_t n, float* __restrict__ d_rgb, float* __restrict__ loss) {
  __shared__ float part[32];
  const float scale = 2.0f / (float)n;
  float acc = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const float d = rgb[i] - gt[i];
    d_rgb[i] = d * scale;
    acc = fmaf(d, d, acc);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (threadIdx.x == 0 && loss != nullptr) *loss = v / (float)n;
  }
}

// ------------------------------------------------------------------ device-resident step state
// (TrainState: stream_common.cuh)
__global__ void __launch_bounds__(256) adam_flat_state_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                              float* __restrict__ m, float* __restrict__ v, int64_t n,
                                                              const TrainState* __restrict__ st, float beta1, float beta2, float eps) {
  const int64_t i4 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= n) return;
  const float t = (float)(st->step + 1);
  const float bc1 = 1.f - powf(beta1, t), bc2_sqrt = sqrtf(1.f - powf(beta2, t));
  const float step_size = st->lr / bc1;
  const bool vec = i4 + 3 < n && ((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0);
  if (vec) {   // the flat buffers of the Trainer: 16-byte aligned, padded to multiples of 4
    float4 pp = *reinterpret_cast<float4*>(p + i4), mm = *reinterpret_cast<float4*>(m + i4), vv = *reinterpret_cast<float4*>(v + i4);
    const float4 gg = *reinterpret_cast<const float4*>(g + i4);
    float* pa = &pp.x; float* ma = &mm.x; float* va = &vv.x; const float* ga = &gg.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      ma[k] = beta1 * ma[k] + (1.f - beta1) * ga[k];
      va[k] = beta2 * va[k] + (1.f - beta2) * ga[k] * ga[k];
      pa[k] -= step_size * ma[k] / (sqrtf(va[k]) / bc2_sqrt + eps);
    }
    *reinterpret_cast<float4*>(p + i4) = pp; *reinterpret_cast<float4*>(m + i4) = mm; *reinterpret_cast<float4*>(v + i4) = vv;
    return;
  }
  for (int64_t i = i4; i < n && i < i4 + 4; ++i) {
    const float gi = g[i];
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] -= step_size * mi / (sqrtf(vi) / bc2_sqrt + eps);
  }
}

// ------------------------------------------------- gradient all-reduce fused into Adam (NVLink peer memory)
// Data-parallel training (SURVEY 8e): instead of an NCCL all-reduce followed by the optimizer kernel, every rank's
// Adam kernel reads the flat gradient of ALL ranks straight out of their HBM over NVLink / NVSwitch (the buffers
// are mapped into each process through CUDA IPC), sums them in rank order (identical on every rank, so the
// replicas stay bit-identical), divides by the world size and applies the update to its own replica.  2.38 MB per
// peer per step: a few microseconds of NVLink time, no separate collective, and the whole step stays ONE CUDA graph.
//   entry : block 0 tells every peer "my gradients of step `epoch` are complete" (release, system scope); every block
//           waits until all peers said so (acquire, system scope)
//   exit  : the last block to finish tells every peer "I am done reading yours" and waits for the same from them, so
//           that stream order protects this rank's gradient buffer from its own next step
// flags of rank r (device memory of r, written remotely): [0, kMaxPeers) ready epochs, [kMaxPeers, 2 kMaxPeers) done
// epochs, [2 kMaxPeers] block counter.
constexpr int kMaxPeers = 8;
struct PeerPtrs {
  const float* grad[kMaxPeers];
  uint32_t* flags[kMaxPeers];
};
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_relaxed_sys_f4(const float* p) {   // never served from a stale (non-coherent) L1 line
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
// Bounded spin: a rank that never arrives must surface as a launch error, not as a hung GPU.
__device__ __forceinline__ void wait_epoch(const uint32_t* flag, uint32_t epoch, int tag) {
  uint64_t t0 = 0;
  uint32_t it = 0;
  while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
    if ((++it & 0x3FFu) == 0u) {
      uint64_t now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 20000000000ull) {
        printf("nb200: peer flag wait timed out (block %d thread %d tag %d epoch %u)\n", blockIdx.x, threadIdx.x, tag, epoch);
        __trap();
      }
    }
  }
}

__global__ void __launch_bounds__(256) adam_allreduce_p2p_kernel(float* __restrict__ p, PeerPtrs peers, int rank, int world,
                                                                 float* __restrict__ m, float* __restrict__ v, int64_t n,
                                                                 const TrainState* __restrict__ st, float beta1, float beta2, float eps) {
  const uint32_t epoch = (uint32_t)(st->step + 1);
  uint32_t* mine = peers.flags[rank];
  if (blockIdx.x == 0 && (int)threadIdx.x < world) {
    __threadfence_system();                                   // this rank's gradient writes (earlier kernels) before the flag
    st_release_sys(peers.flags[threadIdx.x] + rank, epoch);   // flags[r][ready + me] = epoch
  }
  if ((int)threadIdx.x < world) wait_epoch(mine + threadIdx.x, epoch, 1);
  __syncthreads();
  const float t = (float)(st->step + 1);
  const float bc1 = 1.f - powf(beta1, t), bc2_sqrt = sqrtf(1.f - powf(beta2, t));
  const float step_size = st->lr / bc1, inv_world = 1.f / (float)world;
  const int64_t n4 = n >> 2;                                  // the flat buffers are padded to multiples of 4 floats
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += (int64_t)gridDim.x * blockDim.x) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r) {                     // rank order: the same sum on every rank
      if (r < world) {
        const float4 x = ld_relaxed_sys_f4(peers.grad[r] + 4 * q);
        g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
      }
    }
    float4 pp = reinterpret_cast<float4*>(p)[q], mm = reinterpret_cast<float4*>(m)[q], vv = reinterpret_cast<float4*>(v)[q];
    float* pa = &pp.x; float* ma = &mm.x; float* va = &vv.x; float* ga = &g.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gi = ga[k] * inv_world;
      ma[k] = beta1 * ma[k] + (1.f - beta1) * gi;
      va[k] = beta2 * va[k] + (1.f - beta2) * gi * gi;
      pa[k] -= step_size * ma[k] / (sqrtf(va[k]) / bc2_sqrt + eps);
    }
    reinterpret_cast<float4*>(p)[q] = pp; reinterpret_cast<float4*>(m)[q] = mm; reinterpret_cast<float4*>(v)[q] = vv;
  }
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(mine + 2 * kMaxPeers, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {
    if ((int)threadIdx.x < world) {
      __threadfence_system();
      st_release_sys(peers.flags[threadIdx.x] + kMaxPeers + rank, epoch);    // "I am done reading your gradients"
      wait_epoch(mine + kMaxPeers + threadIdx.x, epoch, 2);                  // everyone is done reading mine
    }
    if (threadIdx.x == 0) mine[2 * kMaxPeers] = 0u;
  }
}

__global__ void train_state_advance_kernel(TrainState* st, uint64_t select_inc, uint64_t sample_inc, float lr_decay) {
  st->select_offset += select_inc;
  st->sample_offset += sample_inc;
  st->step += 1;
  st->lr *= lr_decay;       // train.py:56-57
}

}  // namespace nb200

// ------------------------------------------------------------------------------ video frames
// rgb [n,3] fp32 -> u8 [n,3]: clip to [0,1] (utils/rendering.py:146), swap to BGR (cv2.cvtColor, :158), multiply by
// 255 in fp32 and truncate (numpy astype(uint8), :159).  One thread per 4 pixels: three float4 loads, three
// 32-bit stores (48 B in, 12 B out, both fully coalesced).
__device__ __forceinline__ uint32_t to_u8(float v) {
  return (uint32_t)__float2int_rz(__fmul_rn(fminf(fmaxf(v, 0.f), 1.f), 255.f));
}
__global__ void __launch_bounds__(256) frame_to_u8_kernel(const float* __restrict__ rgb, int64_t n, int bgr,
                                                          uint8_t* __restrict__ out, bool vec_ok) {
  const int64_t nquads = (n + 3) >> 2;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nquads; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p0 = q << 2;
    if (vec_ok && p0 + 3 < n) {
      const float4* src = reinterpret_cast<const float4*>(rgb + p0 * 3);
      const float4 a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);
      const float v[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
      uint32_t w[3] = {0u, 0u, 0u};
#pragma unroll
      for (int k = 0; k < 12; ++k) {
        const int px = k / 3, ch = k % 3;
        const int o = px * 3 + (bgr ? 2 - ch : ch);
        w[o >> 2] |= to_u8(v[k]) << (8 * (o & 3));
      }
      uint32_t* dst = reinterpret_cast<uint32_t*>(out + p0 * 3);
      dst[0] = w[0]; dst[1] = w[1]; dst[2] = w[2];
    } else {
      for (int64_t p = p0; p < n && p < p0 + 4; ++p)
        for (int ch = 0; ch < 3; ++ch) out[p * 3 + (bgr ? 2 - ch : ch)] = (uint8_t)to_u8(__ldg(rgb + p * 3 + ch));
    }
  }
}

extern "C" {

int nb200_frame_to_u8(const float* rgb, int64_t n_pixels, int bgr, uint8_t* out, nb200_stream_t stream) {
  using namespace nb200;
  if (n_pixels < 0) return NB200_ERR_ARG;
  if (n_pixels == 0) return NB200_OK;
  if (!rgb || !out) return NB200_ERR_ARG;
  const bool vec_ok = (((uintptr_t)rgb & 15) | ((uintptr_t)out & 3)) == 0;
  const int64_t blocks = ceil_div64(ceil_div64(n_pixels, 4), 256);
  const int grid = (int)(blocks < (int64_t)sm_count() * 16 ? blocks : (int64_t)sm_count() * 16);
  frame_to_u8_kernel<<<grid, 256, 0, as_stream(stream)>>>(rgb, n_pixels, bgr, out, vec_ok);
  NB_LAUNCH_CHECK("frame_to_u8_kernel");
  return NB200_OK;
}

int nb200_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step, float lr,
                    float beta1, float beta2, float eps, nb200_stream_t stream) {
  using namespace nb200;
  if (!param || !grad || !exp_avg || !exp_avg_sq || n < 0 || step < 1) return NB200_ERR_ARG;
  if (n == 0) return NB200_OK;
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2_sqrt = sqrtf(1.f - powf(beta2, (float)step));
  adam_flat_kernel<<<(unsigned)ceil_div64(ceil_div64(n, 4), 256), 256, 0, as_stream(stream)>>>(
      param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, bc1, bc2_sqrt);
  NB_LAUNCH_CHECK("adam_flat_kernel");
  return NB200_OK;
}

int nb200_generate_rays(const float* poses, int P, int H, int W, float f, int64_t ray_begin,
                        int64_t n_rays, float* rays, nb200_stream_t stream) {
  using namespace nb200;
  if (P <= 0 || H <= 0 || W <= 0 || !(f > 0.f) || ray_begin < 0 || n_rays < 0 ||
      ray_begin + n_rays > (int64_t)P * H * W)
    return NB200_ERR_ARG;
  if (n_rays == 0) return NB200_OK;
  if (!poses || !rays || ((uintptr_t)rays & 7)) return NB200_ERR_ARG;  // float2 stores
  const int64_t blocks = ceil_div64(n_rays, 256);
  const int grid = (int)(blocks < (int64_t)sm_count() * 16 ? blocks : (int64_t)sm_count() * 16);
  generate_rays_kernel<<<grid, 256, 0, as_stream(stream)>>>(poses, H, W, f, ray_begin, n_rays, rays);
  NB_LAUNCH_CHECK("generate_rays_kernel");
  return NB200_OK;
}

int nb200_stratified_ts(const float* u, uint64_t seed, uint64_t offset, int64_t B, int N, float tn,
                        float tf, float* ts, nb200_stream_t stream) {
  using namespace nb200;
  if (B < 0 || N < 1) return NB200_ERR_ARG;
  const int64_t total = B * (int64_t)N;
  if (total == 0) return NB200_OK;
  if (!ts) return NB200_ERR_ARG;
  const int64_t blocks = ceil_div64(ceil_div64(total, 4), 256);
  const int grid = (int)(blocks < (int64_t)sm_count() * 16 ? blocks : (int64_t)sm_count() * 16);
  const bool aligned = (((uintptr_t)ts | (uintptr_t)u) & 15) == 0;
  if (N % 4 == 0 && N <= 1024 && aligned) {
    const int64_t threads = (int64_t)grid * 256;
    const int64_t stride = threads - threads % (N >> 2);
    if (u)
      stratified_ts_quad_kernel<true><<<grid, 256, 0, as_stream(stream)>>>(u, seed, offset, total >> 2, N, stride, tn, tf, ts, nullptr);
    else
      stratified_ts_quad_kernel<false><<<grid, 256, 0, as_stream(stream)>>>(u, seed, offset, total >> 2, N, stride, tn, tf, ts, nullptr);
  } else {
    stratified_ts_kernel<<<grid, 256, 0, as_stream(stream)>>>(u, seed, offset, total, N, tn, tf, ts, aligned);
  }
  NB_LAUNCH_CHECK("stratified_ts_kernel");
  return NB200_OK;
}

int nb200_select_rays(const float* rays_table, const float* gt_table, int64_t n_table, uint64_t seed,
                      uint64_t offset, int64_t B, float* rays, float* gt, int64_t* ids, nb200_stream_t stream) {
  using namespace nb200;
  if (B < 0 || n_table <= 0) return NB200_ERR_ARG;
  if (B == 0) return NB200_OK;
  if (!rays_table || !rays || (gt_table && !gt)) return NB200_ERR_ARG;
  if ((((uintptr_t)rays_table | (uintptr_t)rays) & 7) != 0) return NB200_ERR_ARG;
  select_rays_kernel<<<(unsigned)ceil_div64(B, 256), 256, 0, as_stream(stream)>>>(rays_table, gt_table, n_table, seed, offset,
                                                                                B, rays, gt, ids, nullptr);
  NB_LAUNCH_CHECK("select_rays_kernel");
  return NB200_OK;
}

int nb200_mse_loss_grad(const float* rgb, const float* gt, int64_t B, float* d_rgb, float* loss, nb200_stream_t stream) {
  using namespace nb200;
  if (B <= 0 || !rgb || !gt || !d_rgb) return NB200_ERR_ARG;
  mse_loss_grad_kernel<<<1, 1024, 0, as_stream(stream)>>>(rgb, gt, B * 3, d_rgb, loss);
  NB_LAUNCH_CHECK("mse_loss_grad_kernel");
  return NB200_OK;
}

// ---- variants that read the per-step quantities from a device-resident nb200 train state (CUDA graphs)
int nb200_train_state_init(void* state, uint64_t select_offset, uint64_t sample_offset, int64_t step, float lr,
                           nb200_stream_t stream) {
  using namespace nb200;
  if (!state) return NB200_ERR_ARG;
  TrainState h = {select_offset, sample_offset, step, lr, 0.f};
  // the source must outlive the async copy: pass by value through a kernel-free, stream-ordered memset + small memcpys
  NB_CUDA_CHECK(cudaMemcpyAsync(state, &h, sizeof(h), cudaMemcpyHostToDevice, as_stream(stream)));
  NB_CUDA_CHECK(cudaStreamSynchronize(as_stream(stream)));   // one-time set-up call
  return NB200_OK;
}

int nb200_train_state_advance(void* state, uint64_t select_inc, uint64_t sample_inc, float lr_decay, nb200_stream_t stream) {
  using namespace nb200;
  if (!state) return NB200_ERR_ARG;
  train_state_advance_kernel<<<1, 1, 0, as_stream(stream)>>>(reinterpret_cast<TrainState*>(state), select_inc, sample_inc, lr_decay);
  NB_LAUNCH_CHECK("train_state_advance_kernel");
  return NB200_OK;
}

int nb200_select_rays_state(const float* rays_table, const float* gt_table, int64_t n_table, uint64_t seed, const void* state,
                            int64_t B, float* rays, float* gt, int64_t* ids, nb200_stream_t stream) {
  using namespace nb200;
  if (B < 0 || n_table <= 0 || !state) return NB200_ERR_ARG;
  if (B == 0) return NB200_OK;
  if (!rays_table || !rays || (gt_table && !gt)) return NB200_ERR_ARG;
  if ((((uintptr_t)rays_table | (uintptr_t)rays) & 7) != 0) return NB200_ERR_ARG;
  select_rays_kernel<<<(unsigned)ceil_div64(B, 256), 256, 0, as_stream(stream)>>>(
      rays_table, gt_table, n_table, seed, 0, B, rays, gt, ids, &reinterpret_cast<const TrainState*>(state)->select_offset);
  NB_LAUNCH_CHECK("select_rays_kernel");
  return NB200_OK;
}

int nb200_stratified_ts_state(uint64_t seed, const void* state, int64_t B, int N, float tn, float tf, float* ts,
                              nb200_stream_t stream) {
  using namespace nb200;
  if (B < 0 || N < 4 || (N & 3) || N > 1024 || !state) return NB200_ERR_ARG;   // quad kernel only
  const int64_t total = B * (int64_t)N;
  if (total == 0) return NB200_OK;
  if (!ts || ((uintptr_t)ts & 15)) return NB200_ERR_ARG;
  const int64_t blocks = ceil_div64(ceil_div64(total, 4), 256);
  const int grid = (int)(blocks < (int64_t)sm_count() * 16 ? blocks : (int64_t)sm_count() * 16);
  const int64_t threads = (int64_t)grid * 256;
  const int64_t stride = threads - threads % (N >> 2);
  stratified_ts_quad_kernel<false><<<grid, 256, 0, as_stream(stream)>>>(
      nullptr, seed, 0, total >> 2, N, stride, tn, tf, ts, &reinterpret_cast<const TrainState*>(state)->sample_offset);
  NB_LAUNCH_CHECK("stratified_ts_quad_kernel");
  return NB200_OK;
}

int nb200_adam_step_state(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const void* state,
                          float beta1, float beta2, float eps, nb200_stream_t stream) {
  using namespace nb200;
  if (!param || !grad || !exp_avg || !exp_avg_sq || n < 0 || !state) return NB200_ERR_ARG;
  if (n == 0) return NB200_OK;
  adam_flat_state_kernel<<<(unsigned)ceil_div64(ceil_div64(n, 4), 256), 256, 0, as_stream(stream)>>>(
      param, grad, exp_avg, exp_avg_sq, n, reinterpret_cast<const TrainState*>(state), beta1, beta2, eps);
  NB_LAUNCH_CHECK("adam_flat_state_kernel");
  return NB200_OK;
}


int nb200_adam_allreduce_p2p(float* param, const float* const* peer_grads, uint32_t* const* peer_flags, int rank, int world,
                             float* exp_avg, float* exp_avg_sq, int64_t n, const void* state, float beta1, float beta2,
                             float eps, nb200_stream_t stream) {
  using namespace nb200;
  if (!param || !peer_grads || !peer_flags || !exp_avg || !exp_avg_sq || !state || n < 0) return NB200_ERR_ARG;
  if (world < 1 || world > kMaxPeers || rank < 0 || rank >= world) return NB200_ERR_UNSUPPORTED;
  if ((n & 3) || (((uintptr_t)param | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15)) return NB200_ERR_ARG;
  PeerPtrs pp;
  for (int r = 0; r < kMaxPeers; ++r) {
    pp.grad[r] = r < world ? peer_grads[r] : nullptr;
    pp.flags[r] = r < world ? peer_flags[r] : nullptr;
    if (r < world && (!pp.grad[r] || !pp.flags[r] || ((uintptr_t)pp.grad[r] & 15))) return NB200_ERR_ARG;
  }
  if (n == 0) return NB200_OK;
  // every block spins on the peers at entry: keep the grid within one wave so that no block waits for a slot
  const int64_t blocks = ceil_div64(n >> 2, 256);
  const int grid = (int)(blocks < (int64_t)sm_count() * 4 ? blocks : (int64_t)sm_count() * 4);
  adam_allreduce_p2p_kernel<<<grid, 256, 0, as_stream(stream)>>>(param, pp, rank, world, exp_avg, exp_avg_sq, n,
                                                                reinterpret_cast<const TrainState*>(state), beta1, beta2, eps);
  NB_LAUNCH_CHECK("adam_allreduce_p2p_kernel");
  return NB200_OK;
}

}  // extern "C"
