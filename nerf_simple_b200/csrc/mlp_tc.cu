// NB200_BF16 precision: fused positional-encoding + NeRF MLP on tcgen05 / TMEM (sm_100a).
//   forward  <- utils/xyz.py:16-36 + utils/nets.py:34-43 (+ utils/rendering.py:31-40 in rays mode)
//   backward <- autograd of the same (parameter gradients only)
//
// This file owns the packed weight image (pre-swizzled bf16 UMMA operand slabs + fp32 tail), the
// saved-tensor layout and the host entry points.  The kernels live in
//   mlp_chain.cuh  : chain_kernel<FwdEpi> / chain_kernel<DgradEpi> -- persistent 2-CTA clusters,
//                    tcgen05.mma.cta_group::2, two tiles in flight per CTA, weights by tensor-map TMA
//   mlp_tc_bwd.cuh : wgrad (MN-major UMMA operands, dW resident in TMEM) and the head gradients
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <type_traits>
#include <utility>

#include "common.cuh"
#include "stream_common.cuh"
#include "tc_common.cuh"

namespace nb200 {
using namespace tc;

// ------------------------------------------------------------------ packed weight image
constexpr int kNumMmaLayers = 10;  // L0_0..L0_4, skip, L1_0, L1_1, layers_2, color_fc.0
constexpr int kMaxSlabs = 48;
// NB200_BF16 folds layers_2 into color_fc.0.  layers_2 has no activation (utils/nets.py:41-42), so
//   color_fc.0(cat[layers_2(h7), posd]) = (Wc0[:, :256] Wg) h7 + Wc0[:, 256:] posd + (Wc0[:, :256] bg + bc0):
// the folded weight Wf = Wc0[:, :256] Wg (128 x 256) and bias bf are formed in fp32 at pack time and rounded to bf16
// once, so a sample costs 9 MMA layers instead of 10 (-11 % of the FLOPs) and `g` is never rounded to bf16.
// Backward: delta_h7 = delta_c1 Wf (one 128 -> 256 layer instead of two), and with Gm = delta_c1^T h7 (128 x 256, ONE
// wgrad item) the chain rule gives dWc0[:, :256] = Gm Wg^T + s bg^T, dWg = Wc0[:, :256]^T Gm, dbg = Wc0[:, :256]^T s,
// dbc0 = s (s = column sums of delta_c1): two tiny fp32 GEMMs (fold_grads_kernel) replace the 256 x 256 wgrad item of
// layers_2 and the HBM round trip of g and delta_g.  NB200_BF16_LAYERWISE keeps every layer of the reference as its
// own MMA layer.
constexpr int kNumFoldLayers = kNumMmaLayers - 1;
constexpr int kLayerFold = 100;    // SlabDesc::layer of a slab packed from the folded fp32 weight in the packed buffer's tail
constexpr int kFoldBiasRow = 10;   // bias row of the folded color_fc.0

struct SlabDesc {
  uint32_t off;     // byte offset of the slab image in the packed buffer
  uint32_t bytes;   // n * 128
  uint16_t n;       // operand rows (output features): 256 or 128
  uint16_t wcol0;   // first weight column (input feature) covered
  uint16_t kvalid;  // valid columns (rest zero padded up to 64)
  uint16_t ldw;     // row pitch of the fp32 weight
  uint8_t ml;       // MMA layer index 0..9
  uint8_t layer;    // Layer enum (index into the 24 parameter pointers / 2)
  uint8_t src;      // A operand: 0 = activation buffer K-block `kb`, 1 = encoding buffer
  uint8_t kb;
  uint8_t ksteps;   // number of K=16 MMAs
  uint8_t first;    // first slab of its layer (accumulator is overwritten)
  uint8_t last;     // last slab of its layer (commit to acc_full)
  uint8_t flags;    // kSlabTransposed | kSlabLo | kSlabBothA (the struct stays 24 bytes: the MMA warp's issue loop reads it
                    // through the uniform datapath, and a 28-byte stride cost the forward kernel 13 %)
};
constexpr uint8_t kSlabTransposed = 1;  // image(n,k) = W[(wcol0+k)*ldw + n] (dgrad operand) instead of W[n*ldw + wcol0+k]
constexpr uint8_t kSlabLo = 2;          // bf16x3: image of the residual W - bf16(W) instead of bf16(W)
constexpr uint8_t kSlabBothA = 4;       // bf16x3: this slab multiplies A_hi and then A_lo (else A_hi only)
static_assert(sizeof(SlabDesc) == 24, "SlabDesc layout");

struct PackedLayout {
  int num_fwd;
  SlabDesc fwd[kMaxSlabs];
  int num_bwd;
  SlabDesc bwd[kMaxSlabs];  // dgrad chain: transposed weight images, 9 MMA layers
  // folded chains: the tables of the 9-layer forward and the 8-layer delta chain (entries shared with fwd / bwd point
  // at the same images), and the 6 slabs that exist only in the folded form (Wf: 4 forward + 2 transposed)
  int num_fwdf;
  SlabDesc fwdf[kMaxSlabs];
  int num_bwdf;
  SlabDesc bwdf[kMaxSlabs];
  int num_fold;
  SlabDesc fold[8];
  uint32_t f32_off;  // fp32 section: bias[11][256] | wsig[256] | bsig(+pad 4) | wc1[3][128] | bc1[3](+pad) | fold tail
  uint32_t total_bytes;
  // NB200_BF16X3 (error-compensated bf16): its own packed buffer = per K-block a hi slab bf16(W) and a lo slab
  // bf16(W - bf16(W)), then the same fp32 tail, then the delta chain's transposed slabs in the same hi / lo pairs
  int num_fwd3;
  SlabDesc fwd3[2 * kMaxSlabs];
  uint32_t f32_off3;
  uint32_t total_bytes3;
  int num_bwd3;
  SlabDesc bwd3[2 * kMaxSlabs];   // (behind every older field: the bf16 kernels' constant-bank offsets do not move)
};
constexpr int kF32Bias = 0, kF32WSig = 2816, kF32BSig = 3072, kF32WC1 = 3076, kF32BC1 = 3460,
              kF32Floats = 3520;
// fold tail (bf16 image only): Wf [128][256] | Wg^T [256][256] | Wc0[:, :256] [128][256] | bg [256], all fp32
constexpr int kF32Wf = kF32Floats, kF32WgT = kF32Wf + 128 * 256, kF32Wc0g = kF32WgT + 256 * 256, kF32Bg = kF32Wc0g + 128 * 256,
              kF32FloatsFold = kF32Bg + 256;

__host__ __device__ constexpr int mma_layer_of(int ml) {
  return ml <= 4 ? L0_0 + ml : (ml == 5 ? L_SKIP : (ml <= 7 ? L1_0 + (ml - 6) : (ml == 8 ? L_2 : L_C0)));
}

struct LayoutBuilder {
  SlabDesc* arr;
  uint32_t off;
  int s;
  constexpr void add(int ml, int layer, int transposed, int n, int wcol0, int kvalid, int ldw, int src, int kb, int ksteps,
                     int lo = 0, int amode = 0) {
    SlabDesc& d = arr[s++];
    d.off = off; d.bytes = (uint32_t)n * 128u; d.n = (uint16_t)n; d.wcol0 = (uint16_t)wcol0;
    d.kvalid = (uint16_t)kvalid; d.ldw = (uint16_t)ldw; d.ml = (uint8_t)ml; d.layer = (uint8_t)layer;
    d.src = (uint8_t)src; d.kb = (uint8_t)kb; d.ksteps = (uint8_t)ksteps; d.first = 0; d.last = 0;
    d.flags = (uint8_t)((transposed ? kSlabTransposed : 0) | (lo ? kSlabLo : 0) | (amode ? kSlabBothA : 0));
    off += d.bytes;
  }
};

// dgrad chain (mlp_bwd.cuh): MMA layer bl = 1..9 computes delta_in = delta_out @ W (W un-transposed
// [out,in]); its B operand image is W^T: image(n = in-feature, k = out-feature).
__host__ __device__ constexpr int bwd_layer_of(int bl) {
  return bl == 1 ? L_C0 : (bl == 2 ? L_2 : (bl == 3 ? L1_1 : (bl == 4 ? L1_0 : (bl == 5 ? L_SKIP : L0_4 - (bl - 6)))));
}

constexpr PackedLayout make_layout() {
  PackedLayout lay{};
  LayoutBuilder b{lay.fwd, 0, 0};
  for (int ml = 0; ml < kNumMmaLayers; ++ml) {
    const int first = b.s, ly = mma_layer_of(ml);
    if (ml == 0) {
      b.add(ml, ly, 0, 256, 0, kPosX, kPosX, 1, 0, 4);
    } else if (ml == 5) {  // cat([h, posx]) (utils/nets.py:38)
      for (int kb = 0; kb < 4; ++kb) b.add(ml, ly, 0, 256, kb * 64, 64, kHidden + kPosX, 0, kb, 4);
      b.add(ml, ly, 0, 256, 256, kPosX, kHidden + kPosX, 1, 0, 4);
    } else if (ml == 9) {  // cat([g, posd]) (utils/nets.py:42), 128 outputs
      for (int kb = 0; kb < 4; ++kb) b.add(ml, ly, 0, 128, kb * 64, 64, kHidden + kPosD, 0, kb, 4);
      b.add(ml, ly, 0, 128, 256, kPosD, kHidden + kPosD, 1, 0, 2);
    } else {
      for (int kb = 0; kb < 4; ++kb) b.add(ml, ly, 0, 256, kb * 64, 64, kHidden, 0, kb, 4);
    }
    lay.fwd[first].first = 1;
    lay.fwd[b.s - 1].last = 1;
  }
  lay.num_fwd = b.s;
  // dgrad slabs: n = 256 input features (rows of the image), k-blocks over the output features
  LayoutBuilder t{lay.bwd, b.off, 0};
  for (int bl = 1; bl <= 9; ++bl) {
    const int first = t.s, ly = bwd_layer_of(bl);
    const int ldw = (ly == L_C0) ? kHidden + kPosD : (ly == L_SKIP ? kHidden + kPosX : kHidden);
    const int nkb = (bl == 1) ? 2 : 4;  // color_fc.0 has 128 outputs
    for (int kb = 0; kb < nkb; ++kb) t.add(bl, ly, 1, 256, kb * 64, 64, ldw, 0, kb, 4);
    lay.bwd[first].first = 1;
    lay.bwd[t.s - 1].last = 1;
  }
  lay.num_bwd = t.s;
  // the slabs of the folded weight: forward image (n = c1 feature, k = h7 feature), then transposed for the delta chain
  LayoutBuilder f{lay.fold, t.off, 0};
  for (int kb = 0; kb < 4; ++kb) f.add(9, kLayerFold, 0, 128, kb * 64, 64, kHidden, 0, kb, 4);
  for (int kb = 0; kb < 2; ++kb) f.add(2, kLayerFold, 1, 256, kb * 64, 64, kHidden, 0, kb, 4);
  lay.num_fold = f.s;
  {
    int n = 0;
    for (int i = 0; i < lay.num_fwd; ++i)
      if (lay.fwd[i].ml < 8) lay.fwdf[n++] = lay.fwd[i];
    for (int kb = 0; kb < 4; ++kb) lay.fwdf[n++] = lay.fold[kb];
    lay.fwdf[n - 4].first = 1;
    lay.fwdf[n++] = lay.fwd[lay.num_fwd - 1];   // color_fc.0 <- posd (last slab of the layer)
    lay.num_fwdf = n;
    n = 0;
    for (int kb = 0; kb < 2; ++kb) lay.bwdf[n++] = lay.fold[4 + kb];
    lay.bwdf[0].first = 1; lay.bwdf[1].last = 1;
    for (int i = 0; i < lay.num_bwd; ++i)
      if (lay.bwd[i].ml >= 3) lay.bwdf[n++] = lay.bwd[i];
    lay.num_bwdf = n;
  }
  lay.f32_off = f.off;
  lay.total_bytes = f.off + kF32FloatsFold * (uint32_t)sizeof(float);
  // bf16x3: every forward slab twice (hi: consumed with A_hi and A_lo; lo: with A_hi), in consumption order
  LayoutBuilder x{lay.fwd3, 0, 0};
  for (int i = 0; i < lay.num_fwd; ++i) {
    const SlabDesc& f = lay.fwd[i];
    for (int lo = 0; lo < 2; ++lo) {
      x.add(f.ml, f.layer, 0, f.n, f.wcol0, f.kvalid, f.ldw, f.src, f.kb, f.ksteps, lo, lo ? 0 : 1);
      lay.fwd3[x.s - 1].first = (uint8_t)(f.first && lo == 0);
      lay.fwd3[x.s - 1].last = (uint8_t)(f.last && lo == 1);
    }
  }
  lay.num_fwd3 = x.s;
  lay.f32_off3 = x.off;
  // bf16x3 delta chain: every transposed slab of `bwd` twice (hi: consumed with delta_hi and delta_lo; lo: with
  // delta_hi), behind the fp32 tail, so that the forward slabs and the tail keep their offsets
  LayoutBuilder y{lay.bwd3, x.off + kF32Floats * (uint32_t)sizeof(float), 0};
  for (int i = 0; i < lay.num_bwd; ++i) {
    const SlabDesc& d = lay.bwd[i];
    for (int lo = 0; lo < 2; ++lo) {
      y.add(d.ml, d.layer, 1, d.n, d.wcol0, d.kvalid, d.ldw, d.src, d.kb, d.ksteps, lo, lo ? 0 : 1);
      lay.bwd3[y.s - 1].first = (uint8_t)(d.first && lo == 0);
      lay.bwd3[y.s - 1].last = (uint8_t)(d.last && lo == 1);
    }
  }
  lay.num_bwd3 = y.s;
  lay.total_bytes3 = y.off;
  return lay;
}

// The one description of the packed image.  The weight producers and the packer walk its constant-bank copy; the MMA
// warp's compile-time schedule (mlp_chain.cuh: sched_slab) is read from it while compiling.
constexpr PackedLayout kLayout = make_layout();
__constant__ __align__(16) PackedLayout c_layout = kLayout;

// Everything CUDA caches per device (function attributes, the architecture check) is keyed by the current device, so
// one process can drive several GPUs; the caches are guarded by one mutex.
constexpr int kMaxDevices = 64;
static int g_arch[kMaxDevices];
static std::mutex g_mu;
static int current_device(int* dev) {
  NB_CUDA_CHECK(cudaGetDevice(dev));
  return (*dev >= 0 && *dev < kMaxDevices) ? NB200_OK : NB200_ERR_UNSUPPORTED;
}

struct ParamPtrs { const float* p[24]; };

// kPackSplit blocks per slab: fp32 weight -> bf16 SWIZZLE_128B operand image [n rows x 64 k-columns].
// (It runs once per optimizer step; one block per slab left half of the SMs idle: 12.5 us.)
constexpr int kPackSplit = 4;
template <bool kX3>
__global__ void __launch_bounds__(256) pack_slabs_kernel(ParamPtrs P, uint8_t* __restrict__ packed) {
  const int slab = (int)blockIdx.x / kPackSplit, part = (int)blockIdx.x % kPackSplit;
  const bool is_bwd = !kX3 && slab >= c_layout.num_fwd;
  const bool is_fold = !kX3 && slab >= c_layout.num_fwd + c_layout.num_bwd;
  const SlabDesc d = kX3 ? (slab < c_layout.num_fwd3 ? c_layout.fwd3[slab] : c_layout.bwd3[slab - c_layout.num_fwd3])
                         : (is_fold ? c_layout.fold[slab - c_layout.num_fwd - c_layout.num_bwd]
                                    : (is_bwd ? c_layout.bwd[slab - c_layout.num_fwd] : c_layout.fwd[slab]));
  // the folded weight was written to the packed buffer's fp32 tail by fold_weights_kernel (same stream, before this kernel)
  const float* W = is_fold ? reinterpret_cast<const float*>(packed + c_layout.f32_off) + kF32Wf : P.p[2 * d.layer];
  for (int item = part * blockDim.x + threadIdx.x; item < d.n * 8; item += blockDim.x * kPackSplit) {
    const int n = item >> 3, j = item & 7;
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float v[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = j * 8 + 2 * e + h;
        v[h] = 0.f;
        if (k < d.kvalid)
          v[h] = (d.flags & kSlabTransposed) ? __ldg(W + (size_t)(d.wcol0 + k) * d.ldw + n) : __ldg(W + (size_t)n * d.ldw + d.wcol0 + k);
        if (kX3 && (d.flags & kSlabLo)) v[h] -= __bfloat162float(__float2bfloat16_rn(v[h]));   // residual of the hi image
      }
      w[e] = pack_bf16x2(v[0], v[1]);
    }
    *reinterpret_cast<uint4*>(packed + d.off + sw128_off(n, j)) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__global__ void __launch_bounds__(256) pack_f32_kernel(ParamPtrs P, float* __restrict__ f) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kF32Floats) return;
  float v = 0.f;
  if (i >= kF32Bias + kFoldBiasRow * 256 && i < kF32WSig) return;   // the folded bias row belongs to fold_weights_kernel
  if (i < kF32WSig) {
    const int ml = i >> 8, j = i & 255;
    const int layer = mma_layer_of(ml);
    const int n = (ml == 9) ? 128 : 256;
    v = (j < n) ? P.p[2 * layer + 1][j] : 0.f;
  } else if (i < kF32BSig) {
    v = P.p[2 * L_SIGMA][i - kF32WSig];
  } else if (i == kF32BSig) {
    v = P.p[2 * L_SIGMA + 1][0];
  } else if (i >= kF32WC1 && i < kF32WC1 + 384) {
    v = P.p[2 * L_C1][i - kF32WC1];
  } else if (i >= kF32BC1 && i < kF32BC1 + 3) {
    v = P.p[2 * L_C1 + 1][i - kF32BC1];
  }
  f[i] = v;
}

// One 32 x 64 tile of C (+)= A B in fp32 on CUDA cores, 256 threads (thread = 2 rows x 4 columns), K in chunks of 32
// through shared memory with the next chunk's global loads in flight during the FMAs.  A(m, k) = a[m lda + k], or
// a[k lda + m] when kTransA.  The fold / un-fold GEMMs are 8-17 MFLOP: what matters is their latency inside the step
// (one thread per output with a 256-long dependent FMA chain took 35 us and 20 us; these take a few us).
template <bool kTransA, bool kAccum>
__device__ __forceinline__ void sgemm_tile_32x64(const float* __restrict__ a, int lda, const float* __restrict__ b, int ldb,
                                                 float* __restrict__ c, int ldc, int K, int m0, int n0, const float* __restrict__ r1a,
                                                 const float* __restrict__ r1b, float (*sA)[33], float (*sB)[64]) {
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  float ra[4], rb[8];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int idx = t + 256 * r;
      const int m = kTransA ? (idx & 31) : (idx >> 5), k = kTransA ? (idx >> 5) : (idx & 31);
      ra[r] = kTransA ? __ldg(a + (size_t)(k0 + k) * lda + m0 + m) : __ldg(a + (size_t)(m0 + m) * lda + k0 + k);
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int idx = t + 256 * r;
      rb[r] = __ldg(b + (size_t)(k0 + (idx >> 6)) * ldb + n0 + (idx & 63));
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < K; k0 += 32) {
    __syncthreads();   // the previous chunk has been consumed
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int idx = t + 256 * r;
      sA[kTransA ? (idx & 31) : (idx >> 5)][kTransA ? (idx >> 5) : (idx & 31)] = ra[r];
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int idx = t + 256 * r;
      sB[idx >> 6][idx & 63] = rb[r];
    }
    __syncthreads();
    if (k0 + 32 < K) fetch(k0 + 32);
#pragma unroll
    for (int kk = 0; kk < 32; ++kk) {
      const float a0 = sA[2 * ty][kk], a1 = sA[2 * ty + 1][kk];
      const float4 bv = *reinterpret_cast<const float4*>(&sB[kk][4 * tx]);
      acc[0][0] = fmaf(a0, bv.x, acc[0][0]); acc[0][1] = fmaf(a0, bv.y, acc[0][1]);
      acc[0][2] = fmaf(a0, bv.z, acc[0][2]); acc[0][3] = fmaf(a0, bv.w, acc[0][3]);
      acc[1][0] = fmaf(a1, bv.x, acc[1][0]); acc[1][1] = fmaf(a1, bv.y, acc[1][1]);
      acc[1][2] = fmaf(a1, bv.z, acc[1][2]); acc[1][3] = fmaf(a1, bv.w, acc[1][3]);
    }
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int m = m0 + 2 * ty + r;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int n = n0 + 4 * tx + q;
      float v = acc[r][q];
      if (r1a) v = fmaf(__ldg(r1a + m), __ldg(r1b + n), v);   // + rank-1 term
      float* dst = c + (size_t)m * ldc + n;
      *dst = kAccum ? *dst + v : v;
    }
  }
}

// Folded weight and bias in fp32 (see the top of the file), plus the fp32 copies the gradient un-folding reads.
// blocks 0..15: Wf = Wc0[:, :256] Wg in 32 x 64 tiles; blocks 16..31: bf (one warp per row); the rest: copies.
constexpr int kFoldWBlocks = 16 + 16 + 96;
__global__ void __launch_bounds__(256) fold_weights_kernel(ParamPtrs P, float* __restrict__ f) {
  __shared__ float sA[32][33];
  __shared__ __align__(16) float sB[32][64];
  const float* Wc0 = P.p[2 * L_C0];
  const float* Wg = P.p[2 * L_2];
  const float* bg = P.p[2 * L_2 + 1];
  constexpr int ldc = kHidden + kPosD;
  const int b = (int)blockIdx.x;
  if (b < 16) {
    sgemm_tile_32x64<false, false>(Wc0, ldc, Wg, kHidden, f + kF32Wf, kHidden, kHidden, (b >> 2) * 32, (b & 3) * 64, nullptr, nullptr, sA, sB);
  } else if (b < 32) {
    const int i = (b - 16) * 8 + ((int)threadIdx.x >> 5), lane = (int)threadIdx.x & 31;
    float acc = 0.f;
    for (int k = lane; k < kHidden; k += 32) acc = fmaf(__ldg(Wc0 + i * ldc + k), __ldg(bg + k), acc);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0) {
      f[kF32Bias + kFoldBiasRow * 256 + i] = acc + __ldg(P.p[2 * L_C0 + 1] + i);
      f[kF32Bias + kFoldBiasRow * 256 + 128 + i] = 0.f;
    }
  } else {
    for (int t = (b - 32) * 256 + (int)threadIdx.x; t < 256 * 256; t += 96 * 256) {
      f[kF32WgT + t] = __ldg(Wg + (t & 255) * kHidden + (t >> 8));   // [k][j] = Wg[j][k]
      if (t < 128 * 256) f[kF32Wc0g + t] = __ldg(Wc0 + (t >> 8) * ldc + (t & 255));
      if (t < 256) f[kF32Bg + t] = __ldg(bg + t);
    }
  }
}

// ------------------------------------------------------------------------- tile geometry
constexpr int kTileM = 128;                               // samples per tile (= TMEM lanes)
constexpr uint32_t kABytes = 65536, kEBytes = 16384;      // activation tile 128x256 bf16, encoding tile 128x64 bf16

// saved activations (training): tensors 0..7 = h0..h7, 8 = g (256 cols, 64 KB per tile; unwritten in the folded chain), 9 = c1
// (128 cols, 32 KB per tile), 10 = posx (64 cols, 16 KB), 11 = posd (32 of 64 cols, 16 KB).  Every
// tile is stored as [K-block][128 rows x 128 B SWIZZLE_128B], i.e. exactly the UMMA operand image
// the backward kernels bulk-copy back into shared memory (K-major for dgrad, MN-major for wgrad).
constexpr size_t kSavedDataTileBytes = 9 * 65536 + 32768 + 16384 + 16384;
// ReLU bit masks (training), written by the forward epilogue behind the saved tiles and read by the delta chain
// instead of the 64 KB activation tiles themselves: one bit per element, 16 B per (row, column half) for h0..h7
// (mask tensors 0..7, 4 KB per tile) and 8 B per (row, column half) for c1 (mask tensor 8, 2 KB per tile).
// Within a 16-column step the bit of column 2k is bit k and the bit of column 2k+1 is bit 8+k of a 16-bit field
// (what one HSET2 + LOP3 per bf16 pair produces and one SHIFT + PRMT per pair expands back into a word mask).
constexpr size_t kMaskTileBytes = 8 * 4096 + 2048;
constexpr size_t kSavedTileBytes = kSavedDataTileBytes + kMaskTileBytes;
__host__ __device__ __forceinline__ size_t mask_tensor_off(int t, int64_t num_tiles) {
  return (kSavedDataTileBytes + (size_t)t * 4096) * (size_t)num_tiles;
}
__host__ __device__ __forceinline__ size_t saved_tensor_off(int t, int64_t num_tiles) {
  const size_t per_tile = t < 9 ? (size_t)t * 65536 : (t == 9 ? 9 * 65536 : (t == 10 ? 9 * 65536 + 32768 : 9 * 65536 + 49152));
  return per_tile * (size_t)num_tiles;
}
__host__ __device__ __forceinline__ size_t saved_tile_bytes(int t) {
  return t < 9 ? 65536 : (t == 9 ? 32768 : 16384);
}
// bf16x3 training: the data tensors above once for the hi images bf16(x) and once for the lo images bf16(x - hi) (lo
// tensor t at kSavedDataTileBytes * T + saved_tensor_off(t, T)), then the same mask tensors, formed from the fp32 values
constexpr size_t kSavedTileBytes3 = 2 * kSavedDataTileBytes + kMaskTileBytes;
__host__ __device__ __forceinline__ size_t mask_tensor_off3(int t, int64_t num_tiles) {
  return (2 * kSavedDataTileBytes + (size_t)t * 4096) * (size_t)num_tiles;
}

// Encode 3 coordinates with L levels into the bf16 operand row `r` of a SWIZZLE_128B image:
// cols [x0,x1,x2, per coordinate: sin(2^i x), cos(2^i x) ...], zero padded to NCH*8 columns.
// Level 0 uses the accurate sincosf; higher levels the double-angle recurrence (abs. error
// <= 2^i * 1e-7, far below bf16 resolution).
template <int L, int J0, int J1>
__device__ __forceinline__ void encode_row(const float* x, uint32_t img_base, uint32_t r, uint8_t* gsave) {
  // 64 columns = 8 chunks of 16 bytes; this call stores chunks [J0, J1) (columns beyond 3+6L are zero)
  float f[64];
#pragma unroll
  for (int i = 0; i < 64; ++i) f[i] = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    f[c] = x[c];
    float s, co;
    sincosf(x[c], &s, &co);
#pragma unroll
    for (int i = 0; i < L; ++i) {
      f[3 + c * 2 * L + 2 * i] = s;
      f[3 + c * 2 * L + 2 * i + 1] = co;
      const float s2 = 2.f * s * co;
      co = fmaf(-2.f * s, s, 1.f);
      s = s2;
    }
  }
#pragma unroll
  for (int j = J0; j < J1; ++j) {
    const uint32_t w0 = pack_bf16x2(f[8 * j], f[8 * j + 1]), w1 = pack_bf16x2(f[8 * j + 2], f[8 * j + 3]),
                   w2 = pack_bf16x2(f[8 * j + 4], f[8 * j + 5]), w3 = pack_bf16x2(f[8 * j + 6], f[8 * j + 7]);
    st_shared_v4(img_base + sw128_off(r, j), w0, w1, w2, w3);
    if (gsave) *reinterpret_cast<uint4*>(gsave + sw128_off(r, j)) = make_uint4(w0, w1, w2, w3);
  }
}

#include "mlp_tc_bwd.cuh"
#include "mlp_chain.cuh"

// ------------------------------------------------------------------------------ host API
// `precision` selects the tensor-core mode: NB200_BF16 (layers_2 folded into color_fc.0), NB200_BF16_LAYERWISE or
// NB200_BF16X3.  The two bf16 modes share the packed image and the saved / scratch layouts.
size_t tc_packed_bytes(int precision) { return precision == NB200_BF16X3 ? kLayout.total_bytes3 : kLayout.total_bytes; }
// Training tensors are laid out for an EVEN number of 128-sample tiles: the chain kernels work on pair-tiles
// (one tile per CTA of a cluster), so with an odd tile count the second CTA of the last pair still writes a
// (zero-gradient) tile image, which must not alias tile 0 of the next tensor.
static int64_t train_tiles(int64_t M) { return (ceil_div64(M, kTileM) + 1) & ~(int64_t)1; }
// bf16x3: saved = hi data | lo data | masks; scratch = hi deltas | lo deltas | pad images
size_t tc_saved_bytes(int precision, int64_t M) {
  return (size_t)train_tiles(M) * (precision == NB200_BF16X3 ? kSavedTileBytes3 : kSavedTileBytes);
}
// padded staging of the three weight gradients whose rows are not 16-byte multiples (283, 319, 63
// columns): wgrad flushes into [rows x 320] / [rows x 64] images with vector reductions, and
// unpad_add_kernel folds them into the real gradients (the scalar-atomic flush of those three layers
// was 4x slower and left the CTAs holding them ~80 us behind the rest)
constexpr int kPadPitchWide = 320, kPadPitchX = 64;
constexpr size_t kPadC0 = 0, kPadSkip = kPadC0 + 128 * kPadPitchWide, kPadL00 = kPadSkip + 256 * kPadPitchWide,
                 kPadFoldS = kPadL00 + 256 * kPadPitchX,   // folded chain: column sums of delta_c1 (128 floats)
                 kPadFloats = kPadFoldS + 128;
size_t tc_scratch_bytes(int precision, int64_t M, int train) {
  const size_t delta_sets = precision == NB200_BF16X3 ? 2 : 1;
  return train ? (size_t)train_tiles(M) * delta_sets * kDeltaTileBytes + kPadFloats * sizeof(float) : 0;
}

// grad[r, c] += pad[r, c] for the three padded images (one thread per padded float4 group)
// (folded chain: columns 0..255 of the color_fc.0 image hold Gm = delta_c1^T h7, un-folded by fold_grads_kernel)
__global__ void __launch_bounds__(256) unpad_add_kernel(const float* __restrict__ pad, float* __restrict__ gC0,
                                                        float* __restrict__ gSkip, float* __restrict__ gL00, int fold) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // float index into the pad buffer
  if (i >= (int)kPadFoldS) return;
  float* g; int r, c, ncols;
  if (i < (int)kPadSkip) { r = i / kPadPitchWide; c = i - r * kPadPitchWide; g = gC0; ncols = kHidden + kPosD; if (fold && c < kHidden) return; }
  else if (i < (int)kPadL00) { const int j = i - (int)kPadSkip; r = j / kPadPitchWide; c = j - r * kPadPitchWide; g = gSkip; ncols = kHidden + kPosX; }
  else { const int j = i - (int)kPadL00; r = j / kPadPitchX; c = j - r * kPadPitchX; g = gL00; ncols = kPosX; }
  if (c < ncols) g[(size_t)r * ncols + c] += pad[i];
}

// Folded chain: gradients of color_fc.0[:, :256], layers_2 and their biases from Gm = delta_c1^T h7 (pad image of
// color_fc.0, columns 0..255) and s = column sums of delta_c1 (see the top of the file).  `f` = the packed buffer's
// fp32 tail (Wg^T, Wc0[:, :256], bg as they were at pack time).  blocks 0..15: dWc0[:, :256] += Gm Wg^T + s bg^T;
// blocks 16..47: dWg += Wc0[:, :256]^T Gm; block 48: dbg += Wc0[:, :256]^T s and dbc0 += s.
constexpr int kFoldGBlocks = 16 + 32 + 1;
__global__ void __launch_bounds__(256) fold_grads_kernel(const float* __restrict__ pad, const float* __restrict__ f,
                                                         float* __restrict__ gC0, float* __restrict__ gbC0,
                                                         float* __restrict__ gL2, float* __restrict__ gbL2) {
  __shared__ float sA[32][33];
  __shared__ __align__(16) float sB[32][64];
  const float* Gm = pad + kPadC0;
  const float* sv = pad + kPadFoldS;
  const int b = (int)blockIdx.x;
  if (b < 16) {
    sgemm_tile_32x64<false, true>(Gm, kPadPitchWide, f + kF32WgT, kHidden, gC0, kHidden + kPosD, kHidden, (b >> 2) * 32, (b & 3) * 64,
                                  sv, f + kF32Bg, sA, sB);
  } else if (b < 48) {
    const int u = b - 16;
    sgemm_tile_32x64<true, true>(f + kF32Wc0g, kHidden, Gm, kPadPitchWide, gL2, kHidden, 128, (u >> 2) * 32, (u & 3) * 64, nullptr, nullptr,
                                 sA, sB);
  } else {
    const int j = (int)threadIdx.x;
    float acc = 0.f;
#pragma unroll 8
    for (int i = 0; i < 128; ++i) acc = fmaf(__ldg(f + kF32Wc0g + i * kHidden + j), __ldg(sv + i), acc);
    gbL2[j] += acc;
    if (j < 128) gbC0[j] += __ldg(sv + j);
  }
}

int tc_pack_weights(const float* const* P, void* packed, int precision, cudaStream_t s) {
  const bool x3 = precision == NB200_BF16X3;
  ParamPtrs pp;
  for (int i = 0; i < 24; ++i) pp.p[i] = P[i];
  const int nslabs = x3 ? kLayout.num_fwd3 + kLayout.num_bwd3 : kLayout.num_fwd + kLayout.num_bwd + kLayout.num_fold;
  if (!x3) {
    fold_weights_kernel<<<kFoldWBlocks, 256, 0, s>>>(pp, reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(packed) + kLayout.f32_off));
    NB_LAUNCH_CHECK("fold_weights_kernel");
  }
  if (x3) pack_slabs_kernel<true><<<nslabs * kPackSplit, 256, 0, s>>>(pp, reinterpret_cast<uint8_t*>(packed));
  else pack_slabs_kernel<false><<<nslabs * kPackSplit, 256, 0, s>>>(pp, reinterpret_cast<uint8_t*>(packed));
  NB_LAUNCH_CHECK("pack_slabs_kernel");
  pack_f32_kernel<<<(kF32Floats + 255) / 256, 256, 0, s>>>(
      pp, reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(packed) + (x3 ? kLayout.f32_off3 : kLayout.f32_off)));
  NB_LAUNCH_CHECK("pack_f32_kernel");
  return NB200_OK;
}

static int check_arch() {
  int dev = 0;
  NB_TRY_RC(current_device(&dev));
  int arch;
  {
    std::lock_guard<std::mutex> lock(g_mu);
    if (g_arch[dev] == 0) g_arch[dev] = nb200_device_arch();
    arch = g_arch[dev];
  }
  if (arch < 0) return NB200_ERR_CUDA;
  return (arch / 10 == 10) ? NB200_OK : NB200_ERR_ARCH;
}
// cudaFuncSetAttribute is per device: `done` holds one kernel's flag per device
template <class Kernel>
static int set_smem_once(bool (&done)[kMaxDevices], Kernel* kernel, uint32_t bytes) {
  int dev = 0;
  NB_TRY_RC(current_device(&dev));
  std::lock_guard<std::mutex> lock(g_mu);
  if (done[dev]) return NB200_OK;
  NB_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  done[dev] = true;
  return NB200_OK;
}

// Biases and head weights are read from the packed buffer's fp32 tail in global memory (staged through shared memory
// by the kernels): nothing per-net lives in the constant bank, so any number of nets can run concurrently from
// different streams or threads (coarse + fine, two trainers) without sharing state, and a launch needs no copy in
// front of it.

// Tensor maps over the packed weight image (plain [rows x 64 bf16] view, no TMA swizzle: the image
// is pre-swizzled), cached per packed buffer.  cuTensorMapEncodeTiled is fetched through the runtime
// so the library does not link against libcuda.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
struct TmapPair { const void* packed; int dev; uint32_t rows; CUtensorMap m128, m64; };
static int get_tmaps(const void* packed, TmapPair* out, bool x3) {   // returns a COPY: the cache entry may be recycled by another thread
  int dev = 0;
  NB_TRY_RC(current_device(&dev));
  std::lock_guard<std::mutex> lock(g_mu);
  static TmapPair cache[8];
  static int used = 0, next = 0;
  // keyed by the image's row count too: torch's allocator hands a freed bf16 buffer's address to a bf16x3 buffer
  // (the bf16x3 map spans the whole buffer: its delta-chain slabs lie behind the fp32 tail)
  const uint32_t rows = (x3 ? kLayout.total_bytes3 : kLayout.f32_off) / 128;
  for (int i = 0; i < used; ++i)
    if (cache[i].packed == packed && cache[i].dev == dev && cache[i].rows == rows) { *out = cache[i]; return NB200_OK; }
  static EncodeTiledFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    NB_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) return NB200_ERR_CUDA;
    encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  TmapPair& t = cache[next];
  next = (next + 1) % 8;
  if (used < 8) ++used;
  t.packed = nullptr;
  const cuuint64_t gdim[2] = {64, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {128};
  const cuuint32_t estride[2] = {1, 1};
  for (int k = 0; k < 2; ++k) {
    const cuuint32_t box[2] = {64, k == 0 ? 128u : 64u};
    CUresult r = encode(k == 0 ? &t.m128 : &t.m64, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(packed), gdim, gstride,
                        box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "cuTensorMapEncodeTiled failed (%d)", (int)r);
      return NB200_ERR_CUDA;
    }
  }
  t.packed = packed;
  t.dev = dev;
  t.rows = rows;
  *out = t;
  return NB200_OK;
}

// A cluster works on `slots` pair-tiles at a time (one per in-flight tile of each CTA); with two, two pair-tiles per
// cluster keep the ping-pong busy.
static int chain_grid(int64_t T, int slots) {
  const int64_t PT = (T + 1) / 2;         // 256-row pair-tiles
  const int64_t want = (PT + slots - 1) / slots;
  const int64_t maxc = sm_count() / 2;
  const int64_t clusters = want < maxc ? (want > 0 ? want : 1) : maxc;
  return (int)(2 * clusters);
}

template <class Epi>
static int launch_chain(const typename Epi::Params& p, cudaStream_t s) {
  static bool smem_set[kMaxDevices];
  NB_TRY_RC(set_smem_once(smem_set, chain_kernel<Epi>, kCSmemLaunch));
  chain_kernel<Epi><<<chain_grid(p.num_tiles, Epi::kSlots), kCThreads, kCSmemLaunch, s>>>(p);
  NB_LAUNCH_CHECK("chain_kernel");
  return NB200_OK;
}

// What every forward chain launch shares: the weight tensor maps, the input and the tile count.
static int fwd_params(FwdEpiParams& p, int precision, int in_mode, const float* in0, const float* in1, int64_t M, int N,
                      int64_t T, const void* packed) {
  memset(&p, 0, sizeof(p));
  TmapPair tm;
  NB_TRY_RC(get_tmaps(packed, &tm, precision == NB200_BF16X3));
  p.tmap128 = tm.m128; p.tmap64 = tm.m64;
  p.in_mode = in_mode; p.in0 = in0; p.in1 = in1; p.M = M; p.N = N;
  p.nshift = (N > 0 && (N & (N - 1)) == 0) ? __builtin_ctz((unsigned)N) : -1;
  p.packed = reinterpret_cast<const uint8_t*>(packed);
  p.num_tiles = T;
  return NB200_OK;
}

// NB200_BF16X3 runs error-compensated bf16 on the same chain skeleton (one tile in flight per CTA, three MMA passes per
// K-block: A_hi W_hi + A_lo W_hi + A_hi W_lo, fp32 accumulation in TMEM): fp32-class accuracy on the tensor cores.
// With `saved` (training) its kernel also stores the hi and lo image of every layer input and the ReLU masks
// (kSavedTileBytes3 per tile of train_tiles(M)); its outputs are the inference kernel's, bit for bit.
int tc_forward(int precision, int in_mode, const float* in0, const float* in1, int64_t M, int N, const void* packed,
               float* out, void* saved, cudaStream_t s) {
  NB_TRY_RC(check_arch());
  FwdEpiParams p;
  NB_TRY_RC(fwd_params(p, precision, in_mode, in0, in1, M, N, saved ? train_tiles(M) : ceil_div64(M, kTileM), packed));
  p.out = out; p.saved = reinterpret_cast<uint8_t*>(saved);
#ifdef NB200_DEV   // developer probe of the bf16 chains (synchronises, allocates, prints): never in the shipped library
  if (precision != NB200_BF16X3) { const char* e = getenv("NB200_DBG"); p.dbg = e ? atoi(e) : 0; }
  if (p.dbg & 8) {
    static unsigned long long* ctr = nullptr;
    if (!ctr) { cudaMalloc(&ctr, 512); cudaMemset(ctr, 0, 512); }
    unsigned long long h[64];
    cudaMemcpy(h, ctr, 512, cudaMemcpyDeviceToHost);   // counters of the previous launch (debug only; syncs)
    printf("nb200 dbg: mma-warp cycles wait_act=%llu total=%llu | epilogue warp 0: layers=%llu wait_acc=%llu prologue=%llu | producer wait_empty=%llu | epilogue warp 0: reclaim (inside layers)=%llu stage_bias=%llu after_publish=%llu\n",
           h[0], h[3], h[4], h[5], h[6], h[7], h[12], h[13], h[14]);
    printf("nb200 dbg: epilogue warp 0 per layer, busy | wait_acc (share of total):");
    for (int l = 0; l < 10; ++l) printf(" L%d %.1f|%.1f", l, 100.0 * (double)h[16 + l] / (double)(h[3] ? h[3] : 1), 100.0 * (double)h[32 + l] / (double)(h[3] ? h[3] : 1));
    printf("\n");
    cudaMemset(ctr, 0, 512);
    p.dbg_counters = ctr;
  }
#endif
  if (precision == NB200_BF16_LAYERWISE) return !saved ? launch_chain<FwdEpi<false>>(p, s) : launch_chain<FwdEpi<true>>(p, s);
  if (precision == NB200_BF16) return !saved ? launch_chain<FwdEpi<false, false, true>>(p, s) : launch_chain<FwdEpi<true, false, true>>(p, s);
  return !saved ? launch_chain<FwdEpi3<false>>(p, s) : launch_chain<FwdEpi3<true>>(p, s);
}

// Fused render: sampler -> posenc + MLP -> compositing in ONE kernel; per-sample (r,g,b,sigma) and the
// sample depths never reach HBM.  rays == nullptr: rays are generated from (poses, H, W, f, ray_begin).
// ts == nullptr: Philox sample depths (same stream as nb200_stratified_ts with the same seed/offset).
int tc_render(int precision, const float* rays, const float* poses, int H, int W, float f, int64_t ray_begin, const float* ts,
              uint64_t seed, uint64_t offset, int64_t B, int N, float tn, float tf, const void* packed, float* rgb, float* disp,
              float* acc, cudaStream_t s) {
  NB_TRY_RC(check_arch());
  const int64_t M = B * N;
  FwdEpiParams p;
  NB_TRY_RC(fwd_params(p, precision, rays ? NB200_IN_RAYS : kInCamera, rays, ts, M, N, ceil_div64(M, kTileM), packed));
  p.rgb = rgb; p.disp = disp; p.acc = acc; p.B = B;
  p.sampler = ts ? 0 : 1; p.seed = seed; p.offset = offset; p.tn = tn; p.tf = tf;
  p.poses = poses; p.H = H; p.W = W; p.f = f; p.ray_begin = ray_begin;
  return precision == NB200_BF16_LAYERWISE ? launch_chain<FwdEpi<false, true>>(p, s) : launch_chain<FwdEpi<false, true, true>>(p, s);
}

// One wgrad item: dW (+)= (delta tensor dt of `ds`)^T (saved tensor st of `sv`), rows of the layer's weight from col0.
static void wgrad_item(WItem& w, const uint8_t* ds, const uint8_t* sv, int64_t T, float* pad, float* const* G, int dt, int st,
                       int layer, int ldw, int col0, int ncols, int nrows, bool bias) {
  w.a_ptr = ds + delta_tensor_off(dt, T);
  w.a_tile_bytes = dt == 0 ? 32768u : 65536u;
  w.a_chunks = dt == 0 ? 2 : 4;
  w.b_ptr = sv + saved_tensor_off(st, T);
  w.b_tile_bytes = (uint32_t)saved_tile_bytes(st);
  w.b_chunks = st >= 10 ? 1 : 4;
  w.n_mma = st >= 10 ? 64 : 256;
  w.dW = G[2 * layer]; w.db = bias ? G[2 * layer + 1] : nullptr;
  w.ldw = ldw; w.col0 = col0; w.ncols = ncols; w.nrows = nrows;
  if (ldw & 3) {  // unaligned rows: flush the whole (zero-padded) accumulator into the padded image
    w.dW = pad + (layer == L_C0 ? kPadC0 : (layer == L_SKIP ? kPadSkip : kPadL00));
    w.ldw = layer == L0_0 ? kPadPitchX : kPadPitchWide;
    w.ncols = w.n_mma;
  }
  w.cost = (w.a_chunks + w.b_chunks) * 16;
  w.head = 0; w.x_ptr = nullptr; w.x_tile_bytes = 0; w.x_chunks = 0; w.hW = nullptr; w.hb = nullptr;
}
// the sigma (1) / colour (2) head gradients ride on the item that stages their input (h7 / an extra c1 slab)
static void wgrad_head(WItem& w, const uint8_t* sv, int64_t T, float* const* G, int which) {
  const int layer = which == 1 ? L_SIGMA : L_C1;
  w.head = which; w.hW = G[2 * layer]; w.hb = G[2 * layer + 1];
  if (which == 2) {
    w.x_ptr = sv + saved_tensor_off(9, T); w.x_tile_bytes = (uint32_t)saved_tile_bytes(9); w.x_chunks = 2;
    w.cost += w.x_chunks * 16;
  }
}
// Relative time per tile of each item kind, MEASURED per CTA on B200 (global-timer trace of the mixed
// kernel; bytes alone mis-predict it because small stages are latency-bound in the ring and the head
// items add CUDA-core work before a stage is released): plain 256x256 item = 100.
static void wgrad_costs(WItem* items, int n) {
  for (int i = 0; i < n; ++i) {
    WItem& w = items[i];
    const int chunks = w.a_chunks + w.b_chunks + w.x_chunks;
    int c = chunks == 8 ? 100 : (chunks == 6 ? 85 : (w.db ? 85 : 77));
#ifndef NB_WG_HEAD6_COST
#define NB_WG_HEAD6_COST 130   // same-box A/B of the train step: 90 -> 1.085 ms, 106 -> 1.041, 124 -> 1.020, 140 -> 1.021
#endif
    if (w.head == 1) c = chunks == 8 ? 124 : NB_WG_HEAD6_COST;   // (the 6-chunk carrier of the folded chain)
    if (w.head == 2) c = 83;
    w.cost = c;
  }
}

template <bool kX3>
static int launch_wgrad(const WItem* items, int n, int64_t T, int64_t M, const float* d_out, cudaStream_t s) {
  std::conditional_t<kX3, WgradParams3, WgradParams> p;
  memset(&p, 0, sizeof(p));
  memcpy(p.items, items, (size_t)n * sizeof(WItem));
  p.num_items = n; p.T = T; p.M = M; p.d_out = d_out;
  static bool smem_set[kMaxDevices];
  NB_TRY_RC(set_smem_once(smem_set, mlp_wgrad_tc_kernel<kX3>, kWgSmemLaunch));
  mlp_wgrad_tc_kernel<kX3><<<sm_count(), kWgThreads, kWgSmemLaunch, s>>>(p);
  NB_LAUNCH_CHECK("mlp_wgrad_tc_kernel");
  return NB200_OK;
}

// The (delta tensor, input tensor) pairs of the layer-by-layer chain, in the order wgrad splits and sums them.  `head`:
// the sigma (1) / colour (2) head gradients ride on that item.
struct WPair { int dt, st, layer, ldw, col0, ncols, nrows; bool bias; int head; };
constexpr WPair kWPairs[] = {
    {0, 8, L_C0, kHidden + kPosD, 0, kHidden, kHidden / 2, true, 0},         // color_fc.0 <- g
    {0, 11, L_C0, kHidden + kPosD, kHidden, kPosD, kHidden / 2, false, 2},   // color_fc.0 <- posd; color_fc.2 <- c1
    {1, 7, L_2, kHidden, 0, kHidden, kHidden, true, 1},                      // layers_2   <- h7;   sigma_fc   <- h7
    {2, 6, L1_1, kHidden, 0, kHidden, kHidden, true, 0},                     // layers_1.2 <- h6
    {3, 5, L1_0, kHidden, 0, kHidden, kHidden, true, 0},                     // layers_1.0 <- h5
    {4, 4, L_SKIP, kHidden + kPosX, 0, kHidden, kHidden, true, 0},           // skip       <- h4
    {4, 10, L_SKIP, kHidden + kPosX, kHidden, kPosX, kHidden, false, 0},     // skip       <- posx
    {5, 3, L0_4, kHidden, 0, kHidden, kHidden, true, 0},                     // layers_0.8 <- h3
    {6, 2, L0_3, kHidden, 0, kHidden, kHidden, true, 0},
    {7, 1, L0_2, kHidden, 0, kHidden, kHidden, true, 0},
    {8, 0, L0_1, kHidden, 0, kHidden, kHidden, true, 0},
    {9, 10, L0_0, kPosX, 0, kPosX, kHidden, true, 0},                        // layers_0.0 <- posx
};
static_assert(sizeof(kWPairs) / sizeof(WPair) == kMaxWItems, "one wgrad item per pair");

// Backward: the delta chain (chain_kernel<DgradEpi> / <DgradEpi3>), then wgrad over the pairs above.
// NB200_BF16: Gm = delta_c1^T h7 (pad image of color_fc.0, with the column sums of delta_c1 as its "bias") replaces
// color_fc.0 <- g and layers_2 <- h7 and carries the sigma head; fold_grads_kernel un-folds it.
// NB200_BF16X3: hi / lo deltas, and every pair as three items, dW = d_hi^T a_hi + d_lo^T a_hi + d_hi^T a_lo.  The bias
// sums ride on the two items that stage a_hi (sum d_hi + sum d_lo); of the two carriers of each head (hi and lo) only
// the hi one adds the head-bias sums.
int tc_backward(int precision, int64_t M, const void* packed, const float* d_out, const void* saved, float* const* G,
                void* scratch, size_t scratch_bytes, cudaStream_t s) {
  NB_TRY_RC(check_arch());
  if (!scratch || scratch_bytes < tc_scratch_bytes(precision, M, 1)) return NB200_ERR_WORKSPACE;
  const bool x3 = precision == NB200_BF16X3, fold = precision == NB200_BF16;
  const int64_t T = train_tiles(M);
  const uint8_t* sv = reinterpret_cast<const uint8_t*>(saved);
  uint8_t* ds = reinterpret_cast<uint8_t*>(scratch);
  const uint8_t* sv_lo = sv + kSavedDataTileBytes * (size_t)T;   // bf16x3 only
  const uint8_t* ds_lo = ds + kDeltaTileBytes * (size_t)T;       // bf16x3 only
  float* pad = reinterpret_cast<float*>(ds + (x3 ? 2 : 1) * kDeltaTileBytes * (size_t)T);
  NB_CUDA_CHECK(cudaMemsetAsync(pad, 0, kPadFloats * sizeof(float), s));
  // 1. delta chain
  BwdParams bp;
  memset(&bp, 0, sizeof(bp));
  TmapPair tm;
  NB_TRY_RC(get_tmaps(packed, &tm, x3));
  bp.tmap128 = tm.m128; bp.tmap64 = tm.m64;
  bp.M = M; bp.num_tiles = T; bp.packed = reinterpret_cast<const uint8_t*>(packed); bp.saved = sv;
  bp.d_out = d_out; bp.dscr = ds;
  NB_TRY_RC(x3 ? launch_chain<DgradEpi3>(bp, s) : (fold ? launch_chain<DgradEpi<true>>(bp, s) : launch_chain<DgradEpi<false>>(bp, s)));
  // 2. weight gradients
  WItem items[kMaxWItems3];
  int n = 0;
  for (const WPair& q : kWPairs) {
    if (fold && q.layer == L_2) continue;
    const bool gm = fold && q.st == 8;   // color_fc.0 <- g becomes Gm = delta_c1^T h7
    const int st = gm ? 7 : q.st, head = gm ? 1 : q.head;
    for (int k = 0; k < (x3 ? 3 : 1); ++k) {   // bf16x3: d_hi^T a_hi, d_lo^T a_hi, d_hi^T a_lo
      WItem& w = items[n++];
      wgrad_item(w, k == 1 ? ds_lo : ds, k == 2 ? sv_lo : sv, T, pad, G, q.dt, st, q.layer, q.ldw, q.col0, q.ncols, q.nrows,
                 q.bias && k < 2);
      if (gm) w.db = pad + kPadFoldS;   // column sums of delta_c1 (un-folded below)
      if (head && k != 1) wgrad_head(w, k == 2 ? sv_lo : sv, T, G, head);
      if (head && k == 2) w.hb = nullptr;
    }
  }
  wgrad_costs(items, n);   // the bf16 chain's measured per-kind costs; the three items of a bf16x3 pair were not timed apart
#ifdef NB200_DEV   // developer probe: time one item alone (leaves the other gradients at zero -- never in the shipped library)
  if (!x3) { const char* e = getenv("NB200_WG_ONLY"); if (e) { const int k = atoi(e); if (k >= 0 && k < n) { items[0] = items[k]; n = 1; } } }
#endif
  NB_TRY_RC(x3 ? launch_wgrad<true>(items, n, T, M, d_out, s) : launch_wgrad<false>(items, n, T, M, d_out, s));
  unpad_add_kernel<<<((int)kPadFoldS + 255) / 256, 256, 0, s>>>(pad, G[2 * L_C0], G[2 * L_SKIP], G[2 * L0_0], fold);
  NB_LAUNCH_CHECK("unpad_add_kernel");
  if (fold) {
    fold_grads_kernel<<<kFoldGBlocks, 256, 0, s>>>(
        pad, reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(packed) + kLayout.f32_off), G[2 * L_C0], G[2 * L_C0 + 1],
        G[2 * L_2], G[2 * L_2 + 1]);
    NB_LAUNCH_CHECK("fold_grads_kernel");
  }
  return NB200_OK;
}

}  // namespace nb200
