// Backward of the fused MLP on tcgen05 (included inside namespace nb200 by mlp_tc.cu).
//
//   chain_kernel<DgradEpi> (mlp_chain.cuh): fused delta chain.  Same skeleton as the forward kernel;
//       per 128-sample tile it walks color_fc.0 -> layers_2 -> layers_1 -> skip -> layers_0 backwards,
//       delta_in = (delta_out @ W) * relu'(saved activation), each delta kept in shared memory as
//       the A operand of the next MMA and written once to HBM (bf16 tile image) for wgrad.
//       (DgradEpi<true>, the default: layers_2 is folded into color_fc.0, so delta_h7 comes from delta_c1 in ONE layer
//       and delta_g does not exist -- mlp_tc.cu, top.)
//   mlp_wgrad_tc_kernel : dW = delta^T @ activation for the 12 (delta, input) pairs (11 in the folded chain, where
//       Gm = delta_c1^T h7 replaces the pairs of color_fc.0 <- g and layers_2 <- h7).  Both operands
//       are the saved tile images read as MN-major UMMA operands (K = samples); accumulators live in
//       TMEM across the CTA's whole tile range, bias gradients are column sums taken from the staged
//       delta tiles by otherwise idle warps, one atomic flush per (CTA, layer) segment.
//       The 256->1 sigma head and the 128->3 colour head gradients ride along on those warps (CUDA
//       cores) while h7 / c1 are staged, so the heads need no pass of their own.

// ------------------------------------------------------------------ delta scratch layout
// tensor 0 = delta_c1 (128 cols, 32 KB/tile); tensors 1..9 = delta_g, delta_h7, ..., delta_h0 (64 KB/tile): tensor bl
// is the output of the delta chain's layer bl.  The folded chain keeps this layout and leaves tensor 1 unwritten.
constexpr size_t kDeltaTileBytes = 32768 + 9 * 65536;
__host__ __device__ __forceinline__ size_t delta_tensor_off(int t, int64_t num_tiles) {
  return (t == 0 ? (size_t)0 : (size_t)32768 + (size_t)(t - 1) * 65536) * (size_t)num_tiles;
}
__host__ __device__ __forceinline__ uint32_t delta_tile_bytes(int t) { return t == 0 ? 32768u : 65536u; }

struct BwdParams {
  CUtensorMap tmap128, tmap64;
  int dbg;
  int64_t M;
  int64_t num_tiles;
  const uint8_t* packed;
  const uint8_t* saved;
  const float* d_out;  // [M,4]
  uint8_t* dscr;       // delta scratch
};

// ------------------------------------------------------------------------------- wgrad
__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}

struct WItem {
  const uint8_t* a_ptr;   // delta tensor (tile images): A operand, M = output features
  const uint8_t* b_ptr;   // layer input tensor (tile images): B operand, N = input features
  float* dW;              // gradient of the weight, row pitch ldw, first column col0
  float* db;              // bias gradient or null
  uint32_t a_tile_bytes, b_tile_bytes;
  int ldw, col0, ncols, nrows;
  int a_chunks;           // 64-column chunks of delta: 2 (128 outputs) or 4 (256 outputs)
  int b_chunks;           // 64-column chunks of the input staged: 1 or 4
  int n_mma;              // UMMA N: 256 or 64
  int cost;               // relative cost per tile (KB staged), for the work split
  // head gradients ride along on the CUDA-core warps (no MMA):
  //   head 1: dW_sigma[256] += d_sigma^T . (B operand = h7), db_sigma += sum d_sigma
  //   head 2: dW_c1[3,128] += d_rgb^T . c1, db_c1 += sum d_rgb; c1 (x_chunks = 2) is staged behind
  //           the B chunks only for this purpose
  int head;
  const uint8_t* x_ptr;
  uint32_t x_tile_bytes;
  int x_chunks;
  float* hW;              // gradient of the head weight
  float* hb;              // gradient of the head bias
};
constexpr int kMaxWItems = 12;
constexpr int kMaxWItems3 = 3 * kMaxWItems;   // bf16x3: three items per (delta, input) pair
template <int kItems>
struct WgradParamsT {
  WItem items[kItems];
  int num_items;
  int64_t T;
  int64_t M;
  const float* d_out;     // [M,4] cotangent of (r,g,b,sigma): the head "deltas"
};
using WgradParams = WgradParamsT<kMaxWItems>;
using WgradParams3 = WgradParamsT<kMaxWItems3>;

// A stage holds kWgRows sample rows of up to 4 A chunks and 4 B chunks (64 features x kWgRows x 2 B each).
// (An extra L2 prefetch ahead of the ring was measured: 548 -> 742 us, so there is none.)
#ifndef NB_WG_ROWS
#define NB_WG_ROWS 64
#endif
constexpr int kWgRows = NB_WG_ROWS;                      // 32 or 64
constexpr int kWgSubs = kTileM / kWgRows;                // stages per 128-sample tile
constexpr int kWgStages = 192 / kWgRows;                 // 6 x 32 KB or 3 x 64 KB in flight
constexpr uint32_t kWgChunk = kWgRows * 128u;            // one 64-feature chunk of a stage
constexpr uint32_t kWgHalf = 4u * kWgChunk;              // A region; the B region follows
constexpr uint32_t kWgStageData = 2u * kWgHalf;
constexpr uint32_t kWgStageBytes = kWgStageData + 1024;  // + d_out rows of the stage (16 B each) for the head items
constexpr uint32_t kWgSmemBar = kWgStages * kWgStageBytes;  // 196608
constexpr uint32_t kWgSmemLaunch = kWgSmemBar + 256 + 1024;
constexpr int kWgThreads = 192;  // warp 0 producer, warp 1 MMA, warps 2-5 bias sums + flush

struct WSeg { int item; int64_t t0, t1; };

// Position x in the global cost sequence -> (item, tile).
template <class P>
__device__ __forceinline__ void wg_locate(const P& p, int64_t x, int& item, int64_t& tile) {
  int64_t cum = 0;
  for (int i = 0; i < p.num_items; ++i) {
    const int64_t span = (int64_t)p.items[i].cost * p.T;
    if (x < cum + span) { item = i; tile = (x - cum) / p.items[i].cost; return; }
    cum += span;
  }
  item = p.num_items; tile = 0;
}

// kX3 (bf16x3): the parameter block has room for three items per pair, and an item whose head-bias pointer is null adds
// the head-weight gradient only (the two carriers of h7 / c1, hi and lo, must add db_sigma / db_c1 once).
template <bool kX3>
__global__ void __launch_bounds__(kWgThreads, 1)
mlp_wgrad_tc_kernel(const __grid_constant__ std::conditional_t<kX3, WgradParams3, WgradParams> p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + kWgSmemBar;
  const uint32_t bar_full = bar_base, bar_empty = bar_base + 48, bar_accfull = bar_base + 96,
                 bar_accempty = bar_base + 104, tmem_slot = bar_base + 112;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef NB_WG_TRACE
  const uint64_t trace_t0 = global_timer_ns();
#endif
  if (threadIdx.x == 0) {
    for (int i = 0; i < kWgStages; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1 + 4);  // MMA commit + one arrive per bias warp
    }
    mbar_init(bar_accfull, 1);
    mbar_init(bar_accempty, 128);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  // this CTA's share of the (item, tile) sequence
  int64_t total = 0;
  for (int i = 0; i < p.num_items; ++i) total += (int64_t)p.items[i].cost * p.T;
  const int64_t x0 = total * blockIdx.x / gridDim.x, x1 = total * (blockIdx.x + 1) / gridDim.x;
  int i0, i1;
  int64_t t0, t1;
  wg_locate(p, x0, i0, t0);
  if (blockIdx.x + 1 == gridDim.x) { i1 = p.num_items; t1 = 0; } else wg_locate(p, x1, i1, t1);

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int it = i0; it <= i1 && it < p.num_items; ++it) {
        const WItem& w = p.items[it];
        const int64_t tb = (it == i0) ? t0 : 0, te = (it == i1) ? t1 : p.T;
        for (int64_t tile = tb; tile < te; ++tile) {
          for (int sub = 0; sub < kWgSubs; ++sub) {
            mbar_wait(bar_empty + 8 * stage, phase ^ 1, 900);
            // head items also stage the 32 d_out rows (the global-load latency under a saturated HBM is
            // several stage periods, so they have to travel with the stage)
            const int64_t m0 = tile * kTileM + sub * kWgRows;
            const uint32_t g_bytes = !w.head || m0 >= p.M ? 0u : (uint32_t)((p.M - m0 < kWgRows ? p.M - m0 : kWgRows) * 16);
            mbar_arrive_expect_tx(bar_full + 8 * stage, (uint32_t)(w.a_chunks + w.b_chunks + w.x_chunks) * kWgChunk + g_bytes);
            const uint32_t dst = smem_base + stage * kWgStageBytes;
            if (g_bytes) tma_bulk_g2s(dst + kWgStageData, p.d_out + m0 * 4, g_bytes, bar_full + 8 * stage);
            for (int c = 0; c < w.a_chunks; ++c)
              tma_bulk_g2s(dst + c * kWgChunk, w.a_ptr + (size_t)tile * w.a_tile_bytes + c * 16384 + sub * kWgChunk, kWgChunk,
                           bar_full + 8 * stage);
            for (int c = 0; c < w.b_chunks; ++c)
              tma_bulk_g2s(dst + kWgHalf + c * kWgChunk, w.b_ptr + (size_t)tile * w.b_tile_bytes + c * 16384 + sub * kWgChunk,
                           kWgChunk, bar_full + 8 * stage);
            for (int c = 0; c < w.x_chunks; ++c)
              tma_bulk_g2s(dst + kWgHalf + (w.b_chunks + c) * kWgChunk, w.x_ptr + (size_t)tile * w.x_tile_bytes + c * 16384 + sub * kWgChunk,
                           kWgChunk, bar_full + 8 * stage);
            if (++stage == kWgStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, accempty_parity = 1;  // first wait passes on a fresh barrier
      for (int it = i0; it <= i1 && it < p.num_items; ++it) {
        const WItem& w = p.items[it];
        const int64_t tb = (it == i0) ? t0 : 0, te = (it == i1) ? t1 : p.T;
        if (te <= tb) continue;
        mbar_wait(bar_accempty, accempty_parity, 1000);  // previous segment flushed out of TMEM
        accempty_parity ^= 1;
        tc_fence_after();
        const uint32_t idesc = umma_idesc_bf16(128, w.n_mma, 1, 1);  // both operands MN-major
        const int halves = w.a_chunks >> 1;
        bool first = true;
        for (int64_t tile = tb; tile < te; ++tile) {
          for (int sub = 0; sub < kWgSubs; ++sub) {
            mbar_wait(bar_full + 8 * stage, phase, 1100);
            tc_fence_after();
            const uint32_t sa = smem_base + stage * kWgStageBytes;
#pragma unroll
            for (int ks = 0; ks < kWgRows / 16; ++ks) {  // 16 sample rows per MMA
              const uint64_t bdesc = umma_smem_desc(sa + kWgHalf + ks * 2048, kWgChunk, 1024);
              for (int h = 0; h < halves; ++h)
                umma_bf16(tmem_base + h * 256, umma_smem_desc(sa + h * 2 * kWgChunk + ks * 2048, kWgChunk, 1024), bdesc, idesc,
                          (first && ks == 0) ? 0u : 1u);
            }
            first = false;
            umma_commit(bar_empty + 8 * stage);
            if (++stage == kWgStages) { stage = 0; phase ^= 1; }
          }
        }
        umma_commit(bar_accfull);
      }
    }
  } else {
    // warps 2..5: bias column sums while tiles stream, then TMEM -> atomics flush per segment
    const int q = warp & 3;          // TMEM lane group this warp may read
    const int cw = warp - 2;         // delta chunk this warp sums for the bias gradient
    uint32_t stage = 0, phase = 0, accfull_parity = 0;
    for (int it = i0; it <= i1 && it < p.num_items; ++it) {
      const WItem& w = p.items[it];
      const int64_t tb = (it == i0) ? t0 : 0, te = (it == i1) ? t1 : p.T;
      if (te <= tb) continue;
      float b0 = 0.f, b1 = 0.f;
      const bool do_bias = (w.db != nullptr) && (cw < w.a_chunks);
      float hacc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};     // head 1: [0..1]; head 2: (r,g,b) x 2 columns
      float4 hbias = make_float4(0.f, 0.f, 0.f, 0.f);
      const int head = w.head;
      for (int64_t tile = tb; tile < te; ++tile) {
        for (int sub = 0; sub < kWgSubs; ++sub) {
          mbar_wait(bar_full + 8 * stage, phase, 1200);
#pragma unroll 1
          for (int r32 = 0; r32 < kWgRows; r32 += 32) {     // 32 sample rows at a time (lane <-> row for d_out)
          float4 g = make_float4(0.f, 0.f, 0.f, 0.f);      // d_out row `lane` of these 32 rows
          const uint32_t g_smem = smem_base + stage * kWgStageBytes + kWgStageData + r32 * 16;
          const uint32_t rows_smem = smem_base + stage * kWgStageBytes + r32 * 128;
          if (head) {
            if (tile * kTileM + sub * kWgRows + r32 + lane < p.M)
              asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(g.x), "=f"(g.y), "=f"(g.z), "=f"(g.w)
                           : "r"(g_smem + lane * 16));
            else  // tail of the last tile: rows >= M were not copied; every warp zeroes them for its own reads
              asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};" ::"r"(g_smem + lane * 16), "f"(0.f));
            __syncwarp();
            hbias.x += g.x; hbias.y += g.y; hbias.z += g.z; hbias.w += g.w;
          }
          if (do_bias) {
            const uint32_t base = rows_smem + cw * kWgChunk + (lane & 3) * 4;
#pragma unroll 8
            for (int row = 0; row < 32; ++row) {
              uint32_t v;
              asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(base + row * 128 + ((((uint32_t)lane >> 2) ^ (row & 7)) << 4)));
              b0 += __uint_as_float(v << 16);
              b1 += __uint_as_float(v & 0xFFFF0000u);
            }
          }
          if (head == 1) {
            // warp cw: columns [64 cw, 64 cw + 64) of h7; the d_sigma of a row is a broadcast shared load
            const uint32_t base = rows_smem + kWgHalf + cw * kWgChunk + (lane & 3) * 4;
#pragma unroll
            for (int rb = 0; rb < 32; rb += 8) {   // 8 rows per batch: all loads first, then the FMAs
              uint32_t v[8];
              float gs[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v[i]) : "r"(base + (rb + i) * 128 + ((((uint32_t)lane >> 2) ^ (uint32_t)i) << 4)));
                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(gs[i]) : "r"(g_smem + (rb + i) * 16 + 12));
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                hacc[2 * (i & 1)] = fmaf(gs[i], __uint_as_float(v[i] << 16), hacc[2 * (i & 1)]);
                hacc[2 * (i & 1) + 1] = fmaf(gs[i], __uint_as_float(v[i] & 0xFFFF0000u), hacc[2 * (i & 1) + 1]);
              }
            }
          } else if (head == 2) {
            // warp cw: columns [64 (cw&1), +64) of c1, rows [16 (cw>>1), +16) of the stage
            const uint32_t base = rows_smem + kWgHalf + (w.b_chunks + (cw & 1)) * kWgChunk + (lane & 3) * 4;
#pragma unroll
            for (int rb = 0; rb < 16; rb += 8) {
              const int r0 = (cw >> 1) * 16 + rb;
              uint32_t v[8];
              float4 gq[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v[i]) : "r"(base + (r0 + i) * 128 + ((((uint32_t)lane >> 2) ^ (uint32_t)i) << 4)));
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(gq[i].x), "=f"(gq[i].y), "=f"(gq[i].z), "=f"(gq[i].w)
                             : "r"(g_smem + (r0 + i) * 16));
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float c0 = __uint_as_float(v[i] << 16), c1 = __uint_as_float(v[i] & 0xFFFF0000u);
                hacc[0] = fmaf(gq[i].x, c0, hacc[0]); hacc[1] = fmaf(gq[i].x, c1, hacc[1]);
                hacc[2] = fmaf(gq[i].y, c0, hacc[2]); hacc[3] = fmaf(gq[i].y, c1, hacc[3]);
                hacc[4] = fmaf(gq[i].z, c0, hacc[4]); hacc[5] = fmaf(gq[i].z, c1, hacc[5]);
              }
            }
          }
          }  // r32
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_empty + 8 * stage);
          if (++stage == kWgStages) { stage = 0; phase ^= 1; }
        }
      }
      if (head == 1) {
        const int n = cw * 64 + 2 * lane;
        atomicAdd(w.hW + n, hacc[0] + hacc[2]);          // even + odd row partial sums
        atomicAdd(w.hW + n + 1, hacc[1] + hacc[3]);
        if (cw == 0 && (!kX3 || w.hb)) {
          const float tot = warp_sum_f(hbias.w);
          if (lane == 0) atomicAdd(w.hb, tot);
        }
      } else if (head == 2) {
        const int n = (cw & 1) * 64 + 2 * lane;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          atomicAdd(w.hW + k * 128 + n, hacc[2 * k]);
          atomicAdd(w.hW + k * 128 + n + 1, hacc[2 * k + 1]);
        }
        if (cw == 2 && (!kX3 || w.hb)) {
          const float tr = warp_sum_f(hbias.x), tg = warp_sum_f(hbias.y), tbl = warp_sum_f(hbias.z);
          if (lane == 0) { atomicAdd(w.hb, tr); atomicAdd(w.hb + 1, tg); atomicAdd(w.hb + 2, tbl); }
        }
      }
      if (do_bias) {
        const int n = cw * 64 + 2 * lane;
        if (n < w.nrows) atomicAdd(w.db + n, b0);
        if (n + 1 < w.nrows) atomicAdd(w.db + n + 1, b1);
      }
      mbar_wait(bar_accfull, accfull_parity, 1300);
      accfull_parity ^= 1;
      tc_fence_after();
      const int halves = w.a_chunks >> 1;
      for (int h = 0; h < halves; ++h) {
        const int n = h * 128 + q * 32 + lane;  // output feature (row of dW)
        for (int c = 0; c * 32 < w.n_mma; ++c) {
          uint32_t acc[32];
          tmem_ld32(tmem_base + (((uint32_t)q * 32u) << 16) + h * 256 + c * 32, acc);
          tmem_ld_wait();
          if (n < w.nrows) {
            float* dst = w.dW + (size_t)n * w.ldw + w.col0 + c * 32;
            if (((w.ldw | w.col0) & 3) == 0 && (reinterpret_cast<uintptr_t>(w.dW) & 15) == 0 && c * 32 + 32 <= w.ncols) {
              // 16-byte aligned rows: vector reductions, 4x fewer L2 atomic transactions
#pragma unroll
              for (int i = 0; i < 32; i += 4)
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + i), "f"(__uint_as_float(acc[i])),
                             "f"(__uint_as_float(acc[i + 1])), "f"(__uint_as_float(acc[i + 2])),
                             "f"(__uint_as_float(acc[i + 3]))
                             : "memory");
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (c * 32 + i < w.ncols) atomicAdd(dst + i, __uint_as_float(acc[i]));
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar_accempty);
    }
  }
  tc_fence_before();
  __syncthreads();
#ifdef NB_WG_TRACE
  if (threadIdx.x == 0) printf("WGTRACE %d %d %lld %d %lld %llu %llu\n", (int)blockIdx.x, i0, (long long)t0, i1, (long long)t1, (unsigned long long)global_timer_ns(), (unsigned long long)trace_t0);
#endif
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

