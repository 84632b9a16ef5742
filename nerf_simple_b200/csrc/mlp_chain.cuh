// Fused layer-chain kernel, generation 2 (included inside namespace nb200 by mlp_tc.cu).
//
// Two CTAs of a cluster (one SM pair) run every MMA together: tcgen05.mma.cta_group::2 with
// M = 256 (each CTA owns 128 sample rows and their accumulators in its own TMEM) and the N rows
// of each weight slab split across the pair, so a CTA streams only HALF of every weight slab from
// L2.  The slabs of a layer (<= 4 x 16 KB per CTA) stay resident in a 4-stage ring while BOTH
// in-flight tiles (slots) of the CTA consume them, which cuts the L2->SM weight traffic of the
// first-generation kernel (9.3 KB/sample, L2-bandwidth bound) by ~3.4x.
//
//   warps 0-7 / 8-15 : prologue + epilogue of slot 0 / 1.  Two warps share each TMEM lane group:
//                      thread (warp%4)*32+lane <-> sample row <-> TMEM lane, warps 4-7 of a slot take
//                      the upper half of the accumulator columns (the epilogue is the critical path:
//                      it must finish inside the 2048 cycles the other slot's MMAs take).  Serving ONE slot at a
//                      time with all 16 warps (64 columns per thread) was measured and is slower (DESIGN 4.5).
//   warp  16         : weight producer (TMA tensor-map copy of this CTA's half slab); walks the slab table in the
//                      constant bank.  It is never late: the MMA warp's weight waits do not block.
//   warp  17         : leader CTA: MMA issuer, walking a COMPILE-TIME schedule (one unrolled copy of the issue code
//                      per layer class, runtime slot and ring position).  peer CTA: idle.
//   warps 18, 19     : training kernels only: bulk-store issuer of slot 0 / 1.  The epilogue warps hand a finished
//                      tile image over through an mbarrier (one arrive per warp) and get the buffer back through
//                      another one, instead of two 256-thread bar.syncs and a serial leader thread per layer.
//
// The same skeleton runs the forward chain (FwdEpi) and the backward delta chain (DgradEpi); they
// differ only in the slab schedule and in what the epilogue warps do with each accumulator.
//
// Shared memory (231,680 B, 1 KB aligned): A[2] 2 x 64 KB activation tiles | E[2] 2 x 16 KB encodings (posx, later
// posd + the head-weight table in the free half of its rows) | 4 x 16 KB weight ring | 256 B barriers | 2 x 1 KB
// staged bias rows.  The epilogue issues no constant-bank loads: they were its bottleneck (ADU / MIO path).
constexpr uint32_t kC_A = 0, kC_E = 2 * kABytes, kC_W = kC_E + 2 * kEBytes;
constexpr int kCStages = 4;
constexpr uint32_t kCStageBytes = 16384;
constexpr uint32_t kC_Bar = kC_W + kCStages * kCStageBytes;  // 229376
// behind the barrier block: the biases of the layer whose epilogue comes next, one 1 KB fp32 row per slot (staged by the
// slot's own 256 threads while they wait for the accumulator).  The epilogue reads them with warp-uniform LDS.128;
// constant-bank loads in ANY form (indexed LDC.64, or LDCU.128 into uniform registers when the address is an
// immediate) cost ~1,350 of the ~2,400 cycles a hidden-layer epilogue took.
constexpr uint32_t kC_Bias = kC_Bar + 256;
constexpr uint32_t kCSmemLaunch = kC_Bias + 2 * 1024;   // 231,680 of the 232,448 B a CTA can have: the base must be 1 KB aligned
constexpr int kCThreads = 640;
constexpr int kCProducerWarp = 16, kCMmaWarp = 17, kCStoreWarp0 = 18;
// barrier offsets inside the barrier block
constexpr uint32_t kB_WFull = 0, kB_WPeer = 32, kB_WEmpty = 64, kB_Act = 96, kB_Acc = 112, kB_Tmem = 128, kB_Written = 136,
                   kB_StoreFree = 152;

struct TileCtx {
  int64_t tile;      // 128-row tile index
  int slot;          // which in-flight tile of the CTA
  int half;          // 0: accumulator columns [0,128), 1: [128,256)
  int part;          // single-slot kernels (16 warps on one tile): accumulator columns [64 part, 64 part + 64)
  uint32_t r;        // row in tile == TMEM lane
  uint32_t rowoff;   // r * 128
  uint32_t r7s;      // (r & 7) << 4
  uint32_t a_img, e_img, t_lane;
  uint32_t b_img;    // the slot's staged bias row (shared memory)
  const float* gf;   // the net's fp32 tail (biases, head weights) in global memory: part of the packed buffer
};
__device__ __forceinline__ uint32_t sw_off(const TileCtx& c, uint32_t kb, uint32_t j) {
  return kb * 16384u + c.rowoff + ((j << 4) ^ c.r7s);
}

__device__ __forceinline__ void slot_barrier(int slot) {  // the 256 epilogue threads of one slot
  asm volatile("bar.sync %0, 256;" ::"r"(slot + 1) : "memory");
}

// ---------------------------------------------------------------- compile-time slab schedule
// The MMA warp's issue loop is fully unrolled over (layer, slot, slab): A-operand offsets, instruction descriptors
// and the accumulate flags are immediates, and the only runtime state is the ring position.  (Walking the
// constant-bank SlabDesc table instead cost a chain of dependent indexed LDC + R2UR + LDCU per slab, ~700 cycles of
// MMA-warp time for the 512 cycles of tensor work it issued: the issue warp, not the weights or the epilogue, was
// the bottleneck of every chain kernel.)  The schedule is read from kLayout at compile time, the table whose
// constant-bank copy the producer walks (it is never late), so both see the same slabs in the same order.
#ifdef NB200_DEV
constexpr bool kDevBuild = true;    // cycle counters of the MMA / epilogue / producer warps (NB200_DBG=8), never in the shipped library
#else
constexpr bool kDevBuild = false;
#endif
// The slab tables of PackedLayout; each epilogue names the one it walks (Epi::kTab).
enum SlabTab { kTabFwd, kTabFwdFold, kTabBwd, kTabBwdFold, kTabFwd3, kTabBwd3 };
template <int kTab, class Layout> __host__ __device__ constexpr auto& slab_table(Layout& lay) {
  if constexpr (kTab == kTabFwd) return lay.fwd;
  else if constexpr (kTab == kTabFwdFold) return lay.fwdf;
  else if constexpr (kTab == kTabBwd) return lay.bwd;
  else if constexpr (kTab == kTabBwdFold) return lay.bwdf;
  else if constexpr (kTab == kTabFwd3) return lay.fwd3;
  else return lay.bwd3;
}
template <int kTab> __host__ __device__ constexpr bool sched_is_bwd() { return kTab == kTabBwd || kTab == kTabBwdFold || kTab == kTabBwd3; }
// loop layer l = the l-th run of slabs closed by a `last` flag (the producer walks the table the same way)
template <int kTab> __host__ __device__ constexpr int sched_first(int l) {
  int i = 0;
  for (int k = 0; k < l; ++k, ++i)
    while (!slab_table<kTab>(kLayout)[i].last) ++i;
  return i;
}
template <int kTab> __host__ __device__ constexpr int sched_slabs(int l) {
  int i = sched_first<kTab>(l);
  while (!slab_table<kTab>(kLayout)[i].last) ++i;
  return i - sched_first<kTab>(l) + 1;
}
template <int kTab> __host__ __device__ constexpr SlabDesc sched_slab(int l, int s) {
  return slab_table<kTab>(kLayout)[sched_first<kTab>(l) + s];
}

struct MmaRing { uint32_t stage, phase; };

// Layers with the same slab list share one unrolled copy of the issue code (kept small: the fully unrolled version,
// one copy per layer and slot, was 100 KB of instructions and thrashed the instruction cache of the training kernels).
// Class representatives (loop indices): forward 0 | 1 (all plain 256x256 layers) | 5 (skip) | the last (color_fc.0);
// delta chain 0 | 1.
template <class Epi> __host__ __device__ constexpr int sched_class_rep(int l) {
  return sched_is_bwd<Epi::kTab>() ? (l == 0 ? 0 : 1) : ((l == 0 || l == 5 || l == Epi::kNumLayers - 1) ? l : 1);
}
// The table holds Epi::kNumLayers layers, and each has the slab list (as far as the issue code reads it) of its class
// representative.
template <class Epi> constexpr bool sched_classes_hold() {
  int layers = 0;
  for (const SlabDesc& d : slab_table<Epi::kTab>(kLayout)) layers += d.last;
  if (layers != Epi::kNumLayers) return false;
  for (int l = 0; l < Epi::kNumLayers; ++l) {
    const int rep = sched_class_rep<Epi>(l);
    if (sched_slabs<Epi::kTab>(l) != sched_slabs<Epi::kTab>(rep)) return false;
    for (int s = 0; s < sched_slabs<Epi::kTab>(l); ++s) {
      const SlabDesc a = sched_slab<Epi::kTab>(l, s), b = sched_slab<Epi::kTab>(rep, s);
      if (a.src != b.src || a.kb != b.kb || a.n != b.n || a.ksteps != b.ksteps || (a.flags & kSlabBothA) != (b.flags & kSlabBothA))
        return false;
    }
  }
  return true;
}

template <class Epi, int L, int S>
__device__ __forceinline__ void issue_slab(uint32_t smem_base, uint32_t bar, uint32_t tmem_base, uint64_t desc_hi, uint32_t slot,
                                           bool replay, bool release, MmaRing& r) {
  constexpr SlabDesc sc = sched_slab<Epi::kTab>(L, S);
  constexpr int NS = sched_slabs<Epi::kTab>(L);
  if (!replay) {
    mbar_wait(bar + kB_WFull + 8 * r.stage, r.phase, 400);
    tc_fence_after();
  }
  const uint32_t a_addr = smem_base + (sc.src ? kC_E + slot * kEBytes : kC_A + slot * kABytes + (uint32_t)sc.kb * 16384u);
  const uint64_t adesc = desc_hi | (uint64_t)((a_addr >> 4) & 0x3FFFu);
  const uint64_t bdesc = desc_hi | (uint64_t)(((smem_base + kC_W + r.stage * kCStageBytes) >> 4) & 0x3FFFu);
  constexpr uint32_t idesc = umma_idesc_bf16(256, sc.n, 0, 0);
  const uint32_t d_tmem = tmem_base + slot * 256u;
  if (elect_one()) {
    umma_bf16_2cta(d_tmem, adesc, bdesc, idesc, S == 0 ? 0u : 1u);   // +2 in the address field = +32 bytes
    umma_bf16_2cta(d_tmem, adesc + 2, bdesc + 2, idesc, 1u);
    if (sc.ksteps > 2) {
      umma_bf16_2cta(d_tmem, adesc + 4, bdesc + 4, idesc, 1u);
      umma_bf16_2cta(d_tmem, adesc + 6, bdesc + 6, idesc, 1u);
    }
    if (sc.flags & kSlabBothA) {   // bf16x3: the same B slab against the residual image A_lo (the other slot's buffer)
      const uint64_t alo = adesc + ((sc.src ? kEBytes : kABytes) >> 4);
      umma_bf16_2cta(d_tmem, alo, bdesc, idesc, 1u);
      umma_bf16_2cta(d_tmem, alo + 2, bdesc + 2, idesc, 1u);
      if (sc.ksteps > 2) {
        umma_bf16_2cta(d_tmem, alo + 4, bdesc + 4, idesc, 1u);
        umma_bf16_2cta(d_tmem, alo + 6, bdesc + 6, idesc, 1u);
      }
    }
    if (release) umma_commit_2cta(bar + kB_WEmpty + 8 * r.stage);   // the last user frees the stage
    if (S == NS - 1) umma_commit_2cta(bar + kB_Acc + 8 * slot);
  }
  __syncwarp();
  if (++r.stage == kCStages) { r.stage = 0; r.phase ^= 1; }
}
template <class Epi, int L, int... S>
__device__ __forceinline__ void issue_slabs(std::integer_sequence<int, S...>, uint32_t smem_base, uint32_t bar, uint32_t tmem_base,
                                            uint64_t desc_hi, uint32_t slot, bool replay, bool release, MmaRing& r) {
  (issue_slab<Epi, L, S>(smem_base, bar, tmem_base, desc_hi, slot, replay, release, r), ...);
}
// one layer (of class representative L) for the in-flight tiles: slot 0, then slot 1 against the slabs that are still resident
template <class Epi, int L>
__device__ __forceinline__ void issue_layer(uint32_t smem_base, uint32_t bar, uint32_t tmem_base, uint64_t desc_hi, int nslots, int l,
                                            MmaRing& r, uint32_t (&act_parity)[2], long long& t_act) {
  constexpr int NS = sched_slabs<Epi::kTab>(L);
  using Seq = std::make_integer_sequence<int, NS>;
  const bool shared = (nslots == 2 && NS <= kCStages);   // do both slots consume one copy of the layer's slabs?
  const MmaRing r0 = r;
#pragma unroll 1
  for (int slot = 0; slot < nslots; ++slot) {
#ifdef NB200_DEV
    const long long tw0 = clock64();
#endif
    if (slot == 0) { mbar_wait(bar + kB_Act, act_parity[0], 300 + l); act_parity[0] ^= 1; }
    else { mbar_wait(bar + kB_Act + 8, act_parity[1], 350 + l); act_parity[1] ^= 1; }
#ifdef NB200_DEV
    t_act += clock64() - tw0;
#endif
    tc_fence_after();
    const bool replay = shared && slot == 1;   // the slabs are already resident from slot 0's pass
    if (replay) r = r0;
    issue_slabs<Epi, L>(Seq{}, smem_base, bar, tmem_base, desc_hi, (uint32_t)slot, replay, !(shared && slot == 0), r);
  }
}

template <class Epi>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kCThreads, 1)
chain_kernel(const __grid_constant__ typename Epi::Params p) {
  static_assert(sched_classes_hold<Epi>(), "a layer's slab list differs from its class representative's, or the table's layer count from the epilogue's");
  extern __shared__ __align__(1024) uint8_t chain_smem[];
  const uint32_t smem_base = smem_u32(chain_smem);
  if (smem_base & 1023u) {   // the SWIZZLE_128B images need it, and there is no slack left to round up
    if (threadIdx.x == 0) printf("nb200: dynamic shared memory base 0x%x is not 1 KB aligned\n", smem_base);
    __trap();
  }
  const uint32_t bar = smem_base + kC_Bar;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();

  if (threadIdx.x == 0) {
    for (int i = 0; i < kCStages; ++i) {
      mbar_init(bar + kB_WFull + 8 * i, 1);
      mbar_init(bar + kB_WPeer + 8 * i, 1);
      mbar_init(bar + kB_WEmpty + 8 * i, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar + kB_Act + 8 * s, 16 * (3 - Epi::kSlots));   // one elected arrive per epilogue warp (8 or 16 warps x 2 CTAs)
      mbar_init(bar + kB_Acc + 8 * s, 1);
      mbar_init(bar + kB_Written + 8 * s, 8 * (3 - Epi::kSlots));   // this CTA's 8 (16) epilogue warps of the slot: "tile image complete"
      mbar_init(bar + kB_StoreFree + 8 * s, 1);  // the slot's store warp: "the bulk store has read the image"
    }
    fence_mbar_init();
  }
  if (warp == kCMmaWarp) tmem_alloc_2cta(bar + kB_Tmem, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(bar + kB_Tmem));

  // pair-tiles (256 rows) of this cluster: pt = cluster + k * num_clusters; slot = k & 1
  const int64_t PT = (p.num_tiles + 1) / 2;
  const int64_t C = num_clusters_x(), cid = cluster_id_x();
  const int64_t my_pt = (cid < PT) ? (PT - cid + C - 1) / C : 0;
  const SlabDesc* slabs = slab_table<Epi::kTab>(c_layout);

  if (warp < 16) {
    // ============================ prologue + epilogue of one slot ============================
    const int slot = Epi::kSlots == 2 ? warp >> 3 : 0;
    TileCtx c;
    c.slot = slot;
    c.half = (warp >> 2) & 1;
    c.part = warp >> 2;
    c.r = (uint32_t)(warp & 3) * 32u + (uint32_t)lane;
    c.rowoff = c.r * 128u;
    c.r7s = (c.r & 7u) << 4;
    c.a_img = smem_base + kC_A + slot * kABytes;
    c.e_img = smem_base + kC_E + slot * kEBytes;
    c.t_lane = tmem_base + (((uint32_t)(warp & 3) * 32u) << 16) + (uint32_t)slot * 256u;
    c.b_img = smem_base + kC_Bias + (uint32_t)slot * 1024u;
    c.gf = reinterpret_cast<const float*>(p.packed + (Epi::kTab == kTabFwd3 || Epi::kTab == kTabBwd3 ? c_layout.f32_off3 : c_layout.f32_off));
    const uint32_t act_remote = mapa_shared(bar + kB_Act + 8 * slot, 0);  // leader's act_ready[slot]
    uint32_t acc_parity = 0, free_parity = 0;
    typename Epi::State st;
    bool first_step = true;
    long long t_epi = 0, t_accw = 0, t_pro = 0, t_reclaim = 0, t_after = 0, t_stage = 0;
    // hand a finished tile image to the MMA warp (leader's act barrier) and, in the training kernels, to this slot's
    // store warp; `to_mma` is false after the last layer of a tile
    auto publish = [&](bool to_mma) {
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (Epi::kBulkStore) mbar_arrive(bar + kB_Written + 8 * slot);
        if (to_mma) mbar_arrive_cluster(act_remote);
      }
    };
    // the biases of layer l -> the slot's staging row: one constant load + store per thread, between two barriers of
    // the slot's 256 threads (everybody has finished with the previous row / the new row is visible).  Called right
    // after a publish, i.e. while the slot would wait for its next accumulator anyway.
    // `v` is this thread's element of the row, fetched EARLY (before the epilogue that precedes the staging) from the
    // packed buffer's fp32 tail in global memory: coalesced and L2-resident, where 256 DIFFERENT constant-bank
    // addresses per slot serialise in the constant cache (~1,000 cycles per staged row).
    const uint32_t bias_t = threadIdx.x & 255u;
    auto fetch_bias = [&](int l) -> float { return Epi::kStageBias ? __ldg(c.gf + kF32Bias + Epi::bias_row(l) * 256 + (int)bias_t) : 0.f; };
    auto stage_bias = [&](float v) {
      if (!Epi::kStageBias) return;
      if (Epi::kSlots == 2) slot_barrier(slot); else asm volatile("bar.sync 1, 512;" ::: "memory");
      if (Epi::kSlots == 2 || threadIdx.x < 256u) asm volatile("st.shared.f32 [%0], %1;" ::"r"(c.b_img + bias_t * 4u), "f"(v) : "memory");
      if (Epi::kSlots == 2) slot_barrier(slot); else asm volatile("bar.sync 1, 512;" ::: "memory");
    };
    // before overwriting A[slot] / E[slot]: the bulk store of the previous image must have read it
    auto reclaim = [&]() {
      if (Epi::kBulkStore && !first_step) {
        mbar_wait(bar + kB_StoreFree + 8 * slot, free_parity, 500);
        free_parity ^= 1;
      }
      first_step = false;
    };
    Epi::init_slot(c);   // once per kernel, by the slot's 256 threads
    for (int64_t k = slot; k < my_pt; k += Epi::kSlots) {
      c.tile = 2 * (cid + k * C) + rank;
      // the delta chain walks the tiles in REVERSE: the forward pass wrote the saved activations of the last
      // tiles last, so they are the ones still in L2 when the backward starts
      if (Epi::kReverseTiles) c.tile = 2 * (PT - 1 - (cid + k * C)) + rank;
      reclaim();
      long long tq0 = 0;
      if constexpr (Epi::kHasDbg && kDevBuild) tq0 = clock64();
      const float bias0 = fetch_bias(0);
      Epi::begin_tile(p, st, c);
      publish(true);
      stage_bias(bias0);
      if constexpr (Epi::kHasDbg && kDevBuild) t_pro += clock64() - tq0;
      for (int l = 0; l < Epi::kNumLayers; ++l) {
        Epi::prefetch(p, st, c, l);  // global loads that do not depend on the accumulator
        if constexpr (Epi::kHasDbg && kDevBuild) tq0 = clock64();
        mbar_wait(bar + kB_Acc + 8 * slot, acc_parity, 100 + l);
        acc_parity ^= 1;
        tc_fence_after();
        long long tq1 = 0;
        if constexpr (Epi::kHasDbg && kDevBuild) { tq1 = clock64(); t_accw += tq1 - tq0; }
        reclaim();
        if constexpr (Epi::kHasDbg && kDevBuild) t_reclaim += clock64() - tq1;
        const float bias_next = fetch_bias(l + 1 < Epi::kNumLayers ? l + 1 : l);
        Epi::layer(p, st, c, l);
        if (Epi::kBulkStore || l + 1 < Epi::kNumLayers) publish(l + 1 < Epi::kNumLayers);
        if constexpr (Epi::kHasDbg && kDevBuild) {
          const long long tq2 = clock64();
          t_epi += tq2 - tq1;
          if ((p.dbg & 8) && threadIdx.x == 0 && rank == 0 && p.dbg_counters) {   // per-layer split (fire-and-forget reds)
            atomicAdd(p.dbg_counters + 16 + l, (unsigned long long)(tq2 - tq1));
            atomicAdd(p.dbg_counters + 32 + l, (unsigned long long)(tq1 - tq0));
          }
        }
        long long tq3 = 0;
        if constexpr (Epi::kHasDbg && kDevBuild) tq3 = clock64();
        if (l + 1 < Epi::kNumLayers) stage_bias(bias_next);
        long long tq4 = 0;
        if constexpr (Epi::kHasDbg && kDevBuild) { tq4 = clock64(); t_stage += tq4 - tq3; }
        Epi::after_publish(p, st, c, l);
        if constexpr (Epi::kHasDbg && kDevBuild) t_after += clock64() - tq4;
      }
    }
    if constexpr (Epi::kHasDbg && kDevBuild) {
      if ((p.dbg & 8) && threadIdx.x == 0 && rank == 0 && p.dbg_counters) {   // warp 0 of the leader CTA
        atomicAdd(p.dbg_counters + 4, (unsigned long long)t_epi);
        atomicAdd(p.dbg_counters + 5, (unsigned long long)t_accw);
        atomicAdd(p.dbg_counters + 6, (unsigned long long)t_pro);
        atomicAdd(p.dbg_counters + 12, (unsigned long long)t_reclaim);
        atomicAdd(p.dbg_counters + 13, (unsigned long long)t_stage);
        atomicAdd(p.dbg_counters + 14, (unsigned long long)t_after);
      }
    }
    if (Epi::kBulkStore && !first_step) mbar_wait(bar + kB_StoreFree + 8 * slot, free_parity, 501);   // last store read its image
  } else if (warp == kCProducerWarp) {
    // ==================================== weight producer ====================================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      long long t_pempty = 0;
      for (int64_t pr = 0; pr * Epi::kSlots < my_pt; ++pr) {
        const int nslots = (Epi::kSlots == 2 && my_pt - 2 * pr >= 2) ? 2 : 1;
        int s0 = 0;
        for (int l = 0; l < Epi::kNumLayers; ++l) {
          int s1 = s0;
          while (!slabs[s1].last) ++s1;
          const int reps = (nslots == 2 && s1 - s0 + 1 <= kCStages) ? 1 : nslots;  // shared by both slots?
          for (int rep = 0; rep < reps; ++rep) {
            for (int s = s0; s <= s1; ++s) {
              const uint32_t half = slabs[s].bytes >> 1;
              if constexpr (Epi::kHasDbg && kDevBuild) {
                const long long tp0 = clock64();
                mbar_wait(bar + kB_WEmpty + 8 * stage, phase ^ 1, 200);
                const long long tp1 = clock64();
                t_pempty += tp1 - tp0;
              } else
              mbar_wait(bar + kB_WEmpty + 8 * stage, phase ^ 1, 200);
              // both CTAs signal the LEADER's barrier: it expects the whole slab (two halves)
              if (rank == 0) mbar_arrive_expect_tx(bar + kB_WFull + 8 * stage, slabs[s].bytes);
              const int32_t row0 = (int32_t)(slabs[s].off >> 7) + (int32_t)(rank * (half >> 7));
              tma_tensor2d_g2s_2cta(smem_base + kC_W + stage * kCStageBytes, half == 16384u ? &p.tmap128 : &p.tmap64, 0, row0,
                                    mapa_shared(bar + kB_WFull + 8 * stage, 0));
              if (++stage == kCStages) { stage = 0; phase ^= 1; }
            }
          }
          s0 = s1 + 1;
        }
      }
      if constexpr (Epi::kHasDbg && kDevBuild) {
        if ((p.dbg & 8) && rank == 0 && p.dbg_counters) atomicAdd(p.dbg_counters + 7, (unsigned long long)t_pempty);
      }
    }
  } else if (warp >= kCStoreWarp0) {
    // ============================ bulk-store issuer of one slot (training) ============================
    // (single-slot kernels: warp 18 stores, warp 19 idles; store_tile issues every image of the hand-off, e.g. hi and lo)
    if (Epi::kBulkStore && lane == 0 && (Epi::kSlots == 2 || warp == kCStoreWarp0)) {
      const int slot = warp - kCStoreWarp0;
      TileCtx c;
      c.slot = slot;
      c.a_img = smem_base + kC_A + slot * kABytes;
      c.e_img = smem_base + kC_E + slot * kEBytes;
      uint32_t parity = 0;
      for (int64_t k = slot; k < my_pt; k += Epi::kSlots) {
        c.tile = 2 * (cid + k * C) + rank;
        if (Epi::kReverseTiles) c.tile = 2 * (PT - 1 - (cid + k * C)) + rank;
        for (int l = -1; l < Epi::kNumLayers; ++l) {
          mbar_wait(bar + kB_Written + 8 * slot, parity, 600 + l);
          parity ^= 1;
          Epi::store_tile(p, c, l);          // shared -> global through the TMA engine
          tma_bulk_store_wait_read();
          mbar_arrive(bar + kB_StoreFree + 8 * slot);
        }
      }
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all writes complete before the CTA exits
    }
  } else if (rank != 0) {
    // peer CTA: nothing to issue (its MMAs are issued by the leader, its TMA signals the leader)
  } else {
    // ================================ leader CTA: MMA issuer ================================
    // The whole warp walks the schedule convergently (one unrolled copy of the issue code per layer class); one
    // elected lane issues the tcgen05 instructions.
    MmaRing ring{0u, 0u};
    uint32_t act_parity[2] = {0u, 0u};
    long long t_act = 0;
#ifdef NB200_DEV
    const long long t_begin = clock64();
#endif
    const uint64_t desc_hi = umma_smem_desc(0, 16, 1024);  // LBO/SBO/version/swizzle bits
    for (int64_t pr = 0; pr * Epi::kSlots < my_pt; ++pr) {
      const int nslots = (Epi::kSlots == 2 && my_pt - 2 * pr >= 2) ? 2 : 1;
#pragma unroll 1
      for (int l = 0; l < Epi::kNumLayers; ++l) {
        const int rep = sched_class_rep<Epi>(l);
        if (rep == 0) issue_layer<Epi, 0>(smem_base, bar, tmem_base, desc_hi, nslots, l, ring, act_parity, t_act);
        else if (rep == 1) issue_layer<Epi, 1>(smem_base, bar, tmem_base, desc_hi, nslots, l, ring, act_parity, t_act);
        else if (!sched_is_bwd<Epi::kTab>() && rep == 5) issue_layer<Epi, 5>(smem_base, bar, tmem_base, desc_hi, nslots, l, ring, act_parity, t_act);
        else if (!sched_is_bwd<Epi::kTab>()) issue_layer<Epi, Epi::kNumLayers - 1>(smem_base, bar, tmem_base, desc_hi, nslots, l, ring, act_parity, t_act);
      }
    }
#ifdef NB200_DEV
    if constexpr (Epi::kHasDbg && kDevBuild) {
      if ((p.dbg & 8) && lane == 0 && p.dbg_counters) {
        atomicAdd(p.dbg_counters + 0, (unsigned long long)t_act);
        atomicAdd(p.dbg_counters + 3, (unsigned long long)(clock64() - t_begin));
      }
    }
#endif
  }
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();
  if (warp == kCMmaWarp) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

// ============================================================================ forward
struct FwdEpiParams {
  CUtensorMap tmap128, tmap64;  // packed weight image as [rows x 128 B], boxes of 128 / 64 rows
  int dbg;
  unsigned long long* dbg_counters;
  int in_mode;
  const float* in0;
  const float* in1;
  int64_t M;
  int N;
  int nshift;      // log2(N) when N is a power of two, else -1 (sample -> ray index without a 64-bit division)
  const uint8_t* packed;
  float* out;
  uint8_t* saved;  // null for inference
  int64_t num_tiles;
  // fused render (FwdEpi<false, true>): sampler -> MLP -> compositing in one kernel, N in {32, 64, 128}
  float* rgb;        // [B,3]
  float* disp;       // [B]
  float* acc;        // [B]
  int64_t B;
  int sampler;       // 0: sample depths from in1 [B,N]; 1: Philox(seed, offset) like stratified_ts_quad_kernel
  uint64_t seed, offset;
  float tn, tf;
  const float* poses;  // in_mode == kInCamera: rays come from (poses [P,4,4], H, W, f, ray_begin + ray)
  int H, W;
  float f;
  int64_t ray_begin;
};
constexpr int kInCamera = 2;  // internal input mode of the fused render kernel

// (origin, direction) of ray `ray`: a row of the rays tensor, or generated from the camera
__device__ __forceinline__ void load_ray_chain(const FwdEpiParams& p, int64_t ray, float (&o)[6]) {
  if (p.in_mode == kInCamera) {
    camera_ray(p.poses, p.H, p.W, p.f, p.ray_begin + ray, o);
  } else {
    const float2* q = reinterpret_cast<const float2*>(p.in0 + ray * 6);
    const float2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y; o[4] = c.x; o[5] = c.y;
  }
}

template <bool kRender>
__device__ __forceinline__ void load_query_chain(const FwdEpiParams& p, int64_t m, float v[6], float& t) {
  if (!kRender && p.in_mode == NB200_IN_POINTS) {
    const float2* q = reinterpret_cast<const float2*>(p.in0 + m * 6);
    const float2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y;
    t = 0.f;
  } else {
    const int64_t ray = p.nshift >= 0 ? (m >> p.nshift) : m / p.N;
    float o[6];
    if (kRender) {
      load_ray_chain(p, ray, o);
      t = p.sampler ? philox_sample_depth(m, (int)(m - ray * p.N), p.N, p.tn, p.tf, p.seed, p.offset) : __ldg(p.in1 + m);
    } else {
      const float2* q = reinterpret_cast<const float2*>(p.in0 + ray * 6);
      const float2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
      o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y; o[4] = c.x; o[5] = c.y;
      t = __ldg(p.in1 + m);
    }
    const float dx = o[3], dy = o[4], dz = o[5];
    v[0] = __fadd_rn(o[0], __fmul_rn(dx, t));  // utils/rendering.py:34-36 (d un-normalised)
    v[1] = __fadd_rn(o[1], __fmul_rn(dy, t));
    v[2] = __fadd_rn(o[2], __fmul_rn(dz, t));
    const float inv = 1.0f / sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx)));  // :37
    v[3] = dx * inv; v[4] = dy * inv; v[5] = dz * inv;
  }
}

// Fused render: composite one ray of the tile from the (r,g,b,sigma) / depth rows staged in shared
// memory.  One warp, lane l owns the S = N/32 consecutive samples l*S..l*S+S-1: the same arithmetic,
// in the same order, as composite_fwd_kernel<S, ., ., true, false, 1> (utils/rendering.py:60-83).
template <int S>
__device__ __forceinline__ void composite_staged_ray(const FwdEpiParams& p, uint32_t stage_o, uint32_t stage_t, int ray_local,
                                                     int64_t ray, int lane) {
  constexpr int N = 32 * S;
  float4 o[S];
  float t[S];
  const uint32_t row0 = (uint32_t)(ray_local * N + lane * S);
#pragma unroll
  for (int j = 0; j < S; ++j) {
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(o[j].x), "=f"(o[j].y), "=f"(o[j].z), "=f"(o[j].w) : "r"(stage_o + (row0 + j) * 16u));
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(t[j]) : "r"(stage_t + (row0 + j) * 4u));
  }
  float rd[6];
  load_ray_chain(p, ray, rd);
  const float norm = unit_dir_norm(rd[3], rd[4], rd[5]);
  const float t_next_lane = __shfl_down_sync(0xffffffffu, t[0], 1);
  float a[S], pre[S];
  float run = 1.f;
#pragma unroll
  for (int j = 0; j < S; ++j) {
    const bool last = (j == S - 1 && lane == 31);
    const float tn = (j == S - 1) ? t_next_lane : t[j + 1 < S ? j + 1 : j];
    const float d = last ? 1e10f : __fsub_rn(tn, t[j]);                             // :60-61
    const float delta = __fmul_rn(d, norm);                                         // :62
    const float e = transmit_factor(o[j].w, delta);                                 // :67
    a[j] = __fsub_rn(1.f, e);
    const float fac = __fadd_rn(__fsub_rn(1.f, a[j]), 1e-10f);                      // :68
    pre[j] = run;
    run *= fac;
  }
  float pr = run;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const float v = __shfl_up_sync(0xffffffffu, pr, d);
    pr *= (lane >= d) ? v : 1.f;
  }
  float ex = __shfl_up_sync(0xffffffffu, pr, 1);
  ex = lane == 0 ? 1.f : ex;
  float sr = 0.f, sg = 0.f, sb = 0.f, sd = 0.f, sa = 0.f;
#pragma unroll
  for (int j = 0; j < S; ++j) {
    const float w = a[j] * (ex * pre[j]);
    sr = fmaf(w, o[j].x, sr); sg = fmaf(w, o[j].y, sg); sb = fmaf(w, o[j].z, sb);
    sd = fmaf(w, t[j], sd);
    sa += w;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    sr += __shfl_xor_sync(0xffffffffu, sr, d); sg += __shfl_xor_sync(0xffffffffu, sg, d);
    sb += __shfl_xor_sync(0xffffffffu, sb, d); sd += __shfl_xor_sync(0xffffffffu, sd, d);
    sa += __shfl_xor_sync(0xffffffffu, sa, d);
  }
  if (lane == 0) {
    p.rgb[ray * 3] = sr; p.rgb[ray * 3 + 1] = sg; p.rgb[ray * 3 + 2] = sb;
    p.disp[ray] = disparity(sd, sa);
    p.acc[ray] = sa;
  }
}

// Head weights in shared memory.  While E[slot] carries posd (K = 32: logical chunks 0..3 of every 128-byte row), the
// other 64 bytes of each row are free; the forward kernels keep w_sigma, color_fc.2's weight and the two head biases
// there (644 floats, written next to the posd encoding, once per tile), because the constant-bank loads of the head
// weights made the sigma-head layer 2.7x and the colour layer 2.5x as long as a plain hidden layer.
// Table float i lives in logical chunk 4 + (i/4)%4 of row i/16 (SWIZZLE_128B image, like everything else in E).
constexpr uint32_t kTabWSig = 0, kTabWC1 = 256, kTabBC1 = 640, kTabBSig = 643, kTabFloats = 644;
__host__ __device__ constexpr uint32_t tab_off(uint32_t i) {
  return (i >> 4) * 128u + (((4u + ((i >> 2) & 3u)) ^ ((i >> 4) & 7u)) << 4) + (i & 3u) * 4u;
}
__device__ __forceinline__ float4 tab_ld4(uint32_t e_img, uint32_t i) {   // i % 4 == 0, warp-uniform
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(e_img + tab_off(i)));
  return v;
}

// 16 accumulator columns + their (staged) biases -> [ReLU] -> two 16-byte chunks of the next layer's bf16 A operand.
// ReLU is fused into the fp32->bf16x2 conversion (cvt.rn.relu.bf16x2.f32), the biases are added two at a time
// (add.f32x2).  NB_PROBE_* builds are timing probes with wrong results (scripts/build_variants.sh).
template <bool kRelu, bool kSigma, bool kSave>
__device__ __forceinline__ void epi_cols16(const TileCtx& c, const uint32_t (&a)[16], int col0, const float4 (&bq)[4], float& sigma) {
  const uint32_t kb = (uint32_t)col0 >> 6, j0 = ((uint32_t)col0 >> 3) & 7u;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    float x[8];
#ifdef NB_PROBE_NOBIAS   // timing probe only (wrong results)
    const float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
#else
    const float4 b0 = bq[2 * j], b1 = bq[2 * j + 1];
#endif
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(a[8 * j + e]);
    add_f32x2(x[0], x[1], b0.x, b0.y); add_f32x2(x[2], x[3], b0.z, b0.w);
    add_f32x2(x[4], x[5], b1.x, b1.y); add_f32x2(x[6], x[7], b1.z, b1.w);
    if (kSigma) {  // sigma head reads the (ReLU'd, fp32) layers_1 output (utils/nets.py:40)
      const float4 s0 = tab_ld4(c.e_img, kTabWSig + (uint32_t)(col0 + 8 * j)), s1 = tab_ld4(c.e_img, kTabWSig + (uint32_t)(col0 + 8 * j + 4));
      const float ws[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
#pragma unroll
      for (int e = 0; e < 8; ++e) sigma = fmaf(fmaxf(x[e], 0.f), ws[e], sigma);
    }
    uint32_t w0, w1, w2, w3;
    if (kRelu) {
      w0 = pack_bf16x2_relu(x[0], x[1]); w1 = pack_bf16x2_relu(x[2], x[3]);
      w2 = pack_bf16x2_relu(x[4], x[5]); w3 = pack_bf16x2_relu(x[6], x[7]);
    } else {
      w0 = pack_bf16x2(x[0], x[1]); w1 = pack_bf16x2(x[2], x[3]);
      w2 = pack_bf16x2(x[4], x[5]); w3 = pack_bf16x2(x[6], x[7]);
    }
    const uint32_t o = sw_off(c, kb, j0 + j);
#ifdef NB_PROBE_NOSTS   // timing probe only (wrong results)
    if (w0 == 0x12345678u && w1 == w2 && w3 == 0x9abcdef0u) st_shared_v4(c.a_img + o, w0, w1, w2, w3);
#else
    st_shared_v4(c.a_img + o, w0, w1, w2, w3);
#endif
  }
}

// One hidden layer: accumulator (TMEM) + bias -> [ReLU] -> bf16 A operand of the next layer.  Each
// thread converts the 128 columns of its half in 16-column steps, with the TMEM load of the next
// step in flight while the current one is converted (double buffer).
#ifdef NB_PROBE_NOLDTM   // timing probe only (wrong results): no TMEM reads in the hidden-layer epilogue
#define tmem_ld16(addr, arr) do { _Pragma("unroll") for (int i_ = 0; i_ < 16; ++i_) arr[i_] = (addr) + (uint32_t)i_; } while (0)
#endif
// the 16 staged biases of columns [col0, col0 + 16): warp-uniform LDS.128 (broadcast), issued BEFORE the wait for the
// TMEM load they are added to, so that their latency hides behind it
__device__ __forceinline__ void load_bias16(const TileCtx& c, int col0, float4 (&bq)[4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(bq[i].x), "=f"(bq[i].y), "=f"(bq[i].z), "=f"(bq[i].w) : "r"(c.b_img + (uint32_t)(col0 + 4 * i) * 4u));
}
template <bool kRelu, bool kSigma, bool kSave, int kHalf>
__device__ __forceinline__ void epi_hidden_h(const TileCtx& c, float& sigma) {
  constexpr int cbase = kHalf * 128;
  uint32_t a0[16], a1[16];
  float4 bq[4];
  tmem_ld16(c.t_lane + cbase, a0);
#pragma unroll
  for (int q = 0; q < 8; q += 2) {
    load_bias16(c, cbase + q * 16, bq);
    tmem_ld_wait();                                       // a0 (step q) has landed
    tmem_ld16(c.t_lane + cbase + (q + 1) * 16, a1);       // step q+1 in flight
    epi_cols16<kRelu, kSigma, kSave>(c, a0, cbase + q * 16, bq, sigma);
    load_bias16(c, cbase + (q + 1) * 16, bq);
    tmem_ld_wait();                                       // a1 has landed
    if (q + 2 < 8) tmem_ld16(c.t_lane + cbase + (q + 2) * 16, a0);
    epi_cols16<kRelu, kSigma, kSave>(c, a1, cbase + (q + 1) * 16, bq, sigma);
  }
}
// The column half is dispatched to a compile-time constant, so that the shared-memory addresses of the staged biases,
// of the head-weight table and of the swizzled stores are "base + immediate".  (Biases used to be indexed constant-bank
// loads, 8 LDC.64 per 16 columns: they saturated the MIO/ADU path -- 31 % of all warp stall samples of the forward
// kernel sat on them -- and removing the bias path altogether was worth 16 % of the frame time; see DESIGN 4.5.)
template <bool kRelu, bool kSigma, bool kSave>
__device__ __forceinline__ void epi_hidden(const TileCtx& c, float& sigma) {
  if (c.half == 0) epi_hidden_h<kRelu, kSigma, kSave, 0>(c, sigma);
  else epi_hidden_h<kRelu, kSigma, kSave, 1>(c, sigma);
}
#ifdef NB_PROBE_NOLDTM
#undef tmem_ld16
#endif

// kFold: layers_2 folded into color_fc.0 (mlp_tc.cu, top): the chain has 9 layers, loop index 8 is MMA layer 9.
template <bool kSave, bool kRender = false, bool kFold = false>
struct FwdEpi {
  static_assert(!(kSave && kRender), "the fused render kernel is inference only");
  using Params = FwdEpiParams;
  static constexpr bool kHasDbg = true;
  static constexpr bool kBulkStore = kSave;  // training: finished tile images leave through TMA bulk stores
  static constexpr int kTab = kFold ? kTabFwdFold : kTabFwd;
  static constexpr bool kStageBias = true;
  static constexpr int kSlots = 2;
  static constexpr int kNumLayers = kFold ? kNumFoldLayers : kNumMmaLayers;
  static constexpr bool kReverseTiles = false;
  __device__ static constexpr int ml_of(int l) { return (kFold && l == 8) ? 9 : l; }                 // loop index -> MMA layer
  __device__ static constexpr int bias_row(int l) { return (kFold && l == 8) ? kFoldBiasRow : l; }
  struct State {
    float v[6];
    float sigma;
    float t;          // sample depth (fused render)
    int64_t m_raw;
    bool row_valid;
  };
  __device__ static void init_slot(const TileCtx&) {}

  __device__ static void prefetch(const Params&, State&, const TileCtx&, int) {}

  // Training: the ReLU bit masks the delta chain reads (one bit per element of h0..h7 and c1) are formed AFTER the tile
  // image was handed to the MMA warp and the store warp, from the bf16 image in shared memory: the epilogue warps of
  // this slot would otherwise idle until their next accumulator is ready, so the ~130 extra instructions per thread
  // and layer stay off the critical path (inside the epilogue they cost the kernel 11 %).
  __device__ static void after_publish(const Params& p, State& st, const TileCtx& c, int l) {
    const int ml = ml_of(l);
    if (ml == 5) {
      // posx has been consumed by the skip layer's MMAs: the encoding buffer now carries posd (27 -> 64) for color_fc.0,
      // plus the head-weight table in the free half of its rows.  Done here, behind the hand-off of h5, so that it
      // runs while the slot waits for its next accumulator (inside the epilogue it cost ~2,300 cycles of the chain).
      // (only logical chunks 0..3 = K 0..31 are written and read: chunks 4..7 of the rows belong to the table)
      if (c.half == 0) encode_row<kLd, 0, 2>(st.v + 3, c.e_img, c.r, nullptr);
      else encode_row<kLd, 2, 4>(st.v + 3, c.e_img, c.r, nullptr);
#pragma unroll
      for (uint32_t i = threadIdx.x & 255u; i < kTabFloats; i += 256u) {
        const float v = __ldg(c.gf + (i < kTabWC1 ? kF32WSig + (int)i
                                                  : (i < kTabBC1 ? kF32WC1 + (int)(i - kTabWC1) : (i < kTabBSig ? kF32BC1 + (int)(i - kTabBC1) : kF32BSig))));
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(c.e_img + tab_off(i)), "f"(v) : "memory");
      }
    }
    if (!kSave || ml < 0 || ml == 8) return;
    const int64_t T = p.num_tiles;
    if (ml < 8) {
      uint8_t* row = p.saved + mask_tensor_off(ml, T) + (size_t)c.tile * 4096 + ((size_t)(c.half * 128) + c.r) * 16;
      uint32_t m[4];                         // unrolled: no spills, the 16 LDS.128 in flight together (-5 % on the kernel)
#pragma unroll
      for (int q = 0; q < 4; ++q) {          // 32 columns = 4 chunks of 16 B = one mask word
        const uint32_t kb = (uint32_t)(c.half * 2 + (q >> 1)), j0 = (uint32_t)(q & 1) * 4u;
        uint32_t f[2] = {0u, 0u};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t w0, w1, w2, w3;
          asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3) : "r"(c.a_img + sw_off(c, kb, j0 + j)));
          add_pair_flags(f[j >> 1], w0, 4 * (j & 1)); add_pair_flags(f[j >> 1], w1, 4 * (j & 1) + 1);
          add_pair_flags(f[j >> 1], w2, 4 * (j & 1) + 2); add_pair_flags(f[j >> 1], w3, 4 * (j & 1) + 3);
        }
        m[q] = fold_mask16(f[0]) | (fold_mask16(f[1]) << 16);
      }
      *reinterpret_cast<uint4*>(row) = make_uint4(m[0], m[1], m[2], m[3]);
    } else {   // ml == 9: c1, 64 columns per thread = K-block `half` of the image
      uint8_t* row = p.saved + mask_tensor_off(8, T) + (size_t)c.tile * 2048 + ((size_t)(c.half * 128) + c.r) * 8;
      uint32_t m[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        uint32_t f[2] = {0u, 0u};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t w0, w1, w2, w3;
          asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3)
                       : "r"(c.a_img + sw_off(c, (uint32_t)c.half, (uint32_t)(q * 4 + j))));
          add_pair_flags(f[j >> 1], w0, 4 * (j & 1)); add_pair_flags(f[j >> 1], w1, 4 * (j & 1) + 1);
          add_pair_flags(f[j >> 1], w2, 4 * (j & 1) + 2); add_pair_flags(f[j >> 1], w3, 4 * (j & 1) + 3);
        }
        m[q] = fold_mask16(f[0]) | (fold_mask16(f[1]) << 16);
      }
      *reinterpret_cast<uint2*>(row) = make_uint2(m[0], m[1]);
    }
  }

  __device__ static void begin_tile(const Params& p, State& st, const TileCtx& c) {
    st.m_raw = c.tile * kTileM + c.r;
    st.row_valid = st.m_raw < p.M;
    load_query_chain<kRender>(p, st.row_valid ? st.m_raw : p.M - 1, st.v, st.t);
    st.sigma = 0.f;
    // posx -> E[slot] (K = 64); each half of the slot's threads stores 4 of the 8 16-byte chunks
    if (c.half == 0) encode_row<kLp, 0, 4>(st.v, c.e_img, c.r, nullptr);
    else encode_row<kLp, 4, 8>(st.v, c.e_img, c.r, nullptr);
  }

  // one thread per slot, after the slot barrier: tile images shared -> global (saved activations)
  __device__ static void store_tile(const Params& p, const TileCtx& c, int l) {
    const int64_t T = p.num_tiles;
    const int ml = ml_of(l);
    if (ml == -1) tma_bulk_s2g(p.saved + saved_tensor_off(10, T) + (size_t)c.tile * 16384, c.e_img, 16384);        // posx
    else if (ml < 9) tma_bulk_s2g(p.saved + saved_tensor_off(ml, T) + (size_t)c.tile * 65536, c.a_img, 65536);    // h0..h7, g
    else tma_bulk_s2g(p.saved + saved_tensor_off(9, T) + (size_t)c.tile * 32768, c.a_img, 32768);                  // c1
    if (ml == 6) tma_bulk_s2g(p.saved + saved_tensor_off(11, T) + (size_t)c.tile * 16384, c.e_img, 16384);         // posd (encoded behind h5's hand-off)
  }

  __device__ static void layer(const Params& p, State& st, const TileCtx& c, int l) {
    const int ml = ml_of(l);
    if (ml < 9) {
      if (ml == 7) epi_hidden<true, true, kSave>(c, st.sigma);
      else if (ml == 8) epi_hidden<false, false, kSave>(c, st.sigma);  // layers_2: no act.
      else epi_hidden<true, false, kSave>(c, st.sigma);
    } else {
      // color_fc.0 epilogue (128 columns, ReLU; this thread's half = 64 of them) + color_fc.2
      // (128 -> 3) on CUDA cores; the two halves of a row meet through the (now free) E buffer
      float rgb[3] = {0.f, 0.f, 0.f};
#pragma unroll 1
      for (int q = 0; q < 2; ++q) {
        const int col0 = c.half * 64 + q * 32;
        uint32_t a[32];
        tmem_ld32(c.t_lane + col0, a);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float x[8], b[8];
          asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b[0]), "=f"(b[1]), "=f"(b[2]), "=f"(b[3]) : "r"(c.b_img + (uint32_t)(col0 + 8 * j) * 4u));
          asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b[4]), "=f"(b[5]), "=f"(b[6]), "=f"(b[7]) : "r"(c.b_img + (uint32_t)(col0 + 8 * j + 4) * 4u));
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] = fmaxf(__uint_as_float(a[8 * j + e]) + b[e], 0.f);
#pragma unroll
          for (int k = 0; k < 3; ++k) {   // color_fc.2 (128 -> 3), weights from the table in E[slot]
            const float4 w0 = tab_ld4(c.e_img, kTabWC1 + (uint32_t)(k * 128 + col0 + 8 * j)), w1 = tab_ld4(c.e_img, kTabWC1 + (uint32_t)(k * 128 + col0 + 8 * j + 4));
            rgb[k] = fmaf(x[0], w0.x, rgb[k]); rgb[k] = fmaf(x[1], w0.y, rgb[k]); rgb[k] = fmaf(x[2], w0.z, rgb[k]); rgb[k] = fmaf(x[3], w0.w, rgb[k]);
            rgb[k] = fmaf(x[4], w1.x, rgb[k]); rgb[k] = fmaf(x[5], w1.y, rgb[k]); rgb[k] = fmaf(x[6], w1.z, rgb[k]); rgb[k] = fmaf(x[7], w1.w, rgb[k]);
          }
          if (kSave) {  // c1 tile image -> A[slot] K-blocks 0,1 (free after color_fc.0's MMAs), bulk-stored by store_tile
            const uint32_t w0 = pack_bf16x2(x[0], x[1]), w1 = pack_bf16x2(x[2], x[3]), w2 = pack_bf16x2(x[4], x[5]),
                           w3 = pack_bf16x2(x[6], x[7]);
            st_shared_v4(c.a_img + sw_off(c, (uint32_t)c.half, (uint32_t)(q * 4 + j)), w0, w1, w2, w3);
          }
        }
      }
      const uint32_t xaddr = c.e_img + c.r * 16u;
      if (c.half == 1) st_shared_v4(xaddr, __float_as_uint(rgb[0]), __float_as_uint(rgb[1]), __float_as_uint(rgb[2]), __float_as_uint(st.sigma));
      slot_barrier(c.slot);
      if (c.half == 0) {
        float4 o;
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w) : "r"(xaddr));
        const float4 hb = tab_ld4(c.e_img, kTabBC1);   // color_fc.2's bias, sigma_fc's bias
        const float4 res = make_float4(rgb[0] + o.x + hb.x, rgb[1] + o.y + hb.y, rgb[2] + o.z + hb.z, st.sigma + o.w + hb.w);  // (r,g,b,sigma), utils/nets.py:43
        if (kRender) {
          // stage the row for the compositing warps in A[slot]: its last reader (color_fc.0's MMAs) is done and
          // the next writer (layer 0's epilogue of the next tile) runs only after every warp of the slot has
          // arrived for that tile, i.e. after the compositing below
          st_shared_v4(c.a_img + c.r * 16u, __float_as_uint(res.x), __float_as_uint(res.y), __float_as_uint(res.z), __float_as_uint(res.w));
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(c.a_img + 2048u + c.r * 4u), "f"(st.t) : "memory");
        } else if (st.row_valid) {
          reinterpret_cast<float4*>(p.out)[st.m_raw] = res;
        }
      }
      slot_barrier(c.slot);  // E[slot] may be re-encoded for the next tile only after the exchange was read
      if (kRender) {
        const int wq = (int)(threadIdx.x >> 5) & 7, nr = kTileM / p.N;   // warp wq composites ray wq of the tile
        const int64_t ray = c.tile * nr + wq;
        if (wq < nr && ray < p.B) {
          const int lane = (int)threadIdx.x & 31;
          if (p.N == 64) composite_staged_ray<2>(p, c.a_img, c.a_img + 2048u, wq, ray, lane);
          else if (p.N == 128) composite_staged_ray<4>(p, c.a_img, c.a_img + 2048u, wq, ray, lane);
          else composite_staged_ray<1>(p, c.a_img, c.a_img + 2048u, wq, ray, lane);
        }
      }
    }
  }
};

// ============================================================ forward, NB200_BF16X3 (fp32-class accuracy)
// Error-compensated bf16: every activation is kept as a pair of bf16 images, hi = bf16(x) and lo = bf16(x - hi), and
// every weight as (W_hi, W_lo); a K-block costs three MMA passes, A_hi W_hi + A_lo W_hi + A_hi W_lo (the lo x lo term
// is below 2^-16 relative and dropped), all accumulated in fp32 in TMEM.  The lo images live in the buffers the bf16
// kernels use for their second in-flight tile, so ONE tile per CTA is in flight and all 16 epilogue warps work on it
// (four per TMEM lane group, 64 accumulator columns each).  Replaces the 25 TFLOP/s SIMT kernels as the <= 1e-4
// parity mode of utils/nets.py:34-43 for inference.
__device__ __forceinline__ void split_hi_lo(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16x2(x0, x1);
  lo = pack_bf16x2(x0 - __uint_as_float(hi << 16), x1 - __uint_as_float(hi & 0xFFFF0000u));
}
template <int L, int J0, int J1>
__device__ __forceinline__ void encode_row3(const float* x, uint32_t img_hi, uint32_t img_lo, uint32_t r) {
  float f[64];
#pragma unroll
  for (int i = 0; i < 64; ++i) f[i] = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    f[c] = x[c];
#pragma unroll
    for (int i = 0; i < L; ++i) {   // fp32-class mode: every level with the accurate sincosf (no double-angle recurrence)
      float sv, cv;
      sincosf(ldexpf(x[c], i), &sv, &cv);   // (2^i) * x is exact, as in utils/xyz.py:12
      f[3 + c * 2 * L + 2 * i] = sv;
      f[3 + c * 2 * L + 2 * i + 1] = cv;
    }
  }
#pragma unroll
  for (int j = J0; j < J1; ++j) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) split_hi_lo(f[8 * j + 2 * e], f[8 * j + 2 * e + 1], h[e], l[e]);
    st_shared_v4(img_hi + sw128_off(r, j), h[0], h[1], h[2], h[3]);
    st_shared_v4(img_lo + sw128_off(r, j), l[0], l[1], l[2], l[3]);
  }
}

// Bit k / 8+k of a 16-column step's mask field is column 2k / 2k+1 (the layout of the bf16 chain's mask tensors).
__device__ __forceinline__ uint32_t relu_bit(int col_in_step) { return 1u << ((col_in_step >> 1) + 8 * (col_in_step & 1)); }

// kSave (training): the hi and lo images of every layer input leave through the store warp (saved layout: mlp_tc.cu,
// kSavedTileBytes3), and the ReLU masks are formed from the fp32 values in the epilogue.  The outputs are the
// inference kernel's, bit for bit.
template <bool kSave>
struct FwdEpi3 {
  using Params = FwdEpiParams;
  static constexpr bool kHasDbg = false;
  static constexpr bool kBulkStore = kSave;
  static constexpr int kTab = kTabFwd3;
  static constexpr bool kStageBias = true;
  static constexpr int kSlots = 1;
  static constexpr int kNumLayers = kNumMmaLayers;
  static constexpr bool kReverseTiles = false;
  struct State {
    float v[6];
    float sigma;      // this thread's share (64 columns) of the sigma head
    int64_t m_raw;
    bool row_valid;
  };
  __device__ static constexpr int bias_row(int l) { return l; }
  __device__ static void init_slot(const TileCtx&) {}
  __device__ static void prefetch(const Params&, State&, const TileCtx&, int) {}
  __device__ static void after_publish(const Params&, State&, const TileCtx&, int) {}
  // the store warp: layer l's hand-off (l = -1: posx; 0..8: h0..h7, g; 9: c1; posd rides on h5) as hi and lo images
  __device__ static void store_tile(const Params& p, const TileCtx& c, int l) {
    if (!kSave) return;
    const int64_t T = p.num_tiles;
    uint8_t* lo = p.saved + kSavedDataTileBytes * (size_t)T;
    auto put = [&](int t, uint32_t img, uint32_t img_lo) {
      const size_t off = saved_tensor_off(t, T) + (size_t)c.tile * saved_tile_bytes(t);
      tma_bulk_s2g(p.saved + off, img, (uint32_t)saved_tile_bytes(t));
      tma_bulk_s2g(lo + off, img_lo, (uint32_t)saved_tile_bytes(t));
    };
    if (l == -1) put(10, c.e_img, c.e_img + kEBytes);
    else put(l, c.a_img, c.a_img + kABytes);
    if (l == 5) put(11, c.e_img, c.e_img + kEBytes);   // posd, encoded in front of h5's epilogue
  }

  __device__ static void encode(const float* x, const TileCtx& c, bool dirs) {
    const uint32_t hi = c.e_img, lo = c.e_img + kEBytes;
    if (!dirs) {
      if (c.part == 0) encode_row3<kLp, 0, 2>(x, hi, lo, c.r);
      else if (c.part == 1) encode_row3<kLp, 2, 4>(x, hi, lo, c.r);
      else if (c.part == 2) encode_row3<kLp, 4, 6>(x, hi, lo, c.r);
      else encode_row3<kLp, 6, 8>(x, hi, lo, c.r);
    } else {
      if (c.part == 0) encode_row3<kLd, 0, 2>(x, hi, lo, c.r);
      else if (c.part == 1) encode_row3<kLd, 2, 4>(x, hi, lo, c.r);
      else if (c.part == 2) encode_row3<kLd, 4, 6>(x, hi, lo, c.r);
      else encode_row3<kLd, 6, 8>(x, hi, lo, c.r);
    }
  }

  __device__ static void begin_tile(const Params& p, State& st, const TileCtx& c) {
    st.m_raw = c.tile * kTileM + c.r;
    st.row_valid = st.m_raw < p.M;
    float t;
    load_query_chain<false>(p, st.row_valid ? st.m_raw : p.M - 1, st.v, t);
    st.sigma = 0.f;
    encode(st.v, c, false);
  }

  __device__ static void layer(const Params& p, State& st, const TileCtx& c, int ml) {
    if (ml == 5) encode(st.v + 3, c, true);   // posx consumed by the skip layer: the encoding buffers now carry posd
    const uint32_t a_hi = c.a_img, a_lo = c.a_img + kABytes;
    if (ml < 9) {
      const int cbase = c.part * 64;
      const float* ws = c.gf + kF32WSig;   // (read-only global loads at warp-uniform addresses; this mode is not bound by them)
      uint32_t mbits[2] = {0u, 0u};        // kSave: ReLU mask words of this thread's 64 columns (two 16-column steps each)
#pragma unroll 1
      for (int q = 0; q < 4; ++q) {
        const int col0 = cbase + q * 16;
        uint32_t a[16];
        float4 bq[4];
        tmem_ld16(c.t_lane + col0, a);
        load_bias16(c, col0, bq);      // staged bias row of this layer (shared memory), under the TMEM load
        tmem_ld_wait();
        const uint32_t kb = (uint32_t)col0 >> 6, j0 = ((uint32_t)col0 >> 3) & 7u;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          float x[8];
          const float b[8] = {bq[2 * j].x, bq[2 * j].y, bq[2 * j].z, bq[2 * j].w, bq[2 * j + 1].x, bq[2 * j + 1].y, bq[2 * j + 1].z, bq[2 * j + 1].w};
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            x[e] = __uint_as_float(a[8 * j + e]) + b[e];
            if (ml != 8) x[e] = fmaxf(x[e], 0.f);                        // layers_2 has no activation (utils/nets.py:41)
          }
          if (ml == 7) {   // sigma head reads h7 in fp32 (:40)
            const float4 s0 = __ldg(reinterpret_cast<const float4*>(ws + col0 + 8 * j)), s1 = __ldg(reinterpret_cast<const float4*>(ws + col0 + 8 * j + 4));
            st.sigma = fmaf(x[0], s0.x, st.sigma); st.sigma = fmaf(x[1], s0.y, st.sigma); st.sigma = fmaf(x[2], s0.z, st.sigma);
            st.sigma = fmaf(x[3], s0.w, st.sigma); st.sigma = fmaf(x[4], s1.x, st.sigma); st.sigma = fmaf(x[5], s1.y, st.sigma);
            st.sigma = fmaf(x[6], s1.z, st.sigma); st.sigma = fmaf(x[7], s1.w, st.sigma);
          }
          if (kSave && ml != 8) {
            uint32_t f = 0u;
#pragma unroll
            for (int e = 0; e < 8; ++e) f |= x[e] > 0.f ? relu_bit(8 * j + e) : 0u;
            if (q & 2) mbits[1] |= f << (16 * (q & 1)); else mbits[0] |= f << (16 * (q & 1));
          }
          uint32_t h[4], l[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) split_hi_lo(x[2 * e], x[2 * e + 1], h[e], l[e]);
          const uint32_t o = sw_off(c, kb, j0 + j);
          st_shared_v4(a_hi + o, h[0], h[1], h[2], h[3]);
          st_shared_v4(a_lo + o, l[0], l[1], l[2], l[3]);
        }
      }
      if (kSave && ml != 8)   // 8 of the 16 bytes of the (row, column half) entry of mask tensor ml
        *reinterpret_cast<uint2*>(p.saved + mask_tensor_off3(ml, p.num_tiles) + (size_t)c.tile * 4096 +
                                  ((size_t)((c.part >> 1) * 128) + c.r) * 16 + (size_t)(c.part & 1) * 8) = make_uint2(mbits[0], mbits[1]);
    } else {
      // color_fc.0 epilogue (128 columns, 32 per thread, ReLU) + color_fc.2 (128 -> 3) in fp32 on CUDA cores; the four
      // threads of a row meet through the (now free) encoding buffer
      const int col0 = c.part * 32;
      uint32_t a[32];
      tmem_ld32(c.t_lane + col0, a);
      tmem_ld_wait();
      const float4* w4 = reinterpret_cast<const float4*>(c.gf + kF32WC1 + col0);   // color_fc.2's weight, rows 128 floats apart
      float rgb[3] = {0.f, 0.f, 0.f};
      uint32_t mword = 0u;   // kSave: ReLU mask word of this thread's 32 columns of c1
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        float4 bq[4];
        load_bias16(c, col0 + 16 * q, bq);
        uint32_t h[4], lw[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {   // 4 columns at a time
          const float b[4] = {bq[g].x, bq[g].y, bq[g].z, bq[g].w};
          float x[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) x[e] = fmaxf(__uint_as_float(a[16 * q + 4 * g + e]) + b[e], 0.f);
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            const float4 wv = __ldg(w4 + k * 32 + 4 * q + g);
            rgb[k] = fmaf(x[0], wv.x, rgb[k]); rgb[k] = fmaf(x[1], wv.y, rgb[k]);
            rgb[k] = fmaf(x[2], wv.z, rgb[k]); rgb[k] = fmaf(x[3], wv.w, rgb[k]);
          }
          if (kSave) {   // c1 hi / lo images -> K-block part/2 of A[0] / A[1] (free after color_fc.0's MMAs), 8 columns per chunk
#pragma unroll
            for (int e = 0; e < 4; ++e) mword |= x[e] > 0.f ? relu_bit(4 * g + e) << (16 * q) : 0u;
            split_hi_lo(x[0], x[1], h[2 * (g & 1)], lw[2 * (g & 1)]);
            split_hi_lo(x[2], x[3], h[2 * (g & 1) + 1], lw[2 * (g & 1) + 1]);
            if (g & 1) {
              const uint32_t o = sw_off(c, (uint32_t)(c.part >> 1), (uint32_t)((c.part & 1) * 4 + 2 * q + (g >> 1)));
              st_shared_v4(c.a_img + o, h[0], h[1], h[2], h[3]);
              st_shared_v4(c.a_img + kABytes + o, lw[0], lw[1], lw[2], lw[3]);
            }
          }
        }
      }
      if (kSave)   // 4 of the 8 bytes of the (row, column half) entry of mask tensor 8
        *reinterpret_cast<uint32_t*>(p.saved + mask_tensor_off3(8, p.num_tiles) + (size_t)c.tile * 2048 +
                                     ((size_t)((c.part >> 1) * 128) + c.r) * 8 + (size_t)(c.part & 1) * 4) = mword;
      const uint32_t xaddr = c.e_img + ((uint32_t)c.part * 128u + c.r) * 16u;
      if (c.part != 0) st_shared_v4(xaddr, __float_as_uint(rgb[0]), __float_as_uint(rgb[1]), __float_as_uint(rgb[2]), __float_as_uint(st.sigma));
      asm volatile("bar.sync 1, 512;" ::: "memory");
      if (c.part == 0) {
        float4 acc = make_float4(rgb[0], rgb[1], rgb[2], st.sigma);
#pragma unroll
        for (int q = 1; q < 4; ++q) {
          float4 o;
          asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w) : "r"(c.e_img + ((uint32_t)q * 128u + c.r) * 16u));
          acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
        }
        if (st.row_valid)
          reinterpret_cast<float4*>(p.out)[st.m_raw] = make_float4(acc.x + __ldg(c.gf + kF32BC1), acc.y + __ldg(c.gf + kF32BC1 + 1), acc.z + __ldg(c.gf + kF32BC1 + 2),
                                                                   acc.w + __ldg(c.gf + kF32BSig));   // (r,g,b,sigma), utils/nets.py:43
      }
      asm volatile("bar.sync 1, 512;" ::: "memory");   // the encoding buffers may be rewritten for the next tile
    }
  }
};

// ======================================================================= backward (dgrad)
#ifndef NB_DG_L2HINT
#define NB_DG_L2HINT 2   // bit 1: delta stores evict_first (511 -> 501 us).  bit 0 (mask prefetch evict_last, -6 us more) is off:
                          // the evict_last lines outlive the kernel and made the first render after training 2x slower
#endif
// kFold: delta_h7 = delta_c1 Wf in ONE layer (mlp_tc.cu, top): 8 MMA layers, loop index l is bl = l + 2.
template <bool kFold>
struct DgradEpi {
  using Params = BwdParams;
  static constexpr bool kHasDbg = false;
  static constexpr bool kBulkStore = true;
  static constexpr int kTab = kFold ? kTabBwdFold : kTabBwd;
  static constexpr bool kStageBias = false;
  static constexpr int kSlots = 2;
  static constexpr int kNumLayers = kFold ? 8 : 9;  // bl = 1..9 (folded: 2..9)
  static constexpr int kBl0 = kFold ? 2 : 1;        // bl of loop index 0
  static constexpr bool kReverseTiles = true;
  struct State { float4 g; uint4 mask; };
  __device__ static constexpr int bias_row(int l) { return l; }
  __device__ static void after_publish(const Params&, State&, const TileCtx&, int) {}
  // The delta chain has no use for the encoding buffers: E[slot] holds w_sigma (floats 0..255) and color_fc.2's weight
  // (256..639) for the whole kernel, read with warp-uniform LDS.128 instead of constant-bank loads.
  __device__ static void init_slot(const TileCtx& c) {
    for (uint32_t i = threadIdx.x & 255u; i < 640u; i += 256u)
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(c.e_img + i * 4u), "f"(__ldg(c.gf + (i < 256u ? kF32WSig + (int)i : kF32WC1 + (int)(i - 256u)))) : "memory");
    slot_barrier(c.slot);
  }
  __device__ static __forceinline__ float4 head_ld4(const TileCtx& c, uint32_t i) {   // i % 4 == 0, warp-uniform
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(c.e_img + i * 4u));
    return v;
  }

  // The ReLU mask of layer l is this thread's 16-byte row of the bit-mask tensor the forward pass wrote (one bit per
  // element instead of the 64 KB bf16 activation tile): ONE load per thread and layer, issued before the accumulator
  // wait, so its latency is off the epilogue's critical path (the per-thread loads of the activation tile used to
  // account for 25 % of the kernel's stall samples, and for 1.1 GB of DRAM reads per step).
  __device__ static void prefetch(const Params& p, State& st, const TileCtx& c, int l) {
    const int bl = l + kBl0;    // masks with h_{9-bl}: bl=2 -> h7, ..., bl=9 -> h0; bl=1 yields delta_g (no activation)
    if (bl >= 2)
      st.mask = __ldg(reinterpret_cast<const uint4*>(p.saved + mask_tensor_off(9 - bl, p.num_tiles) + (size_t)c.tile * 4096 +
                                                     ((size_t)(c.half * 128) + c.r) * 16));
  }

  __device__ static void begin_tile(const Params& p, State& st, const TileCtx& c) {
    const int64_t T = p.num_tiles;
    const int64_t m_raw = c.tile * kTileM + c.r;
    st.g = make_float4(0.f, 0.f, 0.f, 0.f);  // rows past M carry zero gradient
    if (m_raw < p.M) st.g = __ldg(reinterpret_cast<const float4*>(p.d_out) + m_raw);
    // delta_c1 = (d_rgb @ Wc1) * (c1 > 0)   (color_fc.2 backward, 3 -> 128, CUDA cores)
    const uint2 cbits = __ldg(reinterpret_cast<const uint2*>(p.saved + mask_tensor_off(8, T) + (size_t)c.tile * 2048 +
                                                             ((size_t)(c.half * 128) + c.r) * 8));
    const uint32_t kb = (uint32_t)c.half;  // 128 columns: each half of the slot's threads takes 64
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t o = sw_off(c, kb, j);
      // 8 columns = pairs 4*(j&1) .. +3 of the 16-column step j/2; steps 0,1 in cbits.x, 2,3 in cbits.y
      const uint32_t field = ((j < 4 ? cbits.x : cbits.y) >> (16 * ((j >> 1) & 1))) & 0xFFFFu;
      const int k0 = 4 * (j & 1);
      const uint32_t col = (uint32_t)(c.half * 64 + j * 8);
      float x[8];
      {
        const float4 a0 = head_ld4(c, 256u + col), a1 = head_ld4(c, 256u + col + 4u);
        x[0] = st.g.x * a0.x; x[1] = st.g.x * a0.y; x[2] = st.g.x * a0.z; x[3] = st.g.x * a0.w;
        x[4] = st.g.x * a1.x; x[5] = st.g.x * a1.y; x[6] = st.g.x * a1.z; x[7] = st.g.x * a1.w;
        const float4 b0 = head_ld4(c, 384u + col), b1 = head_ld4(c, 384u + col + 4u);
        x[0] = fmaf(st.g.y, b0.x, x[0]); x[1] = fmaf(st.g.y, b0.y, x[1]); x[2] = fmaf(st.g.y, b0.z, x[2]); x[3] = fmaf(st.g.y, b0.w, x[3]);
        x[4] = fmaf(st.g.y, b1.x, x[4]); x[5] = fmaf(st.g.y, b1.y, x[5]); x[6] = fmaf(st.g.y, b1.z, x[6]); x[7] = fmaf(st.g.y, b1.w, x[7]);
        const float4 c0 = head_ld4(c, 512u + col), c1 = head_ld4(c, 512u + col + 4u);
        x[0] = fmaf(st.g.z, c0.x, x[0]); x[1] = fmaf(st.g.z, c0.y, x[1]); x[2] = fmaf(st.g.z, c0.z, x[2]); x[3] = fmaf(st.g.z, c0.w, x[3]);
        x[4] = fmaf(st.g.z, c1.x, x[4]); x[5] = fmaf(st.g.z, c1.y, x[5]); x[6] = fmaf(st.g.z, c1.z, x[6]); x[7] = fmaf(st.g.z, c1.w, x[7]);
      }
      const uint32_t w0 = pack_bf16x2(x[0], x[1]) & pair_mask_word(field, k0), w1 = pack_bf16x2(x[2], x[3]) & pair_mask_word(field, k0 + 1),
                     w2 = pack_bf16x2(x[4], x[5]) & pair_mask_word(field, k0 + 2), w3 = pack_bf16x2(x[6], x[7]) & pair_mask_word(field, k0 + 3);
      st_shared_v4(c.a_img + o, w0, w1, w2, w3);
    }
  }

  // one thread per slot: delta tile image shared -> global (read back by wgrad)
  __device__ static void store_tile(const Params& p, const TileCtx& c, int l) {
    const int64_t T = p.num_tiles;
#if NB_DG_L2HINT & 2
    const uint64_t pol = l2_policy_evict_first();
    if (l == -1) tma_bulk_s2g_hint(p.dscr + delta_tensor_off(0, T) + (size_t)c.tile * 32768, c.a_img, 32768, pol);   // delta_c1
    else tma_bulk_s2g_hint(p.dscr + delta_tensor_off(l + kBl0, T) + (size_t)c.tile * 65536, c.a_img, 65536, pol);
#else
    if (l == -1) tma_bulk_s2g(p.dscr + delta_tensor_off(0, T) + (size_t)c.tile * 32768, c.a_img, 32768);   // delta_c1
    else tma_bulk_s2g(p.dscr + delta_tensor_off(l + kBl0, T) + (size_t)c.tile * 65536, c.a_img, 65536);
#endif
  }

  // 16 accumulator columns -> masked bf16 delta chunk pair in A[slot] (the next layer's A operand and wgrad's operand)
  template <bool kMasked, bool kSigma>
  __device__ static __forceinline__ void cols16(const TileCtx& c, const uint32_t (&a)[16], int col0, uint32_t field, float gsig) {
    const uint32_t kb = (uint32_t)col0 >> 6, j0 = ((uint32_t)col0 >> 3) & 7u;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      float x[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(a[8 * j + e]);
      if (kSigma) {   // + d_sigma * w_sigma (sigma head reads h7)
        const float4 s0 = head_ld4(c, (uint32_t)(col0 + 8 * j)), s1 = head_ld4(c, (uint32_t)(col0 + 8 * j + 4));
        x[0] = fmaf(gsig, s0.x, x[0]); x[1] = fmaf(gsig, s0.y, x[1]); x[2] = fmaf(gsig, s0.z, x[2]); x[3] = fmaf(gsig, s0.w, x[3]);
        x[4] = fmaf(gsig, s1.x, x[4]); x[5] = fmaf(gsig, s1.y, x[5]); x[6] = fmaf(gsig, s1.z, x[6]); x[7] = fmaf(gsig, s1.w, x[7]);
      }
      uint32_t w0 = pack_bf16x2(x[0], x[1]), w1 = pack_bf16x2(x[2], x[3]), w2 = pack_bf16x2(x[4], x[5]),
               w3 = pack_bf16x2(x[6], x[7]);
      if (kMasked) {
        w0 &= pair_mask_word(field, 4 * j); w1 &= pair_mask_word(field, 4 * j + 1);
        w2 &= pair_mask_word(field, 4 * j + 2); w3 &= pair_mask_word(field, 4 * j + 3);
      }
      st_shared_v4(c.a_img + sw_off(c, kb, j0 + j), w0, w1, w2, w3);
    }
  }
  // this thread's 128 columns in 16-column steps, the TMEM load of the next step in flight while the current one is
  // converted (the single-buffered 32-column loads left the load latency exposed four times per layer)
  template <bool kMasked, bool kSigma>
  __device__ static __forceinline__ void layer_t(State& st, const TileCtx& c) {
    const int cbase = c.half * 128;
    uint32_t a0[16], a1[16];
    tmem_ld16(c.t_lane + cbase, a0);
#pragma unroll
    for (int q = 0; q < 8; q += 2) {
      const uint32_t mw = q == 0 ? st.mask.x : (q == 2 ? st.mask.y : (q == 4 ? st.mask.z : st.mask.w));   // two 16-column steps
      tmem_ld_wait();
      tmem_ld16(c.t_lane + cbase + (q + 1) * 16, a1);
      cols16<kMasked, kSigma>(c, a0, cbase + q * 16, mw & 0xFFFFu, st.g.w);
      tmem_ld_wait();
      if (q + 2 < 8) tmem_ld16(c.t_lane + cbase + (q + 2) * 16, a0);
      cols16<kMasked, kSigma>(c, a1, cbase + (q + 1) * 16, mw >> 16, st.g.w);
    }
  }

  __device__ static void layer(const Params&, State& st, const TileCtx& c, int l) {
    // ReLU mask (bit per element, loaded in prefetch): bl=2 -> h7, ..., bl=9 -> h0; bl=1 yields delta_g (no activation)
    const int bl = l + kBl0;
    if (bl == 1) layer_t<false, false>(st, c);
    else if (bl == 2) layer_t<true, true>(st, c);
    else layer_t<true, false>(st, c);
  }
};

// ================================================================ backward (dgrad), NB200_BF16X3
// The delta chain in error-compensated bf16, on FwdEpi3's skeleton: one tile per CTA, 16 epilogue warps at 64 accumulator
// columns each, delta_hi in A[0] and delta_lo in A[1].  Slabs come from the bwd3 table (hi then lo per K-block), so
// delta_in = delta_hi W_hi + delta_lo W_hi + delta_hi W_lo in fp32 in TMEM; every delta is formed in fp32 (the
// colour head, the sigma-head term, the ReLU mask of the forward's fp32 values) and split into hi / lo once.  The
// store warp writes both images of every delta to the scratch (hi tensors, then lo tensors, in the bf16 layout).
struct DgradEpi3 {
  using Params = BwdParams;
  static constexpr bool kHasDbg = false;
  static constexpr bool kBulkStore = true;
  static constexpr int kTab = kTabBwd3;
  static constexpr bool kStageBias = false;
  static constexpr int kSlots = 1;
  static constexpr int kNumLayers = 9;   // bl = 1..9
  static constexpr bool kReverseTiles = true;
  struct State { float4 g; uint2 mask; };
  __device__ static constexpr int bias_row(int l) { return l; }
  __device__ static void after_publish(const Params&, State&, const TileCtx&, int) {}
  // E[0] holds w_sigma (floats 0..255) and color_fc.2's weight (256..639) for the whole kernel
  __device__ static void init_slot(const TileCtx& c) {
    for (uint32_t i = threadIdx.x; i < 640u; i += 512u)
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(c.e_img + i * 4u), "f"(__ldg(c.gf + (i < 256u ? kF32WSig + (int)i : kF32WC1 + (int)(i - 256u)))) : "memory");
    asm volatile("bar.sync 1, 512;" ::: "memory");
  }
  __device__ static __forceinline__ float4 head_ld4(const TileCtx& c, uint32_t i) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(c.e_img + i * 4u));
    return v;
  }
  // this thread's 8 bytes (64 columns) of the (row, column half) entry of a mask tensor
  __device__ static void prefetch(const Params& p, State& st, const TileCtx& c, int l) {
    const int bl = l + 1;   // bl=2 -> h7, ..., bl=9 -> h0; bl=1 yields delta_g (no activation)
    if (bl >= 2)
      st.mask = __ldg(reinterpret_cast<const uint2*>(p.saved + mask_tensor_off3(9 - bl, p.num_tiles) + (size_t)c.tile * 4096 +
                                                     ((size_t)((c.part >> 1) * 128) + c.r) * 16 + (size_t)(c.part & 1) * 8));
  }

  __device__ static void begin_tile(const Params& p, State& st, const TileCtx& c) {
    const int64_t T = p.num_tiles;
    const int64_t m_raw = c.tile * kTileM + c.r;
    st.g = make_float4(0.f, 0.f, 0.f, 0.f);  // rows past M carry zero gradient
    if (m_raw < p.M) st.g = __ldg(reinterpret_cast<const float4*>(p.d_out) + m_raw);
    // delta_c1 = (d_rgb @ Wc1) * (c1 > 0) in fp32: this thread's 32 of the 128 columns
    const uint32_t cbits = __ldg(reinterpret_cast<const uint32_t*>(p.saved + mask_tensor_off3(8, T) + (size_t)c.tile * 2048 +
                                                                   ((size_t)((c.part >> 1) * 128) + c.r) * 8 + (size_t)(c.part & 1) * 4));
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t col = (uint32_t)(c.part * 32 + j * 8);
      const uint32_t field = (cbits >> (16 * (j >> 1))) & 0xFFFFu;
      const int k0 = 4 * (j & 1);
      float x[8];
      const float4 a0 = head_ld4(c, 256u + col), a1 = head_ld4(c, 256u + col + 4u);
      x[0] = st.g.x * a0.x; x[1] = st.g.x * a0.y; x[2] = st.g.x * a0.z; x[3] = st.g.x * a0.w;
      x[4] = st.g.x * a1.x; x[5] = st.g.x * a1.y; x[6] = st.g.x * a1.z; x[7] = st.g.x * a1.w;
      const float4 b0 = head_ld4(c, 384u + col), b1 = head_ld4(c, 384u + col + 4u);
      x[0] = fmaf(st.g.y, b0.x, x[0]); x[1] = fmaf(st.g.y, b0.y, x[1]); x[2] = fmaf(st.g.y, b0.z, x[2]); x[3] = fmaf(st.g.y, b0.w, x[3]);
      x[4] = fmaf(st.g.y, b1.x, x[4]); x[5] = fmaf(st.g.y, b1.y, x[5]); x[6] = fmaf(st.g.y, b1.z, x[6]); x[7] = fmaf(st.g.y, b1.w, x[7]);
      const float4 c0 = head_ld4(c, 512u + col), c1 = head_ld4(c, 512u + col + 4u);
      x[0] = fmaf(st.g.z, c0.x, x[0]); x[1] = fmaf(st.g.z, c0.y, x[1]); x[2] = fmaf(st.g.z, c0.z, x[2]); x[3] = fmaf(st.g.z, c0.w, x[3]);
      x[4] = fmaf(st.g.z, c1.x, x[4]); x[5] = fmaf(st.g.z, c1.y, x[5]); x[6] = fmaf(st.g.z, c1.z, x[6]); x[7] = fmaf(st.g.z, c1.w, x[7]);
      uint32_t h[4], l[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        split_hi_lo(x[2 * e], x[2 * e + 1], h[e], l[e]);
        const uint32_t m = pair_mask_word(field, k0 + e);
        h[e] &= m; l[e] &= m;
      }
      const uint32_t o = sw_off(c, (uint32_t)(c.part >> 1), (uint32_t)((c.part & 1) * 4 + j));
      st_shared_v4(c.a_img + o, h[0], h[1], h[2], h[3]);
      st_shared_v4(c.a_img + kABytes + o, l[0], l[1], l[2], l[3]);
    }
  }

  // the store warp: delta tile images (hi from A[0], lo from A[1]) -> scratch, read back by wgrad
  __device__ static void store_tile(const Params& p, const TileCtx& c, int l) {
    const int64_t T = p.num_tiles;
    const uint64_t pol = l2_policy_evict_first();
    const uint32_t bytes = l == -1 ? 32768u : 65536u;
    const size_t off = delta_tensor_off(l + 1, T) + (size_t)c.tile * bytes;   // l = -1: delta_c1 (tensor 0)
    tma_bulk_s2g_hint(p.dscr + off, c.a_img, bytes, pol);
    tma_bulk_s2g_hint(p.dscr + kDeltaTileBytes * (size_t)T + off, c.a_img + kABytes, bytes, pol);
  }

  __device__ static void layer(const Params&, State& st, const TileCtx& c, int l) {
    const int bl = l + 1;
    const int cbase = c.part * 64;
#pragma unroll 1
    for (int q = 0; q < 4; ++q) {
      const int col0 = cbase + q * 16;
      uint32_t a[16];
      tmem_ld16(c.t_lane + col0, a);
      tmem_ld_wait();
      const uint32_t field = ((q & 2) ? st.mask.y : st.mask.x) >> (16 * (q & 1)) & 0xFFFFu;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(a[8 * j + e]);
        if (bl == 2) {   // + d_sigma * w_sigma (the sigma head reads h7)
          const float4 s0 = head_ld4(c, (uint32_t)(col0 + 8 * j)), s1 = head_ld4(c, (uint32_t)(col0 + 8 * j + 4));
          x[0] = fmaf(st.g.w, s0.x, x[0]); x[1] = fmaf(st.g.w, s0.y, x[1]); x[2] = fmaf(st.g.w, s0.z, x[2]); x[3] = fmaf(st.g.w, s0.w, x[3]);
          x[4] = fmaf(st.g.w, s1.x, x[4]); x[5] = fmaf(st.g.w, s1.y, x[5]); x[6] = fmaf(st.g.w, s1.z, x[6]); x[7] = fmaf(st.g.w, s1.w, x[7]);
        }
        uint32_t h[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          split_hi_lo(x[2 * e], x[2 * e + 1], h[e], lo[e]);
          if (bl >= 2) {   // bl=1 yields delta_g: layers_2 has no activation
            const uint32_t m = pair_mask_word(field, 4 * j + e);
            h[e] &= m; lo[e] &= m;
          }
        }
        const uint32_t o = sw_off(c, (uint32_t)c.part, (uint32_t)(2 * q + j));
        st_shared_v4(c.a_img + o, h[0], h[1], h[2], h[3]);
        st_shared_v4(c.a_img + kABytes + o, lo[0], lo[1], lo[2], lo[3]);
      }
    }
  }
};
