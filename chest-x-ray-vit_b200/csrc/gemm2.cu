// CTA-pair (cta_group::2) persistent bf16 GEMM for sm_100a — the main dense-contraction kernel.
//
// One cluster of two CTAs (two SMs of a TPC) owns a 256×BN output tile: each CTA stages its own
// 128 rows of A and HALF of the B tile (BN/2 rows) with TMA, the leader CTA issues
// tcgen05.mma.cta_group::2 (M = 256) which reads both CTAs' shared memory, and each CTA ends up with
// its 128 accumulator rows in its own TMEM.  Compared with the single-CTA kernel in gemm.cu this
// halves the B traffic from L2 and the B reads from shared memory per FLOP.
//
//   warp 0        TMA producer: A half + B half per 64-wide K block into a ring of stages; both CTAs'
//                 loads complete on the LEADER's full barrier
//   warp 1        TMEM allocation (both CTAs); in the leader it issues the MMAs and commits to the
//                 stage-empty barriers (multicast to both CTAs) and the accumulator-full barriers
//   (all 32 lanes of warps 0/1 run the loops so addresses stay in uniform registers, and the issuing
//   instructions sit under elect.sync — ptxas then emits back-to-back UTMALDG / UTCHMMA; under a lane-id
//   test it wraps each of them in an elect/broadcast/retry loop and the MMA-issue warp, not the tensor
//   pipe, paces the main loop: 670 instead of ≈500 cycles per K block)
//   (epilogue warp w may only touch TMEM lanes 32·(w%4)…: quadrant = warp id % 4)
//   warps 2..9    (2..17 in the 16-epilogue-warp instantiation used for fc1 + GELU, template parameter EW)
//                 epilogue: TMEM → registers (one row per thread) → fused math → [32 rows × 64 B] slab in
//                 swizzled smem → TMA store (TMA reduce-add for split-K wgrad); outputs cross smem exactly
//                 twice; residual / multiplier tiles are read two chunks ahead with coalesced loads and
//                 transposed through a spare slab.
//   accumulators  double-buffered in TMEM (2×BN columns) so the epilogue of tile i overlaps the MMAs
//                 of tile i+1.
//   schedule      static round-robin over the pairs; a 256-wide launch may mix 256- and 128-column tiles
//                 (n_full / n_half per 256-row band, full tiles first) so that every pair gets equal work.
//   instantiations  <BN, A_MN, B_MN, AUX, EW, EPI>: AUX = epilogues that read a second matrix.  Separate because the
//                 epilogue lives at the 168-register cap (10 warps → 3 per SM sub-partition); EW = 16 with a compile-time
//                 epilogue EPI lives at 96 (18 warps → 5 on one sub-partition).
// Diagnostics: in builds with -DVITK_GEMM_STAMPS=1, clock stamps per K block / tile / CTA / launch
// (tools/gemm_timeline.py).
#include <cuda.h>

#include <mutex>

#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "sm100_prims.cuh"
#include "tmap.cuh"

namespace vitk {

constexpr int k2BM = 128;            // rows per CTA (256 per pair)
constexpr int k2BK = 64;
constexpr int k2FirstEpiWarp = 2;
// Epilogue warps per CTA (template parameter EW): 8 by default (two per TMEM lane quadrant, each draining half of the
// tile's columns), 16 for the GELU instantiation (four per quadrant, a quarter of the columns each): its epilogue is a
// chain of dependent latencies (TMEM load → 2 MUFU + 13 FP32 per element → pack → shared memory → fence → TMA store)
// that four warps per scheduler hide better than two.
constexpr int threads2(int ew) { return (k2FirstEpiWarp + ew) * 32; }
constexpr int k2ABytes = k2BM * k2BK * 2;                       // 16 KB
// [32 rows × 64 B] slabs per epilogue warp (TMA stores in flight): 2 and 4 measured equal (the epilogue is not waiting
// on its TMA stores)
constexpr int k2Slabs = 2;
constexpr int k2SlabBytes = k2Slabs * 2048;
constexpr int staging_bytes2(int ew) { return ew * k2SlabBytes; }  // 32 KB (8 warps) / 64 KB (16 warps)
constexpr int k2MaxSmem = 227 * 1024;
constexpr int k2BiasBytes = 2 * 2 * 128 * 4;                     // bias slice (≤128 floats) per column half × tile parity
constexpr int k2BarBytes = 256;

template <int BN, int EW = 8>
struct Cfg2 {
  static constexpr int kBHalfRows = BN / 2;
  static constexpr int kBBytes = kBHalfRows * k2BK * 2;
  static constexpr int kStageBytes = k2ABytes + kBBytes;
  // Operand bytes in flight are what hides the ≈3,200-cycle refill round trip (MMA retire → commit →
  // producer wake → TMA → L2 → complete_tx on the leader → MMA wake): measured k-block cadence ≈
  // (512 + 3200) / stages cycles, so every stage that fits in the 227 KB is used.
  // 4, 5 and 6 stages at BN = 256 / 192 measured equal: the K-block cadence is a throughput limit, not a latency one.
  static constexpr int kStagingBytes = staging_bytes2(EW);
  static constexpr int kWantStages = (BN == 256 || BN == 192) ? 6 : 8;
  static constexpr int kFitStages = (k2MaxSmem - kStagingBytes - k2BiasBytes - k2BarBytes) / kStageBytes;
  static constexpr int kStages = kWantStages < kFitStages ? kWantStages : kFitStages;   // 16 epilogue warps: 5 stages at BN = 256 / 192
  static constexpr int kTmemCols = (2 * BN <= 256) ? 256 : 512;
  static constexpr int kSmemBytes = kStages * kStageBytes + kStagingBytes + k2BiasBytes + k2BarBytes;   // no slack: smem_raw is declared 1024-aligned
};

struct Gemm2Params {
  int M, N, K;
  int n_tiles, mn_tiles, k_splits, kb_per_split, kb_total, total_work;
  int n_full, n_half;  // every 256-row band is cut into n_full tiles of BN columns followed by n_half tiles of BN/2 columns
                       // (n_tiles = n_full + n_half); all full tiles come first in the work order
  int epi;
  int has_d2;
  const void* aux;
  long long ld_aux;
  const float* bias;
  int tl_seq;         // launch number since the timeline buffer was set: [7100 + 4·seq + {0,1,2,3}] = min entry, min start,
                      // max end, max exit globaltimer over the CTAs of that launch (slots pre-set by the tool to ±inf)
  long long* tl;      // vitk_debug_timeline buffer (nullptr in production): the leader CTA of pair 0 stamps clock64() per
                      // K block [4i]: producer passed the stage-empty wait, [4i+1]: MMA warp passed the stage-full wait,
                      // [4i+2]: MMAs + commit issued; per tile [4096+4t]: epilogue warp 2 passed acc_full, [+1]: tile drained;
                      // [6000+2c], [6001+2c]: globaltimer (ns) when CTA c starts working / has finished
};
extern long long* g_timeline;
extern int g_timeline_seq;

struct Work2 {
  int m_blk, n0, bn, kb_begin, kb_end;   // n0: first output column, bn: tile width (BN or BN/2)
};
template <int BN>
__device__ __forceinline__ Work2 decode_work2(const Gemm2Params& p, int w) {
  const int ks = w / p.mn_tiles;
  const int t = w - ks * p.mn_tiles;
  Work2 it;
  const int full_items = (p.mn_tiles / p.n_tiles) * p.n_full;
  if (t < full_items) {
    it.m_blk = t / p.n_full;
    it.n0 = (t - it.m_blk * p.n_full) * BN;
    it.bn = BN;
  } else {
    const int th = t - full_items;
    it.m_blk = th / p.n_half;
    it.n0 = p.n_full * BN + (th - it.m_blk * p.n_half) * (BN / 2);
    it.bn = BN / 2;
  }
  it.kb_begin = ks * p.kb_per_split;
  it.kb_end = min(it.kb_begin + p.kb_per_split, p.kb_total);
  return it;
}

// ------------------------------------------------------------------------- slab addressing
// bf16 slab: 32 rows × 64 B, 64-byte swizzle (16-byte chunk j of row r lives at chunk j ^ ((r>>1)&3))
__device__ __forceinline__ uint32_t slab16_off(int r, int j) { return r * 64 + ((j ^ ((r >> 1) & 3)) << 4); }
// f32 slab: 32 rows × 128 B, 128-byte swizzle (chunk j of row r lives at chunk j ^ (r&7))
__device__ __forceinline__ uint32_t slab32_off(int r, int j) { return r * 128 + ((j ^ (r & 7)) << 4); }

__device__ __forceinline__ void st_slab16(uint8_t* slab, int r, const float (&v)[32]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint4 q;
    q.x = pack_bf16x2(v[8 * j + 0], v[8 * j + 1]);
    q.y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
    q.z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]);
    q.w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
    *reinterpret_cast<uint4*>(slab + slab16_off(r, j)) = q;
  }
}
__device__ __forceinline__ void ld_slab16(const uint8_t* slab, int r, float (&a)[32]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint4 q = *reinterpret_cast<const uint4*>(slab + slab16_off(r, j));
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
      a[8 * j + 2 * i] = f.x;
      a[8 * j + 2 * i + 1] = f.y;
    }
  }
}
__device__ __forceinline__ void st_slab32(uint8_t* slab, int r, const float (&v)[32]) {
#pragma unroll
  for (int j = 0; j < 8; ++j)
    *reinterpret_cast<float4*>(slab + slab32_off(r, j)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
__device__ __forceinline__ void add_slab32(const uint8_t* slab, int r, float (&v)[32]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 a = *reinterpret_cast<const float4*>(slab + slab32_off(r, j));
    v[4 * j] += a.x; v[4 * j + 1] += a.y; v[4 * j + 2] += a.z; v[4 * j + 3] += a.w;
  }
}

__device__ __forceinline__ void add_bias32(const float* __restrict__ bias, int col0, float (&v)[32]) {
  const float4* b4 = reinterpret_cast<const float4*>(bias + col0);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 b = __ldg(b4 + i);
    v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
  }
}

// AUX: instantiation for the epilogues that read a residual / multiplier tile (BIAS_RESID_F32, MUL_BF16, DGELU_BF16).
// Two instantiations because the epilogue sits at the 168-register cap (10 warps, 3 per SM sub-partition): the
// aux look-ahead registers and the GELU temporaries never coexist, and with both in one kernel ptxas spilled the
// prefetched bias across the accumulator wait — i.e. stalled on that load once per tile.
// EW: epilogue warps (8 or 16).  EPI: compile-time epilogue (−1: taken from Gemm2Params at run time) — 18 warps put
// five on one SM sub-partition, i.e. a 96-register cap, which only a single epilogue's code fits.
template <int BN, bool A_MN, bool B_MN, bool AUX, int EW = 8, int EPI = -1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(threads2(EW), 1)
gemm2_bf16_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                  const __grid_constant__ CUtensorMap tma_bh,   // K-major B, box of BN/4 rows (half-width tiles)
                  const __grid_constant__ CUtensorMap tma_d, const __grid_constant__ CUtensorMap tma_d2,
                  const Gemm2Params p) {
  // Timeline stamps are compiled in only for the diagnostic build (tools/build_variants.sh stamps "-DVITK_GEMM_STAMPS=1",
  // selected with VITK_LIB): in the production kernel they would cost registers the epilogue does not have.
#ifndef VITK_GEMM_STAMPS
#define VITK_GEMM_STAMPS 0
#endif
  constexpr bool kStamps = VITK_GEMM_STAMPS != 0;
  using Cfg = Cfg2<BN, EW>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kBHalf = Cfg::kBHalfRows;
  constexpr int kParts = EW / 4;                 // column parts of a tile, one per group of four (quadrant) warps
  constexpr int kBiasPart = 256 / kParts;        // bias floats per part and tile parity
  constexpr int k2StagingBytes = Cfg::kStagingBytes;
  static_assert(EW == 8 || EW == 16, "epilogue warps: two or four per TMEM lane quadrant");
  if (kStamps && p.tl != nullptr && threadIdx.x == 0) {   // debug timeline: [6400 + cta] = globaltimer at kernel entry
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.tl[6400 + blockIdx.x] = static_cast<long long>(t);
    if (p.tl_seq < 200) atomicMin(reinterpret_cast<unsigned long long*>(p.tl + 7100 + 4 * p.tl_seq), t);
  }
  extern __shared__ __align__(1024) uint8_t smem_raw[];   // 128-byte-swizzled operand tiles need 1024-byte alignment
  uint8_t* smem = smem_raw;
  uint8_t* staging = smem + kStages * Cfg::kStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + k2StagingBytes + k2BiasBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* acc_full = empty_bar + kStages;     // [2]
  uint64_t* acc_empty = acc_full + 2;           // [2]  (leader's copy is the one waited on)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // rank inside the CTA pair: clusters are (2,1,1), so it is the low bit of blockIdx.x.  (Reading
  // %cluster_ctarank / mapa through inline asm hides their warp-uniformity from the compiler, which then
  // wraps every TMA and MMA issue in an elect-broadcast-retry loop.)
  const uint32_t cta_rank = blockIdx.x & 1u;
  const bool leader = cta_rank == 0;
  const int pair_id = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  const bool stamp = kStamps && p.tl != nullptr && blockIdx.x == 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    if (p.n_half > 0 && !B_MN) tma_prefetch_desc(&tma_bh);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&acc_full[s], 1);
      mbar_init(&acc_empty[s], 2 * EW);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, Cfg::kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_relaxed();      // peer barriers initialised (fence.mbarrier_init above), both TMEM allocations done
  tc_fence_after_sync();
  pdl_wait();                  // the previous kernel's outputs are complete; everything above overlapped its tail
  pdl_launch_dependents();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // broadcast marks it warp-uniform: no per-MMA elect-broadcast-retry loop
  if (kStamps && p.tl != nullptr && threadIdx.x == 0) {   // debug timeline: [6000 + 2·cta] = globaltimer when this CTA starts working
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.tl[6000 + 2 * blockIdx.x] = static_cast<long long>(t);
    if (p.tl_seq < 200) atomicMin(reinterpret_cast<unsigned long long*>(p.tl + 7101 + 4 * p.tl_seq), t);
  }

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    // All lanes run the loops of the producer and MMA warps so that stage indices, addresses and
    // descriptors stay warp-uniform (uniform registers); only the issuing instructions are predicated on
    // lane 0.  Under a divergent `if (lane == 0)` the compiler wraps every TMA / MMA in an
    // elect-broadcast-retry loop.
    const bool L = lane == 0;
    // shared::cluster address of the leader's barrier: same offset with the pair's peer bit (bit 24) cleared
    const uint32_t full0_leader = smem_u32(&full_bar[0]) & 0xFEFFFFFFu;
    int stage = 0;
    uint32_t phase = 0;
    int kbi = 0;
    for (int w = pair_id; w < p.total_work; w += num_pairs) {
      const Work2 it = decode_work2<BN>(p, w);
      const int m0 = it.m_blk * (2 * k2BM) + static_cast<int>(cta_rank) * k2BM;
      const bool half = it.bn != BN;                  // half-width tile: this CTA stages BN/4 rows of B
      const int n0 = it.n0 + static_cast<int>(cta_rank) * (it.bn >> 1);
      const uint32_t stage_tx = 2 * (k2ABytes + (half ? Cfg::kBBytes / 2 : Cfg::kBBytes));
      const int kb_begin = it.kb_begin, kb_end = it.kb_end;
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (stamp && L && kbi < 1024) p.tl[4 * kbi] = clock64();
        ++kbi;
        uint8_t* sa = smem + stage * Cfg::kStageBytes;
        uint8_t* sb = sa + k2ABytes;
        const uint32_t bar = full0_leader + stage * 8;
        const int k0 = kb * k2BK;
        if (elect_one()) {                         // elect.sync: ptxas issues the TMA instructions straight from uniform registers
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], stage_tx);
          if (!A_MN) {
            tma_load_2d_pair(sa, &tma_a, bar, k0, m0);
          } else {
#pragma unroll
            for (int g = 0; g < k2BM / 64; ++g) tma_load_2d_pair(sa + g * 8192, &tma_a, bar, m0 + g * 64, k0);
          }
          if (!B_MN) {
            if (half) tma_load_2d_pair(sb, &tma_bh, bar, k0, n0);
            else tma_load_2d_pair(sb, &tma_b, bar, k0, n0);
          } else {
#pragma unroll
            for (int g = 0; g < kBHalf / 64; ++g)
              if (!half || g < kBHalf / 128) tma_load_2d_pair(sb + g * 8192, &tma_b, bar, n0 + g * 64, k0);
          }
        }
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (leader) {
      const bool L = lane == 0;
      constexpr uint32_t idesc_full = umma_idesc_bf16(2 * k2BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      constexpr uint32_t idesc_half = umma_idesc_bf16(2 * k2BM, BN / 2, A_MN ? 1 : 0, B_MN ? 1 : 0);
      constexpr uint32_t a_lbo = A_MN ? 8192u : 0u, b_lbo = B_MN ? 8192u : 0u;
      constexpr uint32_t a_kstep = (A_MN ? 2048u : 32u) >> 4, b_kstep = (B_MN ? 2048u : 32u) >> 4;   // 16-byte units
      const uint64_t a_desc0 = umma_smem_desc(smem_u32(smem), a_lbo, 1024);
      const uint64_t b_desc0 = umma_smem_desc(smem_u32(smem + k2ABytes), b_lbo, 1024);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int kbi = 0;
      int tiles_done = 0;
      for (int w = pair_id; w < p.total_work; w += num_pairs) {
        const Work2 it = decode_work2<BN>(p, w);
        const int kb_begin = it.kb_begin, kb_end = it.kb_end;
        const uint32_t idesc = it.bn == BN ? idesc_full : idesc_half;
        mbar_wait(&acc_empty[acc], acc_phase ^ 1);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after_sync();
          if (stamp && L && kbi < 1024) p.tl[4 * kbi + 1] = clock64();
          const uint64_t soff = static_cast<uint64_t>(stage * (Cfg::kStageBytes >> 4));
          // elect.sync (not `lane == 0`) tells ptxas that exactly one lane issues: it then emits four back-to-back
          // predicated UTCHMMAs on uniform registers.  Under a lane-id branch every MMA is wrapped in an
          // elect/broadcast/retry loop whose latency (≈110 cycles per MMA, 670 per K block) — not the tensor pipe
          // (512) — paced the main loop, for N = 128 and N = 256 alike.
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < k2BK / 16; ++k)
              tc_mma_bf16_pair(d_tmem, a_desc0 + soff + k * a_kstep, b_desc0 + soff + k * b_kstep, idesc,
                               (kb > kb_begin || k > 0) ? 1u : 0u);
            tc_commit_pair(&empty_bar[stage], 3);                         // both CTAs' producers may refill
            if (kb == kb_end - 1) tc_commit_pair(&acc_full[acc], 3);   // both CTAs' epilogues may drain
          }
          if (stamp && L && kbi < 1024) p.tl[4 * kbi + 2] = clock64();
          ++kbi;
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
        ++tiles_done;
      }
      // Teardown guard: the peer CTA's epilogue warps release accumulators with REMOTE arrives on this CTA's
      // acc_empty barriers.  Wait until the last release of each buffer has landed, so that no arrive can still be
      // in flight towards this CTA's shared memory when it exits (the final cluster barrier is execution-only).
#pragma unroll
      for (int bsel = 0; bsel < 2; ++bsel) {
        const int uses = (tiles_done + 1 - bsel) >> 1;          // tiles that used accumulator buffer bsel
        if (uses > 0) mbar_wait(&acc_empty[bsel], (uses - 1) & 1);
      }
    }
    __syncwarp();
  } else if (warp >= k2FirstEpiWarp) {
    // ------------------------------------------------------------------ epilogue (both CTAs)
    // Thread = one accumulator row (TMEM lane).  A chunk is 64 bytes of output per row (32 bf16 or
    // 16 fp32 columns): registers → [32 rows × 64 B] slab in 64-byte-swizzled smem → one TMA store
    // (TMA reduce-add for split-K wgrad), two chunks in flight per warp.  Residual / multiplier tiles
    // are read two chunks ahead with coalesced 128-bit loads (registers) and transposed through a
    // third slab, so the SM's TMA queue carries only operand loads and output stores.
    const int ew = warp - k2FirstEpiWarp;
    const int quad = warp & 3;                // TMEM lane quadrant (= warp id % 4)
    const int part = ew >> 2;                 // which column part of the tile this warp drains
    uint8_t* slabs = staging + ew * k2SlabBytes;            // 2 × 2 KB
    float* bias_base = reinterpret_cast<float*>(staging + k2StagingBytes) + part * (2 * kBiasPart);   // [tile parity][kBiasPart], shared by the 4 warps of this column part
    const int epi = EPI >= 0 ? EPI : p.epi;
    const bool out_f32 = epi == VITK_EPI_BIAS_RESID_F32 || epi == VITK_EPI_ACCUM_F32 || epi == VITK_EPI_STORE_F32;
    const bool has_aux = AUX && (epi == VITK_EPI_BIAS_RESID_F32 || epi == VITK_EPI_MUL_BF16 || epi == VITK_EPI_DGELU_BF16);
    const bool has_bias = p.bias != nullptr && (epi == VITK_EPI_BIAS_BF16 || epi == VITK_EPI_BIAS_GELU_BF16 ||
                                                epi == VITK_EPI_BIAS_GELUG_BF16 || epi == VITK_EPI_BIAS_RESID_F32);
    const int cw = out_f32 ? 16 : 32;                      // chunk width in columns
    const int cshift = out_f32 ? 4 : 5;                    // log2(cw)
    const int nout = has_aux ? k2Slabs - 1 : k2Slabs;      // output slabs in the ring (the last slab transposes aux)
    const int aux_esize = out_f32 ? 4 : 2;
    const uint32_t acc_empty_leader = smem_u32(&acc_empty[0]) & 0xFEFFFFFFu;
    int acc = 0;
    uint32_t acc_phase = 0;
    int oslot = 0;
    const int rc = lane >> 2, jc = lane & 3;               // coalesced layout: iteration i ↔ row 8i + rc, 16-byte chunk jc

    auto tile_row0 = [&](const Work2& it) { return it.m_blk * (2 * k2BM) + static_cast<int>(cta_rank) * k2BM + quad * 32; };
    auto tile_col0 = [&](const Work2& it) { return it.n0 + part * (it.bn / kParts); };   // this warp's column part of the tile

    uint4 axA[4], axB[4];  // aux chunks in flight (coalesced layout); named, never indexed dynamically, so they stay in registers
    auto load_aux = [&](uint4 (&dst)[4], int row0, int col) {
      const uint8_t* base = reinterpret_cast<const uint8_t*>(p.aux) +
                            (static_cast<long long>(row0) * p.ld_aux + col) * aux_esize + jc * 16;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int row = 8 * i + rc;
        dst[i] = (row0 + row < p.M) ? __ldg(reinterpret_cast<const uint4*>(base + static_cast<long long>(row) * p.ld_aux * aux_esize))
                                    : make_uint4(0, 0, 0, 0);
      }
    };
    // coordinates of the chunk `ahead` (≤ 2) chunks after chunk c of tile `cur`; `nxt` is this CTA's next tile
    // (every tile has ≥ 2 chunks per warp — aux epilogues run with 8 epilogue warps — so the look-ahead never reaches
    // past it); false when past the last tile
    auto chunk_after = [&](const Work2& cur, const Work2& nxt, bool has_next, int c, int ahead, int* row0, int* col) {
      c += ahead;
      const int nch = (cur.bn / kParts) >> cshift;
      if (c < nch) {
        *row0 = tile_row0(cur);
        *col = tile_col0(cur) + c * cw;
        return true;
      }
      if (!has_next) return false;
      *row0 = tile_row0(nxt);
      *col = tile_col0(nxt) + (c - nch) * cw;
      return true;
    };
    // stream_out: store with the L2 evict_first policy (the policy is created here, where it is used: 2 registers the
    // epilogue does not have to spare)
    auto emit = [&](const CUtensorMap* map, int col, int row0, const uint4 (&q)[4], bool stream_out = false) {
      // wait until the store issued `nout` stores ago has finished reading its slab, then reuse it
      if (elect_one()) { if (nout == k2Slabs) tma_store_wait_read<k2Slabs - 1>(); else tma_store_wait_read<k2Slabs - 2>(); }
      __syncwarp();
      uint8_t* slab = slabs + oslot * 2048;
#pragma unroll
      for (int j = 0; j < 4; ++j) *reinterpret_cast<uint4*>(slab + slab16_off(lane, j)) = q[j];
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        if (epi == VITK_EPI_ACCUM_F32) tma_reduce_add_2d(map, slab, col, row0);
        else if (stream_out) tma_store_2d_hint(map, slab, col, row0, l2_policy_evict_first());
        else tma_store_2d(map, slab, col, row0);
        tma_store_commit();
      }
      oslot = (oslot + 1 == nout) ? 0 : oslot + 1;
    };
    auto pack4 = [&](const float* v, uint4 (&q)[4]) {      // 32 floats → 4×16 B of bf16
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        q[j].x = pack_bf16x2(v[8 * j + 0], v[8 * j + 1]);
        q[j].y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
        q[j].z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]);
        q[j].w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
      }
    };

    int w = pair_id;
    int ti = 0;
    Work2 it = decode_work2<BN>(p, w < p.total_work ? w : 0);
    if (has_aux && w < p.total_work) {
      int r0, cc;
      if (chunk_after(it, it, false, 0, 0, &r0, &cc)) load_aux(axA, r0, cc);
      if (chunk_after(it, it, false, 0, 1, &r0, &cc)) load_aux(axB, r0, cc);
    }
    int axi = 0;   // 0: axA holds the current chunk's aux, 1: axB
    for (; w < p.total_work; w += num_pairs) {
      const bool has_next = w + num_pairs < p.total_work;
      const Work2 nxt = decode_work2<BN>(p, has_next ? w + num_pairs : w);
      const int row0 = tile_row0(it), col0 = tile_col0(it);
      const int half_w = it.bn / kParts;                   // columns of this tile that belong to this warp's column part
      const int nchunks = half_w >> cshift;
      // This column half's BN/2 bias values: fetched before the wait, published to smem after it.  The slice is
      // shared by the 4 quadrant warps (identical values) and double-buffered by tile parity; a warp past
      // acc_full(t) knows every warp finished READING the bias of tile t−2, because those reads precede the
      // acc_empty(t−2) arrivals that MMA(t) waited for.
      float* bias_s = bias_base + acc * kBiasPart;
      constexpr int kBiasIters = kBiasPart / 32;
      float bpre[kBiasIters];
      if (has_bias) {
#pragma unroll
        for (int i = 0; i < kBiasIters; ++i) bpre[i] = (lane + 32 * i < half_w) ? __ldg(p.bias + col0 + lane + 32 * i) : 0.f;
      }
      mbar_wait(&acc_full[acc], acc_phase);
      tc_fence_after_sync();
      if (stamp && ew == 0 && lane == 0 && ti < 256) p.tl[4096 + 4 * ti] = clock64();
      if (has_bias) {
#pragma unroll
        for (int i = 0; i < kBiasIters; ++i)
          if (lane + 32 * i < half_w) bias_s[lane + 32 * i] = bpre[i];
        __syncwarp();
      }
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * BN + part * half_w;
#pragma unroll 1
      for (int c = 0; c < nchunks; ++c) {
        const int col = col0 + c * cw;
        uint32_t r[32];
        if (out_f32) {
          uint32_t r16[16];
          tmem_ld_32x16(t_row + c * 16, r16);
#pragma unroll
          for (int i = 0; i < 16; ++i) r[i] = r16[i];
        } else {
          tmem_ld_32x32(t_row + c * 32, r);
        }
        uint4 arow[4] = {};  // this thread's row of the aux chunk (64 B)
        if (has_aux) {
          uint8_t* tslab = slabs + (k2Slabs - 1) * 2048;
          if (axi == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(tslab + slab16_off(8 * i + rc, jc)) = axA[i];
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(tslab + slab16_off(8 * i + rc, jc)) = axB[i];
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) arow[j] = *reinterpret_cast<const uint4*>(tslab + slab16_off(lane, j));
          __syncwarp();
          int r0, cc;
          if (chunk_after(it, nxt, has_next, c, 2, &r0, &cc)) {   // refill the registers just consumed
            if (axi == 0) load_aux(axA, r0, cc); else load_aux(axB, r0, cc);
          }
          axi ^= 1;
        }
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
        if (has_bias) {
          const float4* b4 = reinterpret_cast<const float4*>(bias_s + c * cw);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (i < 4 || !out_f32) {
              const float4 b = b4[i];
              v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
            }
          }
        }
        if (c == nchunks - 1) {           // all TMEM and bias reads of this tile are done: hand the buffer back early
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(acc_empty_leader + acc * 8);
        }
        uint4 q[4];
        switch (epi) {
          case VITK_EPI_STORE_BF16:
          case VITK_EPI_BIAS_BF16:
            pack4(v, q);
            emit(&tma_d, col, row0, q);
            break;
          case VITK_EPI_BIAS_GELU_BF16:        // d = u, d2 = gelu(u)
            if constexpr (AUX) break;
            pack4(v, q);
            emit(&tma_d, col, row0, q);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = gelu_erf(v[i]);
            pack4(v, q);
            emit(&tma_d2, col, row0, q);
            break;
          case VITK_EPI_BIAS_GELUG_BF16: {     // d = gelu(u), d2 = gelu'(u) (optional)
            if constexpr (AUX) break;
            // packed as produced (two results → one bf16x2 word each), so only the packed outputs stay live
            uint4 qg[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t wa[4], wg[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float2 u2 = make_float2(v[8 * j + 2 * i], v[8 * j + 2 * i + 1]);
                const GeluParts2 g = gelu_parts2(u2);
                const float2 d = __ffma2_rn(u2, g.pdf, g.cdf);
                const float2 a = __fmul2_rn(u2, g.cdf);
                wa[i] = pack_bf16x2(a.x, a.y);
                wg[i] = pack_bf16x2(d.x, d.y);
              }
              q[j] = make_uint4(wa[0], wa[1], wa[2], wa[3]);
              qg[j] = make_uint4(wg[0], wg[1], wg[2], wg[3]);
            }
            emit(&tma_d, col, row0, q);
            // GELU' is saved for backward and not read again in this pass: evict_first keeps it from pushing gelu(u),
            // the next GEMM's operand, out of L2.  A/B on the step (profiles/r02_l2_hints_ab.txt): +0.5 %, at the edge
            // of the run-to-run noise; evict_first LOADS of the single-use multiplier / residual / LayerNorm-backward
            // inputs changed nothing and were removed.
            if (p.has_d2) emit(&tma_d2, col, row0, qg, true);
            break;
          }
          case VITK_EPI_MUL_BF16:
          case VITK_EPI_DGELU_BF16: {
            if constexpr (!AUX) break;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t wv[4] = {arow[j].x, arow[j].y, arow[j].z, arow[j].w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&wv[i]));
                v[8 * j + 2 * i] *= (epi == VITK_EPI_MUL_BF16) ? f.x : gelu_erf_grad(f.x);
                v[8 * j + 2 * i + 1] *= (epi == VITK_EPI_MUL_BF16) ? f.y : gelu_erf_grad(f.y);
              }
            }
            pack4(v, q);
            emit(&tma_d, col, row0, q);
            break;
          }
          case VITK_EPI_BIAS_RESID_F32:
            if constexpr (!AUX) break;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              q[j].x = __float_as_uint(v[4 * j] + __uint_as_float(arow[j].x));
              q[j].y = __float_as_uint(v[4 * j + 1] + __uint_as_float(arow[j].y));
              q[j].z = __float_as_uint(v[4 * j + 2] + __uint_as_float(arow[j].z));
              q[j].w = __float_as_uint(v[4 * j + 3] + __uint_as_float(arow[j].w));
            }
            emit(&tma_d, col, row0, q);
            break;
          default:  // VITK_EPI_ACCUM_F32, VITK_EPI_STORE_F32
#pragma unroll
            for (int j = 0; j < 4; ++j)
              q[j] = make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]),
                                __float_as_uint(v[4 * j + 3]));
            emit(&tma_d, col, row0, q);
            break;
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
      if (stamp && ew == 0 && lane == 0 && ti < 256) p.tl[4096 + 4 * ti + 1] = clock64();
      ++ti;
      it = nxt;
    }
    if (elect_one()) tma_store_wait_all<0>();   // smem must outlive the bulk reads; writes complete before exit
  }
  __syncwarp();

  tc_fence_before_sync();
  __syncthreads();
  if (kStamps && p.tl != nullptr && threadIdx.x == 0) {   // [6001 + 2·cta] = globaltimer when all of this CTA's warps are done
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.tl[6001 + 2 * blockIdx.x] = static_cast<long long>(t);
    if (p.tl_seq < 200) atomicMax(reinterpret_cast<unsigned long long*>(p.tl + 7102 + 4 * p.tl_seq), t);
  }
  cluster_sync_relaxed();   // neither CTA may free TMEM / exit while the peer can still reach it
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
    if (kStamps && p.tl != nullptr && lane == 0) {        // [6600 + cta] = globaltimer after the TMEM hand-back, right before exit
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      p.tl[6600 + blockIdx.x] = static_cast<long long>(t);
      if (p.tl_seq < 200) atomicMax(reinterpret_cast<unsigned long long*>(p.tl + 7103 + 4 * p.tl_seq), t);
    }
  }
}

// ------------------------------------------------------------------------- host side
// [32 rows × 64 B] output boxes (32 bf16 or 16 fp32 columns), 64-byte swizzle
static int out_map(CUtensorMap* m, const void* base, bool f32, long long rows, long long cols, long long ld) {
  const uint64_t dims[2] = {static_cast<uint64_t>(cols), static_cast<uint64_t>(rows)};
  const uint64_t str[1] = {static_cast<uint64_t>(ld) * (f32 ? 4 : 2)};
  const uint32_t box[2] = {f32 ? 16u : 32u, 32u};
  return get_tensor_map(m, base, f32 ? TM_F32 : TM_BF16, 2, dims, str, box, TM_SW64);
}

template <int BN, bool A_MN, bool B_MN, bool AUX, int EW = 8, int EPI = -1>
static int launch_gemm2(const vitk_gemm_args& a, const Gemm2Params& p, int pairs, cudaStream_t stream) {
  using Cfg = Cfg2<BN, EW>;
  CUtensorMap ta, tb, tbh, td, td2;
  {
    uint64_t dims[2], str[1];
    uint32_t box[2];
    if (!A_MN) { dims[0] = a.K; dims[1] = a.M; box[0] = k2BK; box[1] = k2BM; }
    else       { dims[0] = a.M; dims[1] = a.K; box[0] = 64;   box[1] = k2BK; }
    str[0] = static_cast<uint64_t>(a.lda) * 2;
    if (int rc = make_tensor_map_bf16(&ta, a.a, 2, dims, str, box)) return rc;
    if (!B_MN) { dims[0] = a.K; dims[1] = a.N; box[0] = k2BK; box[1] = Cfg::kBHalfRows; }
    else       { dims[0] = a.N; dims[1] = a.K; box[0] = 64;   box[1] = k2BK; }
    str[0] = static_cast<uint64_t>(a.ldb) * 2;
    if (int rc = make_tensor_map_bf16(&tb, a.b, 2, dims, str, box)) return rc;
    tbh = tb;
    if (!B_MN && p.n_half > 0) {       // half-width tiles stage BN/4 rows of a K-major B per CTA
      box[1] = Cfg::kBHalfRows / 2;
      if (int rc = make_tensor_map_bf16(&tbh, a.b, 2, dims, str, box)) return rc;
    }
  }
  const bool f32_out = a.epilogue == VITK_EPI_BIAS_RESID_F32 || a.epilogue == VITK_EPI_ACCUM_F32 || a.epilogue == VITK_EPI_STORE_F32;
  if (int rc = out_map(&td, a.d, f32_out, a.M, a.N, a.ldd)) return rc;
  td2 = td;
  if (a.d2 != nullptr) { if (int rc = out_map(&td2, a.d2, false, a.M, a.N, a.ldd)) return rc; }
  auto kern = gemm2_bf16_kernel<BN, A_MN, B_MN, AUX, EW, EPI>;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [&] {
    attr_err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
  });
  if (attr_err != cudaSuccess) return cuda_error(attr_err, "cudaFuncSetAttribute(gemm2 smem)");
  if (cudaError_t e = launch_pdl(kern, dim3(2 * pairs), dim3(threads2(EW)), Cfg::kSmemBytes, stream, ta, tb, tbh, td, td2, p); e != cudaSuccess)
    return cuda_error(e, "gemm2_bf16_kernel launch");
  VITK_LAUNCH_CHECK("gemm2_bf16_kernel");
  return 0;
}

template <int BN, bool AUX>
static int dispatch_major2(const vitk_gemm_args& a, const Gemm2Params& p, int pairs, cudaStream_t s) {
  if (!a.a_mn_major && !a.b_mn_major) return launch_gemm2<BN, false, false, AUX>(a, p, pairs, s);
  if constexpr (!AUX) {          // wgrad layouts (MN-major A) never carry an aux tile
    if (a.a_mn_major && !a.b_mn_major) return launch_gemm2<BN, true, false, false>(a, p, pairs, s);
  }
  if constexpr (BN != 192) {     // an MN-major B half must be whole 64-column TMA boxes
    if (!a.a_mn_major && a.b_mn_major) return launch_gemm2<BN, false, true, AUX>(a, p, pairs, s);
    if constexpr (!AUX) return launch_gemm2<BN, true, true, false>(a, p, pairs, s);
  }
  return set_error(VITK_EINVAL, "gemm2: unsupported operand layout for this tile width / epilogue (tile_n 192 needs a K-major B; "
                                "aux epilogues need a K-major A)");
}

// fc1 forward (+bias, GELU, optional GELU') as a 16-epilogue-warp instantiation with the epilogue fixed at compile time
// (see the kernel's template comment): 2 MUFU + 13 FP32 operations per element are a chain of dependent latencies that
// four warps per scheduler hide better than two — 51.4 → 47.1 µs at M = 9232 (profiles/r02_bench_gemm_ew16.txt), bit-identical
// output (tests/test_gpu_gemm.py::test_sixteen_warp_epilogues_equal_eight_warp).  The same treatment of the multiplier
// and fp32-residual epilogues was measured and dropped: those launches move 128 / 71 MB for 43.6 / 10.9 GF and sit on
// the HBM side of the roofline, not on the epilogue's instruction latency (no change at 49.2 / 28.7 / 47.1 µs).
// Variant 3 keeps the 8-warp instantiation (the reference the 16-warp one is tested against).
static bool launch_heavy2(const vitk_gemm_args& a, const Gemm2Params& p, int bn, int pairs, cudaStream_t s, int* rc) {
  if (a.variant == 3) return false;
  if (a.epilogue == VITK_EPI_BIAS_GELUG_BF16 && !a.a_mn_major && !a.b_mn_major && bn == 256) {
    *rc = launch_gemm2<256, false, false, false, 16, VITK_EPI_BIAS_GELUG_BF16>(a, p, pairs, s);
    return true;
  }
  return false;
}

// cycles a CTA pair spends per 64-wide K block of a tile of `bn` columns (tools/gemm_timeline.py, B200): the MMAs of a
// 256-wide tile occupy the tensor pipe for 4 × 122 cycles; narrower tiles are bound by operand delivery instead.
// 192: A/B on the full step, 440 (192-wide tiles for K-major N = 768) beats 500 (mixed 256+128 there) by 0.9 %.
static double kblock_cycles(int bn) { return bn == 256 ? 500.0 : (bn == 192 ? 440.0 : 390.0); }
constexpr double kTileFixedCycles = 1500.0;   // accumulator hand-over + pipeline refill per tile

static void choose_tiling2(const vitk_gemm_args& a, int pairs, int* bn_out, int* splits_out, int* n_half_out,
                           double* cost_out = nullptr) {
  const long long mt = (a.M + 2 * k2BM - 1) / (2 * k2BM);
  const long long kb_total = (a.K + k2BK - 1) / k2BK;
  double best = 1e30;
  const int cands[3] = {256, 192, 128};
  for (int bn : cands) {
    if (a.N % bn) continue;
    if (a.b_mn_major && bn == 192) continue;
    if (a.tile_n && a.tile_n != bn) continue;
    const long long tiles = mt * (a.N / bn);
    int splits = 1;
    if (a.epilogue == VITK_EPI_ACCUM_F32) {
      if (a.split_k > 0) splits = a.split_k;
      else if (tiles < pairs) {
        splits = static_cast<int>(pairs / tiles);
        const long long cap = kb_total / 4 > 0 ? kb_total / 4 : 1;
        if (splits > cap) splits = static_cast<int>(cap);
        if (splits < 1) splits = 1;
      }
    }
    const long long kb_per = (kb_total + splits - 1) / splits;
    const long long items = tiles * ((kb_total + kb_per - 1) / kb_per);
    const long long waves = (items + pairs - 1) / pairs;
    const double cost = static_cast<double>(waves) * (kb_per * kblock_cycles(bn) + kTileFixedCycles);
    if (cost < best - 1e-9) { best = cost; *bn_out = bn; *splits_out = splits; *n_half_out = 0; }
    // Mixed widths (BN = 256 only): replace some of each band's 256-column tiles by pairs of 128-column tiles so that
    // the static round-robin order gives every CTA pair the same amount of work (e.g. N = 768 on 74 pairs: 3 full
    // tiles per band = 1.5 waves of full tiles; 2 full + 2 half = one full and one half tile for every pair).
    if (bn == 256 && splits == 1 && a.epilogue != VITK_EPI_ACCUM_F32 && a.tile_n == 0) {
      const int n_tiles256 = static_cast<int>(a.N / 256);
      const double cf = kb_total * kblock_cycles(256) + kTileFixedCycles, ch = kb_total * kblock_cycles(128) + kTileFixedCycles;
      for (int nh = 2; nh <= 2 * n_tiles256; nh += 2) {
        const int nf = n_tiles256 - nh / 2;
        const long long full_items = mt * nf, all_items = mt * (nf + nh);
        double worst = 0;
        for (int pr = 0; pr < pairs && pr < all_items; ++pr) {
          double c = 0;
          for (long long w = pr; w < all_items; w += pairs) c += w < full_items ? cf : ch;
          if (c > worst) worst = c;
        }
        if (worst < best - 1e-9) { best = worst; *bn_out = 256; *splits_out = 1; *n_half_out = nh; }
      }
    }
  }
  if (cost_out) *cost_out = best;
}

// Data-gradient GEMMs (K-major A, MN-major B, plain bf16 store) whose M is ragged against the pair kernel's 256-row bands
// can quantise badly on 74 pairs yet perfectly on 148 single CTAs with 128-row bands — ViT-L at batch 8: M = 4616 → 19
// bands × 4 tiles of 256 columns = 76 tiles (two pairs get a second tile) against 37 × 4 = 148 tiles = exactly one wave.
// Measured there (tools/bench_gemm.py, VITK_BG_M=4616 VITK_BG_D=1024 VITK_BG_F=4096): fc1 dgrad 43.2 → 35.7 µs,
// qkv dgrad 35.8 → 28.8 µs, out dgrad 19.5 → 16.5 µs.  Per K block a single CTA (which stages the whole B tile itself)
// costs ≈ 1.1 × the pair kernel's 256-wide block for this operand layout.
static bool single_cta_wins(const vitk_gemm_args& a, double pair_cost, int sms) {
  if (a.variant != 0 || a.tile_n != 0 || a.max_ctas != 0 || a.a_mn_major || !a.b_mn_major || a.epilogue != VITK_EPI_STORE_BF16 ||
      a.N % 256 != 0)
    return false;
  const long long tiles = ((a.M + 127) / 128) * (a.N / 256);
  const long long waves = (tiles + sms - 1) / sms;
  const long long kb = (a.K + k2BK - 1) / k2BK;
  const double cost = static_cast<double>(waves) * (kb * 1.1 * kblock_cycles(256) + kTileFixedCycles);
  return cost < 0.9 * pair_cost;
}

// Called by vitk_gemm_bf16 (gemm.cu) after argument validation.  Returns VITK_EINVAL-free 1 when the
// problem is not eligible for the pair kernel so that the caller falls through to the 1-CTA kernel.
int gemm2_try_launch(const vitk_gemm_args& a, cudaStream_t stream, bool* handled) {
  *handled = false;
  if (a.variant == 1) return 0;
  const bool aux_epi = a.epilogue == VITK_EPI_BIAS_RESID_F32 || a.epilogue == VITK_EPI_MUL_BF16 || a.epilogue == VITK_EPI_DGELU_BF16;
  const bool eligible = a.epilogue != VITK_EPI_PATCH_F32 && a.epilogue != VITK_EPI_UNPATCH_F32 && a.N % 128 == 0 && (a.max_ctas == 0 || a.max_ctas >= 2) &&
                        !(aux_epi && a.a_mn_major) &&     // the aux instantiations exist for K-major A only
                        (a.tile_n == 0 || a.tile_n == 128 || a.tile_n == 192 || a.tile_n == 256) &&
                        !(a.tile_n == 192 && a.b_mn_major);
  if (!eligible) {
    VITK_REQUIRE(a.variant < 2, VITK_EINVAL, "gemm: the CTA-pair kernel does not support this problem (epilogue %d, tile_n %d)",
                 a.epilogue, a.tile_n);
    return 0;
  }
  const int sms = num_sms();
  // max_ctas leaves SMs free for a concurrent NCCL all-reduce (tile choice then balances waves over fewer pairs)
  const int pairs_avail = (a.max_ctas > 0 && a.max_ctas < sms ? a.max_ctas : sms) / 2;
  int bn = 0, splits = 1, n_half = 0;
  double pair_cost = 0;
  choose_tiling2(a, pairs_avail, &bn, &splits, &n_half, &pair_cost);
  if (bn == 0) {
    VITK_REQUIRE(a.variant < 2, VITK_EINVAL, "gemm: no CTA-pair tiling for N=%lld tile_n=%d", (long long)a.N, a.tile_n);
    return 0;
  }
  if (single_cta_wins(a, pair_cost, sms)) return 0;     // falls through to the single-CTA kernel (gemm.cu), 256-wide tiles
  Gemm2Params p;
  p.M = static_cast<int>(a.M); p.N = static_cast<int>(a.N); p.K = static_cast<int>(a.K);
  const int m_tiles = (p.M + 2 * k2BM - 1) / (2 * k2BM);
  p.n_half = n_half;
  p.n_full = p.N / bn - n_half / 2;
  p.n_tiles = p.n_full + p.n_half;
  p.mn_tiles = m_tiles * p.n_tiles;
  p.kb_total = (p.K + k2BK - 1) / k2BK;
  if (splits > p.kb_total) splits = p.kb_total;
  p.kb_per_split = (p.kb_total + splits - 1) / splits;
  p.k_splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  p.total_work = p.mn_tiles * p.k_splits;
  p.epi = a.epilogue;
  p.has_d2 = a.d2 != nullptr;
  p.aux = a.aux;
  p.ld_aux = a.ld_aux;
  p.bias = a.bias;
  p.tl = g_timeline;
  p.tl_seq = g_timeline != nullptr ? g_timeline_seq++ : 0;
  const int pairs = p.total_work < pairs_avail ? p.total_work : pairs_avail;
  *handled = true;
  {
    int rc = 0;
    if (launch_heavy2(a, p, bn, pairs, stream, &rc)) return rc;
  }
  switch (bn) {
    case 256: return aux_epi ? dispatch_major2<256, true>(a, p, pairs, stream) : dispatch_major2<256, false>(a, p, pairs, stream);
    case 192: return aux_epi ? dispatch_major2<192, true>(a, p, pairs, stream) : dispatch_major2<192, false>(a, p, pairs, stream);
    default: return aux_epi ? dispatch_major2<128, true>(a, p, pairs, stream) : dispatch_major2<128, false>(a, p, pairs, stream);
  }
}

}  // namespace vitk

// Host-only view of the tiling decision (no device needed): which tile width, split-K factor and number of
// half-width tiles per 256-row band vitk_gemm_bf16 would use for this problem on a GPU with `sms` SMs.
extern "C" VITK_API int vitk_gemm_plan(const vitk_gemm_args* a, int sms, int* tile_n, int* split_k, int* n_half, int* work_items) {
  using namespace vitk;
  VITK_REQUIRE(a != nullptr && tile_n && split_k && n_half && work_items && sms >= 2, VITK_EINVAL, "gemm_plan: bad argument");
  VITK_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0 && a->N % 128 == 0, VITK_EINVAL, "gemm_plan: the CTA-pair kernel needs N %% 128 == 0");
  const int pairs = (a->max_ctas > 0 && a->max_ctas < sms ? a->max_ctas : sms) / 2;
  int bn = 0, splits = 1, nh = 0;
  choose_tiling2(*a, pairs, &bn, &splits, &nh);
  VITK_REQUIRE(bn != 0, VITK_EINVAL, "gemm_plan: no CTA-pair tiling for N=%lld tile_n=%d", (long long)a->N, a->tile_n);
  const long long m_tiles = (a->M + 2 * k2BM - 1) / (2 * k2BM);
  const long long kb_total = (a->K + k2BK - 1) / k2BK;
  if (splits > kb_total) splits = static_cast<int>(kb_total);
  const long long kb_per = (kb_total + splits - 1) / splits;
  *tile_n = bn;
  *split_k = static_cast<int>((kb_total + kb_per - 1) / kb_per);
  *n_half = nh;
  *work_items = static_cast<int>(m_tiles * (a->N / bn - nh / 2 + nh) * *split_k);
  return 0;
}

