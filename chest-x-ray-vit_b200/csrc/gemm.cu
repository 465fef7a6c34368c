// Persistent warp-specialised bf16 GEMM for sm_100a: TMA → smem ring → tcgen05.mma → TMEM
// (double-buffered accumulator) → fused epilogue.  One CTA per SM, 128×BN output tiles,
// BK = 64.  Replaces aten::addmm / aten::mm on the ViT linear layers (see include/vitk.h).
//
//   warp 0      TMA producer (one elected lane)
//   warp 1      TMEM owner + MMA issuer (lane 0)
//   warps 2..9  epilogue: two warps per TMEM lane quadrant, each takes half of the columns
//
// Operand layouts in shared memory (128-byte swizzle, written by TMA, read by UMMA):
//   K-major  A [128 × 64]  one box {64 k, 128 rows}            16 KB, SBO 1024
//   MN-major A [64 k × 128] two boxes {64 m, 64 k} 8 KB apart        , SBO 1024, LBO 8192
//   (B alike with BN rows / BN/64 boxes).
#include <cuda.h>

#include <mutex>

#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "gemm_host.cuh"
#include "sm100_prims.cuh"

namespace vitk {

constexpr int kBM = 128;
constexpr int kBK = 64;
constexpr int kEpiWarps = 8;
constexpr int kGemmThreads = 64 + kEpiWarps * 32;
constexpr int kABytes = kBM * kBK * 2;  // 16 KB

template <int BN>
struct TileCfg {
  static constexpr int kBBytes = BN * kBK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (BN == 256) ? 4 : (BN == 192 ? 5 : 6);
  static constexpr int kTmemCols = (2 * BN <= 256) ? 256 : 512;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

struct GemmParams {
  int M, N, K;
  int n_tiles, mn_tiles, k_splits, kb_per_split, kb_total, total_work;
  int epi;
  void* d;
  void* d2;
  const float* bias;
  const void* aux;
  long long ldd, ld_aux;
  int rows_in, rows_out, row_off;
};

__device__ __forceinline__ void store_bf16x32(__nv_bfloat16* dst, const float (&v)[32]) {
  uint4* o = reinterpret_cast<uint4*>(dst);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    uint4 q;
    q.x = pack_bf16x2(v[8 * i + 0], v[8 * i + 1]);
    q.y = pack_bf16x2(v[8 * i + 2], v[8 * i + 3]);
    q.z = pack_bf16x2(v[8 * i + 4], v[8 * i + 5]);
    q.w = pack_bf16x2(v[8 * i + 6], v[8 * i + 7]);
    o[i] = q;
  }
}

// One thread, one output row, 32 consecutive columns starting at col0.
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, int row, int col0, float (&v)[32]) {
  const int epi = p.epi;
  if (epi == VITK_EPI_BIAS_BF16 || epi == VITK_EPI_BIAS_GELU_BF16 || epi == VITK_EPI_BIAS_RESID_F32 ||
      epi == VITK_EPI_PATCH_F32 || epi == VITK_EPI_BIAS_GELUG_BF16) {
    if (p.bias != nullptr) {
      const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 b = __ldg(b4 + i);
        v[4 * i + 0] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
      }
    }
  }
  if (row >= p.M) return;
  switch (epi) {
    case VITK_EPI_STORE_BF16:
    case VITK_EPI_BIAS_BF16: {
      store_bf16x32(reinterpret_cast<__nv_bfloat16*>(p.d) + static_cast<long long>(row) * p.ldd + col0, v);
      break;
    }
    case VITK_EPI_BIAS_GELU_BF16: {
      const long long off = static_cast<long long>(row) * p.ldd + col0;
      store_bf16x32(reinterpret_cast<__nv_bfloat16*>(p.d) + off, v);
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = gelu_erf(v[i]);
      store_bf16x32(reinterpret_cast<__nv_bfloat16*>(p.d2) + off, v);
      break;
    }
    case VITK_EPI_BIAS_GELUG_BF16: {
      const long long off = static_cast<long long>(row) * p.ldd + col0;
      float gr[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const GeluParts g = gelu_parts(v[i]);
        gr[i] = fmaf(v[i], g.pdf, g.cdf);
        v[i] *= g.cdf;
      }
      store_bf16x32(reinterpret_cast<__nv_bfloat16*>(p.d) + off, v);
      if (p.d2 != nullptr) store_bf16x32(reinterpret_cast<__nv_bfloat16*>(p.d2) + off, gr);
      break;
    }
    case VITK_EPI_BIAS_RESID_F32:
    case VITK_EPI_PATCH_F32: {
      long long out_row = row, aux_row = row;
      if (epi == VITK_EPI_PATCH_F32) {
        const int g = row / p.rows_in, r = row - g * p.rows_in;
        aux_row = p.row_off + r;
        out_row = static_cast<long long>(g) * p.rows_out + aux_row;
      }
      const float4* a4 = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.aux) + aux_row * p.ld_aux + col0);
      float4* o4 = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.d) + out_row * p.ldd + col0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 a = __ldg(a4 + i);
        o4[i] = make_float4(v[4 * i + 0] + a.x, v[4 * i + 1] + a.y, v[4 * i + 2] + a.z, v[4 * i + 3] + a.w);
      }
      break;
    }
    case VITK_EPI_MUL_BF16:
    case VITK_EPI_DGELU_BF16: {
      const uint4* u4 = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.aux) +
                                                       static_cast<long long>(row) * p.ld_aux + col0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint4 q = __ldg(u4 + i);
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
          v[8 * i + 2 * j + 0] *= (epi == VITK_EPI_MUL_BF16) ? f.x : gelu_erf_grad(f.x);
          v[8 * i + 2 * j + 1] *= (epi == VITK_EPI_MUL_BF16) ? f.y : gelu_erf_grad(f.y);
        }
      }
      store_bf16x32(reinterpret_cast<__nv_bfloat16*>(p.d) + static_cast<long long>(row) * p.ldd + col0, v);
      break;
    }
    case VITK_EPI_ACCUM_F32: {
      float* o = reinterpret_cast<float*>(p.d) + static_cast<long long>(row) * p.ldd + col0;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + 4 * i), "f"(v[4 * i + 0]),
                     "f"(v[4 * i + 1]), "f"(v[4 * i + 2]), "f"(v[4 * i + 3])
                     : "memory");
      }
      break;
    }
    case VITK_EPI_STORE_F32: {
      float4* o4 = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.d) + static_cast<long long>(row) * p.ldd + col0);
#pragma unroll
      for (int i = 0; i < 8; ++i) o4[i] = make_float4(v[4 * i + 0], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      break;
    }
    default: break;
  }
}

// VITK_EPI_UNPATCH_F32 (the input gradient, col2im of dh·Wp), in kernel instantiations of its own: a further case in
// epilogue_chunk costs the existing instantiations 36-40 registers, even left unused.  Row = token t of image g; tokens
// before row_off (CLS) carry no pixels.  Columns col0 … col0+31 are channel c, patch rows ky and ky+1
// (k = c·256 + ky·16 + kx): two 64-byte runs of the NCHW image, whose width is ldd = 16·G (G patches per row) and
// whose height the host passes in p.rows_in.
__device__ __forceinline__ void unpatch_chunk(const GemmParams& p, int row, int col0, const float (&v)[32]) {
  if (row >= p.M) return;
  const int g = row / p.rows_out;
  const int t = row - g * p.rows_out - p.row_off;
  if (t < 0) return;
  const int G = static_cast<int>(p.ldd >> 4);
  const int py = t / G, px = t - py * G;
  const int c = col0 >> 8, ky = (col0 >> 4) & 15;
  float4* o4 = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.d) +
                                         ((static_cast<long long>(g) * 3 + c) * p.rows_in + py * 16 + ky) * p.ldd + px * 16);
  const long long next = p.ldd >> 2;    // one image row, in float4
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    o4[i] = make_float4(v[4 * i + 0], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    o4[next + i] = make_float4(v[16 + 4 * i + 0], v[16 + 4 * i + 1], v[16 + 4 * i + 2], v[16 + 4 * i + 3]);
  }
}

struct WorkItem {
  int m_blk, n_blk, kb_begin, kb_end;
};
__device__ __forceinline__ WorkItem decode_work(const GemmParams& p, int w) {
  // (m,n) tiles fastest so that concurrently resident CTAs share the A row-panel / B panel in L2;
  // K-splits slowest.
  const int ks = w / p.mn_tiles;
  const int t = w - ks * p.mn_tiles;
  WorkItem it;
  it.m_blk = t / p.n_tiles;
  it.n_blk = t - it.m_blk * p.n_tiles;
  it.kb_begin = ks * p.kb_per_split;
  it.kb_end = min(it.kb_begin + p.kb_per_split, p.kb_total);
  return it;
}

template <int BN, bool A_MN, bool B_MN, bool UNPATCH>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                 const GemmParams p) {
  using Cfg = TileCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* acc_full = empty_bar + kStages;   // [2]
  uint64_t* acc_empty = acc_full + 2;         // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&acc_full[s], 1);
      mbar_init(&acc_empty[s], kEpiWarps);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  pdl_wait();
  pdl_launch_dependents();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // broadcast marks it warp-uniform: no per-MMA elect-broadcast-retry loop

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // (all lanes run the loop; the issue sits under elect.sync so ptxas emits the TMA instructions on uniform
    // registers instead of one elect/broadcast/retry loop per instruction)
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int w = blockIdx.x; w < p.total_work; w += gridDim.x) {
        const WorkItem it = decode_work(p, w);
        const int m0 = it.m_blk * kBM, n0 = it.n_blk * BN;
        for (int kb = it.kb_begin; kb < it.kb_end; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + kABytes;
          const int k0 = kb * kBK;
          if (elect_one()) {
            mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes);
            if (!A_MN) {
              tma_load_2d(sa, &tma_a, &full_bar[stage], k0, m0);
            } else {
#pragma unroll
              for (int g = 0; g < kBM / 64; ++g) tma_load_2d(sa + g * 8192, &tma_a, &full_bar[stage], m0 + g * 64, k0);
            }
            if (!B_MN) {
              tma_load_2d(sb, &tma_b, &full_bar[stage], k0, n0);
            } else {
#pragma unroll
              for (int g = 0; g < BN / 64; ++g) tma_load_2d(sb + g * 8192, &tma_b, &full_bar[stage], n0 + g * 64, k0);
            }
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_bf16(kBM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
    constexpr uint32_t a_lbo = A_MN ? 8192u : 0u, b_lbo = B_MN ? 8192u : 0u;
    constexpr uint32_t a_kstep = A_MN ? 2048u : 32u, b_kstep = B_MN ? 2048u : 32u;
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int w = blockIdx.x; w < p.total_work; w += gridDim.x) {
      const WorkItem it = decode_work(p, w);
      mbar_wait(&acc_empty[acc], acc_phase ^ 1);
      tc_fence_after_sync();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = it.kb_begin; kb < it.kb_end; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after_sync();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t sb = sa + kABytes;
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            const uint64_t ad = umma_smem_desc(sa + k * a_kstep, a_lbo, 1024);
            const uint64_t bd = umma_smem_desc(sb + k * b_kstep, b_lbo, 1024);
            tc_mma_bf16(d_tmem, ad, bd, idesc, (kb > it.kb_begin || k > 0) ? 1u : 0u);
          }
          tc_commit(&empty_bar[stage]);                       // smem slot reusable once these MMAs retire
          if (kb == it.kb_end - 1) tc_commit(&acc_full[acc]);  // accumulator complete
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else {
    // ------------------------------------------------------------------ epilogue
    const int ew = warp - 2;
    const int quad = warp & 3;            // TMEM lane quadrant this warp may touch
    const int col_half = ew >> 2;         // which half of the tile's columns
    constexpr int kChunks = BN / 32 / 2;  // 32-column chunks per warp
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int w = blockIdx.x; w < p.total_work; w += gridDim.x) {
      const WorkItem it = decode_work(p, w);
      mbar_wait(&acc_full[acc], acc_phase);
      tc_fence_after_sync();
      const int row = it.m_blk * kBM + quad * 32 + lane;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * BN;
#pragma unroll 1
      for (int c = 0; c < kChunks; ++c) {
        const int cc = col_half * kChunks + c;
        uint32_t r[32];
        tmem_ld_32x32(t_row + cc * 32, r);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
        if constexpr (UNPATCH) unpatch_chunk(p, row, it.n_blk * BN + cc * 32, v);
        else epilogue_chunk(p, row, it.n_blk * BN + cc * 32, v);
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------- host side
template <int BN, bool A_MN, bool B_MN, bool UNPATCH>
static int launch_gemm(const vitk_gemm_args& a, const GemmParams& p, int grid, cudaStream_t stream) {
  using Cfg = TileCfg<BN>;
  CUtensorMap ta, tb;
  if (int rc = operand_map(&ta, a.a, A_MN, a.M, a.K, a.lda, kBM)) return rc;
  if (int rc = operand_map(&tb, a.b, B_MN, a.N, a.K, a.ldb, BN)) return rc;
  auto kern = gemm_bf16_kernel<BN, A_MN, B_MN, UNPATCH>;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [&] {
    attr_err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
  });
  if (attr_err != cudaSuccess) return cuda_error(attr_err, "cudaFuncSetAttribute(gemm smem)");
  if (cudaError_t e = launch_pdl(kern, dim3(grid), dim3(kGemmThreads), Cfg::kSmemBytes, stream, ta, tb, p); e != cudaSuccess)
    return cuda_error(e, "gemm_bf16_kernel launch");
  VITK_LAUNCH_CHECK("gemm_bf16_kernel");
  return 0;
}

template <int BN, bool UNPATCH>
static int dispatch_major(const vitk_gemm_args& a, const GemmParams& p, int grid, cudaStream_t s) {
  if (!a.a_mn_major && !a.b_mn_major) return launch_gemm<BN, false, false, UNPATCH>(a, p, grid, s);
  if (!a.a_mn_major && a.b_mn_major) return launch_gemm<BN, false, true, UNPATCH>(a, p, grid, s);
  if (a.a_mn_major && !a.b_mn_major) return launch_gemm<BN, true, false, UNPATCH>(a, p, grid, s);
  return launch_gemm<BN, true, true, UNPATCH>(a, p, grid, s);
}

// ------------------------------------------------------------------------- launch planning
// Both kernels use 128-row CTA tiles and 64-wide K blocks (kBM, kBK); the pair kernel's tiles are 256-row bands.

// Single-CTA kernel: the N tile that wastes the fewest tile-slots in the last wave (cost ∝ waves × BN).
static int choose_tile_n(long long M, long long N, int sms) {
  const long long mt = (M + kBM - 1) / kBM;
  int best = 128;
  double best_cost = 1e30;
  const int cands[3] = {256, 192, 128};
  for (int bn : cands) {
    if (N % bn) continue;
    const long long tiles = mt * (N / bn);
    const long long waves = (tiles + sms - 1) / sms;
    // BN=128 pays the full A+B smem traffic per 64 MMA cycles (smem-bound) → mild penalty.
    const double cost = static_cast<double>(waves) * bn * (bn == 128 ? 1.10 : 1.0);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
  }
  return best;
}

// cycles a CTA pair spends per 64-wide K block of a tile of `bn` columns (tools/gemm_timeline.py, B200): the MMAs of a
// 256-wide tile occupy the tensor pipe for 4 × 122 cycles; narrower tiles are bound by operand delivery instead.
// 192: A/B on the full step, 440 (192-wide tiles for K-major N = 768) beats 500 (mixed 256+128 there) by 0.9 %.
static double kblock_cycles(int bn) { return bn == 256 ? 500.0 : (bn == 192 ? 440.0 : 390.0); }
constexpr double kTileFixedCycles = 1500.0;   // accumulator hand-over + pipeline refill per tile

// CTA-pair kernel: tile width, split count and half-width tiles per band with the lowest modelled cost (bn = 0 when
// no width fits N and tile_n).
static void choose_tiling2(const vitk_gemm_args& a, int pairs, int* bn_out, int* splits_out, int* n_half_out,
                           double* cost_out) {
  const long long mt = (a.M + 2 * kBM - 1) / (2 * kBM);
  const long long kb_total = (a.K + kBK - 1) / kBK;
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
  *cost_out = best;
}

// Data-gradient GEMMs (K-major A, MN-major B, plain bf16 store) whose M is ragged against the pair kernel's 256-row bands
// can quantise badly on 74 pairs yet perfectly on 148 single CTAs with 128-row bands — ViT-L at batch 8: M = 4616 → 19
// bands × 4 tiles of 256 columns = 76 tiles (two pairs get a second tile) against 37 × 4 = 148 tiles = exactly one wave.
// Measured there (tools/bench_gemm.py, VITK_BG_M=4616 VITK_BG_D=1024 VITK_BG_F=4096): fc1 dgrad 43.2 → 35.7 µs,
// qkv dgrad 35.8 → 28.8 µs, out dgrad 19.5 → 16.5 µs.  Per K block a single CTA (which stages the whole B tile itself)
// costs ≈ 1.1 × the pair kernel's 256-wide block for this operand layout.  The cost is that of 256-wide single-CTA
// tiles; the launch then takes choose_tile_n's width, which is 256 for the model's shapes but can be 128 for others.
static bool single_cta_wins(const vitk_gemm_args& a, double pair_cost, int sms) {
  if (a.variant != 0 || a.tile_n != 0 || a.max_ctas != 0 || a.a_mn_major || !a.b_mn_major || a.epilogue != VITK_EPI_STORE_BF16 ||
      a.N % 256 != 0)
    return false;
  const long long tiles = ((a.M + 127) / 128) * (a.N / 256);
  const long long waves = (tiles + sms - 1) / sms;
  const long long kb = (a.K + kBK - 1) / kBK;
  const double cost = static_cast<double>(waves) * (kb * 1.1 * kblock_cycles(256) + kTileFixedCycles);
  return cost < 0.9 * pair_cost;
}

// K blocks per split and work items once mn_tiles and kb_total are set; the split count is clamped to the K blocks
// and every split is non-empty.
static void set_splits(GemmPlan* p, int splits) {
  if (splits > p->kb_total) splits = p->kb_total;
  p->kb_per_split = (p->kb_total + splits - 1) / splits;
  p->k_splits = (p->kb_total + p->kb_per_split - 1) / p->kb_per_split;
  p->total_work = p->mn_tiles * p->k_splits;
}

int plan_gemm(const vitk_gemm_args& a, int sms, GemmPlan* out) {
  VITK_REQUIRE(a.M > 0 && a.N > 0 && a.K > 0, VITK_EINVAL, "gemm: M,N,K must be positive (%lld,%lld,%lld)",
               (long long)a.M, (long long)a.N, (long long)a.K);
  VITK_REQUIRE(a.M < (1ll << 31) && a.N < (1ll << 31) && a.K < (1ll << 31), VITK_EINVAL, "gemm: dims exceed int32");
  VITK_REQUIRE(a.N % 128 == 0, VITK_EINVAL, "gemm: N=%lld must be a multiple of 128", (long long)a.N);
  VITK_REQUIRE(a.a && a.b && a.d, VITK_EINVAL, "gemm: NULL operand");
  VITK_REQUIRE(aligned16(a.a) && aligned16(a.b) && aligned16(a.d), VITK_EALIGN, "gemm: operands must be 16-byte aligned");
  VITK_REQUIRE(a.lda % 8 == 0 && a.ldb % 8 == 0, VITK_EALIGN, "gemm: lda/ldb must be multiples of 8 elements");
  VITK_REQUIRE(a.lda >= (a.a_mn_major ? a.M : a.K) && a.ldb >= (a.b_mn_major ? a.N : a.K), VITK_EINVAL,
               "gemm: leading dimension smaller than the contiguous extent");
  VITK_REQUIRE(a.epilogue >= 0 && a.epilogue <= VITK_EPI_UNPATCH_F32, VITK_EINVAL, "gemm: unknown epilogue %d", a.epilogue);
  const EpiTraits& epi = kEpiTraits[a.epilogue];
  if (a.epilogue == VITK_EPI_UNPATCH_F32) {
    // d is the fp32 NCHW image [M/rows_out, 3, 16·G, 16·G] of G×G patches; ldd is its width
    VITK_REQUIRE(a.N == 768, VITK_EINVAL, "gemm: UNPATCH_F32 needs N = 768 (3 channels × 16 × 16), got N=%lld", (long long)a.N);
    VITK_REQUIRE(a.row_off >= 0 && a.rows_out > a.row_off && a.rows_out < (1ll << 31), VITK_EINVAL,
                 "gemm: UNPATCH_F32 needs rows_out > row_off >= 0 (rows_out=%lld, row_off=%lld)", (long long)a.rows_out,
                 (long long)a.row_off);
    const long long P = a.rows_out - a.row_off;
    if (a.rows_in == 0) {                    // a square grid of G×G patches
      long long G = 0;
      while ((G + 1) * (G + 1) <= P) ++G;
      VITK_REQUIRE(G * G == P, VITK_EINVAL, "gemm: UNPATCH_F32 needs a square number of patches, got rows_out - row_off = %lld", P);
      VITK_REQUIRE(a.ldd == 16 * G, VITK_EINVAL, "gemm: UNPATCH_F32 needs ldd = image width = 16·%lld, got ldd=%lld", G,
                   (long long)a.ldd);
    } else {                                 // rows_in patches per image row, P / rows_in rows of them
      VITK_REQUIRE(a.rows_in > 0 && P % a.rows_in == 0, VITK_EINVAL,
                   "gemm: UNPATCH_F32 needs rows_in (patches per image row) > 0 dividing rows_out - row_off = %lld, got "
                   "rows_in=%lld", P, (long long)a.rows_in);
      VITK_REQUIRE(a.ldd == 16 * a.rows_in, VITK_EINVAL, "gemm: UNPATCH_F32 needs ldd = image width = 16·%lld, got ldd=%lld",
                   (long long)a.rows_in, (long long)a.ldd);
    }
    VITK_REQUIRE(a.M % a.rows_out == 0, VITK_EINVAL, "gemm: UNPATCH_F32 needs M %% rows_out == 0 (M=%lld, rows_out=%lld)",
                 (long long)a.M, (long long)a.rows_out);
  } else {
    VITK_REQUIRE(a.ldd % (epi.f32_out ? 4 : 8) == 0 && a.ldd >= a.N, VITK_EALIGN, "gemm: ldd=%lld not aligned / too small",
                 (long long)a.ldd);
  }
  if (a.epilogue == VITK_EPI_BIAS_GELU_BF16)
    VITK_REQUIRE(a.d2 != nullptr && aligned16(a.d2), VITK_EINVAL, "gemm: BIAS_GELU needs d2");
  if (a.epilogue == VITK_EPI_BIAS_GELUG_BF16 && a.d2 != nullptr)
    VITK_REQUIRE(aligned16(a.d2), VITK_EALIGN, "gemm: d2 must be 16-byte aligned");
  VITK_REQUIRE(a.variant >= 0 && a.variant <= 3, VITK_EINVAL, "gemm: variant must be 0 (auto), 1 (single-CTA), 2 (CTA pair) or 3 (CTA pair, 8 epilogue warps)");
  if (epi.aux)
    VITK_REQUIRE(a.aux != nullptr && aligned16(a.aux) && a.ld_aux % 8 == 0 && a.ld_aux >= a.N, VITK_EINVAL,
                 "gemm: epilogue %d needs aux with ld_aux >= N, multiple of 8", a.epilogue);
  if (a.epilogue == VITK_EPI_PATCH_F32)
    VITK_REQUIRE(a.rows_in > 0 && a.rows_out >= a.rows_in + a.row_off && a.row_off >= 0, VITK_EINVAL,
                 "gemm: bad PATCH row remap");
  if (a.bias) VITK_REQUIRE(aligned16(a.bias), VITK_EALIGN, "gemm: bias must be 16-byte aligned");
  VITK_REQUIRE(a.split_k >= 0 && (a.split_k <= 1 || a.epilogue == VITK_EPI_ACCUM_F32), VITK_EINVAL,
               "gemm: split_k > 1 requires VITK_EPI_ACCUM_F32");

  GemmPlan& p = *out;
  p.kb_total = static_cast<int>((a.K + kBK - 1) / kBK);

  // The CTA-pair kernel wherever it applies (variant 0, 2, 3), unless the single-CTA kernel quantises better.
  if (a.variant != 1) {
    const bool eligible = epi.pair && (a.max_ctas == 0 || a.max_ctas >= 2) &&
                          !(epi.aux && a.a_mn_major) &&     // the aux instantiations exist for K-major A only
                          (a.tile_n == 0 || a.tile_n == 128 || a.tile_n == 192 || a.tile_n == 256) &&
                          !(a.tile_n == 192 && a.b_mn_major);
    VITK_REQUIRE(eligible || a.variant < 2, VITK_EINVAL,
                 "gemm: the CTA-pair kernel does not support this problem (epilogue %d, tile_n %d)", a.epilogue, a.tile_n);
    // max_ctas leaves SMs free for a concurrent NCCL all-reduce (tile choice then balances waves over fewer pairs)
    const int pairs = (a.max_ctas > 0 && a.max_ctas < sms ? a.max_ctas : sms) / 2;
    int bn = 0, splits = 1, n_half = 0;
    double pair_cost = 0;
    if (eligible) {
      choose_tiling2(a, pairs, &bn, &splits, &n_half, &pair_cost);
      VITK_REQUIRE(bn != 0 || a.variant < 2, VITK_EINVAL, "gemm: no CTA-pair tiling for N=%lld tile_n=%d", (long long)a.N,
                   a.tile_n);
    }
    if (bn != 0 && !single_cta_wins(a, pair_cost, sms)) {
      // fc1 forward (+bias, GELU, optional GELU') runs on 16 epilogue warps with the epilogue fixed at compile time
      // (see the pair kernel's template comment): 2 MUFU + 13 FP32 operations per element are a chain of dependent
      // latencies that four warps per scheduler hide better than two — 51.4 → 47.1 µs at M = 9232
      // (profiles/r02_bench_gemm_ew16.txt), bit-identical output (tests/test_gpu_gemm.py::
      // test_sixteen_warp_epilogues_equal_eight_warp).  The same treatment of the multiplier and fp32-residual
      // epilogues was measured and dropped: those launches move 128 / 71 MB for 43.6 / 10.9 GF and sit on the HBM side
      // of the roofline, not on the epilogue's instruction latency (no change at 49.2 / 28.7 / 47.1 µs).  Variant 3
      // keeps 8 warps (the reference the 16-warp instantiation is tested against).
      const bool ew16 = a.variant != 3 && a.epilogue == VITK_EPI_BIAS_GELUG_BF16 && !a.a_mn_major && !a.b_mn_major && bn == 256;
      p.kernel = ew16 ? GEMM_PAIR_EW16 : GEMM_PAIR;
      p.bn = bn;
      p.n_half = n_half;
      p.n_tiles = static_cast<int>(a.N / bn) - n_half / 2 + n_half;
      p.mn_tiles = static_cast<int>((a.M + 2 * kBM - 1) / (2 * kBM)) * p.n_tiles;
      set_splits(&p, splits);
      p.ctas = 2 * (p.total_work < pairs ? p.total_work : pairs);
      return 0;
    }
  }

  // The single-CTA kernel: variant 1, the epilogues and operand layouts the pair kernel lacks, and ragged data gradients.
  const int bn = a.tile_n ? a.tile_n : choose_tile_n(a.M, a.N, sms);
  VITK_REQUIRE((bn == 128 || bn == 192 || bn == 256) && a.N % bn == 0, VITK_EINVAL, "gemm: tile_n=%d invalid for N=%lld",
               bn, (long long)a.N);
  p.kernel = GEMM_SINGLE_CTA;
  p.bn = bn;
  p.n_half = 0;
  p.n_tiles = static_cast<int>(a.N / bn);
  p.mn_tiles = static_cast<int>((a.M + kBM - 1) / kBM) * p.n_tiles;
  int splits = a.split_k;
  if (splits == 0) {
    splits = 1;
    if (a.epilogue == VITK_EPI_ACCUM_F32 && p.mn_tiles < sms) {
      splits = (sms + p.mn_tiles - 1) / p.mn_tiles;  // fill one wave
      if (splits > p.kb_total / 4) splits = p.kb_total / 4 > 0 ? p.kb_total / 4 : 1;
    }
  }
  set_splits(&p, splits);
  p.ctas = p.total_work < sms ? p.total_work : sms;
  if (a.max_ctas > 0 && p.ctas > a.max_ctas) p.ctas = a.max_ctas;
  return 0;
}

}  // namespace vitk

using namespace vitk;

extern "C" VITK_API int vitk_gemm_bf16(const vitk_gemm_args* args, vitk_stream_t stream_) {
  VITK_REQUIRE(args != nullptr, VITK_EINVAL, "gemm: args is NULL");
  const vitk_gemm_args& a = *args;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  GemmPlan plan;
  if (int rc = plan_gemm(a, num_sms(), &plan)) return rc;
  if (plan.kernel != GEMM_SINGLE_CTA) return launch_pair(a, plan, stream);

  GemmParams p;
  p.M = static_cast<int>(a.M); p.N = static_cast<int>(a.N); p.K = static_cast<int>(a.K);
  p.n_tiles = plan.n_tiles; p.mn_tiles = plan.mn_tiles; p.k_splits = plan.k_splits;
  p.kb_per_split = plan.kb_per_split; p.kb_total = plan.kb_total; p.total_work = plan.total_work;
  p.epi = a.epilogue;
  p.d = a.d; p.d2 = a.d2; p.bias = a.bias; p.aux = a.aux;
  p.ldd = a.ldd; p.ld_aux = a.ld_aux;
  p.rows_in = static_cast<int>(a.rows_in); p.rows_out = static_cast<int>(a.rows_out); p.row_off = static_cast<int>(a.row_off);
  const int grid = plan.ctas;
  const bool unpatch = a.epilogue == VITK_EPI_UNPATCH_F32;
  // UNPATCH_F32 reads rows_in as the image height in pixels: 16 · patches / patches per row (ldd / 16 for a square grid)
  if (unpatch) p.rows_in = static_cast<int>(16 * (a.rows_out - a.row_off) / (a.rows_in ? a.rows_in : a.ldd / 16));
  switch (plan.bn) {
    case 256: return unpatch ? dispatch_major<256, true>(a, p, grid, stream) : dispatch_major<256, false>(a, p, grid, stream);
    case 192: return unpatch ? dispatch_major<192, true>(a, p, grid, stream) : dispatch_major<192, false>(a, p, grid, stream);
    default: return unpatch ? dispatch_major<128, true>(a, p, grid, stream) : dispatch_major<128, false>(a, p, grid, stream);
  }
}

// Host-only view of plan_gemm (no device needed): the launch vitk_gemm_bf16 makes for these arguments on a GPU with
// `sms` SMs.
extern "C" VITK_API int vitk_gemm_plan(const vitk_gemm_args* a, int sms, int* tile_n, int* split_k, int* n_half, int* work_items,
                                       int* kernel, int* ctas) {
  VITK_REQUIRE(a != nullptr && tile_n && split_k && n_half && work_items && kernel && ctas && sms >= 2, VITK_EINVAL,
               "gemm_plan: bad argument");
  GemmPlan plan;
  if (int rc = plan_gemm(*a, sms, &plan)) return rc;
  *tile_n = plan.bn;
  *split_k = plan.k_splits;
  *n_half = plan.n_half;
  *work_items = plan.total_work;
  *kernel = plan.kernel;
  *ctas = plan.ctas;
  return 0;
}
