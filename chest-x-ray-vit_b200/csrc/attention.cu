// Fused flash-style attention for sm_100a (head_dim 64, no mask, no dropout), forward and
// backward, on tcgen05 tensor cores with TMEM accumulators and TMA-fed operands.
// Replaces aten::scaled_dot_product_attention (+ backward) as called from HF
// modeling_vit.py:232-246 / integrations/sdpa_attention.py:92-102.
//
// Layouts: qkv bf16 [B,T,3,H,64] (= fused QKV projection output), o / do bf16 [B,T,H,64],
// lse fp32 [B,H,T].  Q/K/V tiles are 128 rows × 64 (one 128-byte swizzle atom wide):
//   as K-major operand  (contraction over head_dim): rows = M/N index
//   as MN-major operand (contraction over tokens)  : rows = K index, +2048 B per 16 tokens
// so the same TMA tile serves both roles.
//
// forward  : CTA = (128 queries, head, image), 4 softmax warps (thread = query row = TMEM lane) + a control warp; four
//            CTAs per SM (128 TMEM columns each) so one CTA's softmax overlaps the others' MMAs.
// backward : persistent CTAs (one per SM) draw (128 keys, head, image) work items and loop over the query blocks of each;
//            Sᵀ and dPᵀ live in TMEM (lane = key), dV/dK accumulate in TMEM across the loop, dQ partials are reduced
//            into an fp32 workspace with TMA reduce-adds.
#include <cuda.h>
#include <math.h>

#include <atomic>
#include <mutex>

#include "common.cuh"
#include "sm100_prims.cuh"
#include "tmap.cuh"

namespace vitk {

// Optional per-phase timeline (vitk_debug_timeline): CTA (0,0,0) records clock64() stamps.
long long* g_timeline = nullptr;   // also stamped by the CTA-pair GEMM (gemm2.cu)
int g_timeline_seq = 0;            // GEMM launches since the buffer was set (per-launch min/max stamps)
#define VITK_STAMP(slot)                                             \
  do {                                                               \
    if (tl != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && lane == 0) tl[(slot)] = clock64(); \
  } while (0)

constexpr int kTile = 128;   // queries per CTA (fwd) / keys per CTA (bwd) / tokens per inner block
constexpr int kDh = 64;
constexpr int kTileBytes = kTile * kDh * 2;  // 16 KB
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Row `row` of a K-major, 128-byte-swizzled [128 × 128] bf16 tile held as two [128 × 64]
// sub-tiles 16 KB apart: write 32 consecutive columns starting at col0 (multiple of 32).
__device__ __forceinline__ void store_row32_sw128(uint8_t* tile, int row, int col0, const float (&v)[32]) {
  uint8_t* base = tile + (col0 >> 6) * kTileBytes + row * 128;
  const int c0 = (col0 & 63) >> 3;  // first 16-byte chunk inside the 128-byte row
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    uint4 w;
    w.x = pack_bf16x2(v[8 * q + 0], v[8 * q + 1]);
    w.y = pack_bf16x2(v[8 * q + 2], v[8 * q + 3]);
    w.z = pack_bf16x2(v[8 * q + 4], v[8 * q + 5]);
    w.w = pack_bf16x2(v[8 * q + 6], v[8 * q + 7]);
    *reinterpret_cast<uint4*>(base + (((c0 + q) ^ (row & 7)) << 4)) = w;
  }
}

// ============================================================================ forward
// CTA = (128 queries, head, image); 4 softmax warps (thread = query row = TMEM lane) + 1 control warp
// that owns TMA and MMA issue.  Four CTAs per SM: 16 softmax warps keep the MUFU pipe (16 exp2/clk/SM — the unit
// that bounds attention at head_dim 64) fed while each CTA's own score → softmax → P·V chain waits on the tensor core.
//   keys are consumed in sub-blocks of 64:
//   S_u = Q·K_uᵀ       SS-MMA (N = 64) into the CTA's 64 score columns of TMEM
//   P_u (bf16)         written back INTO the consumed S columns (two per 32-bit column) with tcgen05.st
//   O += P_u·V_u       TS-MMA: A = P straight from TMEM, B = V rows from smem (MN-major); O accumulates
//                      in TMEM across all sub-blocks — no per-block read-back, no P round trip via smem
// Softmax is single-pass with a lazily updated reference maximum: probabilities are taken relative to
// m_ref; whenever a 32-column chunk exceeds it by more than 2^16 (always on the first chunk, otherwise
// only for extreme logits) everything accumulated so far is rescaled by 2^(old−new) ≤ 1 — exact
// bookkeeping, m_ref cancels in O/l and in the LSE.  Probabilities are computed SPECULATIVELY against the current
// reference while the chunk maximum is still being reduced (the MUFU pipe starts at once instead of after a 16-deep
// max chain + vote); when the reference does move, the chunk is recomputed from the registers it still sits in.
// The last sub-block issues narrower MMAs (N, K rounded up to 16 valid keys) instead of computing masked columns;
// warps whose 32 query rows all lie beyond T (the padding of the last tile) skip the arithmetic.
// Epilogue: O/l → bf16 → the (now idle) Q tile in shared memory → one TMA store (rows ≥ T clipped by the tensor map).
// (A pair-of-tiles variant — two 128-query tiles ping-ponging on one 128-key K/V stream, N = 128 score MMAs, one CTA
// of 8 softmax warps per SM — measured 60 µs against this kernel's 43: 2 softmax warps per scheduler cannot hide the
// chunk latency, see DESIGN.md §4 and profiles/r02_attn_fwd_pair_timeline.txt.)
constexpr int kFwdSoftmaxThreads = 128;
constexpr int kFwdThreads = kFwdSoftmaxThreads + 32;
constexpr int kSub = 64;                                   // keys per sub-block = one K/V TMA tile
constexpr int kSubBytes = kSub * kDh * 2;                  // 8 KB
constexpr int kFwdSmemQ = 0;
constexpr int kFwdSmemK = kFwdSmemQ + kTileBytes;          // 2 buffers of 64 keys
constexpr int kFwdSmemV = kFwdSmemK + 2 * kSubBytes;       // 2 buffers
constexpr int kFwdSmemBar = kFwdSmemV + 2 * kSubBytes;
constexpr int kFwdSmemBytes = kFwdSmemBar + 128 + 1024;    // ≈ 49 KB → four CTAs per SM
constexpr int kFwdTmemCols = 128;  // S/P: [0,64)   O: [64,128)
constexpr float kLazyMaxLog2 = 16.0f;

__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

__global__ void __launch_bounds__(kFwdThreads, 4)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_kv,
                const __grid_constant__ CUtensorMap tma_o, float* __restrict__ lse, int T, int H, float scale_log2, long long* tl) {
  // tl (vitk_debug_timeline, ≥ 8192 int64): [3·cta + {0,1,2}] = globaltimer at entry / %smid / globaltimer at exit
  const unsigned lin_cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
  if (tl != nullptr && threadIdx.x == 0 && lin_cta < 2000) {
    unsigned long long t; unsigned smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    tl[3 * lin_cta] = static_cast<long long>(t);
    tl[3 * lin_cta + 1] = smid;
  }
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem + kFwdSmemQ;
  uint8_t* sK = smem + kFwdSmemK;
  uint8_t* sV = smem + kFwdSmemV;
  uint64_t* bar_q = reinterpret_cast<uint64_t*>(smem + kFwdSmemBar);
  uint64_t* bar_k = bar_q + 1;      // [2] K tile landed
  uint64_t* bar_v = bar_q + 3;      // [2] V tile landed
  uint64_t* bar_free = bar_q + 5;   // [2] K/V buffer consumed by its P·V
  uint64_t* bar_s = bar_q + 7;      // S ready
  uint64_t* bar_p = bar_q + 8;      // P written by the 4 softmax warps
  uint64_t* bar_o = bar_q + 9;      // last P·V retired
  uint64_t* bar_pv = bar_q + 10;    // P·V(u) retired (phase u): only the rescale path waits on it
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_q + 11);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int nsub = (T + kSub - 1) / kSub;
  const int colq = h * kDh, colk = (H + h) * kDh, colv = (2 * H + h) * kDh;

  if (tid == 0) {
    tma_prefetch_desc(&tma_q);
    tma_prefetch_desc(&tma_kv);
    tma_prefetch_desc(&tma_o);
    for (int i = 0; i < 11; ++i) mbar_init(bar_q + i, i == 8 ? 4 : 1);
    fence_mbar_init();
  }
  if (warp == 4) tmem_alloc(tmem_slot, kFwdTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  pdl_wait();
  pdl_launch_dependents();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // broadcast marks it warp-uniform: no per-MMA elect-broadcast-retry loop
  const uint32_t tmem_o = tmem_base + 64;

  if (warp == 4) {
    // ------------------------------------------------------------------ control warp: TMA + MMA issue
    // Every lane runs this loop so that descriptors and addresses stay warp-uniform (uniform registers), and the
    // issuing instructions sit under elect.sync: ptxas then knows exactly one lane issues and emits back-to-back
    // UTCHMMA / UTMALDG on uniform registers.  Under a lane-id test (`lane == 0`) every MMA is wrapped in an
    // elect/broadcast/retry loop costing ≈100 cycles — several times the 49 cycles an N = 64 MMA occupies the pipe.
    {
      auto load_kv = [&](int u) {
        const int buf = u & 1;
        if (elect_one()) {
          mbar_arrive_expect_tx(&bar_k[buf], kSubBytes);
          tma_load_3d(sK + buf * kSubBytes, &tma_kv, &bar_k[buf], colk, u * kSub, b);
          mbar_arrive_expect_tx(&bar_v[buf], kSubBytes);
          tma_load_3d(sV + buf * kSubBytes, &tma_kv, &bar_v[buf], colv, u * kSub, b);
        }
      };
      if (elect_one()) {
        mbar_arrive_expect_tx(bar_q, kTileBytes);
        tma_load_3d(sQ, &tma_q, bar_q, colq, qb * kTile, b);
      }
      load_kv(0);
      if (nsub > 1) load_kv(1);
      const uint64_t q_desc = umma_smem_desc(smem_u32(sQ), 0, 1024);
      const uint64_t k_desc = umma_smem_desc(smem_u32(sK), 0, 1024);
      const uint64_t v_desc = umma_smem_desc(smem_u32(sV), kSubBytes, 1024);
      auto sub_cols = [&](int u) { return (min(kSub, T - u * kSub) + 15) & ~15; };   // keys sub-block u needs
      auto issue_s = [&](int u) {
        const int buf = u & 1;
        mbar_wait(&bar_k[buf], (u >> 1) & 1);
        tc_fence_after_sync();
        const uint64_t bk = k_desc + static_cast<uint64_t>(buf * (kSubBytes >> 4));
        const uint32_t idesc_s = umma_idesc_bf16(kTile, sub_cols(u), 0, 0);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k) tc_mma_bf16(tmem_base, q_desc + 2 * k, bk + 2 * k, idesc_s, k > 0);
          tc_commit(bar_s);
        }
      };
      mbar_wait(bar_q, 0);
      issue_s(0);
      constexpr uint32_t idesc_pv = umma_idesc_bf16(kTile, kDh, 0, 1);
      for (int u = 0; u < nsub; ++u) {
        const int buf = u & 1;
        const uint32_t ph = (u >> 1) & 1;
        mbar_wait(&bar_v[buf], ph);
        mbar_wait(bar_p, u & 1);
        tc_fence_after_sync();
        const uint64_t bv = v_desc + static_cast<uint64_t>(buf * (kSubBytes >> 4));
        const int ksteps = sub_cols(u) / 16;
        if (elect_one()) {
          if (ksteps == kSub / 16) {           // full sub-block: unrolled, MMAs issue back to back
#pragma unroll
            for (int k = 0; k < kSub / 16; ++k)
              tc_mma_bf16_ts(tmem_o, tmem_base + k * 8, bv + k * 128, idesc_pv, (u > 0 || k > 0) ? 1u : 0u);
          } else {
            for (int k = 0; k < ksteps; ++k)
              tc_mma_bf16_ts(tmem_o, tmem_base + k * 8, bv + k * 128, idesc_pv, (u > 0 || k > 0) ? 1u : 0u);
          }
          tc_commit(bar_pv);
          tc_commit(&bar_free[buf]);
          if (u == nsub - 1) tc_commit(bar_o);
        }
        if (u + 1 < nsub) issue_s(u + 1);     // queued right behind P·V(u): MMAs retire in issue order
        if (u + 2 < nsub) {                   // refill this K/V buffer once its P·V has retired
          mbar_wait(&bar_free[buf], ph);
          load_kv(u + 2);
        }
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ softmax warps
    const uint32_t lane_field = static_cast<uint32_t>(warp * 32) << 16;
    float m_ref = -INFINITY, l_run = 1.f;
    const bool live = qb * kTile + warp * 32 < T;     // false: all 32 query rows of this warp are padding beyond T
    if (live) l_run = 0.f;
    for (int u = 0; u < nsub; ++u) {
      const int nvalid = min(kSub, T - u * kSub);
      const int nchunk = (nvalid + 31) >> 5;
      const uint32_t tm_s = tmem_base + lane_field;
      mbar_wait(bar_s, u & 1);
      tc_fence_after_sync();
      float rs0 = 0.f, rs1 = 0.f;
      for (int c = 0; live && c < nchunk; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(tm_s + c * 32, r);
        tmem_ld_wait();
        const bool full = (c + 1) * 32 <= nvalid;
        uint32_t pk[16];
        float s0 = 0.f, s1 = 0.f;
        float cm = -INFINITY;
        if (full) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {          // speculative: against the reference maximum as it stands
            const float p0 = fast_exp2(fmaf(__uint_as_float(r[2 * i]), scale_log2, -m_ref));
            const float p1 = fast_exp2(fmaf(__uint_as_float(r[2 * i + 1]), scale_log2, -m_ref));
            s0 += p0;
            s1 += p1;
            pk[i] = pack_bf16x2(p0, p1);
          }
#pragma unroll
          for (int i = 0; i < 32; i += 2) cm = fmax3(cm, __uint_as_float(r[i]), __uint_as_float(r[i + 1]));
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (c * 32 + i < nvalid) cm = fmaxf(cm, __uint_as_float(r[i]));
        }
        const float m_c = cm * scale_log2;
        const bool fix = m_c > m_ref + kLazyMaxLog2;
        const bool moved = __any_sync(0xffffffffu, fix);
        if (moved) {
          const float m_new = fix ? m_c : m_ref;
          const float alpha = fix ? fast_exp2(m_ref - m_new) : 1.0f;
          l_run *= alpha;
          rs0 *= alpha;
          rs1 *= alpha;
          if (u > 0) {
            // O holds P·V of sub-blocks < u; P·V(u-1) may still be in flight
            mbar_wait(bar_pv, (u - 1) & 1);
            tc_fence_after_sync();
#pragma unroll 1
            for (int cc = 0; cc < 2; ++cc) {
              uint32_t ro[32];
              tmem_ld_32x32(tmem_o + lane_field + cc * 32, ro);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; ++i) ro[i] = __float_as_uint(__uint_as_float(ro[i]) * alpha);
              tmem_st_32x32(tmem_o + lane_field + cc * 32, ro);
            }
          }
          tmem_st_wait();
#pragma unroll 1
          for (int cc = 0; cc < c; ++cc) {
            uint32_t pq[16];
            tmem_ld_32x16(tm_s + cc * 16, pq);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pq[i]));
              pq[i] = pack_bf16x2(f.x * alpha, f.y * alpha);
            }
            tmem_st_32x16(tm_s + cc * 16, pq);
          }
          m_ref = m_new;
        }
        if (moved || !full) {                       // the reference moved (or a ragged chunk): (re)compute from r
          s0 = s1 = 0.f;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float p0 = fast_exp2(fmaf(__uint_as_float(r[2 * i]), scale_log2, -m_ref));
            float p1 = fast_exp2(fmaf(__uint_as_float(r[2 * i + 1]), scale_log2, -m_ref));
            if (c * 32 + 2 * i >= nvalid) p0 = 0.f;
            if (c * 32 + 2 * i + 1 >= nvalid) p1 = 0.f;
            s0 += p0;
            s1 += p1;
            pk[i] = pack_bf16x2(p0, p1);
          }
        }
        rs0 += s0;
        rs1 += s1;
        tmem_st_32x16(tm_s + c * 16, pk);     // P overwrites S columns already consumed
      }
      l_run += rs0 + rs1;
      tmem_st_wait();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_p);
    }
    mbar_wait(bar_o, 0);
    tc_fence_after_sync();
    const int t = qb * kTile + tid;
    const float inv = 1.0f / l_run;
    // O / l → bf16 → the Q tile's shared memory (every S MMA that read it has retired), 128-byte swizzled rows
    uint8_t* srow = sQ + tid * 128;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t r[32];
      tmem_ld_32x32(tmem_o + lane_field + c * 32, r);
      tmem_ld_wait();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 w;
        w.x = pack_bf16x2(__uint_as_float(r[8 * q + 0]) * inv, __uint_as_float(r[8 * q + 1]) * inv);
        w.y = pack_bf16x2(__uint_as_float(r[8 * q + 2]) * inv, __uint_as_float(r[8 * q + 3]) * inv);
        w.z = pack_bf16x2(__uint_as_float(r[8 * q + 4]) * inv, __uint_as_float(r[8 * q + 5]) * inv);
        w.w = pack_bf16x2(__uint_as_float(r[8 * q + 6]) * inv, __uint_as_float(r[8 * q + 7]) * inv);
        *reinterpret_cast<uint4*>(srow + (((4 * c + q) ^ (tid & 7)) << 4)) = w;
      }
    }
    fence_proxy_async_smem();
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (tid == 0) {
      tma_store_3d(&tma_o, sQ, colq, qb * kTile, b);
      tma_store_commit();
      tma_store_wait_read<0>();
    }
    if (t < T) lse[(static_cast<long long>(b) * H + h) * T + t] = (m_ref + log2f(l_run)) * kLn2;
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kFwdTmemCols);
  }
  if (tl != nullptr && threadIdx.x == 0 && lin_cta < 2000) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    tl[3 * lin_cta + 2] = static_cast<long long>(t);
  }
}

// ============================================================================ backward
// stats[b,h,t] = { lse·log2e, Δ = Σ_d dO·O } for t < T and { +inf, 0 } for the padding rows T ≤ t < Tpad
// (Tpad = multiple of 128), so the main kernel reads them with unconditional aligned float4 loads and
// padded queries get P = exp2(−inf) = 0.  One warp per token row; used for H > 16 heads.
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ o,
                                                         const __nv_bfloat16* __restrict__ d_o, const float* __restrict__ lse,
                                                         int B, int T, int Tpad, int H, float* __restrict__ lse2,
                                                         float* __restrict__ delta) {
  pdl_wait();
  pdl_launch_dependents();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);   // over B·Tpad
  const int lane = threadIdx.x & 31;
  if (row >= B * Tpad) return;
  const int b = row / Tpad, t = row - b * Tpad;
  if (t >= T) {
    for (int hh = lane; hh < H; hh += 32) {
      const long long idx = (static_cast<long long>(b) * H + hh) * Tpad + t;
      lse2[idx] = INFINITY;
      delta[idx] = 0.f;
    }
    return;
  }
  const int D = H * kDh;
  const long long grow = static_cast<long long>(b) * T + t;
  const uint4* po = reinterpret_cast<const uint4*>(o + grow * D);
  const uint4* pd = reinterpret_cast<const uint4*>(d_o + grow * D);
  for (int c0 = 0; c0 < D / 8; c0 += 32) {  // chunk c covers columns [8c, 8c+8) of head c/8
    const int c = c0 + lane;
    const bool valid = c < D / 8;
    float s = 0.f;
    if (valid) {
      const uint4 a = __ldg(po + c), g = __ldg(pd + c);
      const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, gw[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 x = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&aw[i]));
        const float2 y = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&gw[i]));
        s += x.x * y.x + x.y * y.y;
      }
    }
    // 8 consecutive lanes hold one head
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (valid && (lane & 7) == 0) {
      const int hh = c >> 3;
      const long long idx = (static_cast<long long>(b) * H + hh) * Tpad + t;
      delta[idx] = s;
      lse2[idx] = __ldg(lse + (static_cast<long long>(b) * H + hh) * T + t) * kLog2e;
    }
  }
}

// The same for H ≤ 16 heads (NIT = ⌈H/4⌉), organised for bandwidth: a block owns 16 consecutive (padded) token rows of
// one image, a warp two of them with all of their O / dO loads (4·NIT × 16 B per lane) in flight at once, and the
// per-head results cross shared memory so that lse2 / delta are written as 64-byte runs per head instead of one
// 4-byte store per (row, head) with a Tpad·4-byte stride (which cost 37 % extra sector traffic and most of the time).
template <int NIT>
__global__ void __launch_bounds__(256) attn_delta16_kernel(const __nv_bfloat16* __restrict__ o,
                                                           const __nv_bfloat16* __restrict__ d_o, const float* __restrict__ lse,
                                                           int B, int T, int Tpad, int H, float* __restrict__ lse2,
                                                           float* __restrict__ delta) {
  __shared__ float sd[4 * NIT][17];                  // [head][row of the block]
  pdl_wait();
  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = blockIdx.x * 16;                  // over B·Tpad (Tpad is a multiple of 128: a block never straddles images)
  const int b = row0 / Tpad, t0 = row0 - b * Tpad;
  const int D = H * kDh, nchunk = D / 8;             // 16-byte chunks per row; chunk c covers columns [8c, 8c+8) of head c/8
  uint4 a[2][NIT], g[2][NIT];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int t = t0 + 2 * warp + j;
    const long long grow = static_cast<long long>(b) * T + t;
    const uint4* po = reinterpret_cast<const uint4*>(o + grow * D);
    const uint4* pd = reinterpret_cast<const uint4*>(d_o + grow * D);
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int c = it * 32 + lane;
      const bool ok = t < T && c < nchunk;
      a[j][it] = ok ? __ldg(po + c) : make_uint4(0u, 0u, 0u, 0u);
      g[j][it] = ok ? __ldg(pd + c) : make_uint4(0u, 0u, 0u, 0u);
    }
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const uint32_t aw[4] = {a[j][it].x, a[j][it].y, a[j][it].z, a[j][it].w}, gw[4] = {g[j][it].x, g[j][it].y, g[j][it].z, g[j][it].w};
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 x = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&aw[i]));
        const float2 y = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&gw[i]));
        s += x.x * y.x + x.y * y.y;
      }
      s += __shfl_xor_sync(0xffffffffu, s, 1);       // 8 consecutive lanes hold one head (same order as attn_delta_kernel)
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      s += __shfl_xor_sync(0xffffffffu, s, 4);
      if ((lane & 7) == 0) sd[it * 4 + (lane >> 3)][2 * warp + j] = s;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < H * 16; i += 256) {
    const int hh = i >> 4, tl = i & 15, t = t0 + tl;
    const long long idx = (static_cast<long long>(b) * H + hh) * Tpad + t;
    if (t < T) {
      delta[idx] = sd[hh][tl];
      lse2[idx] = __ldg(lse + (static_cast<long long>(b) * H + hh) * T + t) * kLog2e;
    } else {
      delta[idx] = 0.f;
      lse2[idx] = INFINITY;
    }
  }
}

// backward main kernel.  CTA = (128 keys, head, image) looping over the queries in sub-blocks of 64;
// 16 compute warps (TMEM lane quadrant = warp%4 = 32 keys, column group = warp/4 = 16 queries) + 1 control
// warp that owns TMA and MMA issue.  Per sub-block u (buffer x = u&1):
//   Sᵀ_x = K·Qᵀ, dPᵀ_x = V·dOᵀ       SS-MMAs (N = 64) into one of TWO score buffers in TMEM (lane = key)
//   Pᵀ = exp2(Sᵀ·c − lse), dSᵀ = Pᵀ∘(dPᵀ − Δ)   compute warps; both are written back (bf16) INTO the warp's own
//                                    consumed Sᵀ / dPᵀ columns with tcgen05.st, dSᵀ additionally to swizzled smem
//   dV += Pᵀ·dO, dK += dSᵀ·Q          TS-MMAs, A straight from TMEM (no shared-memory A reads)
//   dQ_i = dS·K                      once per 128-query block: SS-MMA, A = the dSᵀ smem tile read MN-major
// MMAs retire in issue order, so the scores of sub-block u+2 are queued right behind dV/dK(/dQ) of u and the
// tensor core works on buffer x while the compute warps work on buffer 1−x.  dQ is double-buffered in TMEM
// and reduced into the fp32 accumulator one block later with per-warp TMA reduce-adds.  Keys ≥ T need no
// masking (their dV/dK rows are never stored, their dQ contribution multiplies zero-filled K rows);
// queries ≥ T have lse = +inf in the padded statistics, hence P = dS = 0.
// Persistent: the grid is one CTA per SM and every CTA walks work items (item = key block × head × image, key block
// fastest): first w = blockIdx.x, then whatever a global atomic counter hands out (gridDim.x, gridDim.x + 1, …) — the
// load warp draws the next item while the current one runs and publishes it to the other warps through shared memory
// (item_ring / bar_id).  A draw instead of a fixed stride because a CTA that starts late (its SM still held by a
// communication kernel of the gradient all-reduce) must not sit on a full share of the work.
// Ring / buffer indices and barrier parities run on GLOBAL counters
// (sub-blocks g, 128-query blocks G, items), so nothing is re-initialised between items: the load warp brings the next
// item's K/V and first Q/dO sub-tiles as soon as the previous item's last MMA has retired (bar_item), the MMA warp
// issues the next item's first score MMAs while the compute warps still drain dQ / dV / dK of the previous one, and
// only the first dV/dK MMA of an item waits for that drain (bar_acc).  This hides the per-CTA prologue (TMEM
// allocation, barrier set-up, the K/V + Q/dO round trip) behind the epilogue: 123.9 → 117.5 µs per layer all-in at
// B = 16.  (Tried on top and dropped, 119.7 µs: K/V double-buffered in shared memory with the next item's scores queued
// right behind the last dQ MMA — the boundary was already hidden behind the compute warps' epilogue, and the variable
// K/V descriptor offsets cost the MMA-issue warp ≈100 cycles per sub-block.)
constexpr int kBwdComputeWarps = 16;
constexpr int kBwdThreads = (kBwdComputeWarps + 2) * 32;   // 16 compute warps + MMA-issue warp + TMA-load warp
constexpr int kQSub = 64;
constexpr int kBwdSmemK = 0;
constexpr int kBwdSmemV = kBwdSmemK + kTileBytes;
constexpr int kBwdSmemQ = kBwdSmemV + kTileBytes;        // ring of 4 sub-tiles of 64 queries (8 KB each)
constexpr int kBwdSmemDO = kBwdSmemQ + 2 * kTileBytes;   // ring of 4 sub-tiles
constexpr int kBwdSmemDSt = kBwdSmemDO + 2 * kTileBytes; // dSᵀ [128 keys × 128 q], one tile per 128-query block parity
constexpr int kBwdSmemDqS = kBwdSmemDSt + 4 * kTileBytes;   // per-warp dQ staging slabs: 16 × [32 q × 16 f32], 64 B swizzle
constexpr int kBwdSmemBar = kBwdSmemDqS + kBwdComputeWarps * 2048;
constexpr int kBwdSmemBytes = kBwdSmemBar + 256 + 1024;   // 16 barriers + the TMEM slot, + alignment slack
// TMEM columns: buffer x: Sᵀ/Pᵀ [128x, 128x+64), dPᵀ/dSᵀ [128x+64, 128x+128); dV [256,320) dK [320,384) dQ[2] [384,512)
constexpr int kBwdTmemCols = 512;

__global__ void __launch_bounds__(kBwdThreads, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tma_qkv, const __grid_constant__ CUtensorMap tma_q64,
                const __grid_constant__ CUtensorMap tma_do64, const __grid_constant__ CUtensorMap tma_dq, const float* __restrict__ lse2, const float* __restrict__ delta,
                __nv_bfloat16* __restrict__ dqkv, int T, int Tpad, int H, int B, float scale, float scale_log2, int* __restrict__ work_counter, long long* tl_arg) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem + kBwdSmemK;
  uint8_t* sV = smem + kBwdSmemV;
  uint8_t* sQ = smem + kBwdSmemQ;
  uint8_t* sDO = smem + kBwdSmemDO;
  uint8_t* sDSt = smem + kBwdSmemDSt;
  uint64_t* bar_kv = reinterpret_cast<uint64_t*>(smem + kBwdSmemBar);
  uint64_t* bar_qd = bar_kv + 1;  // [4] Q / dO sub-tile landed
  uint64_t* bar_s = bar_kv + 5;   // [2] Sᵀ_x, dPᵀ_x ready
  uint64_t* bar_pd = bar_kv + 7;  // [2] Pᵀ_x / dSᵀ_x written by the 16 compute warps
  uint64_t* bar_g = bar_kv + 9;   // every MMA up to and including dQ of a 128-query block retired
  uint64_t* bar_free = bar_kv + 10;  // [4] dV/dK of the sub-block using this Q/dO sub-tile retired
  uint64_t* bar_item = bar_kv + 14;  // every MMA of a work item retired: K/V may be overwritten by the next item's
  uint64_t* bar_acc = bar_kv + 15;   // the 16 compute warps have read dV/dK of a work item out of TMEM
  uint64_t* bar_id = bar_kv + 16;    // [2] the id of work item n (slot n & 1) has been published in item_ring
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_kv + 18);
  volatile int* item_ring = reinterpret_cast<volatile int*>(bar_kv + 18) + 1;   // [2] global work-item index, −1 = no more work

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nq = (T + kTile - 1) / kTile;        // key blocks per (image, head) = 128-query blocks per work item
  const int nsub = (T + kQSub - 1) / kQSub;
  const int total_items = nq * H * B;

  if (tid == 0) {
    tma_prefetch_desc(&tma_qkv);
    tma_prefetch_desc(&tma_q64);
    tma_prefetch_desc(&tma_do64);
    tma_prefetch_desc(&tma_dq);
    for (int i = 0; i < 18; ++i) mbar_init(bar_kv + i, (i == 7 || i == 8 || i == 15) ? kBwdComputeWarps : 1);
    fence_mbar_init();
  }
  if (warp == kBwdComputeWarps) tmem_alloc(tmem_slot, kBwdTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  pdl_wait();
  pdl_launch_dependents();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // broadcast marks it warp-uniform: no per-MMA elect-broadcast-retry loop
  const uint32_t tm_dv = tmem_base + 256, tm_dk = tmem_base + 320, tm_dq = tmem_base + 384;

  if (warp == kBwdComputeWarps) {
    // ------------------------------------------------------------------ control warp: TMA + MMA issue
    // (all lanes run the loop so descriptors stay in uniform registers; the issuing instructions sit under
    // elect.sync so that ptxas emits them back to back instead of one elect/broadcast/retry loop per instruction)
    constexpr uint32_t idesc_sc = umma_idesc_bf16(kTile, kQSub, 0, 0);  // Sᵀ = K·Qᵀ, dPᵀ = V·dOᵀ (N = 64 queries)
    constexpr uint32_t idesc_km = umma_idesc_bf16(kTile, kDh, 0, 1);    // dV += Pᵀ·dO, dK += dSᵀ·Q
    constexpr uint32_t idesc_mm = umma_idesc_bf16(kTile, kDh, 1, 1);    // dQ = dS·K
    constexpr uint32_t kTile16 = kTileBytes >> 4;                        // descriptor address units are 16 B
    const uint64_t k_kmaj = umma_smem_desc(smem_u32(sK), 0, 1024);
    const uint64_t v_kmaj = umma_smem_desc(smem_u32(sV), 0, 1024);
    const uint64_t k_mnmaj = umma_smem_desc(smem_u32(sK), kTileBytes, 1024);
    constexpr uint32_t kSub16 = (kQSub * 128) >> 4;                      // one 64-query sub-tile = 8 KB
    const uint64_t q_kmaj = umma_smem_desc(smem_u32(sQ), 0, 1024);
    const uint64_t do_kmaj = umma_smem_desc(smem_u32(sDO), 0, 1024);
    const uint64_t q_mnmaj = umma_smem_desc(smem_u32(sQ), kQSub * 128, 1024);
    const uint64_t do_mnmaj = umma_smem_desc(smem_u32(sDO), kQSub * 128, 1024);
    const uint64_t dst_mnmaj = umma_smem_desc(smem_u32(sDSt), kTileBytes, 1024);
    auto issue_scores = [&](int u) {             // u: GLOBAL sub-block index
      const int x = u & 1;
      const uint64_t boff = static_cast<uint64_t>((u & 3) * kSub16);
      mbar_wait(&bar_qd[u & 3], (u >> 2) & 1);
      tc_fence_after_sync();
      const uint32_t t_s = tmem_base + x * 128, t_dp = t_s + 64;
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < kDh / 16; ++k) tc_mma_bf16(t_s, k_kmaj + 2 * k, q_kmaj + boff + 2 * k, idesc_sc, k > 0);
#pragma unroll
        for (int k = 0; k < kDh / 16; ++k) tc_mma_bf16(t_dp, v_kmaj + 2 * k, do_kmaj + boff + 2 * k, idesc_sc, k > 0);
        tc_commit(&bar_s[x]);
      }
    };
    int g = 0, G = 0, item = 0;                  // global sub-block / 128-query-block / work-item counters of this CTA
    for (int w = blockIdx.x; w >= 0; ++item) {
    long long* tl = item == 0 ? tl_arg : nullptr;
    mbar_wait(bar_kv, item & 1);
    issue_scores(g);
    if (nsub > 1) issue_scores(g + 1);
    for (int u = 0; u < nsub; ++u, ++g) {
      const int hq = u & 1, x = g & 1;
      const uint64_t boff = static_cast<uint64_t>((g & 3) * kSub16);
      mbar_wait(&bar_pd[x], (g >> 1) & 1);
      if (u == 0 && item > 0) mbar_wait(bar_acc, (item - 1) & 1);   // dV/dK of the previous item have left TMEM
      VITK_STAMP(16 * u + 0);
      tc_fence_after_sync();
      const uint32_t t_p = tmem_base + x * 128, t_ds = t_p + 64;
      const bool block_done = hq == 1 || u == nsub - 1;
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < kQSub / 16; ++k)   // dV[key,d] += Σ_q Pᵀ[key,q]·dO[q,d]; Pᵀ of column group k sits at Sᵀ column 16k
          tc_mma_bf16_ts(tm_dv, t_p + 16 * k, do_mnmaj + boff + 128 * k, idesc_km, (u > 0 || k > 0) ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < kQSub / 16; ++k)   // dK[key,d] += Σ_q dSᵀ[key,q]·Q[q,d]
          tc_mma_bf16_ts(tm_dk, t_ds + 16 * k, q_mnmaj + boff + 128 * k, idesc_km, (u > 0 || k > 0) ? 1u : 0u);
        tc_commit(&bar_free[g & 3]);
        if (block_done) {
#pragma unroll
          for (int k = 0; k < kTile / 16; ++k)   // dQ[q,d] = Σ_key dS[q,key]·K[key,d]; A = dSᵀ smem tile read MN-major
            tc_mma_bf16(tm_dq + (G & 1) * kDh, dst_mnmaj + static_cast<uint64_t>((G & 1) * 2 * kTile16) + 128 * k,
                        k_mnmaj + 128 * k, idesc_mm, k > 0);
          tc_commit(bar_g);
          if (u == nsub - 1) tc_commit(bar_item);
        }
      }
      if (block_done) ++G;
      VITK_STAMP(16 * u + 1);
      if (u + 2 < nsub) issue_scores(g + 2);   // queued right behind: MMAs retire in issue order
      VITK_STAMP(16 * u + 2);
      VITK_STAMP(16 * u + 3);
    }
    mbar_wait(&bar_id[(item + 1) & 1], (item >> 1) & 1);            // the load warp drew the next item long ago (item n is the
                                                                    // ⌊(n−1)/2⌋-th publication on slot n & 1: item 0 is never published)
    w = item_ring[(item + 1) & 1];
    }
    __syncwarp();
  } else if (warp == kBwdComputeWarps + 1) {
    // ------------------------------------------------------------------ load warp: K/V once, then the Q/dO ring.
    // (A separate warp: waiting here for a ring slot to be released — i.e. for dV/dK MMAs to retire — must not
    // hold up the MMA-issue warp, which would stall the whole score → softmax → dV/dK chain of the other buffer.)
    int g = 0, item = 0;
    int drawn = 0;                                         // lane 0: the draw in flight (the index of item + 1)
    if (lane == 0) drawn = static_cast<int>(gridDim.x) + atomicAdd(work_counter, 1);
    for (int w = blockIdx.x; w >= 0; ++item) {
      const int kb = w % nq, h = (w / nq) % H, b = w / (nq * H);
      const int colq = h * kDh, colk = (H + h) * kDh, colv = (2 * H + h) * kDh;
      if (item > 0) mbar_wait(bar_item, (item - 1) & 1);   // the previous item's MMAs no longer read K / V
      if (elect_one()) {
        mbar_arrive_expect_tx(bar_kv, 2 * kTileBytes);
        tma_load_3d(sK, &tma_qkv, bar_kv, colk, kb * kTile, b);
        tma_load_3d(sV, &tma_qkv, bar_kv, colv, kb * kTile, b);
      }
      // publish item + 1 (drawn a whole item ago, so the atomic's round trip — behind the bulk reduce-adds in L2 — is
      // never waited for) and draw item + 2.  Every warp has started item − 1 by now (its MMAs have retired), so slot
      // (item + 1) & 1, last read when item − 1 began, is free.
      int nxt = __shfl_sync(0xffffffffu, drawn, 0);
      nxt = nxt < total_items ? nxt : -1;
      if (lane == 0) {
        item_ring[(item + 1) & 1] = nxt;
        mbar_arrive(&bar_id[(item + 1) & 1]);              // (release: the store above is visible to whoever passes the wait)
        if (nxt >= 0) drawn = static_cast<int>(gridDim.x) + atomicAdd(work_counter, 1);
      }
      for (int u = 0; u < nsub; ++u, ++g) {  // sub-block g → ring slot g&3, last used by sub-block g−4: wait until its dV/dK retired
        const int slot = g & 3;
        if (g >= 4) mbar_wait(&bar_free[slot], ((g - 4) >> 2) & 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&bar_qd[slot], 2 * kQSub * 128);
          tma_load_3d(sQ + slot * (kQSub * 128), &tma_q64, &bar_qd[slot], colq, u * kQSub, b);
          tma_load_3d(sDO + slot * (kQSub * 128), &tma_do64, &bar_qd[slot], colq, u * kQSub, b);
        }
      }
      w = nxt;
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ compute warps
    const int quad = warp & 3, cg = warp >> 2;
    const int key_row = quad * 32 + lane;  // TMEM lane = key (Sᵀ, dPᵀ, dV, dK) or query (dQ)
    const uint32_t lane_field = static_cast<uint32_t>(quad * 32) << 16;
    // this warp's 32 query rows × 16 head-dim columns of dQ_i: TMEM → swizzled slab → one TMA reduce-add into the
    // fp32 accumulator (rows ≥ T are clipped by the tensor map)
    uint8_t* dq_slab = smem + kBwdSmemDqS + warp * 2048;
    int g = 0, item = 0;
    for (int w = blockIdx.x; w >= 0; ++item) {
    long long* tl = item == 0 ? tl_arg : nullptr;
    const int kb = w % nq, h = (w / nq) % H, b = w / (nq * H);
    const int key0 = kb * kTile;
    const int G0 = item * nq;                      // global index of this item's first 128-query block
    const float* stat_lse = lse2 + (static_cast<long long>(b) * H + h) * Tpad + cg * 16;
    const float* stat_dlt = delta + (static_cast<long long>(b) * H + h) * Tpad + cg * 16;
    auto reduce_dq = [&](int i) {                  // i: block index within the item; TMEM buffer / barrier parity by G0 + i
      uint32_t r[16];
      tmem_ld_32x16(tm_dq + ((G0 + i) & 1) * kDh + lane_field + cg * 16, r);
      if (elect_one()) tma_store_wait_read<0>();   // previous block's reduce has finished reading the slab
      __syncwarp();
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 4; ++j)
        *reinterpret_cast<uint4*>(dq_slab + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) =
            make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        tma_reduce_add_3d(&tma_dq, dq_slab, h * kDh + cg * 16, i * kTile + quad * 32, b);
        tma_store_commit();
      }
    };
    // statistics of this warp's 16 queries (padded arrays: unconditional aligned loads), fetched one sub-block ahead
    float4 l4[4], d4[4];
#pragma unroll
    for (int y = 0; y < 4; ++y) {
      l4[y] = __ldg(reinterpret_cast<const float4*>(stat_lse) + y);
      d4[y] = __ldg(reinterpret_cast<const float4*>(stat_dlt) + y);
    }
    for (int u = 0; u < nsub; ++u, ++g) {
      const int i = u >> 1, hq = u & 1, x = g & 1;
      if (warp == 0) VITK_STAMP(16 * u + 8);
      mbar_wait(&bar_s[x], (g >> 1) & 1);
      if (warp == 0) VITK_STAMP(16 * u + 9);
      tc_fence_after_sync();
      const uint32_t t_s = tmem_base + x * 128 + lane_field + cg * 16, t_dp = t_s + 64;
      uint32_t rs[16], rp[16];
      tmem_ld_32x16(t_s, rs);
      tmem_ld_32x16(t_dp, rp);
      tmem_ld_wait();
      if (warp == 0) VITK_STAMP(16 * u + 10);
      uint32_t pk[8], dk[8];
#pragma unroll
      for (int y = 0; y < 4; ++y) {
        const float lv[4] = {l4[y].x, l4[y].y, l4[y].z, l4[y].w}, dv[4] = {d4[y].x, d4[y].y, d4[y].z, d4[y].w};
        float p[4], ds[4];
#pragma unroll
        for (int z = 0; z < 4; ++z) {
          p[z] = fast_exp2(fmaf(__uint_as_float(rs[4 * y + z]), scale_log2, -lv[z]));
          ds[z] = p[z] * (__uint_as_float(rp[4 * y + z]) - dv[z]);
        }
        pk[2 * y] = pack_bf16x2(p[0], p[1]);
        pk[2 * y + 1] = pack_bf16x2(p[2], p[3]);
        dk[2 * y] = pack_bf16x2(ds[0], ds[1]);
        dk[2 * y + 1] = pack_bf16x2(ds[2], ds[3]);
      }
      if (u + 1 < nsub) {           // next sub-block's statistics: in flight during the stores, fences and the next wait
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          l4[y] = __ldg(reinterpret_cast<const float4*>(stat_lse + (u + 1) * kQSub) + y);
          d4[y] = __ldg(reinterpret_cast<const float4*>(stat_dlt + (u + 1) * kQSub) + y);
        }
      }
      if (warp == 0) VITK_STAMP(16 * u + 11);
      tmem_st_32x8(t_s, pk);        // Pᵀ  → this warp's own (consumed) Sᵀ columns: A operand of dV
      tmem_st_32x8(t_dp, dk);       // dSᵀ → this warp's own dPᵀ columns: A operand of dK
      {                             // dSᵀ → smem tile [128 keys × 128 q] (two 64-query halves), A operand of dQ
        // (double-buffered by block parity: dQ of block i may still be pending when block i+1's first half is written)
        uint8_t* rowp = sDSt + ((G0 + i) & 1) * 2 * kTileBytes + hq * kTileBytes + key_row * 128;
        *reinterpret_cast<uint4*>(rowp + (((2 * cg) ^ (key_row & 7)) << 4)) = make_uint4(dk[0], dk[1], dk[2], dk[3]);
        *reinterpret_cast<uint4*>(rowp + (((2 * cg + 1) ^ (key_row & 7)) << 4)) = make_uint4(dk[4], dk[5], dk[6], dk[7]);
      }
      fence_proxy_async_smem();
      tmem_st_wait();
      tc_fence_before_sync();
      __syncwarp();
      if (warp == 0) VITK_STAMP(16 * u + 12);
      if (lane == 0) mbar_arrive(&bar_pd[x]);
      if (hq == 1 && i > 0) {       // dQ of the previous 128-query block: its MMAs were issued two sub-blocks ago
        mbar_wait(bar_g, (G0 + i - 1) & 1);
        tc_fence_after_sync();
        reduce_dq(i - 1);
      }
      if (warp == 0) VITK_STAMP(16 * u + 13);
    }
    if (nq > 1 && (nsub & 1)) {     // an odd tail sub-block skipped the hq == 1 step that drains block nq−2
      mbar_wait(bar_g, (G0 + nq - 2) & 1);
      tc_fence_after_sync();
      reduce_dq(nq - 2);
    }
    mbar_wait(bar_g, (G0 + nq - 1) & 1);
    tc_fence_after_sync();
    reduce_dq(nq - 1);
    // dV (cg 0,1) and dK·scale (cg 2,3) → dqkv[b, key, 2|1, h, :]  (while the last dQ reduce-adds complete)
    {
      const bool is_dv = cg < 2;
      const int c32 = (cg & 1) * 32;
      uint32_t r[32];
      tmem_ld_32x32((is_dv ? tm_dv : tm_dk) + lane_field + c32, r);
      tmem_ld_wait();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc);      // the next item's dV / dK MMAs may overwrite the accumulators
      const float mul = is_dv ? 1.0f : scale;
      const int key = key0 + key_row;
      if (key < T) {
        uint4* dst = reinterpret_cast<uint4*>(dqkv + ((static_cast<long long>(b) * T + key) * 3 + (is_dv ? 2 : 1)) * H * kDh +
                                              h * kDh + c32);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 w;
          w.x = pack_bf16x2(__uint_as_float(r[8 * q + 0]) * mul, __uint_as_float(r[8 * q + 1]) * mul);
          w.y = pack_bf16x2(__uint_as_float(r[8 * q + 2]) * mul, __uint_as_float(r[8 * q + 3]) * mul);
          w.z = pack_bf16x2(__uint_as_float(r[8 * q + 4]) * mul, __uint_as_float(r[8 * q + 5]) * mul);
          w.w = pack_bf16x2(__uint_as_float(r[8 * q + 6]) * mul, __uint_as_float(r[8 * q + 7]) * mul);
          dst[q] = w;
        }
      }
    }
    mbar_wait(&bar_id[(item + 1) & 1], (item >> 1) & 1);
    w = item_ring[(item + 1) & 1];
    }   // work items
    if (elect_one()) tma_store_wait_all<0>();   // the slabs must outlive the bulk reads; the reduce-adds complete before exit
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == kBwdComputeWarps) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kBwdTmemCols);
  }
}

// ============================================================================ attention probabilities
// probs[b,h,i,j] = exp2(S[i,j]·scale_log2 − lse[b,h,i]·log2e) as fp32 [B,H,T,T]: the softmax rows HF's
// eager_attention_forward returns (modeling_vit.py:185-190), recomputed from the qkv buffer and the lse attn_fwd wrote,
// with attn_fwd's scale_log2, so each row is the one whose P·V produced o.  Bound by the HBM write (T² floats per
// head and image, never read again on the GPU), not by the recompute.
// CTA = (128 queries, head, image): a control warp loads Q once and 128-key K blocks through a 3-deep TMA ring and
// issues S_j = Q·K_jᵀ (SS-MMA, M = N = 128) into one of two TMEM buffers, so block j+1's MMA overlaps block j's
// epilogue.  Four epilogue warps (thread = query row = TMEM lane) read 32-column chunks, exponentiate, transpose them
// through a padded [32 × 33] shared-memory slab per warp and store them as 128-byte rows (32 consecutive keys of one
// query) with streaming stores.  Row stride T·4 bytes is not 16-byte aligned for odd T (577), which rules out TMA and
// vector stores.  Keys and queries ≥ T (the zero-filled TMA padding) are never stored.  (Eight epilogue warps per CTA,
// two per TMEM lane quadrant, wrote no faster: see DESIGN.md §4 for what bounds the kernel.)
// ≈81 KB of shared memory → two CTAs per SM, whose 2 × 256 TMEM columns fill the SM's 512.
constexpr int kPrbEpiWarps = 4;
constexpr int kPrbThreads = (kPrbEpiWarps + 1) * 32;        // epilogue warps + control warp
constexpr int kPrbKRing = 3;
constexpr int kPrbSmemQ = 0;
constexpr int kPrbSmemK = kPrbSmemQ + kTileBytes;
constexpr int kPrbSmemStage = kPrbSmemK + kPrbKRing * kTileBytes;    // 4 warps × [32 rows × 33 floats]
constexpr int kPrbStageFloats = 32 * 33;
constexpr int kPrbSmemBar = kPrbSmemStage + kPrbEpiWarps * kPrbStageFloats * 4;
constexpr int kPrbSmemBytes = kPrbSmemBar + 128 + 1024;
constexpr int kPrbTmemCols = 256;                           // two 128-column score buffers

__global__ void __launch_bounds__(kPrbThreads, 2)
attn_probs_kernel(const __grid_constant__ CUtensorMap tma_qk, const float* __restrict__ lse, int T, int H, float scale_log2,
                  float* __restrict__ probs) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem + kPrbSmemQ;
  uint8_t* sK = smem + kPrbSmemK;
  uint64_t* bar_q = reinterpret_cast<uint64_t*>(smem + kPrbSmemBar);
  uint64_t* bar_k = bar_q + 1;        // [3] K block landed
  uint64_t* bar_kfree = bar_q + 4;    // [3] the MMA reading this K slot retired
  uint64_t* bar_s = bar_q + 7;        // [2] scores of this TMEM buffer ready
  uint64_t* bar_tfree = bar_q + 9;    // [2] the 4 epilogue warps have read this TMEM buffer
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_q + 11);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int nkb = (T + kTile - 1) / kTile;

  if (tid == 0) {
    tma_prefetch_desc(&tma_qk);
    for (int i = 0; i < 11; ++i) mbar_init(bar_q + i, (i == 9 || i == 10) ? kPrbEpiWarps : 1);
    fence_mbar_init();
  }
  if (warp == kPrbEpiWarps) tmem_alloc(tmem_slot, kPrbTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  pdl_wait();
  pdl_launch_dependents();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == kPrbEpiWarps) {
    // ------------------------------------------------------------------ control warp: TMA + MMA issue (under elect.sync)
    const int colq = h * kDh, colk = (H + h) * kDh;
    auto load_k = [&](int j) {
      const int s = j % kPrbKRing;
      if (elect_one()) {
        mbar_arrive_expect_tx(&bar_k[s], kTileBytes);
        tma_load_3d(sK + s * kTileBytes, &tma_qk, &bar_k[s], colk, j * kTile, b);
      }
    };
    if (elect_one()) {
      mbar_arrive_expect_tx(bar_q, kTileBytes);
      tma_load_3d(sQ, &tma_qk, bar_q, colq, qb * kTile, b);
    }
    for (int j = 0; j < nkb && j < kPrbKRing; ++j) load_k(j);
    const uint64_t q_desc = umma_smem_desc(smem_u32(sQ), 0, 1024);
    const uint64_t k_desc = umma_smem_desc(smem_u32(sK), 0, 1024);
    constexpr uint32_t idesc = umma_idesc_bf16(kTile, kTile, 0, 0);
    mbar_wait(bar_q, 0);
    for (int j = 0; j < nkb; ++j) {
      const int s = j % kPrbKRing, x = j & 1;
      const uint32_t ph = (j / kPrbKRing) & 1;
      mbar_wait(&bar_k[s], ph);
      if (j >= 2) mbar_wait(&bar_tfree[x], ((j - 2) >> 1) & 1);
      tc_fence_after_sync();
      const uint64_t bk = k_desc + static_cast<uint64_t>(s * (kTileBytes >> 4));
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < kDh / 16; ++k) tc_mma_bf16(tmem_base + x * kTile, q_desc + 2 * k, bk + 2 * k, idesc, k > 0);
        tc_commit(&bar_s[x]);
        tc_commit(&bar_kfree[s]);
      }
      __syncwarp();
      if (j + kPrbKRing < nkb) {
        mbar_wait(&bar_kfree[s], ph);
        load_k(j + kPrbKRing);
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ epilogue warps
    const uint32_t lane_field = static_cast<uint32_t>(warp * 32) << 16;
    const int row0 = qb * kTile + warp * 32;          // first query row of this warp
    const bool live = row0 < T;                        // false: all 32 rows are padding beyond T
    const long long bh = static_cast<long long>(b) * H + h;
    const int my_row = row0 + lane;
    const float lse2 = my_row < T ? __ldg(lse + bh * T + my_row) * kLog2e : 0.f;
    const int nrows = min(32, T - row0);
    float* stage = reinterpret_cast<float*>(smem + kPrbSmemStage) + warp * kPrbStageFloats;
    float* out_rows = probs + (bh * T + row0) * T;      // row row0 of this (image, head)
    for (int j = 0; j < nkb; ++j) {
      const int x = j & 1;
      mbar_wait(&bar_s[x], (j >> 1) & 1);
      tc_fence_after_sync();
      const int nchunk = (min(kTile, T - j * kTile) + 31) >> 5;
      for (int c = 0; live && c < nchunk; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + lane_field + x * kTile + c * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i)     // (≤ 1: a row's maximum can round a few ulp above its lse)
          stage[lane * 33 + i] = fminf(fast_exp2(fmaf(__uint_as_float(r[i]), scale_log2, -lse2)), 1.0f);
        __syncwarp();
        const int col = j * kTile + c * 32 + lane;
        if (col < T) {
#pragma unroll 8
          for (int i = 0; i < nrows; ++i) __stcs(out_rows + static_cast<long long>(i) * T + col, stage[i * 33 + lane]);
        }
        __syncwarp();
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tfree[x]);
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == kPrbEpiWarps) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kPrbTmemCols);
  }
}

// dq_acc fp32 [B,T,H,64] · scale → dqkv[b,t,0,h,:] bf16
__global__ void __launch_bounds__(256) attn_dq_store_kernel(const float* __restrict__ dq_acc, int BT, int H, float scale,
                                                            __nv_bfloat16* __restrict__ dqkv) {
  pdl_wait();
  pdl_launch_dependents();
  const long long i8 = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;  // 8 elements each
  const int D = H * kDh;
  const long long total = static_cast<long long>(BT) * D / 8;
  if (i8 >= total) return;
  const long long row = (i8 * 8) / D;
  const int col = static_cast<int>((i8 * 8) - row * D);
  const float4 a = __ldg(reinterpret_cast<const float4*>(dq_acc) + 2 * i8);
  const float4 c = __ldg(reinterpret_cast<const float4*>(dq_acc) + 2 * i8 + 1);
  uint4 w;
  w.x = pack_bf16x2(a.x * scale, a.y * scale);
  w.y = pack_bf16x2(a.z * scale, a.w * scale);
  w.z = pack_bf16x2(c.x * scale, c.y * scale);
  w.w = pack_bf16x2(c.z * scale, c.w * scale);
  *reinterpret_cast<uint4*>(dqkv + row * 3 * D + col) = w;
}

static int qkv_tensor_map(CUtensorMap* m, const void* base, int64_t B, int64_t T, int64_t row_elems, int rows = kTile) {
  const uint64_t dims[3] = {static_cast<uint64_t>(row_elems), static_cast<uint64_t>(T), static_cast<uint64_t>(B)};
  const uint64_t str[2] = {static_cast<uint64_t>(row_elems) * 2, static_cast<uint64_t>(T) * row_elems * 2};
  const uint32_t box[3] = {kDh, static_cast<uint32_t>(rows), 1};
  return make_tensor_map_bf16(m, base, 3, dims, str, box);
}

static int check_shape(const char* who, int64_t B, int64_t T, int64_t H) {
  VITK_REQUIRE(B > 0 && T > 0 && H > 0 && B < 65536 && H < 65536 && T < (1 << 24), VITK_EINVAL,
               "%s: unsupported shape B=%lld T=%lld H=%lld", who, (long long)B, (long long)T, (long long)H);
  return 0;
}

}  // namespace vitk

using namespace vitk;

extern "C" VITK_API int vitk_attn_fwd(const void* qkv, int64_t B, int64_t T, int64_t H, float scale, void* o, float* lse,
                             vitk_stream_t stream) {
  VITK_REQUIRE(qkv && o && lse, VITK_EINVAL, "attn_fwd: NULL argument");
  if (int rc = check_shape("attn_fwd", B, T, H)) return rc;
  VITK_REQUIRE(aligned16(qkv) && aligned16(o), VITK_EALIGN, "attn_fwd: buffers must be 16-byte aligned");
  VITK_REQUIRE(scale > 0.f, VITK_EINVAL, "attn_fwd: scale must be positive");
  CUtensorMap tm, tm_kv, tm_o;
  if (int rc = qkv_tensor_map(&tm, qkv, B, T, 3 * H * kDh)) return rc;
  if (int rc = qkv_tensor_map(&tm_kv, qkv, B, T, 3 * H * kDh, kSub)) return rc;
  if (int rc = qkv_tensor_map(&tm_o, o, B, T, H * kDh)) return rc;
  static std::atomic<int> attr_done{0};
  if (!attr_done.load()) {
    VITK_CUDA(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFwdSmemBytes));
    attr_done.store(1);
  }
  const dim3 grid(static_cast<unsigned>((T + kTile - 1) / kTile), static_cast<unsigned>(H), static_cast<unsigned>(B));
  VITK_CUDA(launch_pdl(attn_fwd_kernel, grid, dim3(kFwdThreads), kFwdSmemBytes, static_cast<cudaStream_t>(stream), tm, tm_kv,
                       tm_o, lse, static_cast<int>(T), static_cast<int>(H), scale * kLog2e, g_timeline));
  VITK_LAUNCH_CHECK("attn_fwd_kernel");
  return 0;
}

extern "C" VITK_API int vitk_attn_probs(const void* qkv, const float* lse, int64_t B, int64_t T, int64_t H, float scale,
                                        float* probs, vitk_stream_t stream) {
  VITK_REQUIRE(qkv && lse && probs, VITK_EINVAL, "attn_probs: NULL argument");
  if (int rc = check_shape("attn_probs", B, T, H)) return rc;
  VITK_REQUIRE(aligned16(qkv) && (reinterpret_cast<uintptr_t>(lse) & 3u) == 0 && (reinterpret_cast<uintptr_t>(probs) & 3u) == 0,
               VITK_EALIGN, "attn_probs: qkv must be 16-byte aligned, lse and probs 4-byte aligned");
  VITK_REQUIRE(scale > 0.f, VITK_EINVAL, "attn_probs: scale must be positive");
  CUtensorMap tm;
  if (int rc = qkv_tensor_map(&tm, qkv, B, T, 3 * H * kDh)) return rc;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(attn_probs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPrbSmemBytes);
  });
  if (attr_err != cudaSuccess) return cuda_error(attr_err, "cudaFuncSetAttribute(attn_probs smem)");
  const dim3 grid(static_cast<unsigned>((T + kTile - 1) / kTile), static_cast<unsigned>(H), static_cast<unsigned>(B));
  VITK_CUDA(launch_pdl(attn_probs_kernel, grid, dim3(kPrbThreads), kPrbSmemBytes, static_cast<cudaStream_t>(stream), tm, lse,
                       static_cast<int>(T), static_cast<int>(H), scale * kLog2e, probs));
  VITK_LAUNCH_CHECK("attn_probs_kernel");
  return 0;
}

extern "C" VITK_API int vitk_debug_timeline(void* device_buf) {
  g_timeline = static_cast<long long*>(device_buf);
  g_timeline_seq = 0;
  return 0;
}

__global__ void debug_stamp_kernel(long long* dst) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  *dst = static_cast<long long>(t);
}
extern "C" VITK_API int vitk_debug_stamp(int64_t slot, void* stream) {
  VITK_REQUIRE(g_timeline != nullptr && slot >= 0, VITK_EINVAL, "vitk_debug_stamp: no timeline buffer set");
  debug_stamp_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(g_timeline + slot);
  VITK_LAUNCH_CHECK("debug_stamp_kernel");
  return 0;
}

static size_t bwd_stats_bytes(int64_t B, int64_t T, int64_t H) {
  const int64_t Tpad = (T + kTile - 1) / kTile * kTile;
  return (static_cast<size_t>(B) * H * Tpad * sizeof(float) + 255) / 256 * 256;
}
static size_t bwd_dq_bytes(int64_t B, int64_t T, int64_t H) {
  return (static_cast<size_t>(B) * T * H * kDh * sizeof(float) + 255) / 256 * 256;
}
// workspace = fp32 dQ accumulator [B,T,H,64] | work-item counter (256 B, cleared with the accumulator) | lse·log2e [B,H,Tpad] | Δ [B,H,Tpad]
constexpr size_t kBwdCounterBytes = 256;
extern "C" VITK_API size_t vitk_attn_bwd_workspace_bytes(int64_t B, int64_t T, int64_t H) {
  return bwd_dq_bytes(B, T, H) + kBwdCounterBytes + 2 * bwd_stats_bytes(B, T, H);
}

extern "C" VITK_API int vitk_attn_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, int64_t B, int64_t T,
                             int64_t H, float scale, void* dqkv, void* workspace, vitk_stream_t stream) {
  VITK_REQUIRE(qkv && o && d_o && lse && dqkv && workspace, VITK_EINVAL, "attn_bwd: NULL argument");
  if (int rc = check_shape("attn_bwd", B, T, H)) return rc;
  VITK_REQUIRE(aligned16(qkv) && aligned16(o) && aligned16(d_o) && aligned16(dqkv) && aligned16(workspace), VITK_EALIGN,
               "attn_bwd: buffers must be 16-byte aligned");
  VITK_REQUIRE(scale > 0.f, VITK_EINVAL, "attn_bwd: scale must be positive");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t dq_bytes = bwd_dq_bytes(B, T, H);
  const int Tpad = static_cast<int>((T + kTile - 1) / kTile * kTile);
  float* dq_acc = static_cast<float*>(workspace);
  int* work_counter = reinterpret_cast<int*>(static_cast<uint8_t*>(workspace) + dq_bytes);
  float* lse2 = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + dq_bytes + kBwdCounterBytes);
  float* delta = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + dq_bytes + kBwdCounterBytes + bwd_stats_bytes(B, T, H));
  CUtensorMap tm_qkv, tm_q64, tm_do, tm_dq;
  if (int rc = qkv_tensor_map(&tm_qkv, qkv, B, T, 3 * H * kDh)) return rc;
  if (int rc = qkv_tensor_map(&tm_q64, qkv, B, T, 3 * H * kDh, kQSub)) return rc;
  if (int rc = qkv_tensor_map(&tm_do, d_o, B, T, H * kDh, kQSub)) return rc;
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(H * kDh), static_cast<uint64_t>(T), static_cast<uint64_t>(B)};
    const uint64_t str[2] = {static_cast<uint64_t>(H * kDh) * 4, static_cast<uint64_t>(T) * H * kDh * 4};
    const uint32_t box[3] = {16, 32, 1};
    if (int rc = get_tensor_map(&tm_dq, dq_acc, TM_F32, 3, dims, str, box, TM_SW64)) return rc;
  }
  static std::atomic<int> attr_done{0};
  if (!attr_done.load()) {
    VITK_CUDA(cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBwdSmemBytes));
    attr_done.store(1);
  }
  VITK_CUDA(cudaMemsetAsync(dq_acc, 0, dq_bytes + kBwdCounterBytes, s));
  const int BT = static_cast<int>(B * T);
  {
    const __nv_bfloat16* po = static_cast<const __nv_bfloat16*>(o);
    const __nv_bfloat16* pdo = static_cast<const __nv_bfloat16*>(d_o);
    const dim3 g16(static_cast<unsigned>(B * Tpad / 16)), g8((static_cast<int>(B) * Tpad + 7) / 8);
    if (H > 16) VITK_CUDA(launch_pdl(attn_delta_kernel, g8, dim3(256), 0, s, po, pdo, lse, (int)B, (int)T, Tpad, (int)H, lse2, delta));
    else if (H > 12) VITK_CUDA(launch_pdl(attn_delta16_kernel<4>, g16, dim3(256), 0, s, po, pdo, lse, (int)B, (int)T, Tpad, (int)H, lse2, delta));
    else if (H > 8) VITK_CUDA(launch_pdl(attn_delta16_kernel<3>, g16, dim3(256), 0, s, po, pdo, lse, (int)B, (int)T, Tpad, (int)H, lse2, delta));
    else if (H > 4) VITK_CUDA(launch_pdl(attn_delta16_kernel<2>, g16, dim3(256), 0, s, po, pdo, lse, (int)B, (int)T, Tpad, (int)H, lse2, delta));
    else VITK_CUDA(launch_pdl(attn_delta16_kernel<1>, g16, dim3(256), 0, s, po, pdo, lse, (int)B, (int)T, Tpad, (int)H, lse2, delta));
  }
  VITK_LAUNCH_CHECK("attn_delta_kernel");
  const long long items = ((T + kTile - 1) / kTile) * H * B;
  VITK_REQUIRE(items < (1ll << 30), VITK_EINVAL, "attn_bwd: too many (key block, head, image) work items");
  const long long ctas = items > num_sms() ? num_sms() : items;
  VITK_CUDA(launch_pdl(attn_bwd_kernel, dim3(static_cast<unsigned>(ctas)), dim3(kBwdThreads), kBwdSmemBytes, s, tm_qkv, tm_q64, tm_do, tm_dq,
                       static_cast<const float*>(lse2), static_cast<const float*>(delta), static_cast<__nv_bfloat16*>(dqkv), (int)T, Tpad,
                       (int)H, (int)B, scale, scale * kLog2e, work_counter, g_timeline));
  VITK_LAUNCH_CHECK("attn_bwd_kernel");
  const long long n8 = static_cast<long long>(BT) * H * kDh / 8;
  VITK_CUDA(launch_pdl(attn_dq_store_kernel, dim3(static_cast<unsigned>((n8 + 255) / 256)), dim3(256), 0, s,
                       static_cast<const float*>(dq_acc), BT, (int)H, scale, static_cast<__nv_bfloat16*>(dqkv)));
  VITK_LAUNCH_CHECK("attn_dq_store_kernel");
  return 0;
}
