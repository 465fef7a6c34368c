// Host side shared by the two GEMM kernels: per-epilogue facts, the launch plan (plan_gemm in gemm.cu decides every
// vitk_gemm_bf16 launch), the operand tensor maps and the CTA-pair launcher (gemm2.cu).
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "tmap.cuh"

namespace vitk {

// Indexed by vitk_epilogue.  Host code only: the kernels keep their own expressions of these facts, because the pair
// kernel's epilogues sit at 168- and 96-register caps that a rewritten test can push them over.
struct EpiTraits {
  bool f32_out;   // d is fp32
  bool aux;       // reads the aux matrix (the pair kernel has separate AUX instantiations)
  bool pair;      // the CTA-pair kernel implements it
};
constexpr EpiTraits kEpiTraits[] = {
    /* STORE_BF16      */ {false, false, true},
    /* BIAS_BF16       */ {false, false, true},
    /* BIAS_GELU_BF16  */ {false, false, true},
    /* BIAS_RESID_F32  */ {true, true, true},
    /* PATCH_F32       */ {true, true, false},
    /* DGELU_BF16      */ {false, true, true},
    /* ACCUM_F32       */ {true, false, true},
    /* STORE_F32       */ {true, false, true},
    /* BIAS_GELUG_BF16 */ {false, false, true},
    /* MUL_BF16        */ {false, true, true},
    /* UNPATCH_F32     */ {true, false, false},
};
static_assert(sizeof(kEpiTraits) / sizeof(kEpiTraits[0]) == VITK_EPI_UNPATCH_F32 + 1, "one row per epilogue");

enum GemmKernel {
  GEMM_SINGLE_CTA = 1,   // gemm_bf16_kernel, 128-row tiles
  GEMM_PAIR = 2,         // gemm2_bf16_kernel, 256-row tiles, 8 epilogue warps
  GEMM_PAIR_EW16 = 3,    // gemm2_bf16_kernel with 16 epilogue warps and BIAS_GELUG_BF16 fixed at compile time
};

struct GemmPlan {
  int kernel;         // GemmKernel
  int bn;             // tile width in columns
  int n_half;         // pair kernel: tiles per band that are bn/2 wide (the last n_half of n_tiles); 0 otherwise
  int n_tiles, mn_tiles, kb_total, kb_per_split, k_splits, total_work;   // as in GemmParams / Gemm2Params
  int ctas;           // grid size in CTAs
};

// Validates a vitk_gemm_bf16 call (the operand pointers' values only, never what they point to) and decides its
// launch on a GPU with `sms` SMs.
int plan_gemm(const vitk_gemm_args& a, int sms, GemmPlan* out);

int launch_pair(const vitk_gemm_args& a, const GemmPlan& plan, cudaStream_t stream);   // gemm2.cu

// bf16 operand A (rows = M) or B (rows = N), 128-byte swizzle, 64-wide K boxes.  K-major: dims {K, rows}, box
// {64, box_rows}; MN-major: dims {rows, K}, box {64, 64} (an MN-major tile is staged as several boxes).
inline int operand_map(CUtensorMap* m, const void* base, bool mn_major, long long rows, long long K, long long ld,
                       uint32_t box_rows) {
  const uint64_t dims[2] = {static_cast<uint64_t>(mn_major ? rows : K), static_cast<uint64_t>(mn_major ? K : rows)};
  const uint64_t str[1] = {static_cast<uint64_t>(ld) * 2};
  const uint32_t box[2] = {64, mn_major ? 64u : box_rows};
  return make_tensor_map_bf16(m, base, 2, dims, str, box);
}

}  // namespace vitk
