// Position-embedding resize for inputs of another size than the checkpoint's (HF interpolate_pos_encoding,
// modeling_vit.py:60-99): row 0 (CLS) is copied, rows 1.. are a gh0×gw0 grid resized bicubically to gh×gw, and the
// exact adjoint of that map for the backward.
//
// The 1-D map is torch's upsample_bicubic2d with align_corners=False and no scale factor: output index o of n_out reads
// source coordinate s = (o + 0.5)·n_in/n_out − 0.5 (not clamped), taps floor(s) − 1 … floor(s) + 2 clamped to
// [0, n_in − 1], cubic convolution weights with A = −0.75 (ATen UpSample.h, upsample_get_cubic_coefficients).  The
// integer and fractional parts of s come from exact integer arithmetic, s = ((2o + 1)·n_in − n_out) / (2·n_out), so the
// weights are within an ulp of the fp64 ones whatever the grid size.
#include <cuda_runtime.h>

#include "common.cuh"

namespace vitk {

__device__ __forceinline__ void cubic_taps(int o, int n_in, int n_out, int (&idx)[4], float (&w)[4]) {
  const long long num = (2ll * o + 1) * n_in - n_out, den = 2ll * n_out;
  long long q = num / den;
  if (num < 0 && q * den != num) --q;                                  // floor, not truncation
  const float t = static_cast<float>(num - q * den) / static_cast<float>(den);
  constexpr float A = -0.75f;
  const float x1 = t, x2 = 1.f - t;
  w[0] = ((A * (x1 + 1.f) - 5.f * A) * (x1 + 1.f) + 8.f * A) * (x1 + 1.f) - 4.f * A;
  w[1] = ((A + 2.f) * x1 - (A + 3.f)) * x1 * x1 + 1.f;
  w[2] = ((A + 2.f) * x2 - (A + 3.f)) * x2 * x2 + 1.f;
  w[3] = ((A * (x2 + 1.f) - 5.f * A) * (x2 + 1.f) + 8.f * A) * (x2 + 1.f) - 4.f * A;
#pragma unroll
  for (int k = 0; k < 4; ++k) idx[k] = static_cast<int>(min(max(q - 1 + k, 0ll), static_cast<long long>(n_in - 1)));
}

// One block per output row, one thread per 4 channels.  Each thread derives the same 8 weights of its output position
// (a few dozen instructions, cheaper than a shared-memory round trip) and contracts separably in a fixed order:
// out = Σ_a wy[a] · (Σ_b wx[b] · pos[iy[a], ix[b]]).
__global__ void pos_interp_kernel(const float4* __restrict__ pos, int gh0, int gw0, int gh, int gw, int D4,
                                  float4* __restrict__ out) {
  const int t = blockIdx.x, c = threadIdx.x;
  if (c >= D4) return;
  if (t == 0) {
    out[c] = __ldg(pos + c);
    return;
  }
  const int oy = (t - 1) / gw, ox = (t - 1) - oy * gw;
  int iy[4], ix[4];
  float wy[4], wx[4];
  cubic_taps(oy, gh0, gh, iy, wy);
  cubic_taps(ox, gw0, gw, ix, wx);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* row = pos + (1ll + static_cast<long long>(iy[a]) * gw0) * D4 + c;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const float4 v = __ldg(row + static_cast<long long>(ix[b]) * D4);
      r.x = fmaf(wx[b], v.x, r.x); r.y = fmaf(wx[b], v.y, r.y); r.z = fmaf(wx[b], v.z, r.z); r.w = fmaf(wx[b], v.w, r.w);
    }
    acc.x = fmaf(wy[a], r.x, acc.x); acc.y = fmaf(wy[a], r.y, acc.y);
    acc.z = fmaf(wy[a], r.z, acc.z); acc.w = fmaf(wy[a], r.w, acc.w);
  }
  out[static_cast<long long>(t) * D4 + c] = acc;
}

// Adjoint as a gather: one block per INPUT row, one thread per 4 channels, so every dpos element has one owner and no
// atomics are needed.  The block first builds the columns Wy[:, iy] and Wx[:, ix] of the dense 1-D matrices (clamped taps
// folded in) in shared memory, with the range of output rows / columns where they can be non-zero; then
// dpos[iy, ix] += Σ_oy Wy[oy, iy] · (Σ_ox Wx[ox, ix] · dout[oy, ox]) in ascending order — the same bits on every run.
__global__ void pos_interp_bwd_kernel(const float4* __restrict__ dout, int gh, int gw, int gh0, int gw0, int D4,
                                      float4* __restrict__ dpos) {
  extern __shared__ float wcol[];              // [gh] column iy of Wy, then [gw] column ix of Wx
  __shared__ int lo_y, hi_y, lo_x, hi_x;
  const int t = blockIdx.x, c = threadIdx.x;
  if (t == 0) {
    if (c < D4) {
      const float4 g = __ldg(dout + c);
      float4 d = dpos[c];
      d.x += g.x; d.y += g.y; d.z += g.z; d.w += g.w;
      dpos[c] = d;
    }
    return;
  }
  const int iy = (t - 1) / gw0, ix = (t - 1) - iy * gw0;
  if (c == 0) {
    lo_y = gh; hi_y = -1; lo_x = gw; hi_x = -1;
  }
  __syncthreads();
  float* wy_col = wcol;
  float* wx_col = wcol + gh;
  for (int o = c; o < gh + gw; o += blockDim.x) {
    const bool is_y = o < gh;
    const int oo = is_y ? o : o - gh;
    int idx[4];
    float w[4];
    cubic_taps(oo, is_y ? gh0 : gw0, is_y ? gh : gw, idx, w);
    const int want = is_y ? iy : ix;
    float s = 0.f;
    bool hit = false;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (idx[k] == want) {
        s += w[k];
        hit = true;
      }
    wcol[o] = s;
    if (hit) {
      atomicMin(is_y ? &lo_y : &lo_x, oo);
      atomicMax(is_y ? &hi_y : &hi_x, oo);
    }
  }
  __syncthreads();
  if (c >= D4) return;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int oy = lo_y; oy <= hi_y; ++oy) {
    const float wy = wy_col[oy];
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* row = dout + (1ll + static_cast<long long>(oy) * gw) * D4 + c;
    for (int ox = lo_x; ox <= hi_x; ++ox) {
      const float wx = wx_col[ox];
      const float4 v = __ldg(row + static_cast<long long>(ox) * D4);
      r.x = fmaf(wx, v.x, r.x); r.y = fmaf(wx, v.y, r.y); r.z = fmaf(wx, v.z, r.z); r.w = fmaf(wx, v.w, r.w);
    }
    acc.x = fmaf(wy, r.x, acc.x); acc.y = fmaf(wy, r.y, acc.y);
    acc.z = fmaf(wy, r.z, acc.z); acc.w = fmaf(wy, r.w, acc.w);
  }
  float4* d = dpos + static_cast<long long>(t) * D4 + c;
  float4 v = *d;
  v.x += acc.x; v.y += acc.y; v.z += acc.z; v.w += acc.w;
  *d = v;
}

static int check_interp_args(const char* what, const void* src, const void* dst, int64_t gh0, int64_t gw0, int64_t gh,
                             int64_t gw, int64_t D) {
  VITK_REQUIRE(src && dst, VITK_EINVAL, "%s: NULL argument", what);
  VITK_REQUIRE(gh0 >= 1 && gw0 >= 1 && gh >= 1 && gw >= 1 && gh0 <= 4096 && gw0 <= 4096 && gh <= 4096 && gw <= 4096 &&
                   gh0 * gw0 < (1ll << 24) && gh * gw < (1ll << 24),
               VITK_EINVAL, "%s: grids must be 1..4096 on each side with fewer than 2^24 positions (%lldx%lld -> %lldx%lld)",
               what, (long long)gh0, (long long)gw0, (long long)gh, (long long)gw);
  VITK_REQUIRE(D >= 4 && D <= 4096 && D % 4 == 0, VITK_EINVAL, "%s: D=%lld must be a multiple of 4 in [4, 4096]", what,
               (long long)D);
  VITK_REQUIRE(aligned16(src) && aligned16(dst), VITK_EALIGN, "%s: buffers must be 16-byte aligned", what);
  return 0;
}

}  // namespace vitk

using namespace vitk;

extern "C" VITK_API int vitk_pos_interp(const float* pos, int64_t gh0, int64_t gw0, int64_t gh, int64_t gw, int64_t D, float* out,
                                        vitk_stream_t stream) {
  if (int rc = check_interp_args("pos_interp", pos, out, gh0, gw0, gh, gw, D)) return rc;
  const int D4 = static_cast<int>(D / 4);
  pos_interp_kernel<<<static_cast<unsigned>(1 + gh * gw), (D4 + 31) / 32 * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(pos), (int)gh0, (int)gw0, (int)gh, (int)gw, D4, reinterpret_cast<float4*>(out));
  VITK_LAUNCH_CHECK("pos_interp_kernel");
  return 0;
}

extern "C" VITK_API int vitk_pos_interp_bwd(const float* dout, int64_t gh, int64_t gw, int64_t gh0, int64_t gw0, int64_t D,
                                            float* dpos, vitk_stream_t stream) {
  if (int rc = check_interp_args("pos_interp_bwd", dout, dpos, gh0, gw0, gh, gw, D)) return rc;
  const int D4 = static_cast<int>(D / 4);
  const size_t smem = static_cast<size_t>(gh + gw) * sizeof(float);      // <= 32 KB
  pos_interp_bwd_kernel<<<static_cast<unsigned>(1 + gh0 * gw0), (D4 + 31) / 32 * 32, smem, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(dout), (int)gh, (int)gw, (int)gh0, (int)gw0, D4, reinterpret_cast<float4*>(dpos));
  VITK_LAUNCH_CHECK("pos_interp_bwd_kernel");
  return 0;
}
