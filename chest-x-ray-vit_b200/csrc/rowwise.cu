// HBM-bound kernels of the path: input normalisation + im2col, LayerNorm fwd/bwd, bias-gradient
// column sums, embedding glue, fp32→bf16 parameter shadow.  All use 128-bit coalesced accesses and
// warp-shuffle reductions; fp32 statistics throughout.
#include <cuda_bf16.h>

#include "common.cuh"

namespace vitk {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ uint32_t bf2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unbf2(uint32_t w) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w));
}

// ------------------------------------------------------------------------- patchify
struct NormConst {
  float mean[3], std[3];
};

// thread = one 16-pixel row (ky) of one patch; consecutive threads = consecutive ky of the same
// patch, so for each channel 16 threads write 512 contiguous bytes of one im2col row.
__global__ void __launch_bounds__(256) patchify_u8_kernel(const uint8_t* __restrict__ gray, int B, int H, int W,
                                                          NormConst nc, __nv_bfloat16* __restrict__ out) {
  const int PW = W / 16, PH = H / 16;
  const long long total = static_cast<long long>(B) * PH * PW * 16;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int ky = static_cast<int>(idx & 15);
  const long long patch = idx >> 4;
  const int px = static_cast<int>(patch % PW);
  const long long t = patch / PW;
  const int py = static_cast<int>(t % PH);
  const int b = static_cast<int>(t / PH);
  const uint4 raw = __ldg(reinterpret_cast<const uint4*>(gray + (static_cast<long long>(b) * H + py * 16 + ky) * W + px * 16));
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
  float g[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) g[i] = __fdiv_rn(static_cast<float>((w[i >> 2] >> (8 * (i & 3))) & 0xffu), 255.0f);
  __nv_bfloat16* orow = out + patch * 768 + ky * 16;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    uint32_t pk[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      // (g/255 − mean)/std with IEEE sub and div: bit-identical to ToTensor+Normalize in fp32
      const float a = __fdiv_rn(__fsub_rn(g[2 * i], nc.mean[c]), nc.std[c]);
      const float d = __fdiv_rn(__fsub_rn(g[2 * i + 1], nc.mean[c]), nc.std[c]);
      pk[i] = bf2(a, d);
    }
    uint4* o = reinterpret_cast<uint4*>(orow + c * 256);
    o[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    o[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
  }
}

// fp32 NCHW drop-in input: thread = (patch, c, ky), 16 floats in, 16 bf16 out.
__global__ void __launch_bounds__(256) patchify_f32_kernel(const float* __restrict__ pix, int B, int H, int W,
                                                           __nv_bfloat16* __restrict__ out) {
  const int PW = W / 16, PH = H / 16;
  const long long total = static_cast<long long>(B) * PH * PW * 48;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int j = static_cast<int>(idx % 48);  // c*16 + ky
  const int c = j >> 4, ky = j & 15;
  const long long patch = idx / 48;
  const int px = static_cast<int>(patch % PW);
  const long long t = patch / PW;
  const int py = static_cast<int>(t % PH);
  const int b = static_cast<int>(t / PH);
  const float4* src = reinterpret_cast<const float4*>(pix + ((static_cast<long long>(b) * 3 + c) * H + py * 16 + ky) * W + px * 16);
  uint32_t pk[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 v = __ldg(src + i);
    pk[2 * i] = bf2(v.x, v.y);
    pk[2 * i + 1] = bf2(v.z, v.w);
  }
  uint4* o = reinterpret_cast<uint4*>(out + patch * 768 + j * 16);
  o[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  o[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
}

// ------------------------------------------------------------------------- horizontal flip (training augmentation)
// thread = one pair of mirrored 16-byte chunks of a row (or the middle chunk when W/16 is odd): load both, reverse the
// bytes of each, store them swapped.  Images whose mask byte is 0 are skipped by whole blocks (blockIdx.y = image).
__device__ __forceinline__ uint4 reverse16(uint4 v) {
  return make_uint4(__byte_perm(v.w, 0, 0x0123), __byte_perm(v.z, 0, 0x0123), __byte_perm(v.y, 0, 0x0123), __byte_perm(v.x, 0, 0x0123));
}
__global__ void __launch_bounds__(256) hflip_u8_kernel(uint8_t* __restrict__ gray, const uint8_t* __restrict__ mask, int H, int W) {
  const int b = blockIdx.y;
  if (mask[b] == 0) return;
  const int n = W / 16, pairs = (n + 1) / 2;                 // chunks per row; (left, right) pairs incl. a self-paired middle chunk
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(H) * pairs) return;
  const int row = static_cast<int>(idx / pairs), c = static_cast<int>(idx - static_cast<long long>(row) * pairs);
  uint4* r = reinterpret_cast<uint4*>(gray + (static_cast<long long>(b) * H + row) * W);
  const int m = n - 1 - c;
  const uint4 left = r[c];
  if (m == c) {
    r[c] = reverse16(left);
  } else {
    const uint4 right = r[m];
    r[c] = reverse16(right);
    r[m] = reverse16(left);
  }
}

// ------------------------------------------------------------------------- LayerNorm
// One warp per row; lane owns float4 chunks lane, lane+32, ... (VPL of them; D = 128·VPL).
template <int VPL>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const float* __restrict__ x, long long ldx,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            float eps, int M, long long rs, __nv_bfloat16* __restrict__ y,
                                                            float* __restrict__ mean, float* __restrict__ rstd) {
  // rs: logical row r is written to physical row r·rs of y / mean / rstd (x has its own ldx); rs = T keeps the CLS rows
  // of a [B,T,D] tensor in place
  constexpr int D = VPL * 128;
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<long long>(row) * ldx);
  float4 v[VPL];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    v[i] = __ldg(xr + lane + 32 * i);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mu = warp_sum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float r = rsqrtf(warp_sum(q) * (1.0f / D) + eps);
  if (lane == 0) {
    if (mean) mean[row * rs] = mu;
    if (rstd) rstd[row * rs] = r;
  }
  uint2* yr = reinterpret_cast<uint2*>(y + static_cast<long long>(row) * rs * D);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const float4 g = __ldg(g4 + lane + 32 * i), bb = __ldg(b4 + lane + 32 * i);
    const float o0 = (v[i].x - mu) * r * g.x + bb.x, o1 = (v[i].y - mu) * r * g.y + bb.y;
    const float o2 = (v[i].z - mu) * r * g.z + bb.z, o3 = (v[i].w - mu) * r * g.w + bb.w;
    yr[lane + 32 * i] = make_uint2(bf2(o0, o1), bf2(o2, o3));
  }
}

// dx = dres + r·(g − mean(g) − x̂·mean(g·x̂)), g = dy·γ.  A PAIR of warps owns a row (each warp half of the
// columns; the two row sums are exchanged through shared memory with a 64-thread named barrier), so a thread
// keeps only half of the dγ / dβ / Σdx partials and of the row in registers: ~60 registers instead of 174,
// 4× the resident warps of the one-warp-per-row version, which is what an HBM-bound kernel needs.  Pairs walk
// rows with a grid stride; one smem reduction + one atomicAdd per column per block at the end.
// rs: logical row r lives at physical row r·rs of dy / dres / dx / mean / rstd (x has its own ldx); rs = T walks
// only the CLS rows of a [B,T,D] tensor.
constexpr int kLnBwdBlocks = 2;   // resident blocks per SM the register budget is cut for (3 or 4 spilled and were slower)
template <int VPL>
__global__ void __launch_bounds__(256, kLnBwdBlocks) layernorm_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const float* __restrict__ x,
                                                               long long ldx, const float* __restrict__ mean,
                                                               const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                               const __nv_bfloat16* __restrict__ dres, int M, long long rs,
                                                               __nv_bfloat16* __restrict__ dx, float* __restrict__ dgamma,
                                                               float* __restrict__ dbeta, float* __restrict__ dxsum) {
  constexpr int D = VPL * 128;
  constexpr int kSplit = (VPL % 2 == 0) ? 2 : 1;   // warps per row
  constexpr int V = VPL / kSplit;                   // float4 chunks per lane
  pdl_wait();
  pdl_launch_dependents();
  extern __shared__ float red[];                    // [row slots][D] reused for dγ, dβ and Σdx
  __shared__ float2 xch[2][8];                      // [row parity][warp]: partial (Σg, Σg·x̂) of each warp
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int slot = warp / kSplit, half = warp % kSplit, nslots = nwarps / kSplit;
  const int c0 = half * V * 32 + lane;              // this lane's float4 chunks: c0 + 32·i
  const float4* gam4 = reinterpret_cast<const float4*>(gamma);
  float4 dg[V], db[V], dsx[V];
#pragma unroll
  for (int i = 0; i < V; ++i) {
    dg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    db[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    dsx[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // software pipeline: the next row's x / dy / dres are in flight while this row is reduced and written (24 more
  // registers than loading each row when it is reached)
  const int row_step = gridDim.x * nslots;
  int row = blockIdx.x * nslots + slot;
  float4 xn[V];
  uint2 dn[V], rn[V];
  auto fetch = [&](int rw) {
    const long long pr = static_cast<long long>(rw) * rs;
    const float4* xr = reinterpret_cast<const float4*>(x + static_cast<long long>(rw) * ldx);
    const uint2* dyr = reinterpret_cast<const uint2*>(dy + pr * D);
#pragma unroll
    for (int i = 0; i < V; ++i) {
      xn[i] = __ldg(xr + c0 + 32 * i);
      dn[i] = __ldg(dyr + c0 + 32 * i);
      rn[i] = dres ? __ldg(reinterpret_cast<const uint2*>(dres + pr * D) + c0 + 32 * i) : make_uint2(0u, 0u);
    }
  };
  if (row < M) fetch(row);
  int parity = 0;
  for (; row < M; row += row_step, parity ^= 1) {
    const long long prow = static_cast<long long>(row) * rs;
    const float mu = __ldg(mean + prow), r = __ldg(rstd + prow);
    float4 xv[V];
    uint2 dw[V], rw_[V];
#pragma unroll
    for (int i = 0; i < V; ++i) { xv[i] = xn[i]; dw[i] = dn[i]; rw_[i] = rn[i]; }
    if (row + row_step < M) fetch(row + row_step);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const float4 gm = __ldg(gam4 + c0 + 32 * i);
      const float2 d01 = unbf2(dw[i].x), d23 = unbf2(dw[i].y);
      const float h0 = (xv[i].x - mu) * r, h1 = (xv[i].y - mu) * r, h2 = (xv[i].z - mu) * r, h3 = (xv[i].w - mu) * r;
      const float g0 = d01.x * gm.x, g1 = d01.y * gm.y, g2 = d23.x * gm.z, g3 = d23.y * gm.w;
      s1 += (g0 + g1) + (g2 + g3);
      s2 += (g0 * h0 + g1 * h1) + (g2 * h2 + g3 * h3);
      dg[i].x += d01.x * h0; dg[i].y += d01.y * h1; dg[i].z += d23.x * h2; dg[i].w += d23.y * h3;
      db[i].x += d01.x; db[i].y += d01.y; db[i].z += d23.x; db[i].w += d23.y;
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (kSplit == 2) {   // both warps of the pair take the same trip count, so the named barrier is always matched
      if (lane == 0) xch[parity][warp] = make_float2(s1, s2);
      asm volatile("bar.sync %0, 64;" ::"r"(1 + slot) : "memory");
      const float2 o = xch[parity][warp ^ 1];
      s1 += o.x;
      s2 += o.y;
    }
    const float m1 = s1 * (1.0f / D), m2 = s2 * (1.0f / D);
    uint2* dxr = reinterpret_cast<uint2*>(dx + prow * D);
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const float4 gm = __ldg(gam4 + c0 + 32 * i);
      const float2 d01 = unbf2(dw[i].x), d23 = unbf2(dw[i].y);
      const float h0 = (xv[i].x - mu) * r, h1 = (xv[i].y - mu) * r, h2 = (xv[i].z - mu) * r, h3 = (xv[i].w - mu) * r;
      const float2 a = unbf2(rw_[i].x), b = unbf2(rw_[i].y);
      const float o0 = r * (d01.x * gm.x - m1 - h0 * m2) + a.x, o1 = r * (d01.y * gm.y - m1 - h1 * m2) + a.y;
      const float o2 = r * (d23.x * gm.z - m1 - h2 * m2) + b.x, o3 = r * (d23.y * gm.w - m1 - h3 * m2) + b.y;
      const uint2 packed = make_uint2(bf2(o0, o1), bf2(o2, o3));
      dxr[c0 + 32 * i] = packed;
      if (dxsum != nullptr) {   // column sums of the bf16 values actually stored (what the wgrad GEMM will read)
        const float2 s01 = unbf2(packed.x), s23 = unbf2(packed.y);
        dsx[i].x += s01.x; dsx[i].y += s01.y; dsx[i].z += s23.x; dsx[i].w += s23.y;
      }
    }
  }
  // block reduction of the per-slot partials
  float4* red4 = reinterpret_cast<float4*>(red);
  const int npass = dxsum != nullptr ? 3 : 2;
  for (int pass = 0; pass < npass; ++pass) {
#pragma unroll
    for (int i = 0; i < V; ++i) red4[slot * (D / 4) + c0 + 32 * i] = pass == 0 ? dg[i] : (pass == 1 ? db[i] : dsx[i]);
    __syncthreads();
    float* dst = pass == 0 ? dgamma : (pass == 1 ? dbeta : dxsum);
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
      float s = 0.f;
      for (int w = 0; w < nslots; ++w) s += red[w * D + c];
      atomicAdd(dst + c, s);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------- column sums
// grid (N/256, row_chunks); thread owns 8 consecutive columns (one uint4), 8 row lanes per block.
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const __nv_bfloat16* __restrict__ x, int M, int N, long long ldx,
                                                          int rows_per_block, float* __restrict__ out) {
  __shared__ float red[8][256];
  pdl_wait();
  pdl_launch_dependents();
  const int cg = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int col = blockIdx.x * 256 + cg * 8;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = col < N ? min(M, r0 + rows_per_block) : 0;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int r = r0 + rl; r < r1; r += 8) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(x + static_cast<long long>(r) * ldx + col));
    const float2 a = unbf2(q.x), b = unbf2(q.y), c = unbf2(q.z), d = unbf2(q.w);
    acc[0] += a.x; acc[1] += a.y; acc[2] += b.x; acc[3] += b.y;
    acc[4] += c.x; acc[5] += c.y; acc[6] += d.x; acc[7] += d.y;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) red[rl][cg * 8 + i] = acc[i];
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
  if (blockIdx.x * 256 + threadIdx.x < N) atomicAdd(out + blockIdx.x * 256 + threadIdx.x, s);
}

// ------------------------------------------------------------------------- embeddings glue
__global__ void embed_cls_kernel(const float* __restrict__ cls, const float* __restrict__ pos, int B, int T, int D,
                                 float* __restrict__ h) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * D) return;
  const int b = i / D, d = i - b * D;
  h[static_cast<long long>(b) * T * D + d] = cls[d] + pos[d];
}

// thread = 8 columns; a block walks tokens t = blockIdx.x, blockIdx.x + gridDim.x, …  dpos[t] += Σ_b dh[b,t]; t=0 → dcls;
// t≥1 → dbias, dpatch copy.  The bias partials stay in registers across the block's tokens, so dbias sees one atomic
// per column per BLOCK — with one block per token 576 atomics piled up on each of only 768 addresses (24 cache
// lines) and that serialisation was most of the kernel's 51 µs.
__global__ void __launch_bounds__(128) embed_bwd_kernel(const __nv_bfloat16* __restrict__ dh, int B, int T, int D,
                                                        float* __restrict__ dpos, float* __restrict__ dcls,
                                                        float* __restrict__ dbias, __nv_bfloat16* __restrict__ dpatch) {
  for (int c8 = threadIdx.x; c8 < D / 8; c8 += blockDim.x) {
    float bias_acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int t = blockIdx.x; t < T; t += gridDim.x) {
      float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int b0 = 0; b0 < B; b0 += 8) {          // 8 images' loads in flight per thread
        uint4 q[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          q[j] = (b0 + j < B) ? __ldg(reinterpret_cast<const uint4*>(dh + (static_cast<long long>(b0 + j) * T + t) * D) + c8)
                              : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (b0 + j >= B) break;
          if (t > 0) reinterpret_cast<uint4*>(dpatch + (static_cast<long long>(b0 + j) * (T - 1) + (t - 1)) * D)[c8] = q[j];
          const float2 a = unbf2(q[j].x), bb = unbf2(q[j].y), c = unbf2(q[j].z), d = unbf2(q[j].w);
          acc[0] += a.x; acc[1] += a.y; acc[2] += bb.x; acc[3] += bb.y;
          acc[4] += c.x; acc[5] += c.y; acc[6] += d.x; acc[7] += d.y;
        }
      }
      float* pp = dpos + static_cast<long long>(t) * D + c8 * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) pp[i] += acc[i];  // (t, column) has exactly one owner
      if (t == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dcls[c8 * 8 + i] += acc[i];
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) bias_acc[i] += acc[i];
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) atomicAdd(dbias + c8 * 8 + i, bias_acc[i]);
  }
}

// ------------------------------------------------------------------------- parameter shadow
__global__ void __launch_bounds__(256) cast_f32_bf16_kernel(const float4* __restrict__ src, uint4* __restrict__ dst,
                                                            long long n8) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 a = __ldg(src + 2 * i), b = __ldg(src + 2 * i + 1);
    dst[i] = make_uint4(bf2(a.x, a.y), bf2(a.z, a.w), bf2(b.x, b.y), bf2(b.z, b.w));
  }
}

template <int VPL>
static int ln_fwd_launch(const float* x, long long ldx, const float* gamma, const float* beta, float eps, int M, long long rs,
                         __nv_bfloat16* y, float* mean, float* rstd, cudaStream_t s) {
  VITK_CUDA(launch_pdl(layernorm_fwd_kernel<VPL>, dim3((M + 7) / 8), dim3(256), 0, s, x, ldx, gamma, beta, eps, M, rs, y, mean, rstd));
  VITK_LAUNCH_CHECK("layernorm_fwd_kernel");
  return 0;
}
template <int VPL>
static int ln_bwd_launch(const __nv_bfloat16* dy, const float* x, long long ldx, const float* mean, const float* rstd,
                         const float* gamma, const __nv_bfloat16* dres, int M, long long rs, __nv_bfloat16* dx, float* dgamma,
                         float* dbeta, float* dxsum, cudaStream_t s) {
  const int warps = 8;
  const int slots = (VPL % 2 == 0) ? warps / 2 : warps;      // rows in flight per block (a warp pair per row)
  int grid = num_sms() * kLnBwdBlocks;
  const int need = (M + slots - 1) / slots;
  if (grid > need) grid = need;
  const size_t smem = static_cast<size_t>(slots) * VPL * 128 * sizeof(float);
  VITK_CUDA(launch_pdl(layernorm_bwd_kernel<VPL>, dim3(grid), dim3(warps * 32), smem, s, dy, x, ldx, mean, rstd, gamma, dres, M, rs, dx,
                       dgamma, dbeta, dxsum));
  VITK_LAUNCH_CHECK("layernorm_bwd_kernel");
  return 0;
}

}  // namespace vitk

using namespace vitk;

extern "C" VITK_API int vitk_patchify_u8(const uint8_t* gray, int64_t B, int64_t H, int64_t W, int64_t patch,
                                const float* host_mean, const float* host_std, void* out, vitk_stream_t stream) {
  VITK_REQUIRE(gray && out && host_mean && host_std, VITK_EINVAL, "patchify_u8: NULL argument");
  VITK_REQUIRE(patch == 16, VITK_EINVAL, "patchify_u8: only patch_size 16 is supported (got %lld)", (long long)patch);
  VITK_REQUIRE(B > 0 && H > 0 && W > 0 && H % 16 == 0 && W % 16 == 0, VITK_EINVAL, "patchify_u8: bad image shape");
  VITK_REQUIRE(aligned16(gray) && aligned16(out), VITK_EALIGN, "patchify_u8: buffers must be 16-byte aligned");
  NormConst nc;
  for (int c = 0; c < 3; ++c) {
    nc.mean[c] = host_mean[c];
    nc.std[c] = host_std[c];
    VITK_REQUIRE(nc.std[c] != 0.f, VITK_EINVAL, "patchify_u8: std[%d] is zero", c);
  }
  const long long total = B * (H / 16) * (W / 16) * 16;
  patchify_u8_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      gray, static_cast<int>(B), static_cast<int>(H), static_cast<int>(W), nc, static_cast<__nv_bfloat16*>(out));
  VITK_LAUNCH_CHECK("patchify_u8_kernel");
  return 0;
}

extern "C" VITK_API int vitk_hflip_u8(uint8_t* gray, const uint8_t* mask, int64_t B, int64_t H, int64_t W, vitk_stream_t stream) {
  VITK_REQUIRE(gray && mask, VITK_EINVAL, "hflip_u8: NULL argument");
  VITK_REQUIRE(B > 0 && B < 65536 && H > 0 && W > 0 && W % 16 == 0 && H < (1 << 20) && W < (1 << 20), VITK_EINVAL, "hflip_u8: bad image shape (W must be a multiple of 16)");
  VITK_REQUIRE(aligned16(gray), VITK_EALIGN, "hflip_u8: the image buffer must be 16-byte aligned");
  const long long per_image = H * ((W / 16 + 1) / 2);
  hflip_u8_kernel<<<dim3(static_cast<unsigned>((per_image + 255) / 256), static_cast<unsigned>(B)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      gray, mask, static_cast<int>(H), static_cast<int>(W));
  VITK_LAUNCH_CHECK("hflip_u8_kernel");
  return 0;
}

extern "C" VITK_API int vitk_patchify_f32(const float* pix, int64_t B, int64_t H, int64_t W, int64_t patch, void* out,
                                 vitk_stream_t stream) {
  VITK_REQUIRE(pix && out, VITK_EINVAL, "patchify_f32: NULL argument");
  VITK_REQUIRE(patch == 16, VITK_EINVAL, "patchify_f32: only patch_size 16 is supported (got %lld)", (long long)patch);
  VITK_REQUIRE(B > 0 && H > 0 && W > 0 && H % 16 == 0 && W % 16 == 0, VITK_EINVAL, "patchify_f32: bad image shape");
  VITK_REQUIRE(aligned16(pix) && aligned16(out), VITK_EALIGN, "patchify_f32: buffers must be 16-byte aligned");
  const long long total = B * (H / 16) * (W / 16) * 48;
  patchify_f32_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      pix, static_cast<int>(B), static_cast<int>(H), static_cast<int>(W), static_cast<__nv_bfloat16*>(out));
  VITK_LAUNCH_CHECK("patchify_f32_kernel");
  return 0;
}

extern "C" VITK_API int vitk_layernorm_fwd_rows(const float* x, int64_t ldx, const float* gamma, const float* beta, float eps,
                                       int64_t M, int64_t D, int64_t row_stride, void* y, float* mean, float* rstd,
                                       vitk_stream_t stream) {
  VITK_REQUIRE(x && gamma && beta && y, VITK_EINVAL, "layernorm_fwd: NULL argument");
  VITK_REQUIRE(M > 0 && M < (1ll << 31) && row_stride >= 1, VITK_EINVAL, "layernorm_fwd: bad M / row_stride");
  VITK_REQUIRE(ldx >= D && ldx % 4 == 0 && aligned16(x) && aligned16(y) && aligned16(gamma) && aligned16(beta),
               VITK_EALIGN, "layernorm_fwd: alignment");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* yy = static_cast<__nv_bfloat16*>(y);
  const long long rs = row_stride;
  switch (D) {
    case 128: return ln_fwd_launch<1>(x, ldx, gamma, beta, eps, (int)M, rs, yy, mean, rstd, s);
    case 256: return ln_fwd_launch<2>(x, ldx, gamma, beta, eps, (int)M, rs, yy, mean, rstd, s);
    case 512: return ln_fwd_launch<4>(x, ldx, gamma, beta, eps, (int)M, rs, yy, mean, rstd, s);
    case 768: return ln_fwd_launch<6>(x, ldx, gamma, beta, eps, (int)M, rs, yy, mean, rstd, s);
    case 1024: return ln_fwd_launch<8>(x, ldx, gamma, beta, eps, (int)M, rs, yy, mean, rstd, s);
    default: return set_error(VITK_EINVAL, "layernorm_fwd: hidden size %lld unsupported (128,256,512,768,1024)", (long long)D);
  }
}

extern "C" VITK_API int vitk_layernorm_fwd(const float* x, int64_t ldx, const float* gamma, const float* beta, float eps,
                                  int64_t M, int64_t D, void* y, float* mean, float* rstd, vitk_stream_t stream) {
  return vitk_layernorm_fwd_rows(x, ldx, gamma, beta, eps, M, D, 1, y, mean, rstd, stream);
}

extern "C" VITK_API int vitk_layernorm_bwd(const void* dy, const float* x, int64_t ldx, const float* mean, const float* rstd,
                                  const float* gamma, const void* dres, int64_t M, int64_t D, void* dx, float* dgamma,
                                  float* dbeta, float* dxsum, vitk_stream_t stream) {
  return vitk_layernorm_bwd_rows(dy, x, ldx, mean, rstd, gamma, dres, M, D, 1, dx, dgamma, dbeta, dxsum, stream);
}

extern "C" VITK_API int vitk_layernorm_bwd_rows(const void* dy, const float* x, int64_t ldx, const float* mean, const float* rstd,
                                       const float* gamma, const void* dres, int64_t M, int64_t D, int64_t row_stride,
                                       void* dx, float* dgamma, float* dbeta, float* dxsum, vitk_stream_t stream) {
  VITK_REQUIRE(dy && x && mean && rstd && gamma && dx && dgamma && dbeta, VITK_EINVAL, "layernorm_bwd: NULL argument");
  VITK_REQUIRE(row_stride >= 1, VITK_EINVAL, "layernorm_bwd: row_stride must be >= 1");
  const long long rs = row_stride;
  VITK_REQUIRE(M > 0 && M < (1ll << 31), VITK_EINVAL, "layernorm_bwd: bad M");
  VITK_REQUIRE(ldx >= D && ldx % 4 == 0 && aligned16(x) && aligned16(dy) && aligned16(dx) && aligned16(gamma) &&
                   (dres == nullptr || aligned16(dres)),
               VITK_EALIGN, "layernorm_bwd: alignment");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const __nv_bfloat16* dyy = static_cast<const __nv_bfloat16*>(dy);
  const __nv_bfloat16* rr = static_cast<const __nv_bfloat16*>(dres);
  __nv_bfloat16* dxx = static_cast<__nv_bfloat16*>(dx);
  switch (D) {
    case 128: return ln_bwd_launch<1>(dyy, x, ldx, mean, rstd, gamma, rr, (int)M, rs, dxx, dgamma, dbeta, dxsum, s);
    case 256: return ln_bwd_launch<2>(dyy, x, ldx, mean, rstd, gamma, rr, (int)M, rs, dxx, dgamma, dbeta, dxsum, s);
    case 512: return ln_bwd_launch<4>(dyy, x, ldx, mean, rstd, gamma, rr, (int)M, rs, dxx, dgamma, dbeta, dxsum, s);
    case 768: return ln_bwd_launch<6>(dyy, x, ldx, mean, rstd, gamma, rr, (int)M, rs, dxx, dgamma, dbeta, dxsum, s);
    case 1024: return ln_bwd_launch<8>(dyy, x, ldx, mean, rstd, gamma, rr, (int)M, rs, dxx, dgamma, dbeta, dxsum, s);
    default: return set_error(VITK_EINVAL, "layernorm_bwd: hidden size %lld unsupported", (long long)D);
  }
}

extern "C" VITK_API int vitk_colsum_bf16(const void* x, int64_t M, int64_t N, int64_t ldx, float* out, vitk_stream_t stream) {
  VITK_REQUIRE(x && out, VITK_EINVAL, "colsum: NULL argument");
  VITK_REQUIRE(M > 0 && N > 0 && N % 8 == 0 && M < (1ll << 31) && N < (1ll << 31), VITK_EINVAL,
               "colsum: N=%lld must be a positive multiple of 8", (long long)N);
  VITK_REQUIRE(ldx % 8 == 0 && ldx >= N && aligned16(x), VITK_EALIGN, "colsum: alignment");
  const int col_blocks = static_cast<int>((N + 255) / 256);
  int row_chunks = (num_sms() * 4 + col_blocks - 1) / col_blocks;
  int rows_per_block = static_cast<int>((M + row_chunks - 1) / row_chunks);
  rows_per_block = (rows_per_block + 7) / 8 * 8;
  row_chunks = static_cast<int>((M + rows_per_block - 1) / rows_per_block);
  VITK_CUDA(launch_pdl(colsum_bf16_kernel, dim3(col_blocks, row_chunks), dim3(256), 0, static_cast<cudaStream_t>(stream),
                       static_cast<const __nv_bfloat16*>(x), static_cast<int>(M), static_cast<int>(N), static_cast<long long>(ldx),
                       rows_per_block, out));
  VITK_LAUNCH_CHECK("colsum_bf16_kernel");
  return 0;
}

extern "C" VITK_API int vitk_embed_cls(const float* cls, const float* pos, int64_t B, int64_t T, int64_t D, float* h,
                              vitk_stream_t stream) {
  VITK_REQUIRE(cls && pos && h && B > 0 && T > 0 && D > 0, VITK_EINVAL, "embed_cls: bad argument");
  const int n = static_cast<int>(B * D);
  embed_cls_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(cls, pos, (int)B, (int)T, (int)D, h);
  VITK_LAUNCH_CHECK("embed_cls_kernel");
  return 0;
}

extern "C" VITK_API int vitk_embed_bwd(const void* dh, int64_t B, int64_t T, int64_t D, float* dpos, float* dcls, float* dbias,
                              void* dpatch, vitk_stream_t stream) {
  VITK_REQUIRE(dh && dpos && dcls && dbias && dpatch && B > 0 && T > 1, VITK_EINVAL, "embed_bwd: bad argument");
  VITK_REQUIRE(D % 8 == 0 && aligned16(dh) && aligned16(dpatch), VITK_EALIGN, "embed_bwd: alignment");
  const unsigned grid = static_cast<unsigned>(T < num_sms() ? T : num_sms());
  embed_bwd_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(dh), (int)B, (int)T, (int)D, dpos, dcls, dbias, static_cast<__nv_bfloat16*>(dpatch));
  VITK_LAUNCH_CHECK("embed_bwd_kernel");
  return 0;
}

extern "C" VITK_API int vitk_cast_f32_bf16(const float* src, void* dst, int64_t n, vitk_stream_t stream) {
  VITK_REQUIRE(src && dst && n > 0 && n % 8 == 0, VITK_EINVAL, "cast: n must be a positive multiple of 8");
  VITK_REQUIRE(aligned16(src) && aligned16(dst), VITK_EALIGN, "cast: alignment");
  const long long n8 = n / 8;
  long long blocks = (n8 + 255) / 256;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  if (blocks > cap) blocks = cap;
  cast_f32_bf16_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(src), static_cast<uint4*>(dst), n8);
  VITK_LAUNCH_CHECK("cast_f32_bf16_kernel");
  return 0;
}

extern "C" VITK_API int vitk_fill_zero(void* ptr, size_t bytes, vitk_stream_t stream) {
  VITK_REQUIRE(ptr != nullptr, VITK_EINVAL, "fill_zero: NULL");
  VITK_CUDA(cudaMemsetAsync(ptr, 0, bytes, static_cast<cudaStream_t>(stream)));
  return 0;
}
