// Classifier head fused with the loss: final LayerNorm on the CLS rows → Linear(D→C) →
// BCEWithLogits (mean) and the gradient of the loss w.r.t. the logits in ONE forward kernel;
// the backward kernel chains that gradient through the classifier and the LayerNorm of the
// B CLS rows.  Latency-bound (B rows of D floats); one CTA per image.
// Replaces HF modeling_vit.py:455,641-646 + loss_utils.py:110-112.
#include <cuda_bf16.h>

#include <mutex>

#include "common.cuh"

namespace vitk {

constexpr int kHeadThreads = 256;
constexpr int kMaxLabels = 64;
constexpr int kMaxHidden = 8192;   // head_bwd keeps two fp32 rows of D in shared memory: 64 KB at this limit

__device__ __forceinline__ float block_sum(float v, float* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < kHeadThreads / 32; ++w) s += scratch[w];
  return s;
}

__global__ void __launch_bounds__(kHeadThreads)
head_fwd_kernel(const float* __restrict__ h, int B, int T, int D, int C, const float* __restrict__ gamma,
                const float* __restrict__ beta, float eps, const float* __restrict__ Wc, const float* __restrict__ bc,
                const float* __restrict__ labels, float* __restrict__ logits, float* __restrict__ loss,
                float* __restrict__ dlogits, float* __restrict__ mean, float* __restrict__ rstd) {
  extern __shared__ float z[];  // [D] LN output of this CLS row
  __shared__ float scratch[kHeadThreads / 32];
  __shared__ float s_logit[kMaxLabels];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* x = h + static_cast<long long>(b) * T * D;  // CLS row

  float s = 0.f;
  for (int d = tid; d < D; d += kHeadThreads) s += x[d];
  const float mu = block_sum(s, scratch) / D;
  float q = 0.f;
  for (int d = tid; d < D; d += kHeadThreads) { const float c = x[d] - mu; q += c * c; }
  const float r = rsqrtf(block_sum(q, scratch) / D + eps);
  if (tid == 0) {
    if (mean) mean[b] = mu;
    if (rstd) rstd[b] = r;
  }
  for (int d = tid; d < D; d += kHeadThreads) z[d] = (x[d] - mu) * r * gamma[d] + beta[d];
  __syncthreads();
  for (int c = warp; c < C; c += kHeadThreads / 32) {
    float acc = 0.f;
    for (int d = lane; d < D; d += 32) acc += z[d] * Wc[static_cast<long long>(c) * D + d];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      const float l = acc + bc[c];
      s_logit[c] = l;
      logits[b * C + c] = l;
    }
  }
  __syncthreads();
  if (labels == nullptr) return;
  const float inv = 1.0f / (static_cast<float>(B) * C);
  float li = 0.f;
  if (tid < C) {
    const float l = s_logit[tid], y = labels[b * C + tid];
    // max(l,0) − l·y + log1p(exp(−|l|)): the numerically stable form ATen uses
    li = (fmaxf(l, 0.f) - l * y + log1pf(expf(-fabsf(l)))) * inv;
    if (dlogits) dlogits[b * C + tid] = (1.0f / (1.0f + expf(-l)) - y) * inv;
  }
  li = block_sum(li, scratch);
  if (tid == 0) atomicAdd(loss, li);
}

__global__ void __launch_bounds__(kHeadThreads)
head_bwd_kernel(const float* __restrict__ h, const float* __restrict__ mean, const float* __restrict__ rstd,
                const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ Wc, int B,
                int T, int D, int C, const float* __restrict__ dlogits, const float* __restrict__ dloss,
                __nv_bfloat16* __restrict__ dh, float* __restrict__ dWc, float* __restrict__ dbc,
                float* __restrict__ dgamma, float* __restrict__ dbeta) {
  extern __shared__ float sm[];
  float* xh = sm;      // [D]
  float* gz = sm + D;  // [D]
  __shared__ float scratch[kHeadThreads / 32];
  __shared__ float s_dl[kMaxLabels];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* x = h + static_cast<long long>(b) * T * D;
  const float mu = mean[b], r = rstd[b];
  const float gs = dloss ? *dloss : 1.0f;
  if (tid < C) {
    const float dl = dlogits[b * C + tid] * gs;
    s_dl[tid] = dl;
    atomicAdd(dbc + tid, dl);
  }
  __syncthreads();
  float s1 = 0.f, s2 = 0.f;
  for (int d = tid; d < D; d += kHeadThreads) {
    const float n = (x[d] - mu) * r;
    const float zd = n * gamma[d] + beta[d];
    float dz = 0.f;
    for (int c = 0; c < C; ++c) {
      const float dl = s_dl[c];
      dz += dl * Wc[static_cast<long long>(c) * D + d];
      atomicAdd(dWc + static_cast<long long>(c) * D + d, dl * zd);
    }
    atomicAdd(dgamma + d, dz * n);
    atomicAdd(dbeta + d, dz);
    const float g = dz * gamma[d];
    xh[d] = n;
    gz[d] = g;
    s1 += g;
    s2 += g * n;
  }
  const float m1 = block_sum(s1, scratch) / D;
  const float m2 = block_sum(s2, scratch) / D;
  __nv_bfloat16* o = dh + static_cast<long long>(b) * T * D;
  for (int d = tid; d < D; d += kHeadThreads) o[d] = __float2bfloat16_rn(r * (gz[d] - m1 - xh[d] * m2));
}

}  // namespace vitk

using namespace vitk;

extern "C" VITK_API int vitk_head_fwd(const float* h, int64_t B, int64_t T, int64_t D, int64_t C, const float* gamma,
                                      const float* beta, float eps, const float* Wc, const float* bc,
                                      const float* labels, float* logits, float* loss, float* dlogits, float* mean,
                                      float* rstd, vitk_stream_t stream) {
  VITK_REQUIRE(h && gamma && beta && Wc && bc && logits, VITK_EINVAL, "head_fwd: NULL argument");
  VITK_REQUIRE(B > 0 && T > 0 && D > 0 && C > 0 && C <= kMaxLabels && D <= kMaxHidden, VITK_EINVAL,
               "head_fwd: unsupported shape B=%lld T=%lld D=%lld C=%lld", (long long)B, (long long)T, (long long)D,
               (long long)C);
  if (labels) VITK_REQUIRE(loss != nullptr, VITK_EINVAL, "head_fwd: labels given but loss is NULL");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (labels) VITK_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), s));
  head_fwd_kernel<<<static_cast<unsigned>(B), kHeadThreads, D * sizeof(float), s>>>(
      h, (int)B, (int)T, (int)D, (int)C, gamma, beta, eps, Wc, bc, labels, logits, loss, dlogits, mean, rstd);
  VITK_LAUNCH_CHECK("head_fwd_kernel");
  return 0;
}

extern "C" VITK_API int vitk_head_bwd(const float* h, const float* mean, const float* rstd, const float* gamma,
                                      const float* beta, const float* Wc, int64_t B, int64_t T, int64_t D, int64_t C,
                                      const float* dlogits, const float* dloss, void* dh, float* dWc, float* dbc,
                                      float* dgamma, float* dbeta, vitk_stream_t stream) {
  VITK_REQUIRE(h && mean && rstd && gamma && beta && Wc && dlogits && dh && dWc && dbc && dgamma && dbeta, VITK_EINVAL,
               "head_bwd: NULL argument");
  VITK_REQUIRE(B > 0 && T > 0 && D > 0 && C > 0 && C <= kMaxLabels && D <= kMaxHidden, VITK_EINVAL,
               "head_bwd: unsupported shape B=%lld T=%lld D=%lld C=%lld", (long long)B, (long long)T, (long long)D,
               (long long)C);
  // above 48 KB of dynamic shared memory (D > 6144) a launch needs the kernel's opt-in
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(head_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    2 * kMaxHidden * static_cast<int>(sizeof(float)));
  });
  if (attr_err != cudaSuccess) return cuda_error(attr_err, "cudaFuncSetAttribute(head_bwd smem)");
  head_bwd_kernel<<<static_cast<unsigned>(B), kHeadThreads, 2 * D * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      h, mean, rstd, gamma, beta, Wc, (int)B, (int)T, (int)D, (int)C, dlogits, dloss, static_cast<__nv_bfloat16*>(dh),
      dWc, dbc, dgamma, dbeta);
  VITK_LAUNCH_CHECK("head_bwd_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------- evaluation counters
// The reference's compute_metrics (ViT-Training.py:112-118) and final report (:139-146): probs = sigmoid(logits),
// predictions = probs >= 0.5, micro-F1 / per-class precision-recall over the whole evaluation set.  Everything those
// need is four integers per class — TP, FP, FN, TN — accumulated on the device over the batches of an evaluation loop,
// so no logits travel to the host.  sigmoid is evaluated in fp32 as 1/(1+exp(−x)) like ATen's, so the threshold
// comparison sees the same rounding (logits a few ulp below 0 still round to exactly 0.5 and count as positive).
namespace vitk {
constexpr int kMaxCountLabels = 4096;   // [C][4] uint32 counters in shared memory: 64 KB at this limit

__global__ void __launch_bounds__(256)
multilabel_counts_kernel(const float* __restrict__ logits, const float* __restrict__ labels, long long n, int C, float threshold,
                         unsigned long long* __restrict__ counts) {
  extern __shared__ unsigned int s_cnt[];   // [C][4]
  for (int i = threadIdx.x; i < 4 * C; i += blockDim.x) s_cnt[i] = 0;
  __syncthreads();
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const float prob = 1.0f / (1.0f + expf(-logits[i]));
    const bool pred = prob >= threshold, truth = labels[i] >= 0.5f;
    atomicAdd(&s_cnt[4 * c + (pred ? (truth ? 0 : 1) : (truth ? 2 : 3))], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 4 * C; i += blockDim.x)
    if (s_cnt[i]) atomicAdd(&counts[i], static_cast<unsigned long long>(s_cnt[i]));
}
}  // namespace vitk

extern "C" VITK_API int vitk_multilabel_counts(const float* logits, const float* labels, int64_t B, int64_t C, float threshold,
                                               int64_t* counts, vitk_stream_t stream) {
  VITK_REQUIRE(logits && labels && counts && B > 0 && C > 0 && C <= vitk::kMaxCountLabels, VITK_EINVAL,
               "multilabel_counts: bad argument");
  VITK_REQUIRE(threshold > 0.f && threshold < 1.f, VITK_EINVAL, "multilabel_counts: threshold must be in (0, 1)");
  // above 48 KB of dynamic shared memory (C > 3072) a launch needs the kernel's opt-in
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(vitk::multilabel_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    16 * vitk::kMaxCountLabels);
  });
  if (attr_err != cudaSuccess) return vitk::cuda_error(attr_err, "cudaFuncSetAttribute(multilabel_counts smem)");
  const long long n = B * C;
  long long blocks = (n + 255) / 256;
  if (blocks > 4LL * vitk::num_sms()) blocks = 4LL * vitk::num_sms();
  vitk::multilabel_counts_kernel<<<static_cast<unsigned>(blocks), 256, 16 * C, static_cast<cudaStream_t>(stream)>>>(
      logits, labels, n, static_cast<int>(C), threshold, reinterpret_cast<unsigned long long*>(counts));
  VITK_LAUNCH_CHECK("multilabel_counts_kernel");
  return 0;
}
