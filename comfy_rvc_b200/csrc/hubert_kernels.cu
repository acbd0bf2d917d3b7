// First layer of the HuBERT / ContentVec feature encoder (SURVEY.md §8f rank 3): Conv1d(1 -> C, k = 10, stride 5, no bias)
// -> GroupNorm(C groups over C channels = per-channel normalisation over time, affine) -> GELU, as HuggingFace
// `HubertGroupNormConvLayer` computes it (transformers/models/hubert/modeling_hubert.py; reached from
// /root/reference/lib/infer_pack/loaders.py:52-61).  With one input channel the "convolution" is 10 FMAs per output, so it
// is recomputed instead of stored: pass 1 accumulates the K x K Gram matrix of the input windows (from which every channel's
// mean and variance follow), pass 2 recomputes, normalises, applies GELU and writes the fp16 channels-last operand
// [L0][C] of the tensor-core conv stack (conv_tc.cu).  The other front-end layers are ordinary contractions on the
// generic tcgen05 kernel (comfy_rvc_b200/hubert.py).
#include <cuda_fp16.h>

#include "common.cuh"

namespace rvc {
namespace {

constexpr int kFrames = 256;      // output frames per block
constexpr int kMaxK = 16;

// Pass 1: the statistics GroupNorm needs -- per-channel mean and second moment of y[t][c] = sum_k w[c][k] x[t S + k] over time --
// follow from the first and second moments of the INPUT windows: E[y_c] = w_c . m, E[y_c^2] = w_c^T G w_c with m[k] = mean_t x[tS+k],
// G[k][l] = mean_t x[tS+k] x[tS+l].  So the pass accumulates the K x K Gram matrix and the K sums (thread = one (k, l) pair, in double) instead of recomputing all C x L0 outputs: 219 -> ~15 us for 60 s of audio.
// The sums are combined in a fixed order, so that every call gives the same bits: one block writes `stats` itself; with several,
// block j writes its K^2 + K partial sums to slot j of conv0_partials ([K^2 + K][nblk]) and hubert_conv0_reduce_kernel adds the
// slots of each statistic in a fixed order.
// (Double atomics in arrival order differed from call to call in the last bits, and where the variance is a small difference of
// large moments -- a DC offset -- that reached the fp16 output.)
// Partial sums of batch item b: at the first 8-byte boundary of its y16 rows, which pass 2 overwrites afterwards (with several
// blocks L0 > 256, and nblk (K^2 + K) doubles fit in L0 C halves since 2 C >= K^2 + K).
__device__ __forceinline__ double* conv0_partials(void* y16, int b, long long y_bstride) {
  const unsigned long long a = reinterpret_cast<unsigned long long>(reinterpret_cast<__half*>(y16) + (long long)b * y_bstride);
  return reinterpret_cast<double*>((a + 7) & ~7ull);
}

__global__ void hubert_conv0_gram_kernel(const float* __restrict__ x, double* __restrict__ stats, void* y16, long long y_bstride,
                                         long long n, long long L0, int C, int K, int S) {
  extern __shared__ float xs[];
  const int b = blockIdx.y;
  const long long t0 = (long long)blockIdx.x * kFrames;
  const int nt = (int)min((long long)kFrames, L0 - t0);
  const int nx = (nt - 1) * S + K;
  const float* xb = x + (long long)b * n + t0 * S;
  for (int i = threadIdx.x; i < nx; i += blockDim.x) xs[i] = xb[i];
  __syncthreads();
  double* st = stats + (long long)b * 2 * C;                    // [K * K] Gram sums, then [K] sums
  for (int pidx = threadIdx.x; pidx < K * K + K; pidx += blockDim.x) {
    double acc = 0.0;                                           // double: w^T G w cancels heavily for high-pass channels
    if (pidx < K * K) {
      const int k = pidx / K, l = pidx - k * K;
      for (int t = 0; t < nt; ++t) acc = fma((double)xs[t * S + k], (double)xs[t * S + l], acc);
    } else {
      const int k = pidx - K * K;
      for (int t = 0; t < nt; ++t) acc += (double)xs[t * S + k];
    }
    if (gridDim.x == 1) st[pidx] = acc;
    else conv0_partials(y16, b, y_bstride)[(long long)pidx * gridDim.x + blockIdx.x] = acc;
  }
}

// One block per (statistic, batch item): thread t adds slots t, t + 256, ... in order, then a fixed shared-memory tree.
constexpr int kReduceThreads = 256;
__global__ void __launch_bounds__(kReduceThreads)
hubert_conv0_reduce_kernel(double* __restrict__ stats, void* y16, long long y_bstride, int nblk, int C) {
  __shared__ double red[kReduceThreads];
  const int pidx = blockIdx.x, b = blockIdx.y;
  const double* pb = conv0_partials(y16, b, y_bstride) + (long long)pidx * nblk;
  double acc = 0.0;
  for (int j = threadIdx.x; j < nblk; j += kReduceThreads) acc += pb[j];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int h = kReduceThreads / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) stats[(long long)b * 2 * C + pidx] = red[0];
}

// Pass 2: recompute the convolution, normalise with the statistics derived from the Gram matrix, GELU, write fp16 channels-last.
__global__ void hubert_conv0_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ gn_w,
                                    const float* __restrict__ gn_b, const double* __restrict__ stats, __half* __restrict__ y,
                                    long long n, long long L0, int C, int K, int S, float eps, long long y_bstride) {
  extern __shared__ float xs[];                       // (kFrames - 1) * S + K input samples of this chunk
  __shared__ double gram[kMaxK * kMaxK + kMaxK];
  const int b = blockIdx.y;
  const long long t0 = (long long)blockIdx.x * kFrames;
  const int nt = (int)min((long long)kFrames, L0 - t0);
  const int nx = (nt - 1) * S + K;
  const float* xb = x + (long long)b * n + t0 * S;
  for (int i = threadIdx.x; i < nx; i += blockDim.x) xs[i] = xb[i];
  const double* st = stats + (long long)b * 2 * C;
  for (int i = threadIdx.x; i < K * K + K; i += blockDim.x) gram[i] = st[i] / (double)L0;
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float wk[kMaxK];
#pragma unroll
    for (int k = 0; k < kMaxK; ++k) wk[k] = k < K ? w[c * K + k] : 0.f;
    double m = 0.0, e2 = 0.0;
    for (int k = 0; k < K; ++k) {
      m += (double)wk[k] * gram[K * K + k];
      double row = 0.0;
      for (int l = 0; l < K; ++l) row += (double)wk[l] * gram[k * K + l];
      e2 += (double)wk[k] * row;
    }
    const double var = e2 - m * m;                                // biased, like torch.nn.GroupNorm
    const float mean = (float)m;
    const float scale = (float)(1.0 / sqrt((var > 0.0 ? var : 0.0) + (double)eps)) * gn_w[c];
    const float shift = gn_b[c];
    for (int t = 0; t < nt; ++t) {
      const float* xp = xs + t * S;
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < kMaxK; ++k)
        if (k < K) acc = fmaf(wk[k], xp[k], acc);
      const float v = (acc - mean) * scale + shift;
      y[(long long)b * y_bstride + (t0 + t) * C + c] = __float2half_rn(0.5f * v * (1.f + erff(v * 0.70710678118654752f)));
    }
  }
}

}  // namespace

cudaError_t launch_hubert_conv0(const float* x, const float* w, const float* gn_w, const float* gn_b, double* stats, void* y16,
                                int B, long long n, int C, int K, int S, float eps, long long y_bstride, cudaStream_t st) {
  if (!x || !w || !gn_w || !gn_b || !stats || !y16 || B <= 0 || K < 1 || K > kMaxK || S < 1 || n < K || C < 1 || 2 * C < K * K + K)
    return cudaErrorInvalidValue;
  const long long L0 = (n - K) / S + 1;
  const int nblk = (int)((L0 + kFrames - 1) / kFrames);
  const dim3 grid((unsigned)nblk, (unsigned)B);
  const size_t smem = sizeof(float) * ((size_t)(kFrames - 1) * S + K);
  hubert_conv0_gram_kernel<<<grid, 128, smem, st>>>(x, stats, y16, y_bstride, n, L0, C, K, S);
  if (nblk > 1) hubert_conv0_reduce_kernel<<<dim3((unsigned)(K * K + K), (unsigned)B), kReduceThreads, 0, st>>>(stats, y16, y_bstride, nblk, C);
  hubert_conv0_kernel<<<grid, 256, smem, st>>>(x, w, gn_w, gn_b, stats, reinterpret_cast<__half*>(y16), n, L0, C, K, S, eps, y_bstride);
  launch_counter().n += nblk > 1 ? 3 : 2;
  return cudaGetLastError();
}

}  // namespace rvc
