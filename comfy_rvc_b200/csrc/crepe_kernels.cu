// CREPE f0 estimator (torchcrepe's `Crepe`, `preprocess`, `postprocess` and decoders): everything that is not a contraction.
// conv1..conv6 and the classifier run on the generic tcgen05 kernel (conv_tc.cu); this file holds
//   * framing + per-frame normalisation, written straight into conv1's operand layout.  conv1 (1 -> C, k 512, stride 4) is a
//     stride-1 convolution of 8 taps at dilation 16 over 64 overlapping polyphase channels, x[t][c] = frame_pad[4 t + c]
//     (frame_pad = the frame zero-padded by 254 on each side): out[j] = sum_{m < 8} sum_{c < 64} w[64 m + c] x[j + 16 m][c],
//     K = 512 exactly.  (4 polyphase channels and 128 taps would be the same sum, but a K block of the MMA is 64 channels.)
//   * eval-mode BatchNorm (after the ReLU of the conv epilogue) + max_pool (2, 1), written into the next layer's layout;
//   * sigmoid, fmin / fmax masking, argmax / weighted_argmax and the per-frame log-probabilities of the Viterbi decode, and the
//     Viterbi recursion itself (one CTA per decode chunk, float64 like librosa's).
#include <cuda_fp16.h>

#include <algorithm>
#include <cfloat>
#include <cmath>

#include "common.cuh"

namespace rvc {
namespace {

constexpr int kWin = 1024, kBins = 360, kBand = 11, kFrameRows = 368, kFrameC = 64, kConv1Pad = 254;

// ---------------------------------------------------------------- frames ------------------------------------------------
__global__ void __launch_bounds__(256)
crepe_frames_kernel(const float* __restrict__ audio, long long n, long long first, int hop, int pad, __half* __restrict__ out) {
  __shared__ float x[kWin];
  __shared__ double red[2][8];
  const int tid = threadIdx.x;
  const long long f = first + blockIdx.x;
  const long long s0 = f * hop - (pad ? kWin / 2 : 0);
  double s = 0.0;
  for (int i = tid; i < kWin; i += 256) {
    const long long k = s0 + i;
    const float v = (k >= 0 && k < n) ? audio[k] : 0.f;
    x[i] = v;
    s += v;
  }
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((tid & 31) == 0) red[0][tid >> 5] = s;
  __syncthreads();
  double mean = 0.0;
  for (int w = 0; w < 8; ++w) mean += red[0][w];
  mean /= kWin;
  double q = 0.0;
  for (int i = tid; i < kWin; i += 256) {
    const double d = x[i] - mean;
    q += d * d;
  }
  for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  if ((tid & 31) == 0) red[1][tid >> 5] = q;
  __syncthreads();
  double var = 0.0;
  for (int w = 0; w < 8; ++w) var += red[1][w];
  const float meanf = (float)mean;
  const float scale = (float)(1.0 / fmax(1e-10, sqrt(var / (kWin - 1))));     // torch.std: unbiased
  __half* o = out + (size_t)blockIdx.x * kFrameRows * kFrameC;
  for (int v = tid; v < kFrameRows * kFrameC / 8; v += 256) {
    const int t = v / (kFrameC / 8), c0 = (v % (kFrameC / 8)) * 8;
    __align__(16) __half h[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int i = 4 * t + c0 + e - kConv1Pad;
      float y = (i >= 0 && i < kWin) ? (x[i] - meanf) * scale : 0.f;
      y = fminf(fmaxf(y, -65504.f), 65504.f);
      h[e] = __float2half_rn(y);
    }
    *reinterpret_cast<uint4*>(o + (size_t)t * kFrameC + c0) = *reinterpret_cast<const uint4*>(h);
  }
}

// ---------------------------------------------------------------- BatchNorm + max-pool ------------------------------------------
// out[f][q][c] = max(bn(x[f * p_in + in_off + 2 j][c]), bn(x[... + 2 j + 1][c])), j = q - out_off in [0, L / 2); other rows 0.
__global__ void __launch_bounds__(256)
crepe_bn_pool_kernel(const __half* __restrict__ x, const float* __restrict__ scale, const float* __restrict__ shift, __half* __restrict__ out,
                     long long frames, int C, int L, int p_in, int in_off, int p_out, int out_off) {
  const int cv = C / 8;
  const long long total = frames * p_out * cv;
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < total; v += (long long)gridDim.x * blockDim.x) {
    const int c0 = (int)(v % cv) * 8;
    const long long row = v / cv;
    const long long f = row / p_out;
    const int j = (int)(row % p_out) - out_off;
    __align__(16) __half h[8];
    if (j >= 0 && j < L / 2) {
      const __half* a = x + ((size_t)(f * p_in + in_off + 2 * j)) * C + c0;
      __align__(16) __half r0[8], r1[8];
      *reinterpret_cast<uint4*>(r0) = *reinterpret_cast<const uint4*>(a);
      *reinterpret_cast<uint4*>(r1) = *reinterpret_cast<const uint4*>(a + C);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float s = scale[c0 + e], b = shift[c0 + e];
        h[e] = __float2half_rn(fmaxf(__half2float(r0[e]) * s + b, __half2float(r1[e]) * s + b));
      }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) h[e] = __float2half_rn(0.f);
    }
    *reinterpret_cast<uint4*>(out + (size_t)row * C + c0) = *reinterpret_cast<const uint4*>(h);
  }
}

// ---------------------------------------------------------------- per-frame decode ------------------------------------------
// One warp per frame.  lane l holds bins l, l + 32, ... (12 of them, the last 8 lanes' 12th slot empty).
__global__ void __launch_bounds__(256)
crepe_frame_decode_kernel(const float* __restrict__ in, int ld, int from_salience, long long T, int lo, int hi, int mode,
                          const double* __restrict__ dither, const double* __restrict__ wcents, float* __restrict__ sal,
                          int* __restrict__ bins, double* __restrict__ f0, float* __restrict__ period, double* __restrict__ logp) {
  const long long t = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (t >= T) return;
  constexpr int kPer = (kBins + 31) / 32;
  float s[kPer];
  float best = -INFINITY;
  int barg = kBins;
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int b = lane + 32 * i;
    s[i] = 0.f;
    if (b < kBins) {
      const float v = in[t * ld + b];
      s[i] = from_salience ? v : 1.f / (1.f + expf(-v));
      if (sal) sal[t * kBins + b] = s[i];
      if (b >= lo && b < hi && (s[i] > best || barg == kBins)) { best = s[i]; barg = b; }
    }
  }
  for (int o = 16; o; o >>= 1) {                                    // first maximum over the lanes
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oa = __shfl_xor_sync(0xffffffffu, barg, o);
    if (oa < kBins && (barg == kBins || ob > best || (ob == best && oa < barg))) { best = ob; barg = oa; }
  }
  if (mode == 2) {                                                  // Viterbi observations: log(softmax(masked) + tiny)
    const double m = (double)best;
    double e[kPer], sum = 0.0;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      const int b = lane + 32 * i;
      e[i] = (b < kBins && b >= lo && b < hi) ? exp((double)s[i] - m) : 0.0;
      sum += e[i];
    }
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      const int b = lane + 32 * i;
      if (b < kBins) logp[t * kBins + b] = log(e[i] / sum + (double)FLT_MIN);
    }
    return;
  }
  double cents;
  if (mode == 1) {
    // weighted_argmax: window [max(0, b - 4), min(360, b + 5)); torchcrepe applies a (second) sigmoid to the masked salience,
    // sigmoid(-inf) = 0 for masked bins.  Every lane gathers the window through shuffles; lane 0 keeps the result.
    double num = 0.0, den = 0.0;
    for (int k = barg - 4; k < barg + 5; ++k) {
      const int kk = k < 0 ? 0 : (k >= kBins ? kBins - 1 : k);
      float v = 0.f;
#pragma unroll
      for (int i = 0; i < kPer; ++i) {
        const float vi = __shfl_sync(0xffffffffu, s[i], kk & 31);
        if (kk / 32 == i) v = vi;
      }
      if (k < 0 || k >= kBins) continue;
      const double p = (k >= lo && k < hi) ? 1.0 / (1.0 + exp(-(double)v)) : 0.0;
      num += wcents[k] * p;
      den += p;
    }
    cents = num / den;
  } else {
    cents = 20.0 * barg + 1997.3794084376191 + dither[t];
  }
  if (lane == 0) {
    bins[t] = barg;
    f0[t] = 10.0 * pow(2.0, cents / 1200.0);
    if (period) period[t] = best;
  }
}

// ---------------------------------------------------------------- Viterbi --------------------------------------------------
// librosa.sequence.viterbi(softmax, transition) for torchcrepe's transition max(12 - |i - j|, 0) / row sum: log_trans[k][j] is
// ltab[k][j - k + 11] inside the band and log(tiny) = c_out outside.  Outside-band predecessors can only win through the
// global maximum of the previous column (an in-band predecessor is at least that maximum + log(1 / 144) > c_out), so each
// state looks at its 23 band neighbours plus the global first argmax.  Ties: the first (lowest) predecessor, like np.argmax.
__global__ void __launch_bounds__(384)
crepe_viterbi_kernel(const double* __restrict__ logp, const float* __restrict__ sal, long long T, int chunk, const double* __restrict__ ltab,
                     double c_out, double log_init, unsigned short* __restrict__ ptr, const double* __restrict__ dither,
                     int* __restrict__ bins, double* __restrict__ f0, float* __restrict__ period, double* __restrict__ score) {
  __shared__ double val[2][kBins];
  __shared__ double wv[12];
  __shared__ int wi[12];
  const int j = threadIdx.x, lane = j & 31, warp = j >> 5;
  const long long t0 = (long long)blockIdx.x * chunk;
  const long long n = min((long long)chunk, T - t0);
  if (j < kBins) val[0][j] = logp[t0 * kBins + j] + log_init;
  double lt[2 * kBand + 1];
  if (j < kBins) {
#pragma unroll
    for (int d = 0; d < 2 * kBand + 1; ++d) {
      const int k = j + d - kBand;
      lt[d] = (k >= 0 && k < kBins) ? ltab[k * (2 * kBand + 1) + (j - k + kBand)] : 0.0;
    }
  }
  __syncthreads();
  for (long long t = 1; t < n; ++t) {
    const double* prev = val[(t - 1) & 1];
    double* cur = val[t & 1];
    // global first argmax of the previous column
    double bv = j < kBins ? prev[j] : -INFINITY;
    int bi = j < kBins ? j : kBins;
    for (int o = 16; o; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { wv[warp] = bv; wi[warp] = bi; }
    __syncthreads();
    if (j < kBins) {
      double gv = wv[0];
      int gi = wi[0];
      for (int w = 1; w < 12; ++w)
        if (wv[w] > gv) { gv = wv[w]; gi = wi[w]; }                 // warps in ascending bin order: strict > keeps the first
      double best = -INFINITY;
      int arg = -1;
#pragma unroll
      for (int d = 0; d < 2 * kBand + 1; ++d) {
        const int k = j + d - kBand;
        if (k >= 0 && k < kBins) {
          const double c = prev[k] + lt[d];
          if (arg < 0 || c > best) { best = c; arg = k; }
        }
      }
      if (gi - j > kBand || j - gi > kBand) {
        const double c = gv + c_out;
        if (c > best || (c == best && gi < arg)) { best = c; arg = gi; }
      }
      cur[j] = logp[(t0 + t) * kBins + j] + best;
      ptr[(t0 + t) * kBins + j] = (unsigned short)arg;
    }
    __syncthreads();
  }
  if (warp == 0) {
    const double* last = val[(n - 1) & 1];
    double bv = -INFINITY;
    int bi = kBins;
    for (int k = lane; k < kBins; k += 32)
      if (last[k] > bv || bi == kBins) { bv = last[k]; bi = k; }
    for (int o = 16; o; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) {
      score[blockIdx.x] = bv;
      int s = bi;
      for (long long t = n - 1; t >= 0; --t) {
        const long long g = t0 + t;
        bins[g] = s;
        f0[g] = 10.0 * pow(2.0, (20.0 * s + 1997.3794084376191 + dither[g]) / 1200.0);
        if (period) period[g] = sal[g * kBins + s];
        if (t > 0) s = ptr[g * kBins + s];
      }
    }
  }
}

}  // namespace

cudaError_t launch_crepe_frames(const float* audio, long long n, long long first, long long count, int hop, int pad, void* out,
                                cudaStream_t st) {
  if (!audio || !out || n <= 0 || first < 0 || count <= 0 || count > 0x7fffffffLL || hop <= 0 ||
      (reinterpret_cast<uintptr_t>(out) & 15))
    return cudaErrorInvalidValue;
  crepe_frames_kernel<<<(unsigned)count, 256, 0, st>>>(audio, n, first, hop, pad, reinterpret_cast<__half*>(out));
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_crepe_bn_pool(const void* x, const float* scale, const float* shift, void* out, long long frames, int C, int L,
                                 int p_in, int in_off, int p_out, int out_off, cudaStream_t st) {
  if (!x || !scale || !shift || !out || frames <= 0 || C <= 0 || C % 8 || L < 2 || L % 2 || in_off < 0 || in_off + L > p_in ||
      out_off < 0 || out_off + L / 2 > p_out || (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(out) & 15))
    return cudaErrorInvalidValue;
  const long long total = frames * p_out * (C / 8);
  const long long blocks = std::min((total + 255) / 256, 148LL * 16);
  crepe_bn_pool_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const __half*>(x), scale, shift, reinterpret_cast<__half*>(out),
                                                         frames, C, L, p_in, in_off, p_out, out_off);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_crepe_decode(const float* in, int ld, int from_salience, long long T, int chunk, int lo, int hi, int mode,
                                const double* dither, const double* wcents, const double* ltab, double c_out, double log_init,
                                float* sal, double* logp, unsigned short* ptr, int* bins, double* f0, float* period, double* score,
                                cudaStream_t st) {
  if (!in || ld < kBins || T <= 0 || lo < 0 || hi > kBins || lo >= hi || mode < 0 || mode > 2 || !bins || !f0 ||
      (mode != 1 && !dither) || (mode == 1 && !wcents) || (mode == 2 && (!ltab || !logp || !ptr || !score || chunk <= 0 || !sal)) ||
      (period && mode == 2 && !sal))
    return cudaErrorInvalidValue;
  crepe_frame_decode_kernel<<<(unsigned)((T * 32 + 255) / 256), 256, 0, st>>>(in, ld, from_salience, T, lo, hi, mode, dither, wcents,
                                                                              sal, bins, f0, period, logp);
  launch_counter().n++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || mode != 2) return e;
  const long long n_chunks = (T + chunk - 1) / chunk;
  if (n_chunks > 0x7fffffffLL) return cudaErrorInvalidValue;
  crepe_viterbi_kernel<<<(unsigned)n_chunks, 384, 0, st>>>(logp, sal, T, chunk, ltab, c_out, log_init, ptr, dither, bins, f0, period,
                                                           score);
  launch_counter().n++;
  return cudaGetLastError();
}

}  // namespace rvc
