// Device-side pre/post steps of the segmented conversion driver (VC.vc / VC.pipeline):
//   prepare_feats : x2 nearest interpolation of the HuBERT frames + "protect" blend   (vc_infer_pipeline.py:77-95)
//   absmax        : max |x| over the concatenated song                                 (vc_infer_pipeline.py:188)
//   to_int16      : x * 32768 / (max / 0.99), C truncation                             (vc_infer_pipeline.py:188-189)
//   rms_halfblock / rms_fold / rms_gain : the volume-envelope mix `change_rms`      (lib/model_utils.py:39, :183)
//   resample_poly : polyphase FIR resampling of the song                               (vc_infer_pipeline.py:185-186)
// All of them but resample_poly (fp32 FMA bound) are HBM-bound streaming kernels (one pass, 16-byte accesses); they exist so
// that a whole song is converted without a host round trip per segment (the reference syncs and gc's after every segment, :102-112).
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace rvc {
namespace {

// out[t][c] = f[t/2][c] * p + f0[t/2][c] * (1 - p),  p = pitchf[t] < 1 ? protect : 1   (fp32, no contraction:
// the reference evaluates mul, mul, add as separate torch ops)
template <typename TIn>
__global__ void prepare_feats_kernel(const TIn* __restrict__ f, const TIn* __restrict__ f0, const float* __restrict__ pitchf,
                                     float* __restrict__ out, int T, int C, float protect, int use_protect) {
  const long long total = (long long)T * (C / 4);
  const int c4n = C / 4;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(idx / c4n);
    const int c = (int)(idx - (long long)t * c4n) * 4;
    const long long src = (long long)(t >> 1) * C + c;
    float a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = (float)f[src + i];
    if (use_protect) {
      const float pf = pitchf[t];
      // pitchff[pitchf > 0] = 1; pitchff[pitchf < 1] = protect  (second assignment wins for 0 < f0 < 1)
      float p = pf;
      if (pf > 0.f) p = 1.f;
      if (pf < 1.f) p = protect;
      const float q = __fsub_rn(1.f, p);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        b[i] = (float)f0[src + i];
        a[i] = __fadd_rn(__fmul_rn(a[i], p), __fmul_rn(b[i], q));
      }
    }
    *reinterpret_cast<float4*>(out + (long long)t * C + c) = make_float4(a[0], a[1], a[2], a[3]);
  }
}

__global__ void absmax_kernel(const float* __restrict__ x, long long n, unsigned* __restrict__ out_bits) {
  float m = 0.f;
  const long long n4 = n / 4;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = x4[i];
    m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(x[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float sm[32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) atomicMax(out_bits, __float_as_uint(m));   // non-negative floats order like their bit patterns
  }
}

__device__ __forceinline__ short cvt_i16(float v, float audio_max) {
  // numpy: (x * 32768 / audio_max).astype(int16) -- two float32 roundings, then truncation toward zero
  return (short)__float2int_rz(__fdiv_rn(__fmul_rn(v, 32768.f), audio_max));
}

__global__ void to_int16_kernel(const float* __restrict__ x, long long n, const float* __restrict__ absmax, short* __restrict__ out) {
  const float audio_max = __fdiv_rn(*absmax, 0.99f);
  const long long n4 = n / 4;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = x4[i];
    short4 o;
    o.x = cvt_i16(v.x, audio_max); o.y = cvt_i16(v.y, audio_max); o.z = cvt_i16(v.z, audio_max); o.w = cvt_i16(v.w, audio_max);
    *reinterpret_cast<short4*>(out + i * 4) = o;
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = cvt_i16(x[i], audio_max);
}

// Quiet-point search of VC.pipeline (vc_infer_pipeline.py:127-135) for ONE centre: candidates j in [lo, hi), value
// |audio_pad[j] + ... + audio_pad[j + window - 1]| with the sum accumulated left to right in double from +0.0 -- the
// reference's `audio_sum += audio_pad[i : i - window]` order per element, so the sums are bit-identical to numpy's.
// Block b scans its contiguous share of the range and writes its first minimum; the (few) block results are reduced by
// the caller in ascending block order with a strict '<' (first minimum overall, like np.where(seg == seg.min())[0][0]).
__global__ void quiet_point_kernel(const double* __restrict__ a, long long lo, long long hi, int window, double* __restrict__ best_v,
                                   long long* __restrict__ best_j) {
  const long long per = (hi - lo + gridDim.x - 1) / gridDim.x;
  const long long j0 = lo + (long long)blockIdx.x * per;
  const long long j1 = j0 + per < hi ? j0 + per : hi;
  double bv = INFINITY;
  long long bj = -1;
  for (long long j = j0 + threadIdx.x; j < j1; j += blockDim.x) {
    double acc = 0.0;
    for (int i = 0; i < window; ++i) acc = __dadd_rn(acc, a[j + i]);
    const double v = fabs(acc);
    if (v < bv) { bv = v; bj = j; }
  }
  __shared__ double sv[256];
  __shared__ long long sj[256];
  sv[threadIdx.x] = bv; sj[threadIdx.x] = bj;
  __syncthreads();
  for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      const double v2 = sv[threadIdx.x + o];
      const long long j2 = sj[threadIdx.x + o];
      const double v1 = sv[threadIdx.x];
      const long long jj = sj[threadIdx.x];
      if (j2 >= 0 && (jj < 0 || v2 < v1 || (v2 == v1 && j2 < jj))) { sv[threadIdx.x] = v2; sj[threadIdx.x] = j2; }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { best_v[blockIdx.x] = sv[0]; best_j[blockIdx.x] = sj[0]; }
}

// ---- volume-envelope mix (change_rms, lib/model_utils.py:39, called at vc_infer_pipeline.py:183) ----------------------------
// librosa.feature.rms(frame_length = 2 * hop, center=True, pad_mode="constant"): frame f covers half-blocks f - 1 and f, where
// half-block b is samples [b * hop, (b + 1) * hop) of the signal and half-blocks outside it are zero.  So the envelope is
// built from half-block sums, which a piece of the signal (one segment's output) can contribute to on its own.

// One block per half-block the piece touches: out[k] = sum over the piece's samples of half-block offset / hop + k of
// float32(x)^2 (the square rounded to float32 like numpy's `np.power(x, 2, dtype=np.float32)`), accumulated in double.
// Thread t adds the samples at global positions b * hop + t + 256 j in ascending j; a fixed tree then combines the 256
// threads.  The order depends only on which samples of the half-block the piece holds, not on the grid or the piece's
// global offset, so every rank produces the same bits for the same piece.
template <typename T>
__global__ void __launch_bounds__(256) rms_halfblock_kernel(const T* __restrict__ x, long long len, long long offset, int hop,
                                                            double* __restrict__ out) {
  const long long b = offset / hop + blockIdx.x;
  const long long glo = b * hop > offset ? b * hop : offset;                       // global sample range of this block
  const long long ghi = (b + 1) * hop < offset + len ? (b + 1) * hop : offset + len;
  long long g = b * hop + threadIdx.x;
  if (g < glo) g += (glo - g + blockDim.x - 1) / blockDim.x * blockDim.x;
  double acc = 0.0;
#pragma unroll 4
  for (; g < ghi; g += blockDim.x) {
    const float v = (float)x[g - offset];                                           // float64 input: rounded to nearest
    acc = __dadd_rn(acc, (double)__fmul_rn(v, v));
  }
  __shared__ double sm[256];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sm[threadIdx.x] = __dadd_rn(sm[threadIdx.x], sm[threadIdx.x + o]);
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sm[0];
}

// rms[f] = sqrt(mean of frame f) in float32, f < n_hb.  table[r][b] (r < rows, row stride n_hb) holds half-block sums split
// over rows (one row per segment, zero where a segment does not reach); the rows are added in ascending order from +0.0,
// then frame f = hb[f - 1] + hb[f] (hb[-1] = 0), divided by frame_length in double and rounded once to float32.
__global__ void rms_fold_kernel(const double* __restrict__ table, int rows, long long n_hb, int frame_length, float* __restrict__ rms) {
  for (long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x; f < n_hb; f += (long long)gridDim.x * blockDim.x) {
    double a = 0.0, b = 0.0;
    for (int r = 0; r < rows; ++r) {
      if (f > 0) a = __dadd_rn(a, table[(long long)r * n_hb + f - 1]);
      b = __dadd_rn(b, table[(long long)r * n_hb + f]);
    }
    rms[f] = __fsqrt_rn(__double2float_rn(__ddiv_rn(__dadd_rn(a, b), (double)frame_length)));
  }
}

// F.interpolate(env[1][1][n_in], size=N, mode="linear", align_corners=False)[d] exactly as torch's float32 CPU kernel
// rounds it: the source index is one fused multiply-add on float32(d) + 0.5 (with N > 2^24 that sum already rounds), and
// the blend is fma(x0, 1 - lam, x1 * lam).  Explicit intrinsics: a more accurate index misses torch by up to 9 % at N = 86.4 M.
__device__ __forceinline__ float interp_linear(const float* __restrict__ env, int n_in, float scale, long long d) {
  const float t = __fadd_rn(__ll2float_rn(d), 0.5f);
  const float src = fmaxf(__fmaf_rn(t, scale, -0.5f), 0.f);
  const int i0 = min((int)src, n_in - 1);
  const int i1 = min(i0 + 1, n_in - 1);
  const float lam = fminf(fmaxf(__fsub_rn(src, (float)i0), 0.f), 1.f);
  return __fmaf_rn(env[i0], __fsub_rn(1.f, lam), __fmul_rn(env[i1], lam));
}

// x[i] *= pow(e1, 1 - rate) * pow(max(e2, 1e-6), rate - 1) for the samples d = offset + i of a song of N samples:
// e1 / e2 = the input / output envelopes interpolated to N; the exponents are float32(1 - rate) and float32(rate - 1)
// (`torch.tensor(1 - rate)`); the product and the update are single float32 roundings (torch's `*`, numpy's `*=`).
__global__ void rms_gain_kernel(float* __restrict__ x, long long len, long long offset, long long N, const float* __restrict__ e1, int n1,
                                const float* __restrict__ e2, int n2, float p1, float p2) {
  const float fN = __ll2float_rn(N);
  const float s1 = __fdiv_rn((float)n1, fN), s2 = __fdiv_rn((float)n2, fN);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (long long)gridDim.x * blockDim.x) {
    const long long d = offset + i;
    const float v1 = interp_linear(e1, n1, s1, d);
    const float v2 = fmaxf(interp_linear(e2, n2, s2, d), 1e-6f);
    const float gain = __fmul_rn(powf(v1, p1), powf(v2, p2));
    x[i] = __fmul_rn(x[i], gain);
  }
}

// ---- output resampling (resample_sr, vc_infer_pipeline.py:185-186) -----------------------------------------------------------
// y[j] = sum_k tab[r][k] * x[m0 - k], k = 0 .. tpp - 1 in ascending order, one fp32 FMA each, from +0.0, where
// t = j * down + half_len, r = t % up, m0 = t / up and tab[r][k] = up * h[r + k * up] (comfy_rvc_b200/resample.py).  The sum of
// an output depends on nothing but j and the input values, so any split of the output range gives the same bits.
//
// A CTA owns the outputs [J0, J0 + qb * up).  Outputs j and j + up share a phase and their inputs are `down` apart, so a task
// is (phase s, 32 consecutive q): lane L computes j = J0 + s + (32 c + L) * up, every lane reads the same tap (a broadcast
// load) and the inputs x[m0(J0 + s) + (32 c + L) * down - k] from shared memory.  The CTA's input window is staged once, with
// one padding word after every `down` words when down is even, so that those 32 reads fall in 32 different banks.
struct ResampleIn {
  const float* left;
  const float* piece;
  const float* right;
  long long n_left, n_piece, n_right, piece_off, n_song;
};

__device__ __forceinline__ float resample_fetch(const ResampleIn& in, long long m) {
  if (m < 0 || m >= in.n_song) return 0.f;
  const long long rel = m - in.piece_off;
  if (rel < 0) return rel >= -in.n_left ? in.left[in.n_left + rel] : 0.f;
  if (rel < in.n_piece) return in.piece[rel];
  return rel - in.n_piece < in.n_right ? in.right[rel - in.n_piece] : 0.f;
}

constexpr int kResampleThreads = 256;

__global__ void __launch_bounds__(kResampleThreads) resample_poly_kernel(const float* __restrict__ tab, int up, int down, int tpp,
                                                                          long long half_len, ResampleIn in, long long out_lo,
                                                                          long long out_hi, int qb, float* __restrict__ out) {
  extern __shared__ float xs[];
  const int stride = (tpp + 3) & ~3;
  const int pad = (down & 1) ? 0 : 1;
  const long long J0 = out_lo + (long long)blockIdx.x * qb * up;
  const long long w_lo = (J0 * down + half_len) / up - (tpp - 1);                  // first input sample of the window
  const long long w_hi = ((J0 + (long long)up - 1) * down + half_len) / up + (long long)(qb - 1) * down;
  const int nw = (int)(w_hi - w_lo + 1);
  for (int i = threadIdx.x; i < nw; i += kResampleThreads) xs[i + pad * (i / down)] = resample_fetch(in, w_lo + i);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int chunks = qb >> 5;
  for (int task = warp; task < up * chunks; task += kResampleThreads / 32) {
    const int s = task % up, c = task / up;
    const long long js = J0 + s;
    const long long t = js * down + half_len;
    const int r = (int)(t % up);
    const int a = (int)(t / up - w_lo);                                             // local index of m0(js), >= tpp - 1
    const int q = c * 32 + lane;
    const float* __restrict__ tr = tab + (long long)r * stride;
    const float* __restrict__ xl = xs + q * (down + pad);
    int fu = a + pad * (a / down);                                                  // padded address of local index a - k
    int col = a % down;
    float acc = 0.f;
    int k = 0;
    for (; k + 4 <= tpp; k += 4) {
      const float4 w = __ldg(reinterpret_cast<const float4*>(tr + k));
      const float wk[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        acc = __fmaf_rn(wk[u], xl[fu], acc);
        fu -= 1;
        if (col == 0) { fu -= pad; col = down; }
        col -= 1;
      }
    }
    for (; k < tpp; ++k) {
      acc = __fmaf_rn(__ldg(tr + k), xl[fu], acc);
      fu -= 1;
      if (col == 0) { fu -= pad; col = down; }
      col -= 1;
    }
    const long long j = js + (long long)q * up;
    if (j < out_hi) out[j - out_lo] = acc;
  }
}

inline unsigned stream_grid(long long work, int threads) {
  long long blocks = (work + threads - 1) / threads;
  const long long cap = 148 * 8;
  return (unsigned)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

}  // namespace

cudaError_t launch_prepare_feats(const void* f, const void* f0, int dtype, const float* pitchf, float* out, int F, int T, int C,
                                 float protect, int use_protect, cudaStream_t st) {
  if (T <= 0 || C % 4 != 0 || T > 2 * F || (use_protect && (!f0 || !pitchf))) return cudaErrorInvalidValue;
  const unsigned grid = stream_grid((long long)T * (C / 4), 256);
  if (dtype == 0)
    prepare_feats_kernel<float><<<grid, 256, 0, st>>>((const float*)f, (const float*)f0, pitchf, out, T, C, protect, use_protect);
  else if (dtype == 1)
    prepare_feats_kernel<__half><<<grid, 256, 0, st>>>((const __half*)f, (const __half*)f0, pitchf, out, T, C, protect, use_protect);
  else
    return cudaErrorInvalidValue;
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_absmax(const float* x, long long n, float* out, int reset, cudaStream_t st) {
  if (n < 0 || (reinterpret_cast<uintptr_t>(x) & 15)) return cudaErrorInvalidValue;
  if (reset) {
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float), st);
    if (e != cudaSuccess) return e;
  }
  if (n == 0) return cudaSuccess;
  absmax_kernel<<<stream_grid(n / 4 + 1, 256), 256, 0, st>>>(x, n, reinterpret_cast<unsigned*>(out));
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_quiet_point(const double* audio_pad, long long lo, long long hi, int window, double* best_v, long long* best_j,
                               int n_blocks, cudaStream_t st) {
  if (!audio_pad || !best_v || !best_j || hi <= lo || window < 1 || n_blocks < 1 || n_blocks > 65535) return cudaErrorInvalidValue;
  quiet_point_kernel<<<n_blocks, 256, 0, st>>>(audio_pad, lo, hi, window, best_v, best_j);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_to_int16(const float* x, long long n, const float* absmax, short* out, cudaStream_t st) {
  if (n < 0 || (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(out) & 7)) return cudaErrorInvalidValue;
  if (n == 0) return cudaSuccess;
  to_int16_kernel<<<stream_grid(n / 4 + 1, 256), 256, 0, st>>>(x, n, absmax, out);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_rms_halfblock(const void* x, int x_f64, long long len, long long offset, int hop, double* out, cudaStream_t st) {
  if (!x || !out || len < 0 || offset < 0 || hop < 1 || (x_f64 != 0 && x_f64 != 1)) return cudaErrorInvalidValue;
  if (len == 0) return cudaSuccess;
  const long long blocks = (offset + len - 1) / hop - offset / hop + 1;
  if (blocks > 0x7fffffffLL) return cudaErrorInvalidValue;
  if (x_f64)
    rms_halfblock_kernel<double><<<(unsigned)blocks, 256, 0, st>>>((const double*)x, len, offset, hop, out);
  else
    rms_halfblock_kernel<float><<<(unsigned)blocks, 256, 0, st>>>((const float*)x, len, offset, hop, out);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_rms_fold(const double* table, int rows, long long n_hb, int frame_length, float* rms, cudaStream_t st) {
  if (!table || !rms || rows < 1 || n_hb < 1 || frame_length < 1) return cudaErrorInvalidValue;
  rms_fold_kernel<<<stream_grid(n_hb, 128), 128, 0, st>>>(table, rows, n_hb, frame_length, rms);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_rms_gain(float* x, long long len, long long offset, long long N, const float* rms1, long long n1, const float* rms2,
                            long long n2, double rate, cudaStream_t st) {
  if (!x || !rms1 || !rms2 || len < 0 || offset < 0 || N < 1 || offset + len > N || n1 < 1 || n2 < 1 || n1 > 0x7fffffffLL ||
      n2 > 0x7fffffffLL || !std::isfinite(rate))
    return cudaErrorInvalidValue;
  if (len == 0) return cudaSuccess;
  const float p1 = (float)(1.0 - rate), p2 = (float)(rate - 1.0);
  rms_gain_kernel<<<stream_grid(len, 256), 256, 0, st>>>(x, len, offset, N, rms1, (int)n1, rms2, (int)n2, p1, p2);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_resample_poly(const float* tab, int up, int down, int tpp, long long half_len, const float* left, long long n_left,
                                 const float* piece, long long n_piece, const float* right, long long n_right, long long piece_off,
                                 long long n_song, long long out_lo, long long out_hi, float* out, cudaStream_t st) {
  constexpr long long kMaxRate = 1 << 20, kMaxLen = 1LL << 40;
  if (!tab || (reinterpret_cast<uintptr_t>(tab) & 15) || up < 1 || down < 1 || up > kMaxRate || down > kMaxRate || tpp < 1 ||
      half_len < 0 || half_len >= (long long)tpp * up || n_left < 0 || n_piece < 0 || n_right < 0 || piece_off < n_left ||
      n_song > kMaxLen || piece_off + n_piece + n_right > n_song || (n_left && !left) || (n_piece && !piece) ||
      (n_right && !right) || out_lo < 0 || out_hi < out_lo || out_hi > kMaxLen)
    return cudaErrorInvalidValue;
  if (out_hi == out_lo) return cudaSuccess;
  if (!out) return cudaErrorInvalidValue;
  // every input sample the outputs [out_lo, out_hi) reach inside the song must be in [left | piece | right]
  const long long m_first = std::max((out_lo * down + half_len) / up - (tpp - 1), 0LL);
  const long long m_last = std::min(((out_hi - 1) * down + half_len) / up, n_song - 1);
  if (m_first <= m_last && (m_first < piece_off - n_left || m_last >= piece_off + n_piece + n_right)) return cudaErrorInvalidValue;
  // a CTA covers qb * up outputs: about 8 K input words of window, qb a multiple of 32
  const long long qb = std::max(32LL, (8192LL - tpp) / down / 32 * 32);
  const long long nw = qb * down + tpp + 1;                                            // window length bound
  const size_t smem = (size_t)(nw + ((down & 1) ? 0 : nw / down + 1)) * sizeof(float);
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  if (smem > 48 * 1024) {                                                              // per device: set on every such launch
    cudaError_t e = cudaFuncSetAttribute(resample_poly_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const long long blocks = (out_hi - out_lo + qb * up - 1) / (qb * up);
  if (blocks > 0x7fffffffLL) return cudaErrorInvalidValue;
  const ResampleIn in{left, piece, right, n_left, n_piece, n_right, piece_off, n_song};
  resample_poly_kernel<<<(unsigned)blocks, kResampleThreads, smem, st>>>(tab, up, down, tpp, half_len, in, out_lo, out_hi, (int)qb,
                                                                          out);
  launch_counter().n++;
  return cudaGetLastError();
}

}  // namespace rvc
