// Index blend of VC.vc (vc_infer_pipeline.py:59-75) on the device, for IVF-Flat indices searched with nprobe = 1 (IndexFlatL2 is
// one list holding every vector in id order):
//   ivf_assign : coarse step, l = argmin_c ||q - c||^2 (lowest centroid index on an exact tie)
//   ivf_scan   : bucket the queries by list, scan each chosen list exhaustively (direct-form distances, earliest list position on an
//                exact tie), then (score, id) per query; an empty list gives (+inf, -1)
//   index_blend: big_npy[ix] * (w / w), w = (1 / score)^2, optional fp16 rounding, then the index_rate blend with torch's roundings
// All distance arithmetic is fp32 FFMA on the CUDA cores: 16-bit or TF32 operand rounding would change neighbours far more often.
// Cross-CTA merges are a 64-bit atomicMin on (order-preserving key of the fp32 distance) << 32 | (centroid index or list
// position), so every result is the same bits for every grid and every run.
#include <cuda_fp16.h>

#include <cmath>

#include "common.cuh"

namespace rvc {
namespace {

constexpr unsigned long long kNone = ~0ull;

// Unsigned key with the order of the float (negative values below positive ones).
__device__ __forceinline__ unsigned order_key(float v) {
  const unsigned b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_value(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float round_half(float v) { return __half2float(__float2half_rn(v)); }

// Min of a packed key over the 16 lanes of a half warp.
__device__ __forceinline__ unsigned long long halfwarp_min(unsigned long long k) {
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) {
    const unsigned long long t = __shfl_xor_sync(0xffffffffu, k, o);
    k = t < k ? t : k;
  }
  return k;
}

// ---- coarse step ---------------------------------------------------------------------------------------------------------------
// CTA tile: 64 queries x 128 centroids, k staged 32 at a time in shared memory (row-major, stride 33: conflict-free stores and
// reads).  Thread (ty, tx) of 16 x 16 owns queries ty + 16 i (i < 4) and centroids tx + 16 j (j < 8).  Distance up to the
// query's own norm, which is the same for every centroid: ||c||^2 - 2 q.c.
constexpr int kCQ = 64, kCC = 128, kK = 32;

template <typename T>
__global__ void __launch_bounds__(256) ivf_assign_kernel(const T* __restrict__ x, long long ldx, int F, int d,
                                                         const float* __restrict__ cent, const float* __restrict__ cnorm, int nlist,
                                                         unsigned long long* __restrict__ coarse) {
  __shared__ float qs[kCQ][kK + 1];
  __shared__ float cs[kCC][kK + 1];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int q0 = blockIdx.x * kCQ, c0 = blockIdx.y * kCC;
  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < d; k0 += kK) {
#pragma unroll
    for (int e = tid; e < kCQ * kK; e += 256) {
      const int r = e / kK, k = e % kK;
      qs[r][k] = (q0 + r < F && k0 + k < d) ? to_f32(x[(long long)(q0 + r) * ldx + k0 + k]) : 0.f;
    }
#pragma unroll
    for (int e = tid; e < kCC * kK; e += 256) {
      const int r = e / kK, k = e % kK;
      cs[r][k] = (c0 + r < nlist && k0 + k < d) ? cent[(long long)(c0 + r) * d + k0 + k] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < kK; ++k) {
      float q[4], c[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) q[i] = qs[ty + 16 * i][k];
#pragma unroll
      for (int j = 0; j < 8; ++j) c[j] = cs[tx + 16 * j][k];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = __fmaf_rn(q[i], c[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    unsigned long long best = kNone;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = c0 + tx + 16 * j;
      if (c < nlist) {
        const unsigned long long key = ((unsigned long long)order_key(__fmaf_rn(-2.f, acc[i][j], cnorm[c])) << 32) | (unsigned)c;
        best = key < best ? key : best;
      }
    }
    best = halfwarp_min(best);
    const int q = q0 + ty + 16 * i;
    if (tx == 0 && q < F && best != kNone) atomicMin(&coarse[q], best);
  }
}

// ---- grouping -------------------------------------------------------------------------------------------------------------------
__global__ void ivf_hist_kernel(const unsigned long long* __restrict__ coarse, int F, int* __restrict__ qcount) {
  for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < F; f += gridDim.x * blockDim.x)
    atomicAdd(&qcount[(unsigned)(coarse[f] & 0xffffffffu)], 1);
}

// One block: qoff = exclusive scan of the per-list query counts; item_off = exclusive scan of the fine-scan work items per list
// (query chunks x vector ranges; 0 for a list without queries or without vectors).  item_off[nlist] is the total.
constexpr int kFQ = 32, kFV = 64;

__global__ void __launch_bounds__(1024) ivf_plan_kernel(const int* __restrict__ qcount, const int* __restrict__ list_offsets, int nlist,
                                                        int* __restrict__ qoff, long long* __restrict__ item_off) {
  __shared__ long long sq[1024], si[1024];
  __shared__ long long carry_q, carry_i;
  if (threadIdx.x == 0) { carry_q = 0; carry_i = 0; }
  __syncthreads();
  for (int base = 0; base < nlist; base += 1024) {
    const int l = base + threadIdx.x;
    long long nq = 0, ni = 0;
    if (l < nlist) {
      nq = qcount[l];
      const long long nv = list_offsets[l + 1] - list_offsets[l];
      ni = ((nq + kFQ - 1) / kFQ) * ((nv + kFV - 1) / kFV);
    }
    sq[threadIdx.x] = nq;
    si[threadIdx.x] = ni;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                                      // Hillis-Steele inclusive scan
      const long long aq = threadIdx.x >= (unsigned)o ? sq[threadIdx.x - o] : 0;
      const long long ai = threadIdx.x >= (unsigned)o ? si[threadIdx.x - o] : 0;
      __syncthreads();
      sq[threadIdx.x] += aq;
      si[threadIdx.x] += ai;
      __syncthreads();
    }
    if (l < nlist) {
      qoff[l] = (int)(carry_q + sq[threadIdx.x] - nq);
      item_off[l] = carry_i + si[threadIdx.x] - ni;
    }
    __syncthreads();
    if (threadIdx.x == 1023) { carry_q += sq[1023]; carry_i += si[1023]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { qoff[nlist] = (int)carry_q; item_off[nlist] = carry_i; }
}

__global__ void ivf_scatter_kernel(const unsigned long long* __restrict__ coarse, int F, const int* __restrict__ qoff,
                                   int* __restrict__ cursor, int* __restrict__ order) {
  for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < F; f += gridDim.x * blockDim.x) {
    const unsigned l = (unsigned)(coarse[f] & 0xffffffffu);
    order[qoff[l] + atomicAdd(&cursor[l], 1)] = f;
  }
}

// ---- fine step -----------------------------------------------------------------------------------------------------------------
// Persistent grid over the work items of ivf_plan_kernel.  Item -> (list, query chunk, vector range) by a binary search of
// item_off; the CTA computes sum_k (q - v)^2 for up to 32 queries x 64 vectors (thread (ty, tx): queries ty, ty + 16, vectors
// tx + 16 j) and merges each query's best (distance, list position) with atomicMin.  Where the scatter put a query does not
// matter: its result is a min over the same keys.
template <typename T>
__global__ void __launch_bounds__(256) ivf_scan_kernel(const T* __restrict__ x, long long ldx, int d, const int* __restrict__ qcount,
                                                       const int* __restrict__ qoff, const int* __restrict__ order,
                                                       const long long* __restrict__ item_off, int nlist,
                                                       const int* __restrict__ list_offsets, const float* __restrict__ vec,
                                                       unsigned long long* __restrict__ fine) {
  __shared__ float qs[kFQ][kK + 1];
  __shared__ float vs[kFV][kK + 1];
  __shared__ int qrow[kFQ];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const long long total = item_off[nlist];
  for (long long it = blockIdx.x; it < total; it += gridDim.x) {
    int lo = 0, hi = nlist;                                                    // last l with item_off[l] <= it
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (item_off[mid] <= it) lo = mid; else hi = mid;
    }
    const int l = lo;
    const int vbeg = list_offsets[l], nv = list_offsets[l + 1] - vbeg;
    const long long nvr = (nv + kFV - 1) / kFV;
    const long long local = it - item_off[l];
    const int qc = (int)(local / nvr), vr = (int)(local % nvr);
    const int nq_tile = min(kFQ, qcount[l] - qc * kFQ);
    const int v0 = vr * kFV, nv_tile = min(kFV, nv - v0);
    if (tid < kFQ) qrow[tid] = tid < nq_tile ? order[qoff[l] + qc * kFQ + tid] : -1;
    __syncthreads();
    float acc[2][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < d; k0 += kK) {
#pragma unroll
      for (int e = tid; e < kFQ * kK; e += 256) {
        const int r = e / kK, k = e % kK, q = qrow[r];
        qs[r][k] = (q >= 0 && k0 + k < d) ? to_f32(x[(long long)q * ldx + k0 + k]) : 0.f;
      }
#pragma unroll
      for (int e = tid; e < kFV * kK; e += 256) {
        const int r = e / kK, k = e % kK;
        vs[r][k] = (r < nv_tile && k0 + k < d) ? vec[(long long)(vbeg + v0 + r) * d + k0 + k] : 0.f;
      }
      __syncthreads();
#pragma unroll 8
      for (int k = 0; k < kK; ++k) {
        float q[2], v[4];
#pragma unroll
        for (int i = 0; i < 2; ++i) q[i] = qs[ty + 16 * i][k];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = vs[tx + 16 * j][k];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float t = __fsub_rn(q[i], v[j]);
            acc[i][j] = __fmaf_rn(t, t, acc[i][j]);
          }
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      unsigned long long best = kNone;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = tx + 16 * j;
        if (r < nv_tile) {
          const unsigned long long key = ((unsigned long long)order_key(acc[i][j]) << 32) | (unsigned)(v0 + r);
          best = key < best ? key : best;
        }
      }
      best = halfwarp_min(best);
      const int q = qrow[ty + 16 * i];
      if (tx == 0 && q >= 0 && best != kNone) atomicMin(&fine[q], best);
    }
    __syncthreads();                                                           // qrow is rewritten by the next item
  }
}

__global__ void ivf_result_kernel(const unsigned long long* __restrict__ coarse, const unsigned long long* __restrict__ fine, int F,
                                  const int* __restrict__ list_offsets, const long long* __restrict__ labels, float* __restrict__ score,
                                  long long* __restrict__ ix) {
  for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < F; f += gridDim.x * blockDim.x) {
    const unsigned long long k = fine[f];
    if (k == kNone) {                                                          // the query's list holds no vector
      score[f] = __int_as_float(0x7f800000);
      ix[f] = -1;
    } else {
      const unsigned l = (unsigned)(coarse[f] & 0xffffffffu);
      score[f] = key_value((unsigned)(k >> 32));
      ix[f] = labels[list_offsets[l] + (unsigned)(k & 0xffffffffu)];
    }
  }
}

// ---- blend ---------------------------------------------------------------------------------------------------------------------
// vc_infer_pipeline.py:61-75 with each numpy / torch step's own rounding: w = float32(1 / score)^2, weight = w / w (1.0, or NaN for a
// score of 0, +inf, or one that over- / underflows w); g = big_npy[ix] * weight (ix = -1 is the last row, as numpy indexes),
// rounded to fp16 with is_half; out = round(round(g * r) + round(s * f)), each product rounded to its operand's dtype and the sum
// to the promoted dtype, no contraction (torch runs three kernels).  Four channels per thread.
template <typename TF, typename TO>
__global__ void index_blend_kernel(const TF* __restrict__ feats, long long ldf, int F, int d, const float* __restrict__ score,
                                   const long long* __restrict__ ix, const float* __restrict__ vec, const int* __restrict__ pos_of_label,
                                   long long ntotal, int is_half, float r, float s, TO* __restrict__ out) {
  const int d4 = d / 4;
  const long long n = (long long)F * d4;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(e / d4), c = (int)(e % d4) * 4;
    long long j = ix[f];
    if (j < 0) j += ntotal;
    float4 v = make_float4(__int_as_float(0x7fffffff), __int_as_float(0x7fffffff), __int_as_float(0x7fffffff), __int_as_float(0x7fffffff));
    if (j >= 0 && j < ntotal) v = *reinterpret_cast<const float4*>(vec + (long long)pos_of_label[j] * d + c);
    float w = __fdiv_rn(1.f, score[f]);
    w = __fmul_rn(w, w);
    const float weight = __fdiv_rn(w, w);
    const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float g = __fmul_rn(vv[t], weight);
      if (is_half) g = round_half(g);
      g = __fmul_rn(g, r);
      if (is_half) g = round_half(g);
      float h = __fmul_rn(s, to_f32(feats[(long long)f * ldf + c + t]));
      if (sizeof(TF) == 2) h = round_half(h);
      const float o = __fadd_rn(g, h);
      if constexpr (sizeof(TO) == 2) out[(long long)f * d + c + t] = __float2half_rn(o);
      else out[(long long)f * d + c + t] = o;
    }
  }
}

unsigned grid_for(long long work, int threads, int per_sm) {
  long long blocks = (work + threads - 1) / threads;
  const long long cap = (long long)current_num_sms() * per_sm;
  if (blocks > cap) blocks = cap;
  return (unsigned)(blocks > 0 ? blocks : 1);
}

// scratch layout of ivf_scan (8-byte arrays first)
struct ScanScratch {
  unsigned long long* fine;   // [F]
  long long* item_off;        // [nlist + 1]
  int* qcount;                // [nlist]
  int* cursor;                // [nlist]
  int* qoff;                  // [nlist + 1]
  int* order;                 // [F]
};
long long scan_scratch(int F, int nlist, void* base, ScanScratch* s) {
  char* p = static_cast<char*>(base);
  long long off = 0;
  auto take = [&](long long bytes) { char* q = p ? p + off : nullptr; off += (bytes + 15) / 16 * 16; return q; };
  char* fine = take(8LL * F);
  char* item = take(8LL * (nlist + 1));
  char* cnt = take(4LL * 2 * nlist);                                           // qcount | cursor: one memset
  char* qoff = take(4LL * (nlist + 1));
  char* order = take(4LL * F);
  if (s) {
    s->fine = reinterpret_cast<unsigned long long*>(fine);
    s->item_off = reinterpret_cast<long long*>(item);
    s->qcount = reinterpret_cast<int*>(cnt);
    s->cursor = reinterpret_cast<int*>(cnt) + nlist;
    s->qoff = reinterpret_cast<int*>(qoff);
    s->order = reinterpret_cast<int*>(order);
  }
  return off;
}

bool bad_queries(const void* x, int x_dtype, long long ldx, int F, int d) {
  return !x || (x_dtype != 0 && x_dtype != 1) || F < 0 || d < 4 || d % 4 != 0 || ldx < d;
}

}  // namespace

long long ivf_scratch_bytes(int F, int nlist) {
  if (F < 0 || nlist < 1) return -1;
  return scan_scratch(F, nlist, nullptr, nullptr);
}

cudaError_t launch_ivf_assign(const void* x, int x_dtype, long long ldx, int F, int d, const float* cent, const float* cnorm, int nlist,
                              unsigned long long* coarse, cudaStream_t st) {
  if (bad_queries(x, x_dtype, ldx, F, d) || !cent || !cnorm || nlist < 1 || !coarse) return cudaErrorInvalidValue;
  if (F == 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(coarse, 0xff, sizeof(unsigned long long) * F, st);
  if (e != cudaSuccess) return e;
  const dim3 grid((F + kCQ - 1) / kCQ, (nlist + kCC - 1) / kCC);
  if (grid.y > 65535) return cudaErrorInvalidValue;
  if (x_dtype == 0)
    ivf_assign_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(x), ldx, F, d, cent, cnorm, nlist, coarse);
  else
    ivf_assign_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(x), ldx, F, d, cent, cnorm, nlist, coarse);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_ivf_scan(const void* x, int x_dtype, long long ldx, int F, int d, const unsigned long long* coarse, int nlist,
                            const int* list_offsets, const float* vec, const long long* labels, void* scratch, long long scratch_bytes,
                            float* score, long long* ix, cudaStream_t st) {
  if (bad_queries(x, x_dtype, ldx, F, d) || !coarse || nlist < 1 || !list_offsets || !vec || !labels || !scratch || !score || !ix)
    return cudaErrorInvalidValue;
  ScanScratch s;
  if (scratch_bytes < scan_scratch(F, nlist, scratch, &s)) return cudaErrorInvalidValue;
  if (F == 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(s.fine, 0xff, sizeof(unsigned long long) * F, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(s.qcount, 0, sizeof(int) * 2 * nlist, st);
  if (e != cudaSuccess) return e;
  ivf_hist_kernel<<<grid_for(F, 256, 4), 256, 0, st>>>(coarse, F, s.qcount);
  ivf_plan_kernel<<<1, 1024, 0, st>>>(s.qcount, list_offsets, nlist, s.qoff, s.item_off);
  ivf_scatter_kernel<<<grid_for(F, 256, 4), 256, 0, st>>>(coarse, F, s.qoff, s.cursor, s.order);
  const unsigned grid = (unsigned)current_num_sms() * 4;                       // persistent: the item count stays on the device
  if (x_dtype == 0)
    ivf_scan_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(x), ldx, d, s.qcount, s.qoff, s.order, s.item_off, nlist,
                                                 list_offsets, vec, s.fine);
  else
    ivf_scan_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(x), ldx, d, s.qcount, s.qoff, s.order, s.item_off, nlist,
                                                  list_offsets, vec, s.fine);
  ivf_result_kernel<<<grid_for(F, 256, 4), 256, 0, st>>>(coarse, s.fine, F, list_offsets, labels, score, ix);
  launch_counter().n += 5;
  return cudaGetLastError();
}

cudaError_t launch_index_blend(const void* feats, int feats_dtype, long long ldf, int F, int d, const float* score, const long long* ix,
                               const float* vec, const int* pos_of_label, long long ntotal, int is_half, double index_rate, void* out,
                               cudaStream_t st) {
  if (bad_queries(feats, feats_dtype, ldf, F, d) || !score || !ix || !vec || !pos_of_label || ntotal < 1 || !out ||
      (is_half != 0 && is_half != 1) || !std::isfinite(index_rate))
    return cudaErrorInvalidValue;
  if (F == 0) return cudaSuccess;
  const float r = (float)index_rate, s = (float)(1.0 - index_rate);         // `1 - index_rate` in Python double, then the cast
  const unsigned grid = grid_for((long long)F * (d / 4), 256, 8);
  if (feats_dtype == 0)
    index_blend_kernel<float, float><<<grid, 256, 0, st>>>(static_cast<const float*>(feats), ldf, F, d, score, ix, vec, pos_of_label,
                                                           ntotal, is_half, r, s, static_cast<float*>(out));
  else if (is_half)
    index_blend_kernel<__half, __half><<<grid, 256, 0, st>>>(static_cast<const __half*>(feats), ldf, F, d, score, ix, vec, pos_of_label,
                                                             ntotal, is_half, r, s, static_cast<__half*>(out));
  else
    index_blend_kernel<__half, float><<<grid, 256, 0, st>>>(static_cast<const __half*>(feats), ldf, F, d, score, ix, vec, pos_of_label,
                                                            ntotal, is_half, r, s, static_cast<float*>(out));
  launch_counter().n++;
  return cudaGetLastError();
}

}  // namespace rvc
