// tcgen05 / TMEM implicit-GEMM 1-D convolution for sm_100a (fp16 or bf16 operands, fp32 accumulate).
//
//   D[128 time rows][N = C_out tile] (TMEM, fp32) += sum_{k-block} sum_{tap} A_tap[128][64] * W_tap[N][64]^T
//
// Operands are staged by TMA (cp.async.bulk.tensor) into the canonical K-major SWIZZLE_128B layout
// (8 rows x 128 B atoms, SBO = 1024 B) that tcgen05.mma reads at full rate.  A first version of this
// kernel (git history: commit 421ed09) used the no-swizzle "interleave" layout and measured ~256
// tensor-pipe cycles per 128xNx16 MMA independent of N (profiles/r1_conv_tc_shapes_v2.jsonl) -- 4x off
// the N=128 floor.
//
// Activations (MMA operand): 16-bit channels-last [B][L][C]; the TMA tensor map is (C, L, B) so rows
// before 0 / after L-1 and channels >= C are zero-filled by the hardware (conv zero padding and the
// K padding of the 32- and 16-channel stages come for free).
//   a_mode 0: ONE TMA box of 128+halo rows per 64-channel k-block; each tap of the (dilated) kernel is
//             a descriptor whose start address is advanced by tap*dil rows (x128 B).  The hardware
//             applies the 128B swizzle on absolute smem address bits, so base_offset stays 0 (measured:
//             base_offset = rows&7 or -rows&7 both give wrong results, 0 is bit-correct).
//   a_mode 1: one TMA box of 128 rows per (k-block, tap) at row coordinate j0 + off + tap*dil.
// Weights: 16-bit [G][C_out/N][taps][k-blocks][N][64] (K zero-padded to 64), TMA box (64, N); kept
// resident in smem for the whole persistent CTA when all (k-block, tap) tiles fit, else a ring.
// Residual stream / fp32 outputs: planar-vector fp32 [B][C/4][Lp][4] (thread = TMEM lane = time row, so
// every warp-level load/store is one 512 B transaction).
//
// Persistent, warp-specialised (320 threads): warp 0 = TMA producer (one lane), warp 1 = TMEM allocator
// + MMA issuer (one lane), warps 2..9 = two epilogue groups, each owning one of the two TMEM accumulator
// buffers (tile t is drained by group t & 1 while the MMAs of tile t+1 run).
// Replaces the cuDNN calls behind modules.py:295-308 (ResBlock1), models.py:545-551 (conv_pre, ups).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "conv_tc.cuh"
#include "tc_ptx.cuh"

namespace rvc {
namespace {

// Phase timestamps of one launch (tools/trace_generic.py): when a trace buffer is set, a few threads of every CTA record
// globaltimer at fixed points -- 16 slots per CTA.  Null (the default): one predictable branch per point.
__device__ unsigned long long* g_trace = nullptr;
__device__ __forceinline__ void trace_mark(int slot) {
  unsigned long long* t = g_trace;
  if (t) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
    t[(size_t)blockIdx.x * 16 + slot] = now;
  }
}

// Row offset of tap `tap`: 1-D kernels step by `dil`; 2-D kernels (tap_w taps per kernel row, RMVPE's 3 x 3 / 2 x 2 convolutions
// over an image stored as rows of W + 1 pixels) step by `dil` inside a kernel row and by `dil2` between kernel rows.
__host__ __device__ __forceinline__ int tap_row_off(const TcConvDesc& p, int tap) {
  return p.tap_w > 0 ? (tap / p.tap_w) * p.dil2 + (tap % p.tap_w) * p.dil : tap * p.dil;
}
__host__ __device__ __forceinline__ int tap_halo(const TcConvDesc& p) { return p.ntaps > 0 ? tap_row_off(p, p.ntaps - 1) : 0; }
// a_mode 2 ("row slabs", 2-D kernels only): one activation box per (k-block, kernel ROW) at row offset kh * dil2, holding
// 128 + (tap_w - 1) * dil rows; the tap_w taps of that kernel row are descriptor offsets into it.  A 3 x 3 convolution over a wide
// image (W = 128: a_mode 0 would need a 128 + 2 W + 4 row box, a_mode 1 nine boxes and nine wait / commit round trips per tile --
// 3.5 us per 128-row tile at C = 16, profiles/r2_rmvpe_launches_60s_v2.csv) takes three boxes and three waits per tile.
__host__ __device__ __forceinline__ int slab_rows_halo(const TcConvDesc& p) { return p.a_mode == 2 ? (p.tap_w - 1) * p.dil : tap_halo(p); }

constexpr int kEpiWarps = 8;
constexpr int kThreadsTC = 64 + 32 * kEpiWarps;   // producer warp + MMA warp + epilogue warps
constexpr int BM = 128;
constexpr int KBLK = 64;                          // channels per k-block = one 128-byte swizzled row

using namespace tc;

// Generic epilogue (text encoder / flow): channels-last or PV fp32 I/O, embedding gather, scale, gate,
// masks, residual modes.  One pass over 16 accumulator columns of this thread's row.
// `sb`: bias (+ speaker conditioning) of these 16 columns, staged in shared memory before the accumulator was waited for;
// `pre`: the residual (or the running sum of `accum`) of this row's output columns, loaded before that wait as well (null:
// loaded here).  Both used to be global loads issued after the accumulator arrived, one L2 round trip after the other per
// 16-column pass -- ~10 of the 15 us of a one-tile launch (profiles/r2_short_step_T100.md).
__device__ __forceinline__ void epilogue_generic16(const TcConvDesc& p, uint32_t taddr, bool row_ok, bool valid, int b,
                                                   long long orow, int co, const float* sb, const float4* pre) {
  uint32_t r[16];
  tmem_ld16_issue(taddr, r);
  tmem_ld_wait();
  if (!row_ok) return;
  const long long Lout = (long long)p.Lj * p.out_stride;
  float v[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]) + sb[i];
  if (p.gather) {
    const long long gi = p.gidx[(long long)b * p.gidx_bstride + orow];
    const float* gr = p.gather + gi * p.Cout_total + co;
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += __ldg(gr + i);
  }
  if (p.alpha != 1.f) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] *= p.alpha;
  }
  int nout = 16, oc = co;
  if (p.gate) {   // commons.py:211-218 on interleaved (tanh, sigmoid) pairs
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      // sigma(x) = 1 / (1 + 2^(-x log2 e)) on the MUFU pipe (ex2 + rcp, ~1e-6), tanh(a) = 2 sigma(2a) - 1: the result is
      // rounded to fp16 (2.4e-4) right below; the libm forms were ~45 instructions per gate and made this epilogue the
      // longest phase of the flow.in launches (profiles/r2_trace_generic.md)
      const float sa = __fdividef(1.f, 1.f + __expf(-2.f * v[2 * i])), sb_ = __fdividef(1.f, 1.f + __expf(-v[2 * i + 1]));
      v[i] = fmaf(2.f, sa, -1.f) * sb_;
    }
    nout = 8; oc = co >> 1;
  }
  if (p.pre_slope != 1.f) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = lrelu(v[i], p.pre_slope);
  }
  if (p.gelu) {   // exact GELU (torch.nn.functional.gelu default): 0.5 x (1 + erf(x / sqrt(2)))
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.5f * v[i] * (1.f + erff(v[i] * 0.70710678118654752f));
  }
  if (p.mask_pre && !valid) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.f;
  }
  // fp32 side: channels-last rows (ldy32 / ldr32) or planar-vector planes
  const size_t pitch_o = (size_t)p.Lp_out * 16;
  const int ctot = p.gate ? p.Cout_total / 2 : p.Cout_total;
  auto f32_ptr = [&](const float* base, int ld, int c) -> const float* {
    if (p.f32_cl) return base + ((size_t)b * Lout + orow) * ld + c;
    return reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(base) + (size_t)b * (ctot / 4) * pitch_o +
                                          (size_t)(c / 4) * pitch_o + (size_t)(orow + p.padf) * 16);
  };
  const size_t cstep = p.f32_cl ? 4 : pitch_o / 4;   // floats between consecutive 4-channel groups
  if (p.res32) {
    const float* rp = f32_ptr(p.res32, p.ldr32, oc);
#pragma unroll
    for (int k4 = 0; k4 < 4; ++k4)
      if (k4 * 4 < nout) {
        const float4 q = pre ? pre[k4] : *reinterpret_cast<const float4*>(rp + k4 * cstep);
        if (p.res_mode == 2) {
          v[k4 * 4 + 0] = q.x - v[k4 * 4 + 0]; v[k4 * 4 + 1] = q.y - v[k4 * 4 + 1];
          v[k4 * 4 + 2] = q.z - v[k4 * 4 + 2]; v[k4 * 4 + 3] = q.w - v[k4 * 4 + 3];
        } else {
          v[k4 * 4 + 0] += q.x; v[k4 * 4 + 1] += q.y; v[k4 * 4 + 2] += q.z; v[k4 * 4 + 3] += q.w;
        }
      }
  }
  if (p.relu) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
  }
  float* yp = p.y32 ? const_cast<float*>(f32_ptr(p.y32, p.ldy32, oc)) : nullptr;
  if (p.accum) {
#pragma unroll
    for (int k4 = 0; k4 < 4; ++k4)
      if (k4 * 4 < nout) {
        const float4 q = (pre && !p.res32) ? pre[k4] : *reinterpret_cast<const float4*>(yp + k4 * cstep);
        v[k4 * 4 + 0] += q.x; v[k4 * 4 + 1] += q.y; v[k4 * 4 + 2] += q.z; v[k4 * 4 + 3] += q.w;
      }
  }
  if (p.div != 1.f) {
    const float rd = 1.f / p.div;
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = div_exact(v[i], p.div, rd);
  }
  if (p.mask_post && !valid) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.f;
  }
  if (yp) {
#pragma unroll
    for (int k4 = 0; k4 < 4; ++k4)
      if (k4 * 4 < nout)
        *reinterpret_cast<float4*>(yp + k4 * cstep) = make_float4(v[k4 * 4 + 0], v[k4 * 4 + 1], v[k4 * 4 + 2], v[k4 * 4 + 3]);
  }
  if (p.y16) {
    const bool obf = p.out_bf16 != 0;
    const int ld16 = p.ldy16 ? p.ldy16 : ctot;
    unsigned char* y16row = reinterpret_cast<unsigned char*>(p.y16) + (((size_t)b * Lout + orow) * ld16 + oc) * 2;
    const bool z16 = p.mask16 && !valid;
#pragma unroll
    for (int k8 = 0; k8 < 2; ++k8)
      if (k8 * 8 < nout) {
        uint4 o;
        o.x = pack2(obf, lrelu(v[k8 * 8 + 0], p.out_slope), lrelu(v[k8 * 8 + 1], p.out_slope));
        o.y = pack2(obf, lrelu(v[k8 * 8 + 2], p.out_slope), lrelu(v[k8 * 8 + 3], p.out_slope));
        o.z = pack2(obf, lrelu(v[k8 * 8 + 4], p.out_slope), lrelu(v[k8 * 8 + 5], p.out_slope));
        o.w = pack2(obf, lrelu(v[k8 * 8 + 6], p.out_slope), lrelu(v[k8 * 8 + 7], p.out_slope));
        if (z16) o = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(y16row + k8 * 16) = o;
      }
  }
}

// Lean form of the generic epilogue for one whole 128 x 64 tile (the N tile of every text-encoder / flow / HuBERT
// contraction): the four tcgen05.ld of the row are in flight together, every mode flag is tested once per tile instead of
// once per 16-column pass, the row's output addresses are formed once.  The pass-by-pass form above costs ~1700 cycles per
// pass with ONE warp per scheduler running it (a dependent chain of flag tests and 64-bit address arithmetic per pass,
// 3.6 us per tile, profiles/r2_trace_generic.md); it stays for the other N and the modes not listed in `lean_ok`.
__device__ __forceinline__ bool lean_ok(const TcConvDesc& p) {
  return p.N == 64 && p.f32_cl && !p.gather && p.alpha == 1.f && p.pre_slope == 1.f && p.div == 1.f && !p.out_bf16 &&
         p.out_slope == 1.f && !(p.res32 && p.accum) && !(p.gate && (p.res32 || p.accum || p.y32 || p.relu || p.gelu));
}
__device__ __forceinline__ void epilogue_lean64(const TcConvDesc& p, uint32_t taddr, bool row_ok, bool valid, int b, long long orow,
                                                int co, const float* sb, const float4* pre, bool have_pre) {
  uint32_t r[64];
#pragma unroll
  for (int q = 0; q < 4; ++q) tmem_ld16_issue(taddr + 16u * q, r + q * 16);
  tmem_ld_wait();
  if (!row_ok) return;
  const long long Lout = (long long)p.Lj * p.out_stride;
  float v[64];
#pragma unroll
  for (int i = 0; i < 64; i += 4) {
    const float4 bq = *reinterpret_cast<const float4*>(sb + i);
    v[i] = __uint_as_float(r[i]) + bq.x; v[i + 1] = __uint_as_float(r[i + 1]) + bq.y;
    v[i + 2] = __uint_as_float(r[i + 2]) + bq.z; v[i + 3] = __uint_as_float(r[i + 3]) + bq.w;
  }
  const size_t rowi = (size_t)b * Lout + orow;
  if (p.gate) {   // 32 gated channels -> 16-bit only (lean_ok)
    uint4 o[4];
    uint32_t* ow = reinterpret_cast<uint32_t*>(o);
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
      float g2[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float sa = __fdividef(1.f, 1.f + __expf(-2.f * v[2 * (i + e)])), sg = __fdividef(1.f, 1.f + __expf(-v[2 * (i + e) + 1]));
        g2[e] = fmaf(2.f, sa, -1.f) * sg;
      }
      if (p.mask_pre && !valid) { g2[0] = 0.f; g2[1] = 0.f; }
      ow[i >> 1] = pack2(false, g2[0], g2[1]);
    }
    if ((p.mask16 || p.mask_post) && !valid) {
#pragma unroll
      for (int q = 0; q < 4; ++q) o[q] = make_uint4(0, 0, 0, 0);
    }
    if (p.y16) {
      const int ctot = p.Cout_total / 2, ld16 = p.ldy16 ? p.ldy16 : ctot;
      uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(p.y16) + (rowi * ld16 + (co >> 1)) * 2);
#pragma unroll
      for (int q = 0; q < 4; ++q) dst[q] = o[q];
    }
    return;
  }
  if (p.gelu) {   // exact GELU (torch.nn.functional.gelu default)
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = 0.5f * v[i] * (1.f + erff(v[i] * 0.70710678118654752f));
  }
  if (p.mask_pre && !valid) {
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = 0.f;
  }
  if (p.res32) {
    const float4* rp = reinterpret_cast<const float4*>(p.res32 + rowi * p.ldr32 + co);
    if (p.res_mode == 2) {
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const float4 q = have_pre ? pre[k] : rp[k];
        v[4 * k] = q.x - v[4 * k]; v[4 * k + 1] = q.y - v[4 * k + 1]; v[4 * k + 2] = q.z - v[4 * k + 2]; v[4 * k + 3] = q.w - v[4 * k + 3];
      }
    } else {
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const float4 q = have_pre ? pre[k] : rp[k];
        v[4 * k] += q.x; v[4 * k + 1] += q.y; v[4 * k + 2] += q.z; v[4 * k + 3] += q.w;
      }
    }
  }
  if (p.relu) {
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = fmaxf(v[i], 0.f);
  }
  float4* yp = p.y32 ? reinterpret_cast<float4*>(p.y32 + rowi * p.ldy32 + co) : nullptr;
  if (p.accum) {
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 q = have_pre ? pre[k] : yp[k];
      v[4 * k] += q.x; v[4 * k + 1] += q.y; v[4 * k + 2] += q.z; v[4 * k + 3] += q.w;
    }
  }
  if (p.mask_post && !valid) {
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = 0.f;
  }
  if (yp) {
#pragma unroll
    for (int k = 0; k < 16; ++k) yp[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
  }
  if (p.y16) {
    const int ld16 = p.ldy16 ? p.ldy16 : p.Cout_total;
    uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(p.y16) + (rowi * ld16 + co) * 2);
    const bool z16 = p.mask16 && !valid;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      uint4 o;
      o.x = pack2(false, v[8 * k], v[8 * k + 1]); o.y = pack2(false, v[8 * k + 2], v[8 * k + 3]);
      o.z = pack2(false, v[8 * k + 4], v[8 * k + 5]); o.w = pack2(false, v[8 * k + 6], v[8 * k + 7]);
      if (z16) o = make_uint4(0, 0, 0, 0);
      dst[k] = o;
    }
  }
}

template <bool GENERIC>
__global__ void __launch_bounds__(kThreadsTC, 1)
conv_tc_kernel(const TcConvDesc p, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
               const __grid_constant__ CUtensorMap tmY) {
  extern __shared__ unsigned char smem_raw[];
  if (threadIdx.x == 0) trace_mark(0);                                     // CTA started
  // aligned with pointer arithmetic on the __shared__ array (not through an integer cast): the compiler keeps the
  // shared address space and emits LDS/STS instead of generic LD/ST for every access derived from it
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const int halo = slab_rows_halo(p);
  const bool slab = p.a_mode != 1;                             // a_mode 0: one box per k-block; 2: one per (k-block, kernel row)
  const int KH = p.a_mode == 2 ? p.ntaps / p.tap_w : 1;        // activation boxes per k-block
  const int TW = p.a_mode == 2 ? p.tap_w : p.ntaps;            // taps per activation box
  const int R = slab ? ((BM + halo + 7) & ~7) : BM;            // rows per activation box
  const int nkb = (p.Cin + KBLK - 1) / KBLK;
  const uint32_t a_bytes = (uint32_t)R * 128;
  const uint32_t b_bytes = (uint32_t)p.N * 128;
  const int NA = p.na_stages, NB = p.nb_stages;
  const uint32_t a_stride = (a_bytes + 1023) & ~1023u, b_stride = (b_bytes + 1023) & ~1023u;
  // Weight ring of the non-resident case: one ring stage = SG weight tiles (one wait / expect / commit per stage instead of
  // per tile).  The two single-thread loops below are instruction-bound -- ~0.45 us per ring step whatever its bytes and
  // whatever the contention (profiles/r2_trace_generic.md) -- so a stage carries SG consecutive k-blocks of a 1-tap contraction or
  // SG consecutive taps of a k-block; the launcher picks SG (b_group).
  const int SG = (p.b_stationary || p.a_mode == 1 || p.b_group < 1) ? 1 : p.b_group;
  const uint32_t b_slot = (uint32_t)SG * b_stride;          // bytes per ring stage

  unsigned char* slabA = smem;                              // [NA][R][128 B] swizzled
  unsigned char* slabB = smem + (size_t)NA * a_stride;      // [NB][SG][N][128 B] swizzled
  uint64_t* bars = reinterpret_cast<uint64_t*>(slabB + (size_t)NB * b_slot);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + NA;
  uint64_t* b_full = a_empty + NA;
  uint64_t* b_empty = b_full + NB;
  uint64_t* acc_full = b_empty + NB;     // [2]
  uint64_t* acc_empty = acc_full + 2;    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  // 16-bit output staging (tma_out): [8 warps][2 slots][32 rows x 64 B], SWIZZLE_64B
  unsigned char* sE = reinterpret_cast<unsigned char*>(tmem_slot + 4);
  sE += (1024u - (smem_u32(sE) & 1023u)) & 1023u;

  const int n_mt = (p.Lj + BM - 1) / BM;
  const int n_nt = p.Cout_total / p.N;
  const long long total_tiles = (long long)n_mt * n_nt * p.G * p.batch;
  const int my_tiles = (int)((total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
  const bool stat = p.b_stationary != 0;

  if (threadIdx.x == 0) {
    pdl_trigger();
    for (int i = 0; i < NA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < NB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], kEpiWarps / 2); }
    fence_mbarrier_init();
    fence_proxy_async();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW);
  }
  if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);   // two accumulator buffers of N columns (power of two >= 32)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) trace_mark(1);                                     // barriers initialised, TMEM allocated

  // Tile order: phase g fastest, then the N tile, then the M tile.  The G phases (and N tiles) of one M tile run on
  // neighbouring CTAs at the same time, so the activation slab is read from HBM once (L2 hits for the rest) and the
  // row-interleaved outputs of a transposed conv (row = t*G + g: 16-byte pieces of the same 32-byte sectors / 128-byte
  // lines written by different phases) merge in L2 instead of being evicted half-written.
  auto decode = [&](long long t, int& mt, int& nt, int& g, int& b) {
    g = (int)(t % p.G); t /= p.G;
    nt = (int)(t % n_nt); t /= n_nt;
    mt = (int)(t % n_mt);
    b = (int)(t / n_mt);
  };
  // weight row coordinate of tile (g, nt), tap, k-block in the [..][N][64] table
  auto w_row = [&](int g, int nt, int tap, int kb) { return (((g * n_nt + nt) * p.ntaps + tap) * nkb + kb) * p.N; };
  // (tried in round 2: starting the K loop of M tile mt at k-block mt % nkb so that the ~47 CTAs of a launch do not ask L2 for
  //  the same weight tile at the same moment -- no change in the flow / encoder classes, profiles/r2_ab_rings_injgemm.md)

  if (warp == 0) {
    // =========================== producer: TMA global -> swizzled smem ============================
    if (lane == 0) {
      if (stat) {  // all (k-block, tap) weight tiles stay resident for every tile of this CTA
        for (int kb = 0; kb < nkb; ++kb)
          for (int tap = 0; tap < p.ntaps; ++tap) {
            const int sb = kb * p.ntaps + tap;
            mbar_expect_tx(&b_full[sb], b_bytes);
            tma_load_2d(slabB + (size_t)sb * b_stride, &tmW, 0, w_row((int)(blockIdx.x % (unsigned)p.G), 0, tap, kb), &b_full[sb]);
          }
      }
      pdl_wait();                         // activations come from the previous kernel (the weights above do not)
      trace_mark(2);                      // producer may load activations
      int sa = 0, sb = 0;                 // ring slots; phase bits flip on wrap (no div/mod in the loop)
      uint32_t pa = 1, pb = 1;            // producer waits on "empty" with inverted parity
      for (int t = 0; t < my_tiles; ++t) {
        int mt, nt, g, b;
        decode((long long)blockIdx.x + (long long)t * gridDim.x, mt, nt, g, b);
        const int row0 = mt * BM + p.g_off[g];
        // grouped convolutions (HuBERT's positional convolution: 16 groups of 48 channels): N tile nt reads its own input channels
        // [nt * a_nt_stride, + Cin); what a 64-channel box reads beyond them meets the zero K padding of the weight image
        const int ch0 = nt * p.a_nt_stride;
        int wrow = w_row(g, nt, 0, 0);
        if (SG > 1) {                     // grouped ring stages (slab modes, weights not resident)
          if (p.ntaps == 1) {             // a stage = SG consecutive k-blocks; their activation boxes first
            for (int kbg = 0; kbg < nkb; kbg += SG) {
              const int cnt = nkb - kbg < SG ? nkb - kbg : SG;
              for (int kk = 0; kk < cnt; ++kk) {
                mbar_wait(&a_empty[sa], pa);
                mbar_expect_tx(&a_full[sa], a_bytes);
                tma_load_3d(slabA + (size_t)sa * a_stride, &tmA, (kbg + kk) * KBLK + ch0, row0, b, &a_full[sa]);
                if (++sa == NA) { sa = 0; pa ^= 1; }
              }
              mbar_wait(&b_empty[sb], pb);
              mbar_expect_tx(&b_full[sb], (uint32_t)cnt * b_bytes);
              for (int kk = 0; kk < cnt; ++kk)
                tma_load_2d(slabB + (size_t)sb * b_slot + (size_t)kk * b_stride, &tmW, 0, wrow + (kbg + kk) * p.N, &b_full[sb]);
              if (++sb == NB) { sb = 0; pb ^= 1; }
            }
          } else {                        // a stage = SG consecutive taps of one (k-block, activation box)
            for (int kb = 0; kb < nkb; ++kb)
              for (int kh = 0; kh < KH; ++kh) {
                mbar_wait(&a_empty[sa], pa);
                mbar_expect_tx(&a_full[sa], a_bytes);
                tma_load_3d(slabA + (size_t)sa * a_stride, &tmA, kb * KBLK + ch0, row0 + kh * p.dil2, b, &a_full[sa]);
                if (++sa == NA) { sa = 0; pa ^= 1; }
                for (int tg = 0; tg < TW; tg += SG) {
                  const int cnt = TW - tg < SG ? TW - tg : SG;
                  mbar_wait(&b_empty[sb], pb);
                  mbar_expect_tx(&b_full[sb], (uint32_t)cnt * b_bytes);
                  for (int tl = 0; tl < cnt; ++tl)
                    tma_load_2d(slabB + (size_t)sb * b_slot + (size_t)tl * b_stride, &tmW, 0,
                                wrow + ((kh * TW + tg + tl) * nkb + kb) * p.N, &b_full[sb]);
                  if (++sb == NB) { sb = 0; pb ^= 1; }
                }
              }
          }
          continue;
        }
        for (int kb = 0; kb < nkb; ++kb)
         for (int kh = 0; kh < KH; ++kh) {
          if (slab) {
            mbar_wait(&a_empty[sa], pa);
            mbar_expect_tx(&a_full[sa], a_bytes);
            tma_load_3d(slabA + (size_t)sa * a_stride, &tmA, kb * KBLK + ch0, row0 + kh * p.dil2, b, &a_full[sa]);
            if (++sa == NA) { sa = 0; pa ^= 1; }
          }
          for (int tap = kh * TW; tap < kh * TW + TW; ++tap) {
            if (!slab) {
              mbar_wait(&a_empty[sa], pa);
              mbar_expect_tx(&a_full[sa], a_bytes);
              tma_load_3d(slabA + (size_t)sa * a_stride, &tmA, kb * KBLK + ch0, row0 + tap_row_off(p, tap), b, &a_full[sa]);
              if (++sa == NA) { sa = 0; pa ^= 1; }
            }
            if (!stat) {
              mbar_wait(&b_empty[sb], pb);
              mbar_expect_tx(&b_full[sb], b_bytes);
              tma_load_2d(slabB + (size_t)sb * b_stride, &tmW, 0, wrow + (tap * nkb + kb) * p.N, &b_full[sb]);
              if (++sb == NB) { sb = 0; pb ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: warp-uniform control flow, one elected lane issues ==========
    // (keeping the loop uniform lets the compiler hold descriptors in uniform registers; a per-thread
    //  `if (lane == 0)` loop spent ~20 SASS instructions / ~270 cycles per UTCHMMA on R2UR traffic.)
    const uint32_t fmt = p.in_bf16 ? 1u : 0u;
    // instruction descriptor: D=F32 @4, A/B format @7/@10, K-major both, N>>3 @17, M>>4 @24
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(p.N >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    const uint64_t dproto = make_desc_sw128(0, 0);
    const uint32_t d_hi0 = (uint32_t)(dproto >> 32), d_lo0 = (uint32_t)dproto;
    const uint32_t slabA_u = smem_u32(slabA), slabB_u = smem_u32(slabB);
    int sa = 0, sb = 0;
    uint32_t pa = 0, pb = 0;
    if (stat) {   // resident weights: wait once for all (k-block, tap) tiles
      for (int i = 0; i < nkb * p.ntaps; ++i) mbar_wait(&b_full[i], 0);
      tc_fence_after();
    }
    for (int t = 0; t < my_tiles; ++t) {
      const int buf = t & 1;
      mbar_wait(&acc_empty[buf], ((t >> 1) & 1) ^ 1);       // epilogue has drained this accumulator
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * p.N);
      uint32_t accum = 0;
      if (SG > 1) {
        // grouped ring stages: one wait and one commit per stage; inside a stage the loop is warp-uniform with predicated MMAs
        const uint32_t leader = elect_one() ? 1u : 0u;
        const uint32_t b_step = b_stride >> 4;
        if (p.ntaps == 1) {
          for (int kbg = 0; kbg < nkb; kbg += SG) {
            const int cnt = nkb - kbg < SG ? nkb - kbg : SG;
            mbar_wait(&b_full[sb], pb);
            tc_fence_after();
            uint32_t b_lo = d_lo0 + ((slabB_u + (uint32_t)sb * b_slot) >> 4);
            for (int kk = 0; kk < cnt; ++kk) {
              const int kleft = p.Cin - (kbg + kk) * KBLK;
              const int ksteps = kleft >= KBLK ? KBLK / 16 : (kleft + 15) / 16;
              mbar_wait(&a_full[sa], pa);
              tc_fence_after();
              if (t == 0 && kbg == 0 && kk == 0 && lane == 0) trace_mark(3);
              const uint32_t a_lo = d_lo0 + ((slabA_u + (uint32_t)sa * a_stride) >> 4);
              for (int ks = 0; ks < ksteps; ++ks) {
                tc_mma_f16_pred(d_tmem, a_lo + 2u * ks, d_hi0, b_lo + 2u * ks, d_hi0, idesc, accum, leader);
                accum = 1;
              }
              tc_commit_pred(&a_empty[sa], leader);
              if (++sa == NA) { sa = 0; pa ^= 1; }
              b_lo += b_step;
            }
            tc_commit_pred(&b_empty[sb], leader);
            if (++sb == NB) { sb = 0; pb ^= 1; }
          }
        } else {
          const uint32_t a_step = (uint32_t)(p.dil * 128) >> 4;
          const uint32_t a_wrap = (p.tap_w > 0 && KH == 1) ? (uint32_t)((p.dil2 - (p.tap_w - 1) * p.dil) * 128) >> 4 : a_step;
          const int tw = (p.tap_w > 0 && KH == 1) ? p.tap_w : 0x7fffffff;
          for (int kb = 0; kb < nkb; ++kb) {
            const int kleft = p.Cin - kb * KBLK;
            const int ksteps = kleft >= KBLK ? KBLK / 16 : (kleft + 15) / 16;
            for (int kh = 0; kh < KH; ++kh) {
              mbar_wait(&a_full[sa], pa);
              tc_fence_after();
              if (t == 0 && kb == 0 && kh == 0 && lane == 0) trace_mark(3);
              uint32_t a_lo = d_lo0 + ((slabA_u + (uint32_t)sa * a_stride) >> 4);
              int tx = 0;
              for (int tg = 0; tg < TW; tg += SG) {
                const int cnt = TW - tg < SG ? TW - tg : SG;
                mbar_wait(&b_full[sb], pb);
                tc_fence_after();
                uint32_t b_lo = d_lo0 + ((slabB_u + (uint32_t)sb * b_slot) >> 4);
                for (int tl = 0; tl < cnt; ++tl) {
                  for (int ks = 0; ks < ksteps; ++ks) {
                    tc_mma_f16_pred(d_tmem, a_lo + 2u * ks, d_hi0, b_lo + 2u * ks, d_hi0, idesc, accum, leader);
                    accum = 1;
                  }
                  if (++tx == tw) { tx = 0; a_lo += a_wrap; } else { a_lo += a_step; }
                  b_lo += b_step;
                }
                tc_commit_pred(&b_empty[sb], leader);
                if (++sb == NB) { sb = 0; pb ^= 1; }
              }
              tc_commit_pred(&a_empty[sa], leader);
              if (++sa == NA) { sa = 0; pa ^= 1; }
            }
          }
        }
        tc_commit_pred(&acc_full[buf], leader);
        if (t == 0 && lane == 0) trace_mark(4);
        __syncwarp();
        continue;
      }
      for (int kb = 0; kb < nkb; ++kb)
       for (int kh = 0; kh < KH; ++kh) {
        const int kleft = p.Cin - kb * KBLK;
        const int ksteps = kleft >= KBLK ? KBLK / 16 : (kleft + 15) / 16;     // skip the zero-padded K of narrow stages
        const int tap0 = kh * TW;                                            // first tap served by this activation box
        if (slab) {
          mbar_wait(&a_full[sa], pa);
          tc_fence_after();
          if (t == 0 && kb == 0 && lane == 0) trace_mark(3);               // first activation slab has landed
        }
        if (slab && stat) {
          // fast path: nothing to wait for inside the k-block -> every tap is issued back to back.  The loop
          // is warp-uniform (descriptors stay in uniform registers); only the MMA itself is predicated.
          {
            const uint32_t leader = elect_one() ? 1u : 0u;
            uint32_t a_lo = d_lo0 + ((slabA_u + (uint32_t)sa * a_stride) >> 4);
            uint32_t b_lo = d_lo0 + ((slabB_u + (uint32_t)(kb * p.ntaps + tap0) * b_stride) >> 4);
            const uint32_t a_step = (uint32_t)(p.dil * 128) >> 4, b_step = b_stride >> 4;
            // 2-D kernels: after tap_w taps the offset jumps to the next kernel row (no division in the loop)
            const uint32_t a_wrap = (p.tap_w > 0 && KH == 1) ? (uint32_t)((p.dil2 - (p.tap_w - 1) * p.dil) * 128) >> 4 : a_step;
            const int tw = (p.tap_w > 0 && KH == 1) ? p.tap_w : 0x7fffffff;
            int tx = 0;
            for (int tap = 0; tap < TW; ++tap) {
              for (int ks = 0; ks < ksteps; ++ks) {
                tc_mma_f16_pred(d_tmem, a_lo + 2u * ks, d_hi0, b_lo + 2u * ks, d_hi0, idesc, accum, leader);
                accum = 1;
              }
              if (++tx == tw) { tx = 0; a_lo += a_wrap; } else { a_lo += a_step; }
              b_lo += b_step;
            }
            tc_commit_pred(&a_empty[sa], leader);
          }
          __syncwarp();
          accum = 1;
          if (++sa == NA) { sa = 0; pa ^= 1; }
          continue;
        }
        for (int tap = tap0; tap < tap0 + TW; ++tap) {
          uint32_t a_lo;
          if (slab) {
            const int roff = KH > 1 ? (tap - tap0) * p.dil : tap_row_off(p, tap);
            a_lo = d_lo0 + ((slabA_u + (uint32_t)sa * a_stride + (uint32_t)roff * 128u) >> 4);
          } else {
            mbar_wait(&a_full[sa], pa);
            tc_fence_after();
            a_lo = d_lo0 + ((slabA_u + (uint32_t)sa * a_stride) >> 4);
          }
          int wb_slot;
          if (stat) {
            wb_slot = kb * p.ntaps + tap;
          } else {
            wb_slot = sb;
            mbar_wait(&b_full[sb], pb);
            tc_fence_after();
          }
          const uint32_t b_lo = d_lo0 + ((slabB_u + (uint32_t)wb_slot * b_stride) >> 4);
          if (elect_one()) {
            for (int ks = 0; ks < ksteps; ++ks) {   // +32 B per K=16 step inside the 128-byte swizzled row
              tc_mma_f16(d_tmem, a_lo + 2u * ks, d_hi0, b_lo + 2u * ks, d_hi0, idesc, accum);
              accum = 1;
            }
            if (!stat) tc_commit(&b_empty[sb]);
            if (!slab) tc_commit(&a_empty[sa]);
          }
          __syncwarp();
          accum = 1;
          if (!stat) { if (++sb == NB) { sb = 0; pb ^= 1; } }
          if (!slab) { if (++sa == NA) { sa = 0; pa ^= 1; } }
        }
        if (slab) {
          if (elect_one()) tc_commit(&a_empty[sa]);
          __syncwarp();
          if (++sa == NA) { sa = 0; pa ^= 1; }
        }
      }
      if (elect_one()) tc_commit(&acc_full[buf]);
      if (t == 0 && lane == 0) trace_mark(4);                               // first tile: every MMA issued
      __syncwarp();
    }
  } else {
    // ============== epilogue: two groups of 4 warps, group e owns accumulator buffer e ===============
    // (tile t is drained by group t & 1, so consecutive tiles' epilogues overlap and each warp pays the
    //  per-tile fixed cost -- barrier wait, index math, bias -- only every other tile)
    pdl_wait();                                     // residual / mask / gather reads and every output write
    const int eg = (warp - 2) >> 2;                 // epilogue group = accumulator buffer
    const int qd = warp & 3;                        // TMEM lane quadrant this warp may access
    const size_t pitch_o = (size_t)p.Lp_out * 16;
    const long long Lout = (long long)p.Lj * p.out_stride;
    const bool simple = n_nt == 1 && p.G == 1;      // resblock convs: tile -> (batch, m-tile) with one division
    const uint32_t tbase = tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(eg * p.N);
    uint32_t ocnt = 0;                              // staged output boxes so far (tma_out)
    const bool lean = GENERIC && !p.reserved1 && lean_ok(p);   // reserved1: launcher's RVCB200_LEAN_EPI=0 (A/B switch)
    for (int t = eg; t < my_tiles; t += 2) {
      int mt, nt = 0, g = 0, b = 0;
      const unsigned tile = blockIdx.x + (unsigned)t * gridDim.x;
      if (simple) {
        if (p.batch == 1) mt = (int)tile;
        else { b = (int)(tile / (unsigned)n_mt); mt = (int)(tile - (unsigned)b * (unsigned)n_mt); }
      } else {
        decode((long long)tile, mt, nt, g, b);
      }
      const int row = mt * BM + qd * 32 + lane;
      const bool row_ok = row < p.Lj;
      const long long orow = (long long)row * p.out_stride + g;
      float4 pre[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) pre[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      bool have_pre = false;
      bool valid = true;
      float* sb = nullptr;
      if (GENERIC) {
        // everything the epilogue needs from global memory is fetched BEFORE the accumulator is waited for, i.e. under
        // the tile's TMA loads and MMAs: bias + conditioning -> shared memory (one copy per epilogue group), this row's
        // residual / running sum -> registers, the row's mask bit
        sb = reinterpret_cast<float*>(sE) + eg * 256;
        asm volatile("bar.sync %0, 128;" ::"r"(2 + eg) : "memory");        // the group's previous tile no longer reads sb
        const float* cond = p.cond ? p.cond + (size_t)b * p.cond_bstride : nullptr;
        for (int i = qd * 32 + lane; i < p.N; i += 128) sb[i] = __ldg(p.bias + nt * p.N + i) + (cond ? __ldg(cond + nt * p.N + i) : 0.f);
        valid = p.out_len ? (orow < p.out_len[b]) : true;
        if (p.pad_period > 0) valid = valid && (int)(orow % p.pad_period) < p.pad_valid;   // image pad pixels stay zero
        have_pre = p.f32_cl && !p.gate && p.N <= 64 && ((p.res32 != nullptr) != (p.accum != 0)) && row_ok;
        if (have_pre) {
          const float* src = p.res32 ? p.res32 + ((size_t)b * Lout + orow) * p.ldr32 : p.y32 + ((size_t)b * Lout + orow) * p.ldy32;
          src += nt * p.N;
#pragma unroll
          for (int k = 0; k < 16; ++k)
            if (k * 4 < p.N) pre[k] = *reinterpret_cast<const float4*>(src + k * 4);
        }
        asm volatile("bar.sync %0, 128;" ::"r"(2 + eg) : "memory");        // sb is complete
      }
      mbar_wait(&acc_full[eg], (t >> 1) & 1);
      tc_fence_after();
      if (t == 0 && warp == 2 && lane == 0) trace_mark(5);                  // first tile: accumulator complete
      if (GENERIC && lean) {
        epilogue_lean64(p, tbase, row_ok, valid, b, orow, nt * p.N, sb, pre, have_pre);
      } else if (GENERIC) {
#pragma unroll 1
        for (int c0 = 0; c0 < p.N; c0 += 16) {
          float4 pq[4];                                  // this pass's 16 prefetched words (static indices: registers)
          const int ci = c0 >> 4;
#pragma unroll
          for (int k = 0; k < 4; ++k) pq[k] = ci == 0 ? pre[k] : ci == 1 ? pre[4 + k] : ci == 2 ? pre[8 + k] : pre[12 + k];
          epilogue_generic16(p, tbase + (uint32_t)c0, row_ok, valid, b, orow, nt * p.N + c0, sb + c0, have_pre ? pq : nullptr);
        }
      } else {
        const size_t orow16 = (size_t)(orow + p.padf) * 16;
        unsigned char* y32 = p.y32 ? reinterpret_cast<unsigned char*>(p.y32) + (size_t)b * (p.Cout_total / (p.acc_f16 ? 8 : 4)) * pitch_o
                                    : nullptr;
        unsigned char* y16row = p.y16 ? reinterpret_cast<unsigned char*>(p.y16) + ((size_t)b * Lout + orow) * p.Cout_total * 2
                                      : nullptr;
        const unsigned char* r32 =
            p.res32 ? reinterpret_cast<const unsigned char*>(p.res32) + (size_t)b * (p.Cout_total / 4) * pitch_o : nullptr;
        const float* cond = p.cond ? p.cond + (size_t)b * p.cond_bstride : nullptr;
        const unsigned char* r16row =
            p.res16 ? reinterpret_cast<const unsigned char*>(p.res16) + ((size_t)b * Lout + orow) * p.Cout_total * 2 : nullptr;
        if (p.tma_out) {
          // the thread = row mapping makes a direct 16-bit store 32 L2 requests per instruction (phase-interleaved rows
          // on top): stage [32 rows][32 channels] boxes (SWIZZLE_64B) and let TMA write them; the tensor map views the
          // output as [B][Lj][G][C], so a box is one phase of 32 consecutive input rows
          unsigned char* my_stage = sE + (size_t)(warp - 2) * (2 * 2048);
          const uint32_t sw_x = ((uint32_t)lane >> 1) & 3u;
          for (int c0 = 0; c0 < p.N; c0 += 32) {
            unsigned char* box = my_stage + (ocnt & 1u) * 2048;
            if (lane == 0) bulk_wait_read<1>();
            __syncwarp();
            epilogue_chunk<32>(p, tbase + (uint32_t)c0, row_ok, nt * p.N + c0, pitch_o, orow16, y32, y16row, r32, cond, r16row,
                               box + lane * 64, sw_x);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_store_4d(&tmY, box, nt * p.N + c0, g, mt * BM + qd * 32, b);
              bulk_commit();
            }
            ++ocnt;
          }
        } else if (p.N % 32 == 0) {
          for (int c0 = 0; c0 < p.N; c0 += 32)
            epilogue_chunk<32>(p, tbase + (uint32_t)c0, row_ok, nt * p.N + c0, pitch_o, orow16, y32, y16row, r32, cond, r16row);
        } else {
          for (int c0 = 0; c0 < p.N; c0 += 16)
            epilogue_chunk<16>(p, tbase + (uint32_t)c0, row_ok, nt * p.N + c0, pitch_o, orow16, y32, y16row, r32, cond, r16row);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[eg]);
    }
    if (p.tma_out && lane == 0) bulk_wait_all();    // staged stores complete before the CTA's smem goes away
  }
  // ------------------------------------ teardown -------------------------------------------------
  if (warp == 2 && lane == 0) trace_mark(6);                                // first epilogue warp done
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

constexpr size_t kStageBytes = 8 * 2 * 2048 + 1024;   // tma_out staging (+ alignment slack)
constexpr size_t kGenericBiasBytes = 2 * 256 * 4 + 1024;   // generic epilogue: staged bias + conditioning per epilogue group

size_t tc_smem_bytes(const TcConvDesc& d) {
  const int halo = slab_rows_halo(d);
  const int R = d.a_mode != 1 ? ((BM + halo + 7) & ~7) : BM;
  const size_t a = (((size_t)R * 128) + 1023) & ~(size_t)1023;
  const size_t bb = (((size_t)d.N * 128) + 1023) & ~(size_t)1023;
  const size_t sg = (d.b_stationary || d.a_mode == 1 || d.b_group < 1) ? 1 : (size_t)d.b_group;
  return 1024 + d.na_stages * a + d.nb_stages * sg * bb + 8 * (2 * d.na_stages + 2 * d.nb_stages + 4) + 16 + 128 +
         (d.tma_out ? kStageBytes : 0) + (d.generic ? kGenericBiasBytes : 0);
}

// ---- driver entry point for tensor-map encoding (no link-time dependency on libcuda) --------------
using EncodeTiledFn = decltype(&cuTensorMapEncodeTiled);
EncodeTiledFn encode_tiled() {
  static const EncodeTiledFn fn = [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    const bool found = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
                       qres == cudaDriverEntryPointSuccess;
    return found ? reinterpret_cast<EncodeTiledFn>(ptr) : nullptr;
  }();
  return fn;
}

// ---- glue kernels between the fp32 channels-last world and the tensor-core layouts -------------------
__global__ void zero_pads_kernel(unsigned char* base, long long planes, int Lp, int padf, long long L) {
  // zero rows [0, padf) and [padf+L, Lp) of every 16-byte-vector plane
  const long long tail0 = padf + L;
  const int npad = padf + (int)(Lp - tail0);
  const long long total = planes * npad;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long pl = idx / npad;
    const int r = (int)(idx % npad);
    const long long row = r < padf ? r : tail0 + (r - padf);
    *reinterpret_cast<uint4*>(base + (pl * Lp + row) * 16) = make_uint4(0, 0, 0, 0);
  }
}

__global__ void cl32_to_cl16_kernel(const float* __restrict__ x, unsigned char* __restrict__ y16, long long n8, float slope,
                                    bool BF16) {
  // fp32 channels-last -> 16-bit channels-last (same shape), 8 elements per thread
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n8; idx += (long long)gridDim.x * blockDim.x) {
    const float4 a = *reinterpret_cast<const float4*>(x + idx * 8), c = *reinterpret_cast<const float4*>(x + idx * 8 + 4);
    uint4 o;
    o.x = pack2(BF16, lrelu(a.x, slope), lrelu(a.y, slope));
    o.y = pack2(BF16, lrelu(a.z, slope), lrelu(a.w, slope));
    o.z = pack2(BF16, lrelu(c.x, slope), lrelu(c.y, slope));
    o.w = pack2(BF16, lrelu(c.z, slope), lrelu(c.w, slope));
    *reinterpret_cast<uint4*>(y16 + idx * 16) = o;
  }
}

__device__ __forceinline__ void unpack8(const uint4& w, float* f) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&w.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
  const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&w.z)), d = __half22float2(*reinterpret_cast<const __half2*>(&w.w));
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

// x = x32 (planar-vector fp32, the transposed conv's output) + noise_conv(har);  x16 (channels-last 16 bit) =
// cvt(lrelu(x))   (models.py:552-553 + the lrelu of modules.py:297).  HBM-bound: 4 B read + 2 B write per element.
// A block owns tiles of TR time rows x all C channels: planar reads are coalesced along time (thread = row), the
// 16-bit rows are assembled in shared memory (16-byte pieces XOR-swizzled by row) and leave as one contiguous
// TR*C*2-byte copy -- a direct store from the thread = row mapping is 32 L2 requests of 8 bytes per warp instruction.
__global__ void __launch_bounds__(256)
noise_add_tile_kernel(const float* __restrict__ har, const float* __restrict__ wn, const float* __restrict__ nb,
                      unsigned char* __restrict__ x32, unsigned char* __restrict__ x16, int write32, long long L_har,
                      long long L, int C, int k, int s, int pad, int Lp, int padf, float slope, bool BF16, int TR) {
  extern __shared__ __align__(16) unsigned char nsm[];
  const int hs = s + 1;                                            // padded har row: (r, j) -> r*hs + j, conflict-free
  const int n_hrows = TR + (k + s - 1) / s;                        // rows of s samples the tile's taps touch
  float* sw = reinterpret_cast<float*>(nsm);                       // [k][C] + [C]
  float* sh = sw + (size_t)k * C + C;                              // [n_hrows][hs]
  unsigned char* tile = reinterpret_cast<unsigned char*>(sh + (((size_t)n_hrows * hs + 3) & ~(size_t)3));   // [TR][C] 16 bit
  if (threadIdx.x == 0) pdl_trigger();
  for (int i = threadIdx.x; i < k * C; i += blockDim.x) sw[i] = wn[i];
  for (int i = threadIdx.x; i < C; i += blockDim.x) sw[k * C + i] = nb ? nb[i] : 0.f;   // k = 0, nb = null: plain conversion
  pdl_wait();                                                      // x32 comes from the transposed conv just before
  const int b = blockIdx.y;
  const float* hb = har + (long long)b * L_har;
  const int n4 = C / 4, pieces = C / 8;
  const int pmask = pieces >= 8 ? 7 : pieces - 1;
  const long long n_tiles = (L + TR - 1) / TR;
  for (long long tl = blockIdx.x; tl < n_tiles; tl += gridDim.x) {
    const long long t0 = tl * TR;
    __syncthreads();                                               // previous tile fully copied out; weights visible
    const long long h0 = t0 * s - pad;
    if (k > 0)
      for (int i = threadIdx.x; i < n_hrows * s; i += blockDim.x) {
        const long long h = h0 + i;
        sh[(i / s) * hs + (i % s)] = (h >= 0 && h < L_har) ? __ldg(hb + h) : 0.f;
      }
    __syncthreads();
    // one item = 4 rows (TR/4 apart: each of the 4 planar loads is coalesced across the warp) x 4 channels: the 4 loads
    // are in flight together and every weight vector read from shared memory feeds 16 FMAs
    const int RQ = TR / 4;
    for (int idx = threadIdx.x; idx < RQ * n4; idx += blockDim.x) {
      const int rq = idx % RQ, g4 = idx / RQ;
      unsigned char* px0 = x32 + (((long long)b * n4 + g4) * Lp + padf + t0 + rq) * 16;
      float4 xv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        xv[j] = (t0 + rq + j * RQ < L) ? *reinterpret_cast<const float4*>(px0 + (long long)j * RQ * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 bq = *reinterpret_cast<const float4*>(sw + k * C + g4 * 4);
      float a[4][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { a[j][0] = bq.x; a[j][1] = bq.y; a[j][2] = bq.z; a[j][3] = bq.w; }
      const float* hp = sh + rq * hs;                              // tap kk -> har row r + kk / s, column kk % s
      const int hstep = RQ * hs;
      for (int kk = 0, j = 0; kk < k; ++kk) {
        const float4 wq = *reinterpret_cast<const float4*>(sw + kk * C + g4 * 4);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float hv = hp[q * hstep + j];
          a[q][0] = fmaf(hv, wq.x, a[q][0]); a[q][1] = fmaf(hv, wq.y, a[q][1]);
          a[q][2] = fmaf(hv, wq.z, a[q][2]); a[q][3] = fmaf(hv, wq.w, a[q][3]);
        }
        if (++j == s) { j = 0; hp += hs; }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int r = rq + q * RQ;
        if (t0 + r >= L) continue;
        xv[q].x += a[q][0]; xv[q].y += a[q][1]; xv[q].z += a[q][2]; xv[q].w += a[q][3];
        if (write32) *reinterpret_cast<float4*>(px0 + (long long)q * RQ * 16) = xv[q];
        uint2 o;
        o.x = pack2(BF16, lrelu(xv[q].x, slope), lrelu(xv[q].y, slope));
        o.y = pack2(BF16, lrelu(xv[q].z, slope), lrelu(xv[q].w, slope));
        const int piece = (g4 >> 1) ^ (r & pmask);
        *reinterpret_cast<uint2*>(tile + ((size_t)r * pieces + piece) * 16 + (g4 & 1) * 8) = o;
      }
    }
    __syncthreads();
    const long long rows_here = (L - t0) < TR ? (L - t0) : TR;
    uint4* dst = reinterpret_cast<uint4*>(x16 + (((long long)b * L + t0) * C) * 2);
    for (int i = threadIdx.x; i < (int)rows_here * pieces; i += blockDim.x) {
      const int r = i / pieces, pc = i - r * pieces;
      dst[i] = *reinterpret_cast<const uint4*>(tile + ((size_t)r * pieces + (pc ^ (r & pmask))) * 16);
    }
  }
}

// In-place source injection on the 16-bit stream (models.py:552-553 + the lrelu of modules.py:297):
//   x16[b][t][c] <- cvt( lrelu( x16[b][t][c] + nb[c] + sum_k har[b][t*s - pad + k] * wn[k][c] ) )
// x16 arrives as the transposed conv's RAW fp16 output (out_slope 1) and leaves as the stage's first stream tensor.
// Both sides are channels-last, so a thread owns one 16-byte piece (8 channels) of a row and every warp access is
// contiguous; 2 B read + 2 B written per element.  Tiles of TR rows per block; taps, bias and the harmonic-source
// segment of the tile sit in shared memory; one item = 4 rows (TR/4 apart) x 8 channels so that the 4 loads are in
// flight together and every weight vector feeds 32 FMAs.
// ROWS rows per item: 4 for the many-tap stages (every weight vector feeds 32 FMAs), 2 for the few-tap ones, which are
// bound by HBM and want the occupancy instead (121 registers per thread held the 8-tap stage at 16 warps per SM and
// 2.6 TB/s, ncu `gpurun_out/prof_noise.ncu-rep`).  Taps sit in shared memory as [k][2][C/8][4]: the two float4 halves of a
// lane's 8 channels in separate planes, so that a warp's LDS.128 is contiguous (the [k][C] order made every weight load a
// two-way bank conflict: 40 % of the kernel's shared-memory wavefronts).
template <int ROWS>
__global__ void __launch_bounds__(256, ROWS == 4 ? 2 : 4)
noise_add16_kernel(const float* __restrict__ har, const float* __restrict__ wn, const float* __restrict__ nb,
                   unsigned char* __restrict__ x16, long long L_har, long long L, int C, int k, int s, int pad, float slope,
                   int TR) {
  extern __shared__ __align__(16) unsigned char nsm[];
  const int hs = s + 1;
  const int n_hrows = TR + (k + s - 1) / s;
  float* sw = reinterpret_cast<float*>(nsm);                       // [k + 1][2][C/8][4]  (plane k = bias)
  float* sh = sw + (size_t)k * C + C;                              // [n_hrows][hs]
  if (threadIdx.x == 0) pdl_trigger();
  const int pieces = C / 8, RQ = TR / ROWS;
  for (int i = threadIdx.x; i < (k + 1) * (C / 4); i += blockDim.x) {   // one float4 = half of a piece
    const int kk = i / (C / 4), r = i % (C / 4), pc = r >> 1, hf = r & 1;
    const float4 w = __ldg(reinterpret_cast<const float4*>(kk < k ? wn + (size_t)kk * C : nb) + r);
    *reinterpret_cast<float4*>(sw + (size_t)kk * C + (size_t)hf * (C / 2) + pc * 4) = w;
  }
  pdl_wait();
  const int b = blockIdx.y;
  const float* hb = har + (long long)b * L_har;
  const long long n_tiles = (L + TR - 1) / TR;
  for (long long tl = blockIdx.x; tl < n_tiles; tl += gridDim.x) {
    const long long t0 = tl * TR;
    __syncthreads();
    const long long h0 = t0 * s - pad;
    for (int i = threadIdx.x; i < n_hrows * s; i += blockDim.x) {
      const long long h = h0 + i;
      sh[(i / s) * hs + (i % s)] = (h >= 0 && h < L_har) ? __ldg(hb + h) : 0.f;
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < RQ * pieces; idx += blockDim.x) {
      const int pc = idx % pieces, rq = idx / pieces;
      uint4* px0 = reinterpret_cast<uint4*>(x16 + (((long long)b * L + t0 + rq) * C + pc * 8) * 2);
      const long long rstep = (long long)RQ * pieces;              // uint4 elements between the item's rows
      uint4 xv[ROWS];
#pragma unroll
      for (int j = 0; j < ROWS; ++j) xv[j] = (t0 + rq + j * RQ < L) ? px0[j * rstep] : make_uint4(0, 0, 0, 0);
      float a[ROWS][8];
      const float* wp = sw + pc * 4;
      {
        const float4 b0 = *reinterpret_cast<const float4*>(wp + (size_t)k * C), b1 = *reinterpret_cast<const float4*>(wp + (size_t)k * C + C / 2);
#pragma unroll
        for (int j = 0; j < ROWS; ++j) {
          a[j][0] = b0.x; a[j][1] = b0.y; a[j][2] = b0.z; a[j][3] = b0.w; a[j][4] = b1.x; a[j][5] = b1.y; a[j][6] = b1.z; a[j][7] = b1.w;
        }
      }
      const float* hp = sh + rq * hs;
      const int hstep = RQ * hs;
      // taps in runs of one source row (s taps), the run unrolled by four
      for (int k0 = 0; k0 < k; k0 += s, hp += hs) {
        const int run = min(s, k - k0);
#pragma unroll 4
        for (int j = 0; j < run; ++j) {
          const float4 w0 = *reinterpret_cast<const float4*>(wp + (size_t)(k0 + j) * C),
                       w1 = *reinterpret_cast<const float4*>(wp + (size_t)(k0 + j) * C + C / 2);
#pragma unroll
          for (int q = 0; q < ROWS; ++q) {
            const float hv = hp[q * hstep + j];
            a[q][0] = fmaf(hv, w0.x, a[q][0]); a[q][1] = fmaf(hv, w0.y, a[q][1]); a[q][2] = fmaf(hv, w0.z, a[q][2]);
            a[q][3] = fmaf(hv, w0.w, a[q][3]); a[q][4] = fmaf(hv, w1.x, a[q][4]); a[q][5] = fmaf(hv, w1.y, a[q][5]);
            a[q][6] = fmaf(hv, w1.z, a[q][6]); a[q][7] = fmaf(hv, w1.w, a[q][7]);
          }
        }
      }
#pragma unroll
      for (int q = 0; q < ROWS; ++q) {
        if (t0 + rq + q * RQ >= L) continue;
        float f[8];
        unpack8(xv[q], f);
        uint4 o;
        o.x = pack2(false, lrelu(f[0] + a[q][0], slope), lrelu(f[1] + a[q][1], slope));
        o.y = pack2(false, lrelu(f[2] + a[q][2], slope), lrelu(f[3] + a[q][3], slope));
        o.z = pack2(false, lrelu(f[4] + a[q][4], slope), lrelu(f[5] + a[q][5], slope));
        o.w = pack2(false, lrelu(f[6] + a[q][6], slope), lrelu(f[7] + a[q][7], slope));
        px0[q * rstep] = o;
      }
    }
  }
}

__global__ void conv_post_pv_kernel(const unsigned char* __restrict__ x32, const float* __restrict__ w, float* __restrict__ out,
                                    long long L, int C, int k, int Lp, int padf, float slope) {
  // out[b][t] = tanh(sum_{kk,c} lrelu(x[c][t+kk-pad]) * w[kk][c]);  x is PV32 with zero pads
  extern __shared__ float swp[];  // [k][C]
  for (int i = threadIdx.x; i < k * C; i += blockDim.x) swp[i] = w[i];
  __syncthreads();
  const int b = blockIdx.y;
  const int pad = (k - 1) / 2;
  const int n4 = C / 4;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < L; t += (long long)gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int g4 = 0; g4 < n4; ++g4) {
      const unsigned char* pl = x32 + (((long long)b * n4 + g4) * Lp + padf + t - pad) * 16;
      for (int kk = 0; kk < k; ++kk) {
        const float4 v = *reinterpret_cast<const float4*>(pl + (long long)kk * 16);
        const float* wr = swp + kk * C + g4 * 4;
        acc = fmaf(lrelu(v.x, slope), wr[0], acc);
        acc = fmaf(lrelu(v.y, slope), wr[1], acc);
        acc = fmaf(lrelu(v.z, slope), wr[2], acc);
        acc = fmaf(lrelu(v.w, slope), wr[3], acc);
      }
    }
    out[(long long)b * L + t] = tanhf(acc);
  }
}


// out[b][t] = tanh(sum_{kk,c} lrelu(x[c][t+kk-pad]) * w[kk][c]);  x is planar-vector fp16 [B][C/8][Lp][8] with zero pads.
// Instruction-bound (convert + lrelu + FMA per loaded element), so a thread produces 4 consecutive samples from a
// sliding window of KT+3 rows: every 16-byte row piece is loaded, converted and rectified once for the (up to) 4
// outputs it feeds instead of once per output.
template <int KT>
__global__ void conv_post_pv16_kernel(const unsigned char* __restrict__ x16, const float* __restrict__ w, float* __restrict__ out,
                                      long long L, int C, int Lp, int padf, float slope) {
  extern __shared__ float swp[];  // [KT][C]
  if (threadIdx.x == 0) pdl_trigger();
  for (int i = threadIdx.x; i < KT * C; i += blockDim.x) swp[i] = w[i];
  __syncthreads();
  pdl_wait();
  const int b = blockIdx.y;
  constexpr int pad = (KT - 1) / 2;
  constexpr int NO = 4;
  const int n8 = C / 8;
  const long long nq = (L + NO - 1) / NO;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (long long)gridDim.x * blockDim.x) {
    const long long t0 = q * NO;
    float acc[NO] = {0.f, 0.f, 0.f, 0.f};
    for (int g8 = 0; g8 < n8; ++g8) {
      const unsigned char* pl = x16 + (((long long)b * n8 + g8) * Lp + padf + t0 - pad) * 16;
      const float* wg = swp + g8 * 8;
#pragma unroll
      for (int r = 0; r < KT + NO - 1; ++r) {
        float f[8];
        unpack8(*reinterpret_cast<const uint4*>(pl + (long long)r * 16), f);
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = lrelu(f[i], slope);
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          const int kk = r - o;
          if (kk >= 0 && kk < KT) {
            const float4 w0 = *reinterpret_cast<const float4*>(wg + kk * C), w1 = *reinterpret_cast<const float4*>(wg + kk * C + 4);
            acc[o] = fmaf(f[0], w0.x, acc[o]); acc[o] = fmaf(f[1], w0.y, acc[o]); acc[o] = fmaf(f[2], w0.z, acc[o]);
            acc[o] = fmaf(f[3], w0.w, acc[o]); acc[o] = fmaf(f[4], w1.x, acc[o]); acc[o] = fmaf(f[5], w1.y, acc[o]);
            acc[o] = fmaf(f[6], w1.z, acc[o]); acc[o] = fmaf(f[7], w1.w, acc[o]);
          }
        }
      }
    }
    if (t0 + NO <= L) {
      *reinterpret_cast<float4*>(out + (long long)b * L + t0) = make_float4(tanhf(acc[0]), tanhf(acc[1]), tanhf(acc[2]), tanhf(acc[3]));
    } else {
      for (int o = 0; o < NO && t0 + o < L; ++o) out[(long long)b * L + t0 + o] = tanhf(acc[o]);
    }
  }
}

__global__ void pv16_to_cl_kernel(const unsigned char* __restrict__ x16, float* __restrict__ y, long long L, int C, int Lp, int padf) {
  // debug/tap helper: planar-vector fp16 -> fp32 channels-last [B][L][C]
  const int b = blockIdx.y;
  const int n8 = C / 8;
  const long long total = L * n8;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int g8 = (int)(idx / L);
    const long long t = idx % L;
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(x16 + (((long long)b * n8 + g8) * Lp + padf + t) * 16), f);
    float* o = y + ((long long)b * L + t) * C + g8 * 8;
    *reinterpret_cast<float4*>(o) = make_float4(f[0], f[1], f[2], f[3]);
    *reinterpret_cast<float4*>(o + 4) = make_float4(f[4], f[5], f[6], f[7]);
  }
}

__global__ void pv32_to_cl_kernel(const unsigned char* __restrict__ x32, float* __restrict__ y, long long L, int C, int Lp, int padf) {
  // debug/tap helper: PV32 -> channels-last [B][L][C]
  const int b = blockIdx.y;
  const int n4 = C / 4;
  const long long total = L * n4;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int g4 = (int)(idx / L);
    const long long t = idx % L;
    const float4 v = *reinterpret_cast<const float4*>(x32 + (((long long)b * n4 + g4) * Lp + padf + t) * 16);
    *reinterpret_cast<float4*>(y + ((long long)b * L + t) * C + g4 * 4) = v;
  }
}

inline unsigned grid_for(long long total, int threads) {
  long long blocks = (total + threads - 1) / threads;
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

}  // namespace

bool tensor_map_encoder_available() { return encode_tiled() != nullptr; }

bool encode_tensor_map(CUtensorMap* tm, CUtensorMapDataType dt, int rank, const void* base, const cuuint64_t* dims,
                       const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle,
                       CUtensorMapL2promotion l2) {
  const EncodeTiledFn enc = encode_tiled();
  const cuuint32_t elem_strides[5] = {1, 1, 1, 1, 1};
  return enc && enc(tm, dt, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, elem_strides,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

cudaError_t conv_tc_set_trace(void* buf) {
  unsigned long long* p = reinterpret_cast<unsigned long long*>(buf);
  return cudaMemcpyToSymbol(g_trace, &p, sizeof(p));
}

cudaError_t launch_conv_tc(const TcConvDesc& d_in, int B, cudaStream_t st) {
  TcConvDesc d = d_in;
  if (d.N < 16 || d.N > 256 || d.N % 16 != 0 || d.Cin % 8 != 0 || d.Cout_total % d.N != 0 || d.G < 1 || d.G > 16 ||
      d.Lj <= 0 || d.L_in <= 0 || (d.a_mode != 1 && slab_rows_halo(d) > 127) || tap_halo(d) < 0 || d.tap_w < 0 ||
      d.a_mode < 0 || d.a_mode > 2 || (d.a_mode == 2 && d.tap_w <= 0) || d.a_nt_stride < 0 || (d.a_nt_stride > 0 && (!d.generic || d.G != 1)) ||
      (d.tap_w > 0 && (d.ntaps % d.tap_w != 0 || d.dil2 < (d.tap_w - 1) * d.dil)) || d.pad_period < 0 || (d.pad_period > 0 && !d.generic) || (d.accum && !d.y32) || B <= 0 || !d.x16 || !d.w16 ||
      d.a_fp16 || (d.res16 && d.res32) || (d.acc_f16 && (d.generic || d.Cout_total % 8)) || !tc_div_exact(d.div))
    return cudaErrorInvalidValue;
  if (!tensor_map_encoder_available()) return cudaErrorNotSupported;
  {
    static const int lean_on = [] { const char* e = getenv("RVCB200_LEAN_EPI"); return e ? atoi(e) : 1; }();
    d.reserved1 = lean_on ? 0 : 1;
  }
  d.batch = B;
  int cols = 32;
  while (cols < 2 * d.N) cols <<= 1;          // two accumulator buffers
  d.tmem_cols = cols;
  const int nkb = (d.Cin + KBLK - 1) / KBLK;
  const int halo = slab_rows_halo(d);
  const int n_nt = d.Cout_total / d.N;
  const long long tiles = (long long)((d.Lj + BM - 1) / BM) * n_nt * d.G * B;
  {
    // smem policy: weights stationary (loaded once per persistent CTA) when every (k-block, tap) tile
    // fits beside >= 3 activation boxes; otherwise a weight ring.
    const int R = d.a_mode != 1 ? ((BM + halo + 7) & ~7) : BM;
    const size_t a = (((size_t)R * 128) + 1023) & ~(size_t)1023;
    const size_t bb = (((size_t)d.N * 128) + 1023) & ~(size_t)1023;
    // lean epilogue with a 16-bit output in whole 32-column chunks: staged + TMA-stored (see the kernel)
    d.tma_out = (!d.generic && d.y16 && d.N % 32 == 0) ? 1 : 0;
    size_t budget = 208 * 1024 - (d.tma_out ? kStageBytes : 0) - (d.generic ? kGenericBiasBytes : 0);
    // Launches of at most two waves (the text encoder / flow contractions, M = T rows) can be given a small ring so that
    // the CTAs of the NEXT launch fit on the SM beside them and run their prologue under this launch's tail
    // (programmatic dependent launch, RVCB200_PDL=1): RVCB200_SMALL_SMEM_KB=<KB> (0 = off)
    static const int small_kb = [] { const char* e = getenv("RVCB200_SMALL_SMEM_KB"); return e ? atoi(e) : 0; }();
    if (small_kb > 0 && tiles <= 2 * 148 && budget > (size_t)small_kb * 1024) budget = (size_t)small_kb * 1024;
    const int nw = nkb * d.ntaps;
    const int na_max = d.a_mode != 1 ? 6 : 10;
    d.b_stationary = 0;
    // Phase groups (transposed conv, G > 1): with the phase fastest in the tile order and a grid that is a multiple of G,
    // every tile of a CTA has the same phase blockIdx.x % G, so that phase's weights can stay resident as well.  Without
    // it the 128 KB of weights of a 256 -> 128 stride-10 stage are re-streamed from L2 for every 128-row tile (ncu:
    // 196 us, tensor pipe 24 % busy, epilogue warps waiting for the accumulator 31 % of their samples).
    // (the 256 -> 128 stage needs 128 KB of weights + 3 slabs + 32 KB of output staging: it gets the last 10 KB of the SM)
    const size_t budget_s = d.G > 1 ? budget + 10 * 1024 : budget;
    if (n_nt == 1 && nw <= 48 && (size_t)nw * bb + 3 * a <= budget_s && tiles > 2 * 148 && d.G <= 148) {
      d.b_stationary = 1;
      d.nb_stages = nw;
      long long na = (long long)(budget_s - (size_t)nw * bb) / (long long)a;
      d.na_stages = (int)(na > na_max ? na_max : na);
    } else {
      // (ring depths: 5 slabs / 16 weight tiles instead of 3 / 10 changed nothing for the one-tile-per-CTA contractions,
      //  profiles/r2_ab_rings_injgemm.md)
      d.na_stages = d.a_mode == 0 ? (nkb >= 2 ? 3 : 2) : 4;
      // grouped ring stages (slab modes): SG weight tiles per stage, <= 48 KB, at least 3 stages beside the activation boxes.
      // 1-tap contractions group k-blocks (and need SG + 1 activation boxes in flight), the others group the taps of one box.
      static const int max_group = [] { const char* e = getenv("RVCB200_BGROUP"); return e ? atoi(e) : 8; }();
      d.b_group = 1;
      if (d.a_mode != 1 && max_group > 1) {
        const int per_box = d.ntaps == 1 ? nkb : (d.a_mode == 2 ? d.tap_w : d.ntaps);     // tiles that can share a stage
        int sg = per_box < max_group ? per_box : max_group;
        while (sg > 1) {
          if (d.ntaps != 1 && per_box % sg != 0 && per_box > sg) { --sg; continue; }       // even groups (9 taps -> 3, 5 -> 5)
          const int na = d.ntaps == 1 ? sg + 2 : d.na_stages;
          const size_t ring = budget > (size_t)na * a ? budget - (size_t)na * a : 0;
          if ((size_t)sg * bb <= 48 * 1024 && ring / ((size_t)sg * bb) >= 3 && na <= 8) {
            d.b_group = sg;
            d.na_stages = na;
            break;
          }
          --sg;
        }
      }
      long long nb = (long long)(budget - (size_t)d.na_stages * a) / (long long)((size_t)d.b_group * bb);
      d.nb_stages = (int)(nb > 10 ? 10 : (nb < 2 ? 2 : nb));
    }
  }
  const size_t smem = tc_smem_bytes(d);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;

  // tensor maps: activations (C, L_in, B) box (64, R, 1); weights (64, rows) box (64, N); SWIZZLE_128B
  CUtensorMap tmA, tmW, tmY;
  const CUtensorMapDataType dt = d.in_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  {
    const int R = d.a_mode != 1 ? ((BM + halo + 7) & ~7) : BM;
    // (grouped: the channel axis spans every N tile's input channels)
    cuuint64_t dims[3] = {(cuuint64_t)(d.a_nt_stride > 0 ? (long long)d.a_nt_stride * (n_nt - 1) + d.Cin : (long long)d.Cin),
                          (cuuint64_t)d.L_in, (cuuint64_t)B};
    const cuuint64_t ldx = (cuuint64_t)(d.generic && d.ldx16 ? d.ldx16 : d.Cin);
    cuuint64_t strides[2] = {ldx * 2, ldx * 2 * (cuuint64_t)d.L_in};
    cuuint32_t box[3] = {(cuuint32_t)KBLK, (cuuint32_t)R, 1};
    if (!encode_tensor_map(&tmA, dt, 3, d.x16, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return cudaErrorInvalidValue;
    const cuuint64_t wrows = (cuuint64_t)d.G * n_nt * d.ntaps * nkb * d.N;
    cuuint64_t wdims[2] = {(cuuint64_t)KBLK, wrows};
    cuuint64_t wstrides[1] = {(cuuint64_t)KBLK * 2};
    cuuint32_t wbox[2] = {(cuuint32_t)KBLK, (cuuint32_t)d.N};
    if (!encode_tensor_map(&tmW, dt, 2, d.w16, wdims, wstrides, wbox, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return cudaErrorInvalidValue;
  }
  tmY = tmA;
  if (d.tma_out) {   // output viewed as [B][Lj][G][Cout_total] 16-bit; box = 32 channels x 1 phase x 32 rows
    cuuint64_t odims[4] = {(cuuint64_t)d.Cout_total, (cuuint64_t)d.out_stride, (cuuint64_t)d.Lj, (cuuint64_t)B};
    cuuint64_t ostr[3] = {(cuuint64_t)d.Cout_total * 2, (cuuint64_t)d.Cout_total * 2 * d.out_stride,
                          (cuuint64_t)d.Cout_total * 2 * d.out_stride * (cuuint64_t)d.Lj};
    cuuint32_t obox[4] = {32, 1, 32, 1};
    if (!encode_tensor_map(&tmY, d.out_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, d.y16, odims,
                           ostr, obox, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B))
      return cudaErrorInvalidValue;
  }
  static SmemOptIn opt_s, opt_g;
  const int num_sms = current_num_sms();
  if (cudaError_t e = opt_in_smem(conv_tc_kernel<false>, smem, opt_s)) return e;
  if (cudaError_t e = opt_in_smem(conv_tc_kernel<true>, smem, opt_g)) return e;
  unsigned grid = (unsigned)(tiles < num_sms ? tiles : num_sms);            // persistent: one CTA per SM
  if (d.b_stationary && d.G > 1) grid = (unsigned)((num_sms / d.G) * d.G);  // every tile of a CTA has phase blockIdx.x % G
  cudaError_t le = d.generic ? launch_pdl(conv_tc_kernel<true>, dim3(grid), dim3(kThreadsTC), smem, st, d, tmA, tmW, tmY)
                             : launch_pdl(conv_tc_kernel<false>, dim3(grid), dim3(kThreadsTC), smem, st, d, tmA, tmW, tmY);
  launch_counter().n++;
  return le != cudaSuccess ? le : cudaGetLastError();
}

cudaError_t launch_zero_pads(void* base, long long planes, int Lp, int padf, long long L, cudaStream_t st) {
  const long long total = planes * (Lp - L);
  zero_pads_kernel<<<grid_for(total, 256), 256, 0, st>>>(reinterpret_cast<unsigned char*>(base), planes, Lp, padf, L);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_cl32_to_cl16(const float* x, void* y16, long long numel, float slope, bool bf16, cudaStream_t st) {
  if (numel % 8) return cudaErrorInvalidValue;
  cl32_to_cl16_kernel<<<grid_for(numel / 8, 256), 256, 0, st>>>(x, reinterpret_cast<unsigned char*>(y16), numel / 8, slope, bf16);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_noise_add_pv(const float* har, const float* wn, const float* nb, void* x32, void* x16, bool write32, int B,
                                long long L_har, long long L, int C, int k, int s, int pad, int Lp, int padf, float slope,
                                bool bf16, cudaStream_t st) {
  if (C % 8 != 0 || C / 8 > 64 || ((C / 8) & (C / 8 - 1)) != 0 || s < 1 || k < 0 ||
      (k > 0 && (!har || !wn || !nb)))
    return cudaErrorInvalidValue;
  // tile rows: as many as fit beside the taps in ~100 KB (two blocks per SM), at most 128
  int TR = 128;
  auto smem_for = [&](int tr) {
    const size_t nh = (size_t)(tr + (k + s - 1) / s) * (s + 1);
    return sizeof(float) * ((size_t)k * C + C + ((nh + 3) & ~(size_t)3)) + (size_t)tr * C * 2;
  };
  while (TR > 8 && smem_for(TR) > 100 * 1024) TR >>= 1;
  const size_t smem = smem_for(TR);
  static SmemOptIn opt;
  if (cudaError_t e = opt_in_smem(noise_add_tile_kernel, smem, opt)) return e;
  const long long n_tiles = (L + TR - 1) / TR;
  const long long per = smem > 56 * 1024 ? 2 : 4;                  // resident blocks per SM
  dim3 grid((unsigned)(n_tiles < 148 * per ? n_tiles : 148 * per), B);
  cudaError_t le = launch_pdl(noise_add_tile_kernel, grid, dim3(256), smem, st, har, wn, nb, reinterpret_cast<unsigned char*>(x32),
                              reinterpret_cast<unsigned char*>(x16), write32 ? 1 : 0, L_har, L, C, k, s, pad, Lp, padf, slope, bf16,
                              TR);
  launch_counter().n++;
  return le != cudaSuccess ? le : cudaGetLastError();
}

cudaError_t launch_noise_add16(const float* har, const float* wn, const float* nb, void* x16, int B, long long L_har,
                               long long L, int C, int k, int s, int pad, float slope, cudaStream_t st) {
  if (C % 8 != 0 || s < 1 || k < 1 || !har || !wn || !nb || !x16) return cudaErrorInvalidValue;
  // tile rows: ~32 KB of stream per tile (two block-wide barriers per tile), shrunk until taps + source segment fit
  int TR = 512;
  while (TR > 32 && (long long)TR * C > 16384) TR >>= 1;      // (8 K - 64 K elements per tile measured: no difference)
  auto smem_for = [&](int tr) { return sizeof(float) * ((size_t)k * C + C + (size_t)(tr + (k + s - 1) / s) * (s + 1)); };
  while (TR > 8 && smem_for(TR) > 100 * 1024) TR >>= 1;
  const size_t smem = smem_for(TR);
  const bool many = k >= 16;                   // 4 rows per item (FMA-bound stages) or 2 (HBM-bound ones, higher occupancy)
  static SmemOptIn opt4, opt2;
  if (cudaError_t e = many ? opt_in_smem(noise_add16_kernel<4>, smem, opt4) : opt_in_smem(noise_add16_kernel<2>, smem, opt2)) return e;
  const long long n_tiles = (L + TR - 1) / TR;
  const long long per = smem > 56 * 1024 ? 2 : (smem > 24 * 1024 ? 4 : 8);
  dim3 grid((unsigned)(n_tiles < 148 * per ? n_tiles : 148 * per), B);
  unsigned char* xp = reinterpret_cast<unsigned char*>(x16);
  cudaError_t le = many ? launch_pdl(noise_add16_kernel<4>, grid, dim3(256), smem, st, har, wn, nb, xp, L_har, L, C, k, s, pad, slope, TR)
                        : launch_pdl(noise_add16_kernel<2>, grid, dim3(256), smem, st, har, wn, nb, xp, L_har, L, C, k, s, pad, slope, TR);
  launch_counter().n++;
  return le != cudaSuccess ? le : cudaGetLastError();
}

cudaError_t launch_conv_post_pv(const void* x32, const float* w, float* out, int B, long long L, int C, int k, int Lp,
                                int padf, float slope, cudaStream_t st) {
  dim3 grid(grid_for(L, 256), B);
  conv_post_pv_kernel<<<grid, 256, sizeof(float) * k * C, st>>>(reinterpret_cast<const unsigned char*>(x32), w, out, L, C, k, Lp,
                                                                padf, slope);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_conv_post_pv16(const void* x16, const float* w, float* out, int B, long long L, int C, int k, int Lp,
                                  int padf, float slope, cudaStream_t st) {
  if (k != 7 || C % 8 || L % 4) return cudaErrorInvalidValue;     // L = T * upp, upp a multiple of 4 in every configuration
  dim3 grid(grid_for((L + 3) / 4, 256), B);
  cudaError_t le = launch_pdl(conv_post_pv16_kernel<7>, grid, dim3(256), sizeof(float) * k * C, st,
                              reinterpret_cast<const unsigned char*>(x16), w, out, L, C, Lp, padf, slope);
  launch_counter().n++;
  return le != cudaSuccess ? le : cudaGetLastError();
}

cudaError_t launch_pv16_to_cl(const void* src, float* y, int B, long long L, int C, int Lp, int padf, cudaStream_t st) {
  dim3 grid(grid_for(L * (C / 8), 256), B);
  pv16_to_cl_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const unsigned char*>(src), y, L, C, Lp, padf);
  launch_counter().n++;
  return cudaGetLastError();
}

cudaError_t launch_pv32_to_cl(const void* src, float* y, int B, long long L, int C, int Lp, int padf, cudaStream_t st) {
  dim3 grid(grid_for(L * (C / 4), 256), B);
  pv32_to_cl_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const unsigned char*>(src), y, L, C, Lp, padf);
  launch_counter().n++;
  return cudaGetLastError();
}

}  // namespace rvc
