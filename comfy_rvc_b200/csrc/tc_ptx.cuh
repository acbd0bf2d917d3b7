// PTX wrappers (mbarrier, TMA, tcgen05) of every tcgen05 kernel -- conv_tc.cu (generic persistent implicit-GEMM conv),
// rbconv_tc.cu (compile-time specialised resblock conv), rbpair_tc.cu (fused resblock pair), attention_tc.cu (windowed
// attention) -- and the epilogue helpers of the three convolution kernels.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "conv_tc.cuh"

namespace rvc {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(done) : "r"(addr), "r"(parity) : "memory");
  } while (!done);
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ bool elect_one() {   // one lane of a converged warp (elect.sync)
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// descriptors are passed as (lo, hi) 32-bit halves: only the low word (start address) changes per MMA
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                           uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc) : "memory");
}
// Same, executed by every lane of a converged warp but issued only where `leader` is set: the operands
// are computed in warp-uniform control flow so they can live in uniform registers.
__device__ __forceinline__ void tc_mma_f16_pred(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                uint32_t idesc, uint32_t acc, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "setp.ne.b32 q, %7, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc), "r"(leader) : "memory");
}
__device__ __forceinline__ void tc_commit_pred(uint64_t* bar, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(leader) : "memory");
}
// A operand in tensor memory (lane = row, 32-bit column c = elements 2c | 2c+1 of the row's K range), B through a descriptor
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                              uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t"
      "}" ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc) : "memory");
}

// ---- tensor memory: allocation (one warp), loads and stores of this thread's lane ----
// writes the base address to *slot and gives up the right to allocate more, so that the next CTA on the SM may
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols));
}
// r[0..32) / r[0..16) = columns [taddr, +32) / [taddr, +16); the registers are valid only after tmem_ld_wait(), so that
// other loads can be issued in between
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
      "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
      "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// K-major SWIZZLE_128B shared-memory descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
// start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major, 1) | SBO>>4 [32,46) = 1024 B |
// version 1 [46,48) | base_offset [49,52) | layout_type SWIZZLE_128B = 2 [61,64)
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr, uint32_t base_offset) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
         ((uint64_t)(base_offset & 7u) << 49) | (2ull << 61);
}

// Shared-memory loads the compiler may not move: issued between a tcgen05.ld and its wait so that the smem latency (bias,
// residual rows) hides under the TMEM latency instead of stalling the first use after the wait
__device__ __forceinline__ float4 lds_f4(const float* p) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(p)));
  return v;
}
__device__ __forceinline__ uint4 lds_u4(const void* p) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(p)));
  return v;
}

// 16-byte read-only global load that does not allocate in L1 (streamed residuals)
__device__ __forceinline__ uint4 ld_nc_u4(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

// leaky ReLU for 0 < slope <= 1 as multiply + max (2 instructions instead of compare + multiply + select; the same value
// bit for bit, signed zeros included)
__device__ __forceinline__ float lrelu_max(float v, float slope) { return fmaxf(v, v * slope); }

// v[0..8) += x where the 8 fp16 values of `w` hold r = lrelu(x): x = r > 0 ? r : r * neg_scale, computed as
// min(r, r * neg_scale) -- neg_scale >= 1 (1: plain add; 10: the decoder's lrelu_{0.1}-domain stream)
__device__ __forceinline__ void add_res8(float* v, const uint4& w, float neg_scale) {
  const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&w.x));
  const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
  const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&w.z));
  const float2 f3 = __half22float2(*reinterpret_cast<const __half2*>(&w.w));
  const float r[8] = {f0.x, f0.y, f1.x, f1.y, f2.x, f2.y, f3.x, f3.y};
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] += fminf(r[i], r[i] * neg_scale);
}

// v / d rounded to nearest, bit for bit as the IEEE divide, for d in {2, 3, 4} (tc_div_exact) and r = 1.f / d:
// the remainder e = v - q0 * d is exact under the FMA, so one correction step gives the rounded quotient (checked over all
// 2^32 inputs per divisor by tests/test_exact_div.py).  q0 is kept where e is zero -- the sign of -0 (fmaf(+0, r, -0) is
// +0) -- or NaN -- v = +-inf (inf - inf) and v = NaN.  A plain divide is a div.rn.f32: an FCHK slow-path test plus a
// branch per value.
__device__ __forceinline__ float div_exact(float v, float d, float r) {
  const float q0 = __fmul_rn(v, r);
  const float e = __fmaf_rn(-q0, d, v);
  return fabsf(e) > 0.f ? __fmaf_rn(e, r, q0) : q0;
}

// ---- bulk-tensor (TMA) stores from shared memory ----
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* tm, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack2(bool bf16, float a, float b) {
  if (bf16) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}

// One epilogue pass over CH accumulator columns of this thread's row: TMEM -> regs, + bias/cond/residual,
// accumulate, /div, fp32 PV store, lrelu + 16-bit channels-last store.  Loads are issued before use.
template <int CH>
__device__ __forceinline__ void epilogue_chunk(const TcConvDesc& p, uint32_t taddr, bool row_ok, int co, size_t pitch_o,
                                               size_t orow16, unsigned char* y32, unsigned char* y16row,
                                               const unsigned char* r32, const float* cond,
                                               const unsigned char* r16row = nullptr, unsigned char* stage_row = nullptr,
                                               uint32_t sw_x = 0) {
  uint32_t r[CH];
  if constexpr (CH == 32) tmem_ld32_issue(taddr, r);
  else tmem_ld16_issue(taddr, r);
  float4 rr[CH / 4], aa[CH / 4];
  uint4 rh[CH / 8];
  if (row_ok) {
    if (r16row) {
#pragma unroll
      for (int k8 = 0; k8 < CH / 8; ++k8) rh[k8] = *reinterpret_cast<const uint4*>(r16row + (size_t)(co + k8 * 8) * 2);
    }
    if (r32) {
#pragma unroll
      for (int k4 = 0; k4 < CH / 4; ++k4)
        rr[k4] = *reinterpret_cast<const float4*>(r32 + (size_t)(co / 4 + k4) * pitch_o + orow16);
    }
    if (p.accum) {
      if (p.acc_f16) {   // planar-vector fp16: 8 channels per 16-byte row
#pragma unroll
        for (int k8 = 0; k8 < CH / 8; ++k8) {
          const uint4 w = *reinterpret_cast<const uint4*>(y32 + (size_t)(co / 8 + k8) * pitch_o + orow16);
          const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&w.x));
          const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
          const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&w.z));
          const float2 f3 = __half22float2(*reinterpret_cast<const __half2*>(&w.w));
          aa[2 * k8] = make_float4(f0.x, f0.y, f1.x, f1.y);
          aa[2 * k8 + 1] = make_float4(f2.x, f2.y, f3.x, f3.y);
        }
      } else {
#pragma unroll
        for (int k4 = 0; k4 < CH / 4; ++k4)
          aa[k4] = *reinterpret_cast<const float4*>(y32 + (size_t)(co / 4 + k4) * pitch_o + orow16);
      }
    }
  }
  tmem_ld_wait();
  if (!row_ok) return;
  float v[CH];
#pragma unroll
  for (int i = 0; i < CH; ++i) v[i] = __uint_as_float(r[i]) + __ldg(p.bias + co + i);
  if (cond) {
#pragma unroll
    for (int i = 0; i < CH; ++i) v[i] += __ldg(cond + co + i);
  }
  if (r32) {
#pragma unroll
    for (int k4 = 0; k4 < CH / 4; ++k4) {
      v[k4 * 4 + 0] += rr[k4].x; v[k4 * 4 + 1] += rr[k4].y; v[k4 * 4 + 2] += rr[k4].z; v[k4 * 4 + 3] += rr[k4].w;
    }
  }
  if (r16row) {
    const float ns = p.res_neg_scale == 0.f ? 1.f : p.res_neg_scale;
#pragma unroll
    for (int k8 = 0; k8 < CH / 8; ++k8) add_res8(v + k8 * 8, rh[k8], ns);
  }
  if (p.accum) {
#pragma unroll
    for (int k4 = 0; k4 < CH / 4; ++k4) {
      v[k4 * 4 + 0] += aa[k4].x; v[k4 * 4 + 1] += aa[k4].y; v[k4 * 4 + 2] += aa[k4].z; v[k4 * 4 + 3] += aa[k4].w;
    }
  }
  if (p.div != 1.f) {
    const float rd = 1.f / p.div;
#pragma unroll
    for (int i = 0; i < CH; ++i) v[i] = div_exact(v[i], p.div, rd);
  }
  if (y32 && p.acc_f16) {
#pragma unroll
    for (int k8 = 0; k8 < CH / 8; ++k8) {
      uint4 o;
      o.x = pack2(false, v[k8 * 8 + 0], v[k8 * 8 + 1]); o.y = pack2(false, v[k8 * 8 + 2], v[k8 * 8 + 3]);
      o.z = pack2(false, v[k8 * 8 + 4], v[k8 * 8 + 5]); o.w = pack2(false, v[k8 * 8 + 6], v[k8 * 8 + 7]);
      *reinterpret_cast<uint4*>(y32 + (size_t)(co / 8 + k8) * pitch_o + orow16) = o;
    }
  } else if (y32) {
#pragma unroll
    for (int k4 = 0; k4 < CH / 4; ++k4)
      *reinterpret_cast<float4*>(y32 + (size_t)(co / 4 + k4) * pitch_o + orow16) =
          make_float4(v[k4 * 4 + 0], v[k4 * 4 + 1], v[k4 * 4 + 2], v[k4 * 4 + 3]);
  }
  if (y16row) {
    const bool obf = p.out_bf16 != 0;
#pragma unroll
    for (int k8 = 0; k8 < CH / 8; ++k8) {
      uint4 o;
      o.x = pack2(obf, lrelu(v[k8 * 8 + 0], p.out_slope), lrelu(v[k8 * 8 + 1], p.out_slope));
      o.y = pack2(obf, lrelu(v[k8 * 8 + 2], p.out_slope), lrelu(v[k8 * 8 + 3], p.out_slope));
      o.z = pack2(obf, lrelu(v[k8 * 8 + 4], p.out_slope), lrelu(v[k8 * 8 + 5], p.out_slope));
      o.w = pack2(obf, lrelu(v[k8 * 8 + 6], p.out_slope), lrelu(v[k8 * 8 + 7], p.out_slope));
      if (stage_row)   // this lane's row of a SWIZZLE_64B staging box (the caller stores the box with TMA)
        *reinterpret_cast<uint4*>(stage_row + ((((uint32_t)k8) ^ sw_x) << 4)) = o;
      else
        *reinterpret_cast<uint4*>(y16row + (size_t)(co + k8 * 8) * 2) = o;
    }
  }
}

}  // namespace tc
}  // namespace rvc
