// Compile-time specialised tcgen05 convolution for the decoder's ResBlock convs (C_in = C_out = C, zero "same"
// padding, kernel NTAPS, dilation DIL) -- the 72 launches that are >70 % of a synthesis step.
//
// Why a second kernel next to conv_tc.cu: the ncu source view of the generic kernel on the narrow stages
// (profiles/r1_ncu_conv_tc_v5.md) shows the tensor pipe 3-10 % busy, DRAM 23-50 % busy and the single MMA-issuing
// warp executing ~256 SASS instructions per 128-row tile for 6 MMAs (runtime loop bounds, ring arithmetic, R2UR
// traffic): the kernel is bound by per-tile instruction overhead of the issuing warp.  Here
//   * every loop bound, descriptor offset and smem address is a compile-time constant (C, NTAPS, DIL, MSUB),
//   * one "tile" is MSUB x 128 time rows: one activation slab (MSUB*128 + halo rows per 64-channel k-block, loaded
//     by <= 3 TMA boxes) feeds MSUB accumulators, so barrier round trips, ring updates and -- when the weights do
//     not fit in shared memory (C = 128, k = 7/11; C = 256) -- the weight stream are amortised over MSUB x more work,
//   * the epilogue moves its 16-bit residual and output as TMA boxes (the residual one 32-column chunk ahead of the
//     TMEM reads), at every C,
//   * the bias lives in shared memory.
// Layouts, epilogue semantics and the weight packing are those of conv_tc.cu (see its header).
#include "tc_ptx.cuh"

namespace rvc {
namespace {

using namespace tc;

constexpr int kRbThreads = 64 + 32 * 8;   // TMA producer warp, MMA warp, 8 epilogue warps (2 groups of 4)
constexpr int kEpiBox = 2048;             // one epilogue staging box: 32 rows x 32 channels x 16 bit, SWIZZLE_64B
constexpr int kInjFloats = 5 * 64;        // source-injection taps [<= 4][<= 64] + bias [<= 64]

// Shared-memory plan of one instantiation (plain constexpr functions so that MSUB can be chosen by "does it fit").
struct RbPlan {
  int nkb, ks, tile_m, halo, r, nbox, rb, a_bytes, w_bytes, nw, out_slots, epi_bytes, budget, stat, nb, na_fit;
};
constexpr RbPlan rb_plan(int C, int NTAPS, int DIL, int MSUB) {
  RbPlan q{};
  q.nkb = (C + 63) / 64;
  q.ks = C >= 64 ? 4 : C / 16;
  q.tile_m = MSUB * 128;
  q.halo = (NTAPS - 1) * DIL;
  q.r = q.tile_m + q.halo;
  q.nbox = (q.r + 255) / 256;
  q.rb = (((q.r + q.nbox - 1) / q.nbox) + 7) & ~7;
  q.a_bytes = q.nbox * q.rb * 128;
  q.w_bytes = C * 128;
  q.nw = q.nkb * NTAPS;
  // epilogue staging: per warp 2 residual boxes + out_slots output boxes
  q.out_slots = C >= 128 ? 1 : 2;
  q.epi_bytes = 8 * (2 + q.out_slots) * kEpiBox;
  q.budget = 218 * 1024 - q.epi_bytes;
  q.stat = (q.nw * q.w_bytes <= 96 * 1024 && (q.budget - q.nw * q.w_bytes) / q.a_bytes >= 2) ? 1 : 0;
  q.nb = q.stat ? q.nw : (C >= 256 ? 3 : (C == 128 ? 4 : 6));
  q.na_fit = (q.budget - q.nb * q.w_bytes) / q.a_bytes;
  return q;
}
constexpr bool rb_fits(int C, int NTAPS, int DIL, int MSUB) {
  return rb_plan(C, NTAPS, DIL, MSUB).na_fit >= 2 && 2 * MSUB * C <= 512;
}
// largest MSUB <= the preferred one whose rings fit beside the epilogue staging
constexpr int rb_msub(int C, int NTAPS, int DIL) {
  int m = C == 32 ? 4 : (C == 256 ? 1 : 2);
  while (m > 1 && !rb_fits(C, NTAPS, DIL, m)) m >>= 1;
  return m;
}

template <int C, int NTAPS, int DIL, int MSUB>
struct RbCfg {
  static constexpr RbPlan P = rb_plan(C, NTAPS, DIL, MSUB);
  static constexpr int NKB = P.nkb;                        // 64-channel k-blocks (one 128-byte swizzled row each)
  static constexpr int KS = P.ks;                          // K=16 MMA steps per k-block (zero-padded K is skipped)
  static constexpr int TILE_M = P.tile_m;
  static constexpr int HALO = P.halo;
  static constexpr int GOFF = -((NTAPS - 1) / 2) * DIL;    // "same" padding
  static constexpr int NBOX = P.nbox;                      // TMA boxes are <= 256 rows
  static constexpr int RB = P.rb;
  static constexpr uint32_t A_BYTES = (uint32_t)P.a_bytes;
  static constexpr uint32_t W_BYTES = (uint32_t)P.w_bytes; // one (k-block, tap) weight tile [C][64] 16-bit
  static constexpr int NW = P.nw;
  static constexpr bool STAT = P.stat != 0;                // weights resident for the whole CTA
  static constexpr int NB = P.nb;
  static constexpr int NA = P.na_fit > 6 ? 6 : P.na_fit;
  static constexpr int OUT_SLOTS = P.out_slots;
  static constexpr int EPI_WARP_BYTES = (2 + OUT_SLOTS) * kEpiBox;
  static constexpr int EPI_BYTES = P.epi_bytes;
  static constexpr int TMEM_COLS = 2 * MSUB * C;           // two accumulator buffers of MSUB sub-tiles
  static constexpr int NCH = MSUB * (C / 32);              // 32-column epilogue chunks per tile and warp
  static constexpr int NBAR = 2 * NA + 2 * NB + 4 + 16;    // + 8 warps x 2 residual-box barriers
  static constexpr size_t SMEM = 1024 + (size_t)NA * A_BYTES + (size_t)NB * W_BYTES + EPI_BYTES + (C + kInjFloats) * sizeof(float) +
                                 8 * NBAR + 64;
  static_assert(C % 32 == 0 && C <= 256, "C");
  static_assert(NA >= 2, "activation ring too small");
  static_assert(TMEM_COLS <= 512 && (TMEM_COLS & (TMEM_COLS - 1)) == 0 && TMEM_COLS >= 32, "TMEM columns");
  static_assert(SMEM <= 227 * 1024, "shared memory");
  static_assert(RB <= 256 && A_BYTES % 1024 == 0 && W_BYTES % 1024 == 0, "box");
};

template <int C, int NTAPS, int DIL, int MSUB>
__global__ void __launch_bounds__(kRbThreads, 1)
rbconv_tc_kernel(const TcConvDesc p, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                 const __grid_constant__ CUtensorMap tmR, const __grid_constant__ CUtensorMap tmY) {
  using K = RbCfg<C, NTAPS, DIL, MSUB>;
  extern __shared__ unsigned char smem_raw[];
  // aligned with pointer arithmetic on the __shared__ array (not through an integer cast): the compiler keeps the
  // shared address space and emits LDS/STS instead of generic LD/ST for every access derived from it
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* sA = smem;                                       // [NA][SLAB_ROWS][128 B] swizzled
  unsigned char* sW = sA + (size_t)K::NA * K::A_BYTES;            // [NB][C][128 B] swizzled
  unsigned char* sE = sW + (size_t)K::NB * K::W_BYTES;            // [8 warps][2 residual + OUT_SLOTS output boxes][2 KB]
  float* sbias = reinterpret_cast<float*>(sE + K::EPI_BYTES);
  float* sinj = sbias + C;                                        // [inj_k][inj_cn] taps, then [inj_cn] bias
  uint64_t* bars = reinterpret_cast<uint64_t*>(sinj + kInjFloats);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + K::NA;
  uint64_t* b_full = a_empty + K::NA;
  uint64_t* b_empty = b_full + K::NB;
  uint64_t* acc_full = b_empty + K::NB;     // [2]
  uint64_t* acc_empty = acc_full + 2;       // [2]
  uint64_t* res_full = acc_empty + 2;       // [8 warps][2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 16);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const unsigned n_mt = (unsigned)((p.Lj + K::TILE_M - 1) / K::TILE_M);
  const unsigned total_tiles = n_mt * (unsigned)p.batch;

  if (threadIdx.x == 0) {
    pdl_trigger();     // the next kernel's CTAs may take over SMs as ours retire (they block in pdl_wait until we are done)
    for (int i = 0; i < K::NA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < K::NB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
    for (int i = 0; i < 16; ++i) mbar_init(&res_full[i], 1);
    fence_mbarrier_init();
    fence_proxy_async();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW);
  }
  if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)K::TMEM_COLS);
  for (int i = threadIdx.x; i < C; i += kRbThreads) sbias[i] = p.bias[i];
  if (p.inj_har) {
    const int nw = p.inj_k * p.inj_cn;
    for (int i = threadIdx.x; i < nw + p.inj_cn; i += kRbThreads) sinj[i] = i < nw ? p.inj_w[i] : p.inj_b[i - nw];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =========================== producer: TMA global -> swizzled smem ============================
    if (lane == 0) {
      if (K::STAT) {
#pragma unroll 1
        for (int i = 0; i < K::NW; ++i) {            // slot i = kb * NTAPS + tap; packed row = (tap * NKB + kb) * C
          const int kb = i / NTAPS, tap = i - kb * NTAPS;
          mbar_expect_tx(&b_full[i], K::W_BYTES);
          tma_load_2d(sW + (size_t)i * K::W_BYTES, &tmW, 0, (tap * K::NKB + kb) * C, &b_full[i]);
        }
      }
      pdl_wait();                                    // activations come from the previous kernel (weights do not)
      int sa = 0, sb = 0;
      uint32_t pa = 1, pb = 1;                       // producer waits on "empty" with inverted parity
#pragma unroll 1
      for (unsigned tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const unsigned b = tile / n_mt, mt = tile - b * n_mt;
        const int row0 = (int)mt * K::TILE_M + K::GOFF;
#pragma unroll 1
        for (int kb = 0; kb < K::NKB; ++kb) {
          mbar_wait(&a_empty[sa], pa);
          mbar_expect_tx(&a_full[sa], K::A_BYTES);
#pragma unroll
          for (int j = 0; j < K::NBOX; ++j)
            tma_load_3d(sA + (size_t)sa * K::A_BYTES + (size_t)j * K::RB * 128, &tmA, kb * 64, row0 + j * K::RB, (int)b,
                        &a_full[sa]);
          if (++sa == K::NA) { sa = 0; pa ^= 1; }
          if (!K::STAT) {
#pragma unroll 1
            for (int tap = 0; tap < NTAPS; ++tap) {
              mbar_wait(&b_empty[sb], pb);
              mbar_expect_tx(&b_full[sb], K::W_BYTES);
              tma_load_2d(sW + (size_t)sb * K::W_BYTES, &tmW, 0, (tap * K::NKB + kb) * C, &b_full[sb]);
              if (++sb == K::NB) { sb = 0; pb ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ============ MMA issuer: warp-uniform control flow, fully unrolled per k-block, one elected lane issues ========
    // (everything the MMAs consume is warp-uniform -- kernel parameters, loop counters and values broadcast with
    //  __shfl_sync(.., 0) -- so descriptors live in uniform registers: SASS is UMOV/UIADD3 + UTCHMMA per MMA)
    {
      const uint32_t leader = elect_one() ? 1u : 0u;
      const uint32_t fmt = p.in_bf16 ? 1u : 0u;
      // instruction descriptor: D=F32 @4, A/B format @7/@10, K-major both, N>>3 @17, M>>4 @24
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(C >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      const uint64_t dproto = make_desc_sw128(0, 0);
      const uint32_t d_hi = (uint32_t)(dproto >> 32), d_lo0 = (uint32_t)dproto;
      const uint32_t sA_d = __shfl_sync(0xffffffffu, d_lo0 + (smem_u32(sA) >> 4), 0);
      const uint32_t sW_d = __shfl_sync(0xffffffffu, d_lo0 + (smem_u32(sW) >> 4), 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      if (K::STAT) {
#pragma unroll 1
        for (int i = 0; i < K::NW; ++i) mbar_wait(&b_full[i], 0);
        tc_fence_after();
      }
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      uint32_t it = 0;
#pragma unroll 1
      for (unsigned tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const uint32_t buf = it & 1u;
        mbar_wait(&acc_empty[buf], ((it >> 1) & 1u) ^ 1u);       // the epilogue has drained this accumulator buffer
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + buf * (uint32_t)(MSUB * C);
#pragma unroll
        for (int kb = 0; kb < K::NKB; ++kb) {
          mbar_wait(&a_full[sa], pa);
          tc_fence_after();
          const uint32_t a_d = sA_d + (uint32_t)sa * (K::A_BYTES >> 4);
#pragma unroll
          for (int tap = 0; tap < NTAPS; ++tap) {
            uint32_t b_d;
            if (K::STAT) {
              b_d = sW_d + (uint32_t)(kb * NTAPS + tap) * (K::W_BYTES >> 4);
            } else {
              mbar_wait(&b_full[sb], pb);
              tc_fence_after();
              b_d = sW_d + (uint32_t)sb * (K::W_BYTES >> 4);
            }
#pragma unroll
            for (int ms = 0; ms < MSUB; ++ms) {
#pragma unroll
              for (int ks = 0; ks < K::KS; ++ks) {
                // activation rows of sub-tile ms shifted by tap*DIL: +128 B per row inside the swizzled slab
                // (base_offset stays 0, see conv_tc.cu); +32 B per K=16 step inside the 128-byte row
                tc_mma_f16_pred(d_tmem + (uint32_t)(ms * C), a_d + (uint32_t)(((ms * 128 + tap * DIL) * 128 + ks * 32) >> 4),
                                d_hi, b_d + (uint32_t)((ks * 32) >> 4), d_hi, idesc, (kb | tap | ks) != 0 ? 1u : 0u, leader);
              }
            }
            if (!K::STAT) {
              tc_commit_pred(&b_empty[sb], leader);
              if (++sb == K::NB) { sb = 0; pb ^= 1; }
            }
          }
          tc_commit_pred(&a_empty[sa], leader);
          if (++sa == K::NA) { sa = 0; pa ^= 1; }
        }
        tc_commit_pred(&acc_full[buf], leader);
        __syncwarp();
      }
    }
  } else {
    // ============== epilogue: two groups of 4 warps, group e drains accumulator buffer e ==================
    // 16-bit I/O: thread = TMEM lane = time row, so direct global accesses would be 16-byte pieces 2*C bytes apart --
    // 32 L2 requests per warp instruction; measured ~0.37 requests/clk/SM whatever the byte count, the limit of every
    // epilogue-heavy shape (profiles/r1_conv_shapes_v8_*.jsonl).  Instead each warp moves [32 rows][32 channels]
    // boxes with TMA: the residual box lands in a SWIZZLE_64B staging slot (2 slots, loaded one chunk ahead), the
    // 16-bit output box is written to a staging slot by the lanes (conflict-free under the swizzle) and stored by one
    // lane.  The fp16 planar branch sum keeps the direct path: its warp accesses are 512 B contiguous.
    // The chunk loop is unrolled by two only (slot indices stay compile-time): the fully unrolled version was 240 KB of
    // SASS and 39 % of all warp stalls were instruction fetches (ncu source view, profiles/r1_ncu_rbconv_v8.md).
    pdl_wait();                                     // residual / branch sum reads and every output write
    const int eg = (warp - 2) >> 2;
    const int ew = warp - 2;
    const int qd = warp & 3;                        // TMEM lane quadrant this warp may access
    const size_t pitch_o = (size_t)p.Lp_out * 16;   // bytes per planar-vector plane
    const bool obf = p.out_bf16 != 0;
    const float slope = p.out_slope;
    const float div = p.div, rdiv = 1.f / p.div;    // branch mean: exact quotient without a divide (div_exact)
    const float neg_scale = p.res_neg_scale == 0.f ? 1.f : p.res_neg_scale;
    const bool has_r16 = p.res16 != nullptr;
    const bool has_y16 = p.y16 != nullptr;
    const bool has_acc = p.y32 != nullptr;          // planar-vector fp16 branch sum [C/8][Lp][8]
    const bool do_acc = has_acc && p.accum != 0;
    const bool st_acc = has_acc && p.acc_nostore == 0;
    float* const tanh_out = p.tanh_out;             // conv_post mode: column 0 -> tanh -> fp32 [B][Lj], nothing else
    unsigned char* my_stage = sE + (size_t)ew * K::EPI_WARP_BYTES;      // [2 residual][OUT_SLOTS output] boxes
    uint64_t* my_res_full = res_full + ew * 2;
    // byte offset of this lane's 16-byte piece j inside a SWIZZLE_64B box: row = lane (64 B), piece ^= (row >> 1) & 3
    const uint32_t sw_row = (uint32_t)lane * 64u, sw_x = ((uint32_t)lane >> 1) & 3u;
    uint32_t rpar = 0;                              // phase parity of the two residual slots (both flip once per pair)
    uint32_t ocnt = 0;                              // output boxes stored so far
    uint32_t it = (uint32_t)eg;
    constexpr int CPS = C / 32;                     // chunks per 128-row sub-tile (power of two)
#pragma unroll 1
    for (unsigned tile = blockIdx.x + (unsigned)eg * gridDim.x; tile < total_tiles; tile += 2 * gridDim.x, it += 2) {
      const unsigned b = tile / n_mt, mt = tile - b * n_mt;
      const int wrow0 = (int)mt * K::TILE_M + qd * 32;            // first row of this warp's 32-row group (sub-tile 0)
      const int row_base = wrow0 + lane;
      const uint32_t tbase = tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(eg * MSUB * C);
      unsigned char* acc = has_acc ? reinterpret_cast<unsigned char*>(p.y32) + (size_t)b * (C / 8) * pitch_o : nullptr;

      uint4 rq[8];    // branch-sum prefetch, 2 slots x 4 words
      auto issue_box = [&](int ci, int slot) {       // one lane: residual box of chunk ci -> staging slot
        const int ms = ci / CPS, c0 = (ci - ms * CPS) * 32;
        uint64_t* bar = &my_res_full[slot];
        mbar_expect_tx(bar, kEpiBox);
        tma_load_3d(my_stage + slot * kEpiBox, &tmR, c0, wrow0 + ms * 128, (int)b, bar);
      };
      auto load_acc = [&](int ci, int slot) {
        const int ms = ci / CPS, c0 = (ci - ms * CPS) * 32;
        const int row = row_base + ms * 128;
        if (row < p.Lj) {
          const unsigned char* q = acc + (size_t)(c0 / 8) * pitch_o + (size_t)(row + p.padf) * 16;
#pragma unroll
          for (int k = 0; k < 4; ++k) rq[slot * 4 + k] = *reinterpret_cast<const uint4*>(q + (size_t)k * pitch_o);
        }
      };
      // the first residual / branch-sum words are in flight before the MMAs of this tile finish
      if (has_r16 && lane == 0) { issue_box(0, 0); issue_box(1, 1); }
      if (do_acc) load_acc(0, 0);
      mbar_wait(&acc_full[eg], (it >> 1) & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int cp = 0; cp < K::NCH; cp += 2) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int ci = cp + u;
          const int ms = ci / CPS, c0 = (ci - ms * CPS) * 32;
          const int row = row_base + ms * 128;
          const bool row_ok = row < p.Lj;
          if (do_acc && ci + 1 < K::NCH) load_acc(ci + 1, u ^ 1);
          uint32_t r[32];
          tmem_ld32_issue(tbase + (uint32_t)(ms * C + c0), r);
          float4 bq[8];                               // bias: its smem latency hides under the TMEM load
#pragma unroll
          for (int k4 = 0; k4 < 8; ++k4) bq[k4] = lds_f4(sbias + c0 + k4 * 4);
          tmem_ld_wait();
          if (tanh_out) {                             // (warp-uniform) the 128 B a warp stores are contiguous
            if (c0 == 0 && row_ok) tanh_out[(size_t)b * (size_t)p.Lj + row] = tanhf(__uint_as_float(r[0]) + bq[0].x);
            continue;
          }
          float v[32];
#pragma unroll
          for (int k4 = 0; k4 < 8; ++k4) {
            v[k4 * 4 + 0] = __uint_as_float(r[k4 * 4 + 0]) + bq[k4].x;
            v[k4 * 4 + 1] = __uint_as_float(r[k4 * 4 + 1]) + bq[k4].y;
            v[k4 * 4 + 2] = __uint_as_float(r[k4 * 4 + 2]) + bq[k4].z;
            v[k4 * 4 + 3] = __uint_as_float(r[k4 * 4 + 3]) + bq[k4].w;
          }
          if (p.inj_har) {
            // source injection of a dense stride-u transposed conv: columns [c0, c0 + 32) are channels cb.. of phase ph,
            // i.e. of output time row * u + ph
            const int cn = p.inj_cn, ph = c0 / cn, cb = c0 - ph * cn;
            const long long h0 = ((long long)row * (C / cn) + ph) * p.inj_s - p.inj_pad;
            const float* hb = p.inj_har + (size_t)b * (size_t)p.inj_Lhar;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              if (kk < p.inj_k) {
                const long long h = h0 + kk;
                const float hv = (row_ok && h >= 0 && h < p.inj_Lhar) ? __ldg(hb + h) : 0.f;
                const float* wk = sinj + kk * cn + cb;
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                  const float4 wq = *reinterpret_cast<const float4*>(wk + k4 * 4);
                  v[k4 * 4 + 0] = fmaf(hv, wq.x, v[k4 * 4 + 0]); v[k4 * 4 + 1] = fmaf(hv, wq.y, v[k4 * 4 + 1]);
                  v[k4 * 4 + 2] = fmaf(hv, wq.z, v[k4 * 4 + 2]); v[k4 * 4 + 3] = fmaf(hv, wq.w, v[k4 * 4 + 3]);
                }
              }
            }
            const float* bk = sinj + p.inj_k * cn + cb;
#pragma unroll
            for (int k4 = 0; k4 < 8; ++k4) {
              const float4 bq = *reinterpret_cast<const float4*>(bk + k4 * 4);
              v[k4 * 4 + 0] += bq.x; v[k4 * 4 + 1] += bq.y; v[k4 * 4 + 2] += bq.z; v[k4 * 4 + 3] += bq.w;
            }
          }
          if (has_r16) {
            // residual box of this chunk: wait, read this lane's row, hand the slot back, refill it two chunks ahead
            const unsigned char* box = my_stage + u * kEpiBox + sw_row;
            mbar_wait(&my_res_full[u], rpar);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              add_res8(v + k * 8, *reinterpret_cast<const uint4*>(box + ((((uint32_t)k) ^ sw_x) << 4)), neg_scale);
            __syncwarp();
            if (lane == 0 && ci + 2 < K::NCH) issue_box(ci + 2, u);
          }
          if (has_acc) {
            if (do_acc) {
#pragma unroll
              for (int k = 0; k < 4; ++k) add_res8(v + k * 8, rq[u * 4 + k], 1.f);
            }
            if (div != 1.f) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = div_exact(v[i], div, rdiv);
            }
            if (row_ok && st_acc) {
              unsigned char* q = acc + (size_t)(c0 / 8) * pitch_o + (size_t)(row + p.padf) * 16;
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                uint4 o;
                o.x = pack2(false, v[k * 8 + 0], v[k * 8 + 1]); o.y = pack2(false, v[k * 8 + 2], v[k * 8 + 3]);
                o.z = pack2(false, v[k * 8 + 4], v[k * 8 + 5]); o.w = pack2(false, v[k * 8 + 6], v[k * 8 + 7]);
                *reinterpret_cast<uint4*>(q + (size_t)k * pitch_o) = o;
              }
            }
          } else if (div != 1.f) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = div_exact(v[i], div, rdiv);
          }
          if (has_y16) {
            uint4 o[4];
#pragma unroll
            for (int k8 = 0; k8 < 4; ++k8) {
              o[k8].x = pack2(obf, lrelu_max(v[k8 * 8 + 0], slope), lrelu_max(v[k8 * 8 + 1], slope));
              o[k8].y = pack2(obf, lrelu_max(v[k8 * 8 + 2], slope), lrelu_max(v[k8 * 8 + 3], slope));
              o[k8].z = pack2(obf, lrelu_max(v[k8 * 8 + 4], slope), lrelu_max(v[k8 * 8 + 5], slope));
              o[k8].w = pack2(obf, lrelu_max(v[k8 * 8 + 6], slope), lrelu_max(v[k8 * 8 + 7], slope));
            }
            // stage the [32 rows][32 channels] box, then one lane stores it (rows >= L are clipped by the tensor map)
            unsigned char* box = my_stage + (2 + (ocnt % K::OUT_SLOTS)) * kEpiBox;
            if (lane == 0) bulk_wait_read<K::OUT_SLOTS - 1>();      // the store that last used this slot has read it
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 4; ++k) *reinterpret_cast<uint4*>(box + sw_row + ((((uint32_t)k) ^ sw_x) << 4)) = o[k];
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_store_3d(&tmY, box, c0, wrow0 + ms * 128, (int)b);
              bulk_commit();
            }
            ++ocnt;
          }
        }
        if (has_r16) rpar ^= 1u;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[eg]);
    }
    if (lane == 0) bulk_wait_all();     // staged stores complete before the CTA's smem goes away
  }
  // ------------------------------------ teardown -------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)K::TMEM_COLS);
}

template <int C, int NTAPS, int DIL, int MSUB>
cudaError_t launch_one(const TcConvDesc& d, int B, cudaStream_t st) {
  using K = RbCfg<C, NTAPS, DIL, MSUB>;
  if (!tensor_map_encoder_available()) return cudaErrorNotSupported;
  CUtensorMap tmA, tmW, tmR, tmY;
  const CUtensorMapDataType dt = d.in_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  {
    cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)d.L_in, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * (cuuint64_t)d.L_in};
    cuuint32_t box[3] = {64, (cuuint32_t)K::RB, 1};
    if (!encode_tensor_map(&tmA, dt, 3, d.x16, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return cudaErrorInvalidValue;
    cuuint64_t wdims[2] = {64, (cuuint64_t)NTAPS * K::NKB * C};
    cuuint64_t wstrides[1] = {128};
    cuuint32_t wbox[2] = {64, (cuuint32_t)C};
    if (!encode_tensor_map(&tmW, dt, 2, d.w16, wdims, wstrides, wbox, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return cudaErrorInvalidValue;
    // epilogue boxes: [32 rows][32 channels] of the 16-bit channels-last residual / output, SWIZZLE_64B staging
    tmR = tmA;
    tmY = tmA;
    cuuint64_t odims[3] = {(cuuint64_t)C, (cuuint64_t)d.Lj, (cuuint64_t)B};
    cuuint64_t ostrides[2] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * (cuuint64_t)d.Lj};
    cuuint32_t obox[3] = {32, 32, 1};
    if (d.res16 && !encode_tensor_map(&tmR, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, d.res16, odims, ostrides, obox,
                                      CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B))
      return cudaErrorInvalidValue;
    if (d.y16 && !encode_tensor_map(&tmY, d.out_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                                    d.y16, odims, ostrides, obox, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B))
      return cudaErrorInvalidValue;
  }
  static SmemOptIn opt;
  if (cudaError_t e = opt_in_smem(rbconv_tc_kernel<C, NTAPS, DIL, MSUB>, K::SMEM, opt)) return e;
  const int num_sms = current_num_sms();
  TcConvDesc p = d;
  p.batch = B;
  const long long tiles = (long long)((d.Lj + K::TILE_M - 1) / K::TILE_M) * B;
  const unsigned grid = (unsigned)(tiles < num_sms ? tiles : num_sms);      // persistent: one CTA per SM
  cudaError_t le = launch_pdl(rbconv_tc_kernel<C, NTAPS, DIL, MSUB>, dim3(grid), dim3(kRbThreads), K::SMEM, st, p, tmA, tmW, tmR, tmY);
  launch_counter().n++;
  return le != cudaSuccess ? le : cudaGetLastError();
}

template <int C>
cudaError_t launch_c(const TcConvDesc& d, int B, cudaStream_t st) {
  switch (d.ntaps * 16 + d.dil) {
    case 3 * 16 + 1: return launch_one<C, 3, 1, rb_msub(C, 3, 1)>(d, B, st);
    case 3 * 16 + 3: return launch_one<C, 3, 3, rb_msub(C, 3, 3)>(d, B, st);
    case 3 * 16 + 5: return launch_one<C, 3, 5, rb_msub(C, 3, 5)>(d, B, st);
    case 7 * 16 + 1: return launch_one<C, 7, 1, rb_msub(C, 7, 1)>(d, B, st);
    case 7 * 16 + 3: return launch_one<C, 7, 3, rb_msub(C, 7, 3)>(d, B, st);
    case 7 * 16 + 5: return launch_one<C, 7, 5, rb_msub(C, 7, 5)>(d, B, st);
    case 11 * 16 + 1: return launch_one<C, 11, 1, rb_msub(C, 11, 1)>(d, B, st);
    case 11 * 16 + 3: return launch_one<C, 11, 3, rb_msub(C, 11, 3)>(d, B, st);
    case 11 * 16 + 5: return launch_one<C, 11, 5, rb_msub(C, 11, 5)>(d, B, st);
    default: return cudaErrorNotSupported;
  }
}

}  // namespace

bool rbconv_tc_supported(const TcConvDesc& d) {
  if (d.generic || d.G != 1 || d.out_stride != 1 || d.cond != nullptr || d.a_mode != 0) return false;
  if (d.Cin != d.Cout_total || d.N != d.Cin || d.L_in != d.Lj) return false;
  if (!(d.Cin == 32 || d.Cin == 64 || d.Cin == 128 || d.Cin == 256)) return false;
  if (!(d.ntaps == 3 || d.ntaps == 7 || d.ntaps == 11) || !(d.dil == 1 || d.dil == 3 || d.dil == 5)) return false;
  if (d.g_off[0] != -((d.ntaps - 1) / 2) * d.dil) return false;
  if ((d.accum && !d.y32) || !d.x16 || !d.w16 || !d.bias || d.a_fp16) return false;
  if (d.res32 || (d.y32 && !d.acc_f16)) return false;      // fp32 planar residual / output: generic kernel only
  if (d.tanh_out && (d.y16 || d.y32 || d.res16 || d.Cin > 128)) return false;       // conv_post mode: the only output
  if (d.acc_nostore && !(d.y32 && d.accum && d.y16)) return false;
  if (!tc_div_exact(d.div)) return false;
  if (d.inj_har && (!d.inj_w || !d.inj_b || d.inj_k < 1 || d.inj_k > 4 || !(d.inj_cn == 32 || d.inj_cn == 64) ||
                    d.Cin % d.inj_cn != 0 || !d.y16 || d.y32 || d.res16 || d.tanh_out || d.inj_s < 1))
    return false;
  // the epilogue computes lrelu as max(v, v * slope) and the residual expansion as min(r, r * scale)
  if (!(d.out_slope > 0.f && d.out_slope <= 1.f) || !(d.res_neg_scale == 0.f || d.res_neg_scale >= 1.f)) return false;
  return true;
}

// Resblock convolution on the specialised kernel; cudaErrorNotSupported when the shape is not covered
// (the caller falls back to launch_conv_tc).
cudaError_t launch_rbconv_tc(const TcConvDesc& d, int B, cudaStream_t st) {
  if (!rbconv_tc_supported(d) || B <= 0) return cudaErrorNotSupported;
  switch (d.Cin) {
    case 32: return launch_c<32>(d, B, st);
    case 64: return launch_c<64>(d, B, st);
    case 128: return launch_c<128>(d, B, st);
    case 256: return launch_c<256>(d, B, st);
    default: return cudaErrorNotSupported;
  }
}

}  // namespace rvc
