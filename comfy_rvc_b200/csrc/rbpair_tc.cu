// Fused ResBlock1 pair on tcgen05:  x' = x + conv2(lrelu(conv1(lrelu(x))))   (modules.py:295-308, one (c1, c2) pair)
// in ONE kernel, with h = lrelu(conv1(.)) living only in shared memory.
//
// Why: on the narrow decoder stages (C = 64 / 32, L = 1.44 M / 2.88 M rows per 60 s segment) the two launches of a
// pair are bound by the bytes they move through HBM -- conv1 reads the stream and writes h (4 B/element), conv2 reads
// h and the residual and writes the stream (6 B/element); profiles/r1_conv_shapes_v10.jsonl: 4.7-5.9 TB/s on every
// k = 3 shape.  Fused, a pair reads the stream once and writes it once: 4 B/element instead of 10 (6 instead of 12
// for the branch-closing pair, which also carries the planar fp16 branch sum).
//
// Tiling: one tile = TILE_M = MSUB x 128 rows of h.  conv1 reads an activation slab of TILE_M + (k-1) DIL rows (one
// TMA slab, tap = descriptor row offset, as in rbconv_tc.cu) and accumulates MSUB sub-tiles in TMEM; the first
// epilogue group adds the bias, applies lrelu, rounds to the operand format of conv2 and writes h straight into a
// SWIZZLE_128B K-major shared-memory tile (the layout TMA would have produced), zeroing rows outside [0, L) -- the
// zero padding conv2 sees.  conv2 (dilation 1) reads that tile with tap = row offset; its last k-1 output rows would
// need h rows of the next tile, so a tile yields OUT_ROWS = TILE_M - (k-1) valid output rows and tiles advance by
// OUT_ROWS (0.8-4.7 % of the MMA work is recomputed instead of exchanging halos between CTAs).  The second epilogue
// group takes the residual from the activation slab that is still in shared memory (x = r > 0 ? r : 10 r, the
// lrelu-domain stream of DESIGN.md §3), so the residual costs no second global read.
//
// Pipeline per CTA (persistent, 1 CTA/SM): TMA producer warp (NA-slot slab ring), one MMA warp issuing conv1 LA tiles
// ahead of conv2 (conv1(i+LA) before conv2(i)) so the tensor pipe works while epilogue 1 turns accumulator i into h,
// LA+1 conv1 accumulators and 2 conv2 accumulators in TMEM, NH h tiles, 4 + 4 epilogue warps.  A slab slot is released
// only when epilogue 2 has read the residual from it, i.e. a whole conv1 -> h -> conv2 -> epilogue chain after it was
// loaded: with the 3 slots of the first version the HBM latency of the next slab load sat on the critical path
// (profiles/r1_pair_shapes_v1.jsonl: 2.6 TB/s, 490 TFLOP/s on C = 64, k = 3), hence small tiles and deep rings.
// Arithmetic is that of two rbconv_tc launches (same MMA order, same rounding points): the op-level test compares
// the outputs bit for bit.
#include "tc_ptx.cuh"

#include <cstdlib>

namespace rvc {
namespace {

using namespace tc;

// threads: TMA producer warp, MMA warp, E1G x 4 h-epilogue warps, E2G x 4 output-epilogue warps
constexpr int pair_threads(int e1g, int e2g) { return 64 + 32 * (4 * e1g + 4 * e2g); }
constexpr int kPairBox = 2048;              // one output staging box: 32 rows x 32 channels x 16 bit, SWIZZLE_64B
constexpr int kPairSmemMax = 227 * 1024;

// Pipeline shape of one instantiation: rows per tile, h tiles, conv1 look-ahead, output staging slots per warp.
struct PairSel { int msub, nh, la, out_slots, e2g, e1g; };
constexpr PairSel pair_sel(int C, int NTAPS, int variant) {
  if (C == 64) {
    // k = 3: bound by the h-epilogue (profiles/r1_ncu_v16_final.md) -> variant 1 tries a second h-epilogue group
    if (NTAPS == 3) return variant == 0 ? PairSel{1, 2, 2, 1, 2, 1} : PairSel{1, 2, 2, 1, 2, 2};
    // k = 7: 112 KB of weights, bound by MMA issue (profiles/r1_pair_shapes_v4_*.jsonl): one output-epilogue group, the
    // shared memory of the second group's staging goes to a fourth slab instead
    return variant == 0 ? PairSel{1, 1, 1, 1, 1, 1} : PairSel{1, 1, 1, 1, 2, 1};
  }
  if (NTAPS == 3) return variant == 0 ? PairSel{2, 1, 1, 1, 2, 1} : PairSel{1, 2, 2, 1, 2, 2};
  // C = 32, k = 11: 88 KB of weights.  One h tile + four slab slots (measured 192-198 us per pair at L = 2.88 M against
  // 205-231 us as two launches); two h tiles leave three slots at dilation 5 and lose there (241 us):
  // profiles/r2_pair_k11_cfg{0,1}.jsonl.  The shape sits at the shared-memory operand bound of N = 32 MMAs (~0.66 PFLOP/s)
  if (NTAPS == 11) return variant == 0 ? PairSel{1, 1, 1, 1, 2, 1} : PairSel{1, 2, 1, 1, 2, 1};
  return variant == 0 ? PairSel{1, 2, 2, 1, 2, 1} : PairSel{1, 2, 2, 1, 2, 2};
}

struct PairPlan {
  int tile_m, out_rows, halo, r, nbox, rb, a_bytes, h_rows, h_bytes, w_bytes, epi_bytes, nb1, fixed, na, nbar, smem;
};
constexpr PairPlan pair_plan(int C, int NTAPS, int DIL, PairSel s) {
  PairPlan q{};
  q.tile_m = s.msub * 128;
  q.out_rows = q.tile_m - (NTAPS - 1);
  q.halo = (NTAPS - 1) * DIL;
  q.r = q.tile_m + q.halo;
  q.nbox = (q.r + 255) / 256;
  q.rb = (((q.r + q.nbox - 1) / q.nbox) + 7) & ~7;
  q.a_bytes = q.nbox * q.rb * 128;
  q.h_rows = (q.tile_m + NTAPS - 1 + 7) & ~7;
  q.h_bytes = q.h_rows * 128;
  q.w_bytes = C * 128;
  q.epi_bytes = 4 * s.e2g * s.out_slots * s.msub * (C / 32) * kPairBox;      // [warps][sets][boxes of a tile][2 KB]
  q.nb1 = s.la + 1;
  q.fixed = 1024 + s.nh * q.h_bytes + 2 * NTAPS * q.w_bytes + q.epi_bytes + 2 * C * 4 + 8 * (2 * 6 + 1 + 2 * q.nb1 + 4 + 2 * s.nh) + 64;
  q.na = (kPairSmemMax - q.fixed) / q.a_bytes;
  if (q.na > 6) q.na = 6;
  q.nbar = 2 * q.na + 1 + 2 * q.nb1 + 4 + 2 * s.nh;
  q.smem = q.fixed + q.na * q.a_bytes;
  return q;
}

struct PairParams {
  const float* bias1;
  const float* bias2;
  int L, batch;
  int fmt1, fmt2;              // MMA operand formats of conv1 / conv2 (0 = fp16, 1 = bf16); h is stored in fmt2
  float h_slope;               // lrelu slope between the convolutions
  void* y32;                   // planar-vector fp16 branch sum [B][C/8][Lp_out][8] (or null)
  void* y16;                   // 16-bit channels-last output lrelu_{out_slope}(x') (or null)
  int Lp_out, padf, accum, out_bf16;
  int acc_nostore;             // 1: the branch sum is read (accum) but not written back (the decoder's last tensor leaves as y16 only)
  float div, out_slope, res_neg_scale;
};

template <int C, int NTAPS, int DIL, int VAR>
struct PairCfg {
  static constexpr PairSel S = pair_sel(C, NTAPS, VAR);
  static constexpr PairPlan P = pair_plan(C, NTAPS, DIL, S);
  static constexpr int MSUB = S.msub;
  static constexpr int NH = S.nh;                          // h tiles
  static constexpr int LA = S.la;                          // conv1 runs LA tiles ahead of conv2
  static constexpr int NB1 = P.nb1;                        // conv1 accumulator buffers
  static constexpr int NA = P.na;                          // slab ring
  static constexpr int OUT_SLOTS = S.out_slots;
  static constexpr int E2G = S.e2g;                        // output-epilogue groups (alternate tiles)
  static constexpr int E1G = S.e1g;                        // h-epilogue groups (alternate tiles)
  static constexpr int THREADS = pair_threads(S.e1g, S.e2g);
  static_assert(S.e1g == 1 || (S.nh >= 2 && S.la + 1 >= 2), "two h-epilogue groups need two h tiles and two conv1 accumulators");
  static constexpr int KS = C / 16;                        // K=16 MMA steps (C <= 64: one 128-byte swizzled row)
  static constexpr int OUT_ROWS = P.out_rows;
  static constexpr int P2 = (NTAPS - 1) / 2;               // "same" padding of conv2 (dilation 1)
  static constexpr int P1 = ((NTAPS - 1) / 2) * DIL;       // ... of conv1
  static constexpr int NBOX = P.nbox;
  static constexpr int RB = P.rb;
  static constexpr uint32_t A_BYTES = (uint32_t)P.a_bytes;
  static constexpr uint32_t H_BYTES = (uint32_t)P.h_bytes;
  static constexpr uint32_t W_BYTES = (uint32_t)P.w_bytes;
  static constexpr int EPI_BYTES = P.epi_bytes;
  static constexpr int ACC_COLS = MSUB * C;                // one accumulator buffer
  static constexpr int ACC_USED = (NB1 + 2) * ACC_COLS;    // conv1 x NB1, conv2 x 2
  static constexpr int TMEM_COLS = ACC_USED <= 32 ? 32 : ACC_USED <= 64 ? 64 : ACC_USED <= 128 ? 128 : ACC_USED <= 256 ? 256 : 512;
  static constexpr size_t SMEM = (size_t)P.smem;
  static constexpr int TAIL_ROWS = 32 - (NTAPS - 1);       // valid rows of a tile's last 32-row output box
  static constexpr int CPS = C / 32;                       // 32-column epilogue chunks per 128-row sub-tile
  static constexpr int NCH = MSUB * CPS;                   // ... per tile and warp
  static constexpr int GCH = NCH >= 2 ? 2 : 1;             // chunks whose TMEM loads are issued together
  static_assert(C == 32 || C == 64, "C");
  static_assert(ACC_USED <= 512, "TMEM columns");
  static_assert(NA >= LA + 2 && NA >= 2, "slab ring too small for the conv1 look-ahead");
  static_assert(SMEM <= (size_t)kPairSmemMax, "shared memory");
  static_assert(RB <= 256 && A_BYTES % 1024 == 0 && H_BYTES % 1024 == 0 && W_BYTES % 1024 == 0, "box");
  static_assert(NTAPS - 1 < 32 && NCH % GCH == 0 && NCH <= 2, "tail box / chunk groups / epilogue registers");
};

struct Ring { uint32_t i, ph; };
template <int N>
__device__ __forceinline__ void ring_next(Ring& r) {
  if (++r.i == (uint32_t)N) { r.i = 0; r.ph ^= 1u; }
}

template <int C, int NTAPS, int DIL, int VAR>
__global__ void __launch_bounds__(pair_threads(pair_sel(C, NTAPS, VAR).e1g, pair_sel(C, NTAPS, VAR).e2g), 1)
rbpair_tc_kernel(const PairParams p, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW1,
                 const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmY,
                 const __grid_constant__ CUtensorMap tmYt) {
  using K = PairCfg<C, NTAPS, DIL, VAR>;
  constexpr int MSUB = K::MSUB, NA = K::NA, NH = K::NH, LA = K::LA, NB1 = K::NB1;
  extern __shared__ unsigned char smem_raw[];
  // aligned with pointer arithmetic on the __shared__ array (not through an integer cast): the compiler keeps the
  // shared address space and emits LDS/STS instead of generic LD/ST for every access derived from it
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* sA = smem;                                       // [NA][slab rows][128 B] swizzled (TMA)
  unsigned char* sH = sA + (size_t)NA * K::A_BYTES;               // [NH][H_ROWS][128 B] swizzled (written by epilogue 1)
  unsigned char* sW1 = sH + (size_t)NH * K::H_BYTES;              // [NTAPS][C][128 B] swizzled
  unsigned char* sW2 = sW1 + (size_t)NTAPS * K::W_BYTES;
  unsigned char* sE = sW2 + (size_t)NTAPS * K::W_BYTES;           // [4 E2G warps][OUT_SLOTS sets][NCH output boxes][2 KB]
  float* sbias1 = reinterpret_cast<float*>(sE + K::EPI_BYTES);
  float* sbias2 = sbias1 + C;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sbias2 + C);
  uint64_t* a_full = bars;                  // [NA]
  uint64_t* a_empty = a_full + NA;          // [NA]  conv1 MMAs done (1) + the 4 output-epilogue warps (residual reads)
  uint64_t* w_full = a_empty + NA;          // [1]
  uint64_t* acc1_full = w_full + 1;         // [NB1]
  uint64_t* acc1_empty = acc1_full + NB1;   // [NB1]
  uint64_t* acc2_full = acc1_empty + NB1;   // [2]
  uint64_t* acc2_empty = acc2_full + 2;     // [2]
  uint64_t* h_full = acc2_empty + 2;        // [NH]  epilogue 1 has written h (4 warps)
  uint64_t* h_empty = h_full + NH;          // [NH]  conv2 MMAs have read h
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(h_empty + NH);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const unsigned n_mt = (unsigned)((p.L + K::OUT_ROWS - 1) / K::OUT_ROWS);
  const unsigned total_tiles = n_mt * (unsigned)p.batch;

  if (threadIdx.x == 0) {
    pdl_trigger();
    for (int i = 0; i < NA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 5); }
    mbar_init(w_full, 1);
    for (int i = 0; i < NB1; ++i) { mbar_init(&acc1_full[i], 1); mbar_init(&acc1_empty[i], 4); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc2_full[i], 1); mbar_init(&acc2_empty[i], 4); }
    for (int i = 0; i < NH; ++i) { mbar_init(&h_full[i], 4); mbar_init(&h_empty[i], 1); }
    fence_mbarrier_init();
    fence_proxy_async();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW1);
    prefetch_tmap(&tmW2);
  }
  if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)K::TMEM_COLS);
  for (int i = threadIdx.x; i < C; i += K::THREADS) { sbias1[i] = p.bias1[i]; sbias2[i] = p.bias2[i]; }
  // rows [TILE_M, H_ROWS) of an h tile are only ever read for output rows that are discarded; keep them finite
  for (int i = threadIdx.x; i < (int)((size_t)NH * K::H_BYTES / 16); i += K::THREADS)
    reinterpret_cast<uint4*>(sH)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =========================== producer: TMA global -> swizzled smem ============================
    if (lane == 0) {
      mbar_expect_tx(w_full, 2u * NTAPS * K::W_BYTES);
#pragma unroll 1
      for (int tap = 0; tap < NTAPS; ++tap) {
        tma_load_2d(sW1 + (size_t)tap * K::W_BYTES, &tmW1, 0, tap * C, w_full);
        tma_load_2d(sW2 + (size_t)tap * K::W_BYTES, &tmW2, 0, tap * C, w_full);
      }
      pdl_wait();                                    // the stream comes from the previous kernel (weights do not)
      Ring ra{0u, 0u};
#pragma unroll 1
      for (unsigned tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const unsigned b = tile / n_mt, mt = tile - b * n_mt;
        const int row0 = (int)mt * K::OUT_ROWS - K::P2 - K::P1;
        mbar_wait(&a_empty[ra.i], ra.ph ^ 1u);
        mbar_expect_tx(&a_full[ra.i], K::A_BYTES);
#pragma unroll
        for (int j = 0; j < K::NBOX; ++j)
          tma_load_3d(sA + (size_t)ra.i * K::A_BYTES + (size_t)j * K::RB * 128, &tmA, 0, row0 + j * K::RB, (int)b,
                      &a_full[ra.i]);
        ring_next<NA>(ra);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (warp-uniform, one elected lane): conv1(i + LA) is issued before conv2(i) =====
    const uint32_t leader = elect_one() ? 1u : 0u;
    // instruction descriptor: D=F32 @4, A/B format @7/@10, K-major both, N>>3 @17, M>>4 @24
    const uint32_t f1 = p.fmt1 ? 1u : 0u, f2 = p.fmt2 ? 1u : 0u;
    const uint32_t idesc1 = (1u << 4) | (f1 << 7) | (f1 << 10) | ((uint32_t)(C >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    const uint32_t idesc2 = (1u << 4) | (f2 << 7) | (f2 << 10) | ((uint32_t)(C >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    const uint64_t dproto = make_desc_sw128(0, 0);
    const uint32_t d_hi = (uint32_t)(dproto >> 32), d_lo0 = (uint32_t)dproto;
    const uint32_t sA_d = __shfl_sync(0xffffffffu, d_lo0 + (smem_u32(sA) >> 4), 0);
    const uint32_t sH_d = __shfl_sync(0xffffffffu, d_lo0 + (smem_u32(sH) >> 4), 0);
    const uint32_t sW1_d = __shfl_sync(0xffffffffu, d_lo0 + (smem_u32(sW1) >> 4), 0);
    const uint32_t sW2_d = __shfl_sync(0xffffffffu, d_lo0 + (smem_u32(sW2) >> 4), 0);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t n_my = __shfl_sync(0xffffffffu, (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x, 0);
    mbar_wait(w_full, 0);
    tc_fence_after();
    Ring ra{0u, 0u}, r1{0u, 0u}, rh{0u, 0u}, r2{0u, 0u};
#pragma unroll 1
    for (uint32_t it = 0; it < n_my + (uint32_t)LA; ++it) {
      if (it < n_my) {                                // conv1 of my tile `it`
        mbar_wait(&acc1_empty[r1.i], r1.ph ^ 1u);
        mbar_wait(&a_full[ra.i], ra.ph);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + r1.i * (uint32_t)K::ACC_COLS;
        const uint32_t a_d = sA_d + ra.i * (K::A_BYTES >> 4);
#pragma unroll
        for (int tap = 0; tap < NTAPS; ++tap) {
          const uint32_t b_d = sW1_d + (uint32_t)tap * (K::W_BYTES >> 4);
#pragma unroll
          for (int ms = 0; ms < MSUB; ++ms) {
#pragma unroll
            for (int ks = 0; ks < K::KS; ++ks)
              tc_mma_f16_pred(d_tmem + (uint32_t)(ms * C), a_d + (uint32_t)(((ms * 128 + tap * DIL) * 128 + ks * 32) >> 4), d_hi,
                              b_d + (uint32_t)((ks * 32) >> 4), d_hi, idesc1, (tap | ks) != 0 ? 1u : 0u, leader);
          }
        }
        tc_commit_pred(&a_empty[ra.i], leader);
        tc_commit_pred(&acc1_full[r1.i], leader);
        ring_next<NA>(ra);
        ring_next<NB1>(r1);
      }
      if (it >= (uint32_t)LA) {                       // conv2 of my tile `it - LA`: its h is in sH[rh.i]
        mbar_wait(&h_full[rh.i], rh.ph);
        mbar_wait(&acc2_empty[r2.i], r2.ph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + ((uint32_t)NB1 + r2.i) * (uint32_t)K::ACC_COLS;
        const uint32_t h_d = sH_d + rh.i * (K::H_BYTES >> 4);
#pragma unroll
        for (int tap = 0; tap < NTAPS; ++tap) {
          const uint32_t b_d = sW2_d + (uint32_t)tap * (K::W_BYTES >> 4);
#pragma unroll
          for (int ms = 0; ms < MSUB; ++ms) {
#pragma unroll
            for (int ks = 0; ks < K::KS; ++ks)
              tc_mma_f16_pred(d_tmem + (uint32_t)(ms * C), h_d + (uint32_t)(((ms * 128 + tap) * 128 + ks * 32) >> 4), d_hi,
                              b_d + (uint32_t)((ks * 32) >> 4), d_hi, idesc2, (tap | ks) != 0 ? 1u : 0u, leader);
          }
        }
        tc_commit_pred(&h_empty[rh.i], leader);
        tc_commit_pred(&acc2_full[r2.i], leader);
        ring_next<NH>(rh);
        ring_next<2>(r2);
      }
      __syncwarp();
    }
  } else if (warp < 2 + 4 * K::E1G) {
    // ============ epilogue 1: conv1 accumulator -> h = lrelu(. + b1) in the operand format of conv2 -> sH ============
    // E1G groups of 4 warps take alternate tiles (group g: my tiles g, g + E1G, ...).
    const int qd = warp & 3;                        // TMEM lane quadrant this warp may access
    const uint32_t hg = (uint32_t)(warp - 2) >> 2;
    const bool hbf = p.fmt2 != 0;
    const float hs = p.h_slope;
    Ring r1{hg % (uint32_t)NB1, 0u}, rh{hg % (uint32_t)NH, 0u};   // accumulator / h tile of my tile: (g + E1G n) mod ring
#pragma unroll 1
    for (unsigned tile = blockIdx.x + hg * gridDim.x; tile < total_tiles; tile += K::E1G * gridDim.x) {
      const unsigned mt = tile % n_mt;
      const int th0 = (int)mt * K::OUT_ROWS - K::P2 + qd * 32 + lane;     // time index of this lane's h row (sub-tile 0)
      mbar_wait(&acc1_full[r1.i], r1.ph);
      mbar_wait(&h_empty[rh.i], rh.ph ^ 1u);         // conv2 of the tile that last used this h tile has consumed it
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(qd * 32) << 16) + r1.i * (uint32_t)K::ACC_COLS;
      unsigned char* hbuf = sH + (size_t)rh.i * K::H_BYTES;
#pragma unroll
      for (int g0 = 0; g0 < K::NCH; g0 += K::GCH) {
        uint32_t r[K::GCH][32];
#pragma unroll
        for (int u = 0; u < K::GCH; ++u) {
          const int ci = g0 + u, ms = ci / K::CPS, cc = ci - ms * K::CPS;
          tmem_ld32_issue(tbase + (uint32_t)(ms * C + cc * 32), r[u]);
        }
        float4 bq[8];                                 // bias of the first chunk: its smem latency hides under the TMEM load
        {
          const int cc0 = g0 % K::CPS;
#pragma unroll
          for (int k = 0; k < 8; ++k) bq[k] = lds_f4(sbias1 + cc0 * 32 + k * 4);
        }
        tmem_ld_wait();
        if (g0 + K::GCH >= K::NCH) {                  // the accumulator is in registers: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc1_empty[r1.i]);
        }
#pragma unroll
        for (int u = 0; u < K::GCH; ++u) {
          const int ci = g0 + u, ms = ci / K::CPS, cc = ci - ms * K::CPS;
          if (u > 0) {
#pragma unroll
            for (int k = 0; k < 8; ++k) bq[k] = lds_f4(sbias1 + cc * 32 + k * 4);
          }
          const int hrow = ms * 128 + qd * 32 + lane;
          const int th = th0 + ms * 128;
          const bool ok = th >= 0 && th < p.L;       // conv2 pads h with zeros outside [0, L)
          unsigned char* hp = hbuf + (size_t)hrow * 128;
          const uint32_t sx = (uint32_t)hrow & 7u;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float v[8];
            const float4 b0 = bq[2 * k], b1 = bq[2 * k + 1];
            v[0] = __uint_as_float(r[u][k * 8 + 0]) + b0.x; v[1] = __uint_as_float(r[u][k * 8 + 1]) + b0.y;
            v[2] = __uint_as_float(r[u][k * 8 + 2]) + b0.z; v[3] = __uint_as_float(r[u][k * 8 + 3]) + b0.w;
            v[4] = __uint_as_float(r[u][k * 8 + 4]) + b1.x; v[5] = __uint_as_float(r[u][k * 8 + 5]) + b1.y;
            v[6] = __uint_as_float(r[u][k * 8 + 6]) + b1.z; v[7] = __uint_as_float(r[u][k * 8 + 7]) + b1.w;
            uint4 o;
            o.x = pack2(hbf, lrelu_max(v[0], hs), lrelu_max(v[1], hs)); o.y = pack2(hbf, lrelu_max(v[2], hs), lrelu_max(v[3], hs));
            o.z = pack2(hbf, lrelu_max(v[4], hs), lrelu_max(v[5], hs)); o.w = pack2(hbf, lrelu_max(v[6], hs), lrelu_max(v[7], hs));
            if (!ok) o = make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(hp + ((((uint32_t)(cc * 4 + k)) ^ sx) << 4)) = o;
          }
        }
      }
      fence_proxy_async();                           // generic-proxy writes of sH -> visible to the MMA (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&h_full[rh.i]);
#pragma unroll
      for (int e = 0; e < K::E1G; ++e) { ring_next<NB1>(r1); ring_next<NH>(rh); }
    }
  } else {
    // ===== epilogue 2: conv2 accumulator + b2 + residual (from the slab) -> branch sum / 16-bit stream (TMA boxes) =====
    // The warps of this group are the busiest of the CTA (profiles/r1_ncu_rbpair_v2.md: 94 % of their samples are not
    // barrier waits), so the branch-sum words (global loads) are in registers BEFORE the accumulator barrier is waited
    // for, the accumulator is handed back as soon as it is in registers, and the tile's output boxes share one proxy
    // fence and one bulk group.
    // E2G groups of 4 warps take alternate tiles (group g: my tiles g, g + E2G, ...).
    pdl_wait();
    const int ew = warp - (2 + 4 * K::E1G);
    const uint32_t eg = (uint32_t)ew >> 2;
    const int qd = warp & 3;
    const size_t pitch_o = (size_t)p.Lp_out * 16;   // bytes per planar-vector plane
    const bool obf = p.out_bf16 != 0;
    const float slope = p.out_slope;
    const float div = p.div, rdiv = 1.f / p.div;    // branch mean: exact quotient without a divide (div_exact)
    const float neg_scale = p.res_neg_scale == 0.f ? 1.f : p.res_neg_scale;
    const bool has_y16 = p.y16 != nullptr;
    const bool has_acc = p.y32 != nullptr;
    const bool do_acc = has_acc && p.accum != 0;
    const bool st_acc = p.acc_nostore == 0;
    unsigned char* my_stage = sE + (size_t)ew * K::OUT_SLOTS * K::NCH * kPairBox;   // [OUT_SLOTS sets][NCH boxes]
    const uint32_t sw_row = (uint32_t)lane * 64u, sw_x = ((uint32_t)lane >> 1) & 3u;   // SWIZZLE_64B staging box
    uint32_t oset = 0;
    Ring r2{eg & 1u, 0u};                                         // accumulator buffer of my tile: (g + E2G n) mod 2
    Ring ra{eg % (uint32_t)NA, 0u};                               // slab slot of my tile: (g + E2G n) mod NA
#pragma unroll 1
    for (unsigned tile = blockIdx.x + eg * gridDim.x; tile < total_tiles; tile += K::E2G * gridDim.x) {
      const unsigned b = tile / n_mt, mt = tile - b * n_mt;
      const int o0 = (int)mt * K::OUT_ROWS;
      const int wj0 = qd * 32;                                    // first in-tile row of this warp's group (sub-tile 0)
      unsigned char* acc = has_acc ? reinterpret_cast<unsigned char*>(p.y32) + (size_t)b * (C / 8) * pitch_o : nullptr;
      const unsigned char* slab = sA + (size_t)ra.i * K::A_BYTES;
      uint4 aq[K::NCH][4];                                        // branch-sum words of this lane's rows
      if (do_acc) {
#pragma unroll
        for (int ci = 0; ci < K::NCH; ++ci) {
          const int ms = ci / K::CPS, c0 = (ci - ms * K::CPS) * 32;
          const int jl = ms * 128 + wj0 + lane;
          if (jl < K::OUT_ROWS && o0 + jl < p.L) {
            const unsigned char* q = acc + (size_t)(c0 / 8) * pitch_o + (size_t)(o0 + jl + p.padf) * 16;
#pragma unroll
            for (int k = 0; k < 4; ++k) aq[ci][k] = *reinterpret_cast<const uint4*>(q + (size_t)k * pitch_o);
          }
        }
      }
      mbar_wait(&a_full[ra.i], ra.ph);                            // (long complete: orders the slab reads after the TMA writes)
      mbar_wait(&acc2_full[r2.i], r2.ph);
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(qd * 32) << 16) + ((uint32_t)NB1 + r2.i) * (uint32_t)K::ACC_COLS;
      if (has_y16) {
        if (lane == 0) bulk_wait_read<K::OUT_SLOTS - 1>();        // the bulk group that last used this staging set has read it
        __syncwarp();
      }
      unsigned char* stage = my_stage + (size_t)oset * K::NCH * kPairBox;
#pragma unroll
      for (int ci = 0; ci < K::NCH; ++ci) {
        const int ms = ci / K::CPS, cc = ci - ms * K::CPS, c0 = cc * 32;
        const int jl = ms * 128 + wj0 + lane;                     // in-tile output row of this lane
        const int row = o0 + jl;
        const bool row_ok = jl < K::OUT_ROWS && row < p.L;
        uint32_t r[32];                                           // one chunk at a time: 128 registers per thread at 448 threads
        tmem_ld32_issue(tbase + (uint32_t)(ms * C + c0), r);
        float4 bq[8];                                             // bias and residual row: smem latency under the TMEM load
        uint4 rq[4];
        {
          const int srow = jl + K::P2 + K::P1;                    // this lane's time step inside the activation slab
          const unsigned char* rp = slab + (size_t)srow * 128;
          const uint32_t rx = (uint32_t)srow & 7u;
#pragma unroll
          for (int k4 = 0; k4 < 8; ++k4) bq[k4] = lds_f4(sbias2 + c0 + k4 * 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) rq[k] = lds_u4(rp + ((((uint32_t)(cc * 4 + k)) ^ rx) << 4));
        }
        tmem_ld_wait();
        if (ci == K::NCH - 1) {                                   // the accumulator is in registers: hand it back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc2_empty[r2.i]);
        }
        float v[32];
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) {
          v[k4 * 4 + 0] = __uint_as_float(r[k4 * 4 + 0]) + bq[k4].x;
          v[k4 * 4 + 1] = __uint_as_float(r[k4 * 4 + 1]) + bq[k4].y;
          v[k4 * 4 + 2] = __uint_as_float(r[k4 * 4 + 2]) + bq[k4].z;
          v[k4 * 4 + 3] = __uint_as_float(r[k4 * 4 + 3]) + bq[k4].w;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) add_res8(v + k * 8, rq[k], neg_scale);
        if (has_acc) {
          if (do_acc && row_ok) {
#pragma unroll
            for (int k = 0; k < 4; ++k) add_res8(v + k * 8, aq[ci][k], 1.f);
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
          // this lane's row of the [32 rows][32 channels] staging box of chunk ci (conflict-free under the swizzle)
          unsigned char* box = stage + ci * kPairBox + sw_row;
#pragma unroll
          for (int k8 = 0; k8 < 4; ++k8) {
            uint4 o;
            o.x = pack2(obf, lrelu_max(v[k8 * 8 + 0], slope), lrelu_max(v[k8 * 8 + 1], slope));
            o.y = pack2(obf, lrelu_max(v[k8 * 8 + 2], slope), lrelu_max(v[k8 * 8 + 3], slope));
            o.z = pack2(obf, lrelu_max(v[k8 * 8 + 4], slope), lrelu_max(v[k8 * 8 + 5], slope));
            o.w = pack2(obf, lrelu_max(v[k8 * 8 + 6], slope), lrelu_max(v[k8 * 8 + 7], slope));
            *reinterpret_cast<uint4*>(box + ((((uint32_t)k8) ^ sw_x) << 4)) = o;
          }
        }
      }
      if (has_y16) {
        // one lane stores the tile's boxes (rows >= L are clipped by the tensor map; the tile's last 32-row box holds only
        // TAIL_ROWS valid rows and goes through the shorter tensor-map box)
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (int ci = 0; ci < K::NCH; ++ci) {
            const int ms = ci / K::CPS, cc = ci - ms * K::CPS;
            const bool tail = ms == MSUB - 1 && qd == 3;
            tma_store_3d(tail ? &tmYt : &tmY, stage + ci * kPairBox, cc * 32, o0 + ms * 128 + wj0, (int)b);
          }
          bulk_commit();
        }
        if (++oset == (uint32_t)K::OUT_SLOTS) oset = 0;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&a_empty[ra.i]);                 // the residual rows of this slab have been read
#pragma unroll
      for (int e = 0; e < K::E2G; ++e) { ring_next<2>(r2); ring_next<NA>(ra); }
    }
    if (lane == 0) bulk_wait_all();                 // staged stores complete before the CTA's smem goes away
  }
  // ------------------------------------ teardown -------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)K::TMEM_COLS);
}

template <int C, int NTAPS, int DIL, int VAR>
cudaError_t launch_pair_one(const TcConvDesc& d1, const TcConvDesc& d2, int B, cudaStream_t st) {
  using K = PairCfg<C, NTAPS, DIL, VAR>;
  if (!tensor_map_encoder_available()) return cudaErrorNotSupported;
  CUtensorMap tmA, tmW1, tmW2, tmY, tmYt;
  const CUtensorMapDataType dt1 = d1.in_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const CUtensorMapDataType dt2 = d2.in_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const int L = d1.Lj;
  {
    cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)L, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * (cuuint64_t)L};
    cuuint32_t box[3] = {64, (cuuint32_t)K::RB, 1};
    if (!encode_tensor_map(&tmA, dt1, 3, d1.x16, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return cudaErrorInvalidValue;
    cuuint64_t wdims[2] = {64, (cuuint64_t)NTAPS * C};
    cuuint64_t wstrides[1] = {128};
    cuuint32_t wbox[2] = {64, (cuuint32_t)C};
    if (!encode_tensor_map(&tmW1, dt1, 2, d1.w16, wdims, wstrides, wbox, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return cudaErrorInvalidValue;
    if (!encode_tensor_map(&tmW2, dt2, 2, d2.w16, wdims, wstrides, wbox, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return cudaErrorInvalidValue;
    tmY = tmA;
    tmYt = tmA;
    if (d2.y16) {
      const CUtensorMapDataType dto = d2.out_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
      cuuint32_t obox[3] = {32, 32, 1};
      cuuint32_t tbox[3] = {32, (cuuint32_t)K::TAIL_ROWS, 1};
      if (!encode_tensor_map(&tmY, dto, 3, d2.y16, dims, strides, obox, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B))
        return cudaErrorInvalidValue;
      if (!encode_tensor_map(&tmYt, dto, 3, d2.y16, dims, strides, tbox, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B))
        return cudaErrorInvalidValue;
    }
  }
  static SmemOptIn opt;
  if (cudaError_t e = opt_in_smem(rbpair_tc_kernel<C, NTAPS, DIL, VAR>, K::SMEM, opt)) return e;
  const int num_sms = current_num_sms();
  PairParams p{};
  p.bias1 = d1.bias; p.bias2 = d2.bias;
  p.L = L; p.batch = B;
  p.fmt1 = d1.in_bf16; p.fmt2 = d2.in_bf16;
  p.h_slope = d1.out_slope;
  p.y32 = d2.y32; p.y16 = d2.y16;
  p.Lp_out = d2.Lp_out; p.padf = d2.padf; p.accum = d2.accum; p.out_bf16 = d2.out_bf16;
  p.acc_nostore = d2.acc_nostore;
  p.div = d2.div; p.out_slope = d2.out_slope; p.res_neg_scale = d2.res_neg_scale;
  const long long tiles = (long long)((L + K::OUT_ROWS - 1) / K::OUT_ROWS) * B;
  const unsigned grid = (unsigned)(tiles < num_sms ? tiles : num_sms);      // persistent: one CTA per SM
  cudaError_t le = launch_pdl(rbpair_tc_kernel<C, NTAPS, DIL, VAR>, dim3(grid), dim3(K::THREADS), K::SMEM, st, p, tmA, tmW1,
                              tmW2, tmY, tmYt);
  launch_counter().n++;
  return le != cudaSuccess ? le : cudaGetLastError();
}

// RVCB200_PAIR_CFG=1 selects the alternative pipeline shape of pair_sel() (A/B measurements, tools/bench_conv_tc.py --pair)
int pair_variant() {
  const char* e = getenv("RVCB200_PAIR_CFG");
  return e ? atoi(e) : 0;
}

template <int C, int NTAPS, int VAR>
cudaError_t launch_pair_d(const TcConvDesc& d1, const TcConvDesc& d2, int B, cudaStream_t st) {
  switch (d1.dil) {
    case 1: return launch_pair_one<C, NTAPS, 1, VAR>(d1, d2, B, st);
    case 3: return launch_pair_one<C, NTAPS, 3, VAR>(d1, d2, B, st);
    case 5: return launch_pair_one<C, NTAPS, 5, VAR>(d1, d2, B, st);
    default: return cudaErrorNotSupported;
  }
}

template <int C, int NTAPS>
cudaError_t launch_pair_v(const TcConvDesc& d1, const TcConvDesc& d2, int B, cudaStream_t st) {
  return pair_variant() == 1 ? launch_pair_d<C, NTAPS, 1>(d1, d2, B, st) : launch_pair_d<C, NTAPS, 0>(d1, d2, B, st);
}

}  // namespace

// The fused kernel covers a (conv1, conv2) pair when both are resblock shapes of rbconv_tc.cu with C in {32, 64},
// k in {3, 7} -- and k = 11 at C = 32 -- (both weight sets resident in shared memory: C = 64, k = 11 would need 176 KB),
// conv2 has dilation 1 and consumes conv1's 16-bit output,
// the residual is the pair's own input stream, and the output does not alias it (tiles read a halo of the input).
bool rbpair_tc_supported(const TcConvDesc& d1, const TcConvDesc& d2) {
  if (!rbconv_tc_supported(d1) || !rbconv_tc_supported(d2)) return false;
  if (d1.tanh_out || d2.tanh_out || d1.acc_nostore || d1.inj_har || d2.inj_har) return false;
  if (!(d1.Cin == 32 || d1.Cin == 64) || d2.Cin != d1.Cin) return false;
  if (!(d1.ntaps == 3 || d1.ntaps == 7 || (d1.ntaps == 11 && d1.Cin == 32)) || d2.ntaps != d1.ntaps || d2.dil != 1) return false;
  if (d1.Lj != d2.Lj || d1.L_in != d2.L_in) return false;
  if (!d1.y16 || d1.y32 || d1.res16 || d1.accum || d1.div != 1.f) return false;      // conv1: 16-bit store of lrelu(.) only
  if (d2.x16 != d1.y16 || d1.out_bf16 != d2.in_bf16) return false;                   // conv2 consumes h
  if (!d2.res16 || d2.res16 != d1.x16) return false;                                 // residual = the pair's input stream
  if (d2.y16 == d1.x16) return false;                                                // no in-place update (halo reads)
  if (!d2.y16 && !d2.y32) return false;
  return true;
}

cudaError_t launch_rbpair_tc(const TcConvDesc& d1, const TcConvDesc& d2, int B, cudaStream_t st) {
  if (!rbpair_tc_supported(d1, d2) || B <= 0) return cudaErrorNotSupported;
  if (d1.Cin == 32 && d1.ntaps == 11) return launch_pair_v<32, 11>(d1, d2, B, st);
  if (d1.Cin == 32) return d1.ntaps == 3 ? launch_pair_v<32, 3>(d1, d2, B, st) : launch_pair_v<32, 7>(d1, d2, B, st);
  return d1.ntaps == 3 ? launch_pair_v<64, 3>(d1, d2, B, st) : launch_pair_v<64, 7>(d1, d2, B, st);
}

}  // namespace rvc
