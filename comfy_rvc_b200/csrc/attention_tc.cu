// Windowed relative-position self-attention on tcgen05 / TMEM (fp16 operands, fp32 softmax + accumulate).
//
// Restates /root/reference/lib/infer_pack/attentions.py:222-270 in the banded form of SURVEY.md App. D:
//     S[i][j] = q~_i . k_j + [|j-i| <= w] q~_i . Ek[j-i+w]        (q~ = q / sqrt(dk), folded into the q weights)
//     P = softmax_j(S) over keys j < len;   O_i = sum_j P[i][j] v_j + sum_{|j-i|<=w} P[i][j] Ev[j-i+w]
//
// One CTA = 128 queries of one (batch, head).  All four contractions run on the tensor core:
//     R  = Q Ek^T           [128 x 32]   once          (the 21 relative-key logits of every query)
//     S  = Q K^T            [128 x 64]   per key tile
//     O += P V              [128 x 96]   per key tile
//     O += Pband Ev         [128 x 96]   once          (Pband[i][r] = P[i][i+r-w])
// ONE pass over the keys with an online softmax (round 2; the first version made two passes to avoid rescaling the TMEM
// accumulator, and its extra Q K^T was 38 % of the tensor-pipe time of a kernel that ncu showed to be bound by exactly that
// -- an M = 128, N = 64, K = 16 MMA keeps the pipe busy ~63 cycles, twice its math time, from shared memory and from tensor
// memory alike, `profiles/r2_ncu_attention.md`).  A row's running max is raised only when a tile exceeds it by more than
// kTau (probabilities stay <= e^kTau in fp16), so the rescale of O -- tcgen05.ld / multiply / tcgen05.st by the row's own
// softmax thread, after the group's previous P V has completed -- happens in the first tiles only.
//
// Operands: qkv16 [B][T][3*heads*128] = q | k | v, 128 channels per head (96 + zero pad), q pre-scaled; K tiles by TMA
// (K-major, SWIZZLE_128B); V tiles by TMA from the same rows, keys x channels as the projection wrote them, consumed as an
// MN-major B operand (no transposed copy; the `vt` scratch argument of the launcher is unused); ek16 [32][128]; evt16 [128][64].  Q and P are MMA A operands in TENSOR MEMORY (tcgen05.mma TS form: lane = row, a 32-bit column holds two
// fp16 of the row): the softmax threads store their q row once and each tile's probabilities over the head of the tile's own
// S slot, so neither needs shared memory, a swizzle or a proxy fence.
// Warps: 0 = TMA producer (lane 0: K ring, lane 1: V ring), 2..9 = softmax, thread = query row = TMEM lane, in two GROUPS of
// four warps (one per lane quadrant).  Group g takes every second key tile whole (64 columns per thread) and has its OWN
// accumulator O_g, running max and running sum, so the two groups never synchronise inside the key loop; they are combined
// at the end (O_0 is brought to the final scale in tensor memory, the band probabilities are formed from the kept band
// logits at that scale, Pband Ev is accumulated into O_0, O_1 is added in registers).  Three MMA-issuing warps: warp 1 /
// warp 10 issue Q K^T for group 0 / 1, warp 11 issues P V and Pband Ev -- with ONE issuer the kernel was bound by that
// thread's instruction stream (~145 SASS instructions, ~1200 cycles per key tile).
#include "tc_ptx.cuh"

namespace rvc {
namespace {

constexpr int BQ = 128, BKV = 64, DKP = 128, DKV = 96, NSTG = 4, NSTV = 4, MAXREL = 21;   // K ring (= S slots) / V ring depths
constexpr int kThreadsAtt = 64 + 256 + 64;   // producer, Q K^T issuer 0, 8 softmax warps, Q K^T issuer 1, P V issuer
// TMEM columns (512 allocated): one O accumulator per softmax group, the relative-key logits R (aliases the head of O_1,
// dead before the first P V), the Q tile as an MMA A operand (96 fp16 per lane = 48 columns), four S slots; the P tile
// of a key tile (64 fp16 = 32 columns, MMA A operand) overwrites the head of its own S slot.
constexpr uint32_t TM_O = 0, TM_R = 96, TM_Q = 192, TM_S = 256, TM_COLS = 512;
constexpr float kTau = 4.f;                  // a row's running max is raised (and O rescaled) only when exceeded by more than this
constexpr float kLog2e = 1.4426950408889634f;

using namespace tc;

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// SWIZZLE_128B K-major descriptor halves: lo = start>>4 | LBO(1)<<16 ; hi = SBO(1024>>4) | version 1<<14 | SW128 (2)<<29
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr >> 4) & 0x3FFFu) | (1u << 16); }
constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t idesc_f16(int N) {   // D=F32, A=B=F16, K-major, M=128
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(BQ >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  tmem_ld32_issue(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// 64 accumulator columns of this thread's lane: both loads in flight before the one wait
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, float* v) {
  uint32_t r[64];
  tmem_ld32_issue(taddr, r);
  tmem_ld32_issue(taddr + 32, r + 32);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 64; ++i) v[i] = __uint_as_float(r[i]);
}

struct AttSmem {                        // 1024-byte aligned tiles, all [rows][128 B] swizzled
  unsigned char k[NSTG][2][BKV * 128];  // 2 k-blocks of 64 channels
  unsigned char v[NSTV][2][BKV * 128];  // V tile as it lies in q|k|v: 64 keys x (2 blocks of 64 channels), MN-major B operand
  unsigned char pband[BQ * 128];        // P[i][i+r-w], r < 21 (columns >= 21 stay zero)
  unsigned char ek[2][32 * 128];
  unsigned char evt[DKV * 128];
  float rtab[BQ * 24];                  // relative-key logits per query row (dynamic indexing)
  float xch[2][2][BQ];                  // [max | sum][group][row]: exchanged between the two warps of a row
  uint64_t bars[40];
  uint32_t tmem_slot;
};

struct AttArgs {
  const int* len;
  const __half* qkv;    // [B][T][ld]: q | k | v, 128 channels per head
  __half* out;          // [B][T][H]
  int T, n_heads, window, H, ld;
};

__global__ void __launch_bounds__(kThreadsAtt, 1)
attention_tc_kernel(const AttArgs a, const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                    const __grid_constant__ CUtensorMap tmEk, const __grid_constant__ CUtensorMap tmEv) {
  extern __shared__ unsigned char smem_raw[];
  // aligned by pointer arithmetic on the __shared__ array: keeps the shared address space (LDS/STS, not generic LD/ST)
  AttSmem& sm = *reinterpret_cast<AttSmem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * BQ;
  if (threadIdx.x == 0) pdl_trigger();
  pdl_wait();                            // q|k|v come from the kernel just before
  const int L = min(a.len ? a.len[b] : a.T, a.T);
  const int nrel = 2 * a.window + 1;

  if (q0 >= L) {   // padding-only query tile: zeros (uniform early exit, nothing allocated yet)
    for (int idx = threadIdx.x; idx < BQ * (DKV / 8); idx += kThreadsAtt) {
      const int i = idx / (DKV / 8), c = idx % (DKV / 8);
      if (q0 + i < a.T)
        *reinterpret_cast<uint4*>(a.out + ((size_t)b * a.T + q0 + i) * a.H + h * DKV + c * 8) = make_uint4(0, 0, 0, 0);
    }
    return;
  }
  const int ntiles = (L + BKV - 1) / BKV;

  uint64_t* e_full = &sm.bars[0];        // Ek | Ev^T landed
  uint64_t* q_ready = &sm.bars[1];       // Q tile stored to tensor memory by the 8 softmax warps
  uint64_t* r_full = &sm.bars[2];
  uint64_t* pb_full = &sm.bars[3];       // the 4 warps of group 0: O_0 at the final scale, Pband tile written
  uint64_t* o_full = &sm.bars[4];
  uint64_t* pv_all = &sm.bars[5];        // every P V MMA has completed
  uint64_t* k_full = &sm.bars[8];        // [NSTG]   key tile it -> slot it & 3: K stage, S buffer, P buffer
  uint64_t* k_empty = &sm.bars[12];      // [NSTG]
  uint64_t* v_full = &sm.bars[16];       // [NSTV]
  uint64_t* v_empty = &sm.bars[20];      // [NSTV]
  uint64_t* s_full = &sm.bars[24];       // [4]
  uint64_t* pv_done = &sm.bars[28];      // [4]  the P V MMA of the slot's tile has completed: slot (S and P) free, O settled
  uint64_t* p_full = &sm.bars[32];       // [4], the 4 warps of the slot's group

  if (threadIdx.x == 0) {
    mbar_init(e_full, 1); mbar_init(q_ready, 8); mbar_init(r_full, 1); mbar_init(pb_full, 4); mbar_init(o_full, 1); mbar_init(pv_all, 1);
    for (int i = 0; i < NSTG; ++i) {
      mbar_init(&k_full[i], 1); mbar_init(&k_empty[i], 1); mbar_init(&s_full[i], 1); mbar_init(&pv_done[i], 1); mbar_init(&p_full[i], 4);
    }
    for (int i = 0; i < NSTV; ++i) { mbar_init(&v_full[i], 1); mbar_init(&v_empty[i], 1); }
    fence_mbarrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(&sm.tmem_slot, TM_COLS);
  // zero the Pband tile (generic proxy) before anybody can use it
  for (int idx = threadIdx.x; idx < BQ * 8; idx += kThreadsAtt) reinterpret_cast<uint4*>(sm.pband)[idx] = make_uint4(0, 0, 0, 0);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_slot;

  if (warp == 0) {
    // ======================================= TMA producer =======================================
    // lane 0 streams the relative tables and the K tiles, lane 1 the V tiles: two independent rings, so that a full V ring
    // never holds back the K tile the next Q K^T is waiting for
    if (lane == 0) {
      mbar_expect_tx(e_full, 2 * 32 * 128 + DKV * 128);
      for (int kb = 0; kb < 2; ++kb) tma_load_2d(sm.ek[kb], &tmEk, kb * 64, 0, e_full);
      tma_load_2d(sm.evt, &tmEv, 0, 0, e_full);
      int ks = 0;
      uint32_t kp = 1;
      for (int it = 0; it < ntiles; ++it) {
        mbar_wait(&k_empty[ks], kp);
        mbar_expect_tx(&k_full[ks], 2 * BKV * 128);
        for (int kb = 0; kb < 2; ++kb) tma_load_3d(sm.k[ks][kb], &tmK, a.n_heads * DKP + h * DKP + kb * 64, it * BKV, b, &k_full[ks]);
        if (++ks == NSTG) { ks = 0; kp ^= 1; }
      }
    } else if (lane == 1) {
      int vs = 0;
      uint32_t vp = 1;
      for (int t = 0; t < ntiles; ++t) {
        mbar_wait(&v_empty[vs], vp);
        mbar_expect_tx(&v_full[vs], 2 * BKV * 128);
        for (int db = 0; db < 2; ++db) tma_load_3d(sm.v[vs][db], &tmV, 2 * a.n_heads * DKP + h * DKP + db * 64, t * BKV, b, &v_full[vs]);
        if (++vs == NSTV) { vs = 0; vp ^= 1; }
      }
    }
  } else if (warp == 1 || warp == 10) {
    // ============================ Q K^T issuer of softmax group g (warp 1: also R = Q Ek^T) ============================
    const int g = warp == 1 ? 0 : 1;
    const uint32_t id_s = idesc_f16(BKV), id_r = idesc_f16(32);
    const uint32_t q_tm = tmem + TM_Q;                   // A operand: 8 columns per K = 16 step
    mbar_wait(q_ready, 0);
    tc_fence_after();
    if (g == 0) {
      mbar_wait(e_full, 0);
      if (elect_one()) {   // R = Q Ek^T : K = 96 = 4 + 2 MMAs
        for (int ks = 0; ks < 6; ++ks)
          tc_mma_f16_ts(tmem + TM_R, q_tm + 8u * ks, desc_lo(smem_u32(sm.ek[ks >> 2])) + 2u * (ks & 3), kDescHi, id_r, ks ? 1u : 0u);
        tc_commit(r_full);
      }
      __syncwarp();
    }
    // key tile it = g + 2 n lands in slot g + 2 (n & 1)
    const uint32_t k_lo[2] = {desc_lo(smem_u32(sm.k[g][0])), desc_lo(smem_u32(sm.k[g + 2][0]))};
    constexpr uint32_t kKb = (BKV * 128) >> 4;            // second k-block of a stage, in descriptor units
    const int mine = (ntiles - g + 1) / 2;
    auto issue_qk = [&](int n, int odd) {
      const int slot = g + 2 * odd;
      mbar_wait(&k_full[slot], ((uint32_t)n >> 1) & 1u);
      mbar_wait(&pv_done[slot], (((uint32_t)n >> 1) & 1u) ^ 1u);   // P V of the slot's previous tile has read its P
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < 6; ++ks)
          tc_mma_f16_ts(tmem + TM_S + 64u * slot, q_tm + 8u * ks, k_lo[odd] + (ks < 4 ? 0u : kKb) + 2u * (ks & 3), kDescHi, id_s,
                     ks ? 1u : 0u);
        tc_commit(&s_full[slot]);
        tc_commit(&k_empty[slot]);
      }
      __syncwarp();
    };
    int n = 0;
    for (; n + 1 < mine; n += 2) { issue_qk(n, 0); issue_qk(n + 1, 1); }
    if (n < mine) issue_qk(n, 0);
  } else if (warp == 11) {
    // ======================================= P V issuer =========================================
    // V is read where the q|k|v projection wrote it, keys x channels: an MN-major B operand (idesc bit 16; canonical
    // SWIZZLE_128B layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units: 64 channels contiguous, key rows 128 B apart,
    // SBO = 1024 B between groups of 8 keys, LBO = 8192 B between the two 64-channel blocks); N = 96 takes the first
    // block and half of the second.  No transposed copy of V.
    const uint32_t id_o = idesc_f16(DKV), id_ov = id_o | (1u << 16);
    mbar_wait(e_full, 0);                                 // Ev^T
    int vs_ = 0;
    uint32_t vp = 0;
    for (int it = 0; it < ntiles; ++it) {
      const int slot = it & 3;
      mbar_wait(&p_full[slot], ((uint32_t)it >> 2) & 1u); // probabilities of this tile are in tensor memory
      mbar_wait(&v_full[vs_], vp);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t p_tm = tmem + TM_S + 64u * slot;
        const uint32_t v_lo = ((smem_u32(sm.v[vs_][0]) >> 4) & 0x3FFFu) | ((uint32_t)((BKV * 128) >> 4) << 16);
        const uint32_t o_tm = tmem + TM_O + 96u * (it & 1);      // the group's own accumulator
#pragma unroll
        for (int ks = 0; ks < BKV / 16; ++ks)
          tc_mma_f16_ts(o_tm, p_tm + 8u * ks, v_lo + 128u * ks, kDescHi, id_ov, (it > 1 || ks) ? 1u : 0u);   // 16 keys = 2048 B
        tc_commit(&pv_done[slot]);
        tc_commit(&v_empty[vs_]);
      }
      __syncwarp();
      if (++vs_ == NSTV) { vs_ = 0; vp ^= 1; }
    }
    if (elect_one()) tc_commit(pv_all);
    __syncwarp();
    // O_0 += Pband Ev  (K = 32: two MMAs, both operands in shared memory; O_0 and Pband are at the final scale)
    mbar_wait(pb_full, 0);
    tc_fence_after();
    if (elect_one()) {
      const uint32_t p_lo = desc_lo(smem_u32(sm.pband)), e_lo = desc_lo(smem_u32(sm.evt));
      for (int ks = 0; ks < 2; ++ks) tc_mma_f16(tmem + TM_O, p_lo + 2u * ks, kDescHi, e_lo + 2u * ks, kDescHi, id_o, 1u);
      tc_commit(o_full);
    }
    __syncwarp();
  } else {
    // ======================================= softmax warps ======================================
    const int qd = warp & 3;
    const int grp = (warp - 2) >> 2;                    // softmax group: every second key tile, accumulator O_grp
    const int row = qd * 32 + lane;                     // TMEM lane = query row in the tile
    const int qi = q0 + row;
    const uint32_t lane_base = ((uint32_t)(qd * 32) << 16);
    {  // this row's q (pre-scaled, fp16) -> tensor memory: group 0 channels [0, 48), group 1 [48, 96)
      uint32_t qv[24];
      if (qi < a.T) {
        const uint4* src = reinterpret_cast<const uint4*>(a.qkv + ((size_t)b * a.T + qi) * a.ld + h * DKP + grp * 48);
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          const uint4 w = __ldg(src + c);
          qv[c * 4 + 0] = w.x; qv[c * 4 + 1] = w.y; qv[c * 4 + 2] = w.z; qv[c * 4 + 3] = w.w;
        }
      } else {
#pragma unroll
        for (int c = 0; c < 24; ++c) qv[c] = 0u;
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) tmem_st8(tmem + lane_base + TM_Q + grp * 24 + c * 8, qv + c * 8);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(q_ready);
    }
    // relative-key logits of this row -> smem (dynamic indexing by key offset); written by the row's first warp
    mbar_wait(r_full, 0);
    tc_fence_after();
    if (grp == 0) {
      float rv[32];
      tmem_ld32(tmem + lane_base + TM_R, rv);
#pragma unroll
      for (int r = 0; r < 24; ++r) sm.rtab[row * 24 + r] = rv[r];
    }
    tc_fence_before();
    asm volatile("bar.sync 1, 256;" ::: "memory");      // the 8 softmax warps; R (= head of O_1) is dead from here on
    float m_run = -INFINITY, l_run = 0.f;
    const uint32_t o_addr = tmem + lane_base + TM_O + 96u * grp;
    int n = 0;                                          // n-th tile of this group -> slot grp + 2 (n & 1)
    for (int it = grp; it < ntiles; it += 2, ++n) {
      const int j0 = it * BKV;
      const int slot = grp + 2 * (n & 1);
      const uint32_t s_addr = tmem + lane_base + TM_S + 64u * slot;
      mbar_wait(&s_full[slot], ((uint32_t)n >> 1) & 1u);
      tc_fence_after();
      float s[BKV];
      tmem_ld64(s_addr, s);
      if (j0 <= q0 + BQ - 1 + a.window && j0 + BKV - 1 >= q0 - a.window) {
        // band: add the relative-key logit and keep the full logit (each band key belongs to exactly one tile): the
        // probabilities of the Ev term are formed from it at the end, at the final scale
#pragma unroll
        for (int c = 0; c < BKV; ++c) {
          const int r = j0 + c - qi + a.window;
          if ((unsigned)r < (unsigned)nrel) {
            s[c] += sm.rtab[row * 24 + r];
            sm.rtab[row * 24 + r] = s[c];
          }
        }
      }
      if (j0 + BKV > L) {
#pragma unroll
        for (int c = 0; c < BKV; ++c)
          if (j0 + c >= L) s[c] = -INFINITY;
      }
      float m_t = s[0];
#pragma unroll
      for (int c = 1; c < BKV; ++c) m_t = fmaxf(m_t, s[c]);
      if (__any_sync(0xffffffffu, m_t > m_run + kTau)) {
        // raise the running max of the warp's rows; O_grp (settled once the group's previous P V has completed) follows
        const float m_new = fmaxf(m_run, m_t);
        if (n > 0) {
          mbar_wait(&pv_done[grp + 2 * ((n - 1) & 1)], ((uint32_t)(n - 1) >> 1) & 1u);
          tc_fence_after();
          const float sc = ex2f((m_run - m_new) * kLog2e);
          l_run *= sc;
#pragma unroll
          for (int c0 = 0; c0 < DKV; c0 += 32) {
            float o[32];
            tmem_ld32(o_addr + c0, o);
            uint32_t ob[32];
#pragma unroll
            for (int c = 0; c < 32; ++c) ob[c] = __float_as_uint(o[c] * sc);
            tmem_st32(o_addr + c0, ob);
          }
          tmem_st_wait();
        }
        m_run = m_new;
      }
      // probabilities (fp16, two keys per 32-bit column) -> head of this tile's S slot
      const float mb = m_run * kLog2e;
      uint32_t pk[BKV / 2];
#pragma unroll
      for (int c = 0; c < BKV; c += 2) {
        const float p0 = ex2f(fmaf(s[c], kLog2e, -mb)), p1 = ex2f(fmaf(s[c + 1], kLog2e, -mb));
        l_run += p0 + p1;
        __half2 hp = __floats2half2_rn(p0, p1);
        pk[c / 2] = *reinterpret_cast<uint32_t*>(&hp);
      }
      tmem_st32(s_addr, pk);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[slot]);
    }
    // ---- combine the two groups: final row max / row sum, O_0 and the band probabilities at the final scale ----
    sm.xch[0][grp][row] = m_run;
    sm.xch[1][grp][row] = l_run;
    asm volatile("bar.sync 1, 256;" ::: "memory");      // also: every band logit is in rtab
    const float m_o = sm.xch[0][grp ^ 1][row], l_o = sm.xch[1][grp ^ 1][row];
    const int n_o = grp ? (ntiles + 1) / 2 : ntiles / 2;  // tiles of the other group
    const float m_fin = fmaxf(m_run, m_o);
    const float f_me = n > 0 ? ex2f((m_run - m_fin) * kLog2e) : 0.f;
    const float f_o = n_o > 0 ? ex2f((m_o - m_fin) * kLog2e) : 0.f;
    const float lsum = l_run * f_me + l_o * f_o;
    if (grp == 0) {
      mbar_wait(pv_all, 0);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < DKV; c0 += 32) {
        float o[32];
        tmem_ld32(o_addr + c0, o);
        uint32_t ob[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) ob[c] = __float_as_uint(o[c] * f_me);
        tmem_st32(o_addr + c0, ob);
      }
      tmem_st_wait();
      const float mb = m_fin * kLog2e;
      for (int r = 0; r < nrel; ++r) {
        const int j = qi + r - a.window;
        const float pv = (j >= 0 && j < L) ? ex2f(fmaf(sm.rtab[row * 24 + r], kLog2e, -mb)) : 0.f;
        *reinterpret_cast<__half*>(sm.pband + row * 128 + (((r >> 3) ^ (row & 7)) << 4) + (r & 7) * 2) = __float2half_rn(pv);
      }
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(pb_full);
    }
    mbar_wait(o_full, 0);
    tc_fence_after();
    const bool valid = qi < L;
    const float inv = valid ? 1.f / lsum : 0.f;
    const float f1 = grp ? f_me : f_o;                  // scale of O_1 (O_0 is at the final scale already)
    const bool has1 = (grp ? n : n_o) > 0;
    __half* orow = a.out + ((size_t)b * a.T + qi) * a.H + h * DKV;
    // output columns: the row's warp of group 0 stores [0, 64), that of group 1 [64, 96)
#pragma unroll
    for (int c0 = 0; c0 < DKV; c0 += 32) {
      if ((c0 < 64) != (grp == 0)) continue;
      float o[32];
      tmem_ld32(tmem + lane_base + TM_O + c0, o);
      if (has1) {
        float o1[32];
        tmem_ld32(tmem + lane_base + TM_O + 96 + c0, o1);
#pragma unroll
        for (int c = 0; c < 32; ++c) o[c] = fmaf(o1[c], f1, o[c]);
      }
      if (qi < a.T) {
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          uint4 w;
          __half2 h0 = __floats2half2_rn(o[c8 * 8 + 0] * inv, o[c8 * 8 + 1] * inv);
          __half2 h1 = __floats2half2_rn(o[c8 * 8 + 2] * inv, o[c8 * 8 + 3] * inv);
          __half2 h2 = __floats2half2_rn(o[c8 * 8 + 4] * inv, o[c8 * 8 + 5] * inv);
          __half2 h3 = __floats2half2_rn(o[c8 * 8 + 6] * inv, o[c8 * 8 + 7] * inv);
          w.x = *reinterpret_cast<uint32_t*>(&h0); w.y = *reinterpret_cast<uint32_t*>(&h1);
          w.z = *reinterpret_cast<uint32_t*>(&h2); w.w = *reinterpret_cast<uint32_t*>(&h3);
          *reinterpret_cast<uint4*>(orow + c0 + c8 * 8) = w;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

// qkv16: [B][T][3*heads*128] fp16 (q | k | v, 128 channels per head, q pre-scaled); vt: unused (was the V^T scratch);
// ek16 [32][128], evt16 [128][64]; out: [B][T][heads*96] fp16.
cudaError_t launch_attention_tc(const void* qkv16, void* vt, const void* ek16, const void* evt16, const int* len, void* out,
                                int B, int T, int n_heads, int dk, int window, cudaStream_t st) {
  if (dk != DKV || 2 * window + 1 > MAXREL || B <= 0 || T <= 0 || n_heads < 1) return cudaErrorInvalidValue;
  if (!tensor_map_encoder_available()) return cudaErrorNotSupported;
  const int ld = 3 * n_heads * DKP;
  (void)vt;   // the transposed copy of V is no longer made (the scratch argument stays in the ABI)
  CUtensorMap tmK, tmV, tmEk, tmEv;
  {
    const CUtensorMapDataType f16 = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B;
    const CUtensorMapL2promotion l2 = CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
    cuuint64_t dims[3] = {(cuuint64_t)(2 * n_heads * DKP), (cuuint64_t)T, (cuuint64_t)B};   // only the q|k columns are visible
    cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)ld * 2 * (cuuint64_t)T};
    cuuint32_t boxk[3] = {64, BKV, 1};
    if (!encode_tensor_map(&tmK, f16, 3, qkv16, dims, strides, boxk, sw, l2)) return cudaErrorInvalidValue;
    cuuint64_t vd[3] = {(cuuint64_t)ld, (cuuint64_t)T, (cuuint64_t)B};                        // the whole q|k|v row; keys >= T read as zero
    if (!encode_tensor_map(&tmV, f16, 3, qkv16, vd, strides, boxk, sw, l2)) return cudaErrorInvalidValue;
    cuuint64_t ekd[2] = {DKP, 32}, eks[1] = {DKP * 2};
    cuuint32_t boxek[2] = {64, 32};
    if (!encode_tensor_map(&tmEk, f16, 2, ek16, ekd, eks, boxek, sw, l2)) return cudaErrorInvalidValue;
    cuuint64_t evd[2] = {64, DKP}, evs[1] = {64 * 2};
    cuuint32_t boxev[2] = {64, DKV};
    if (!encode_tensor_map(&tmEv, f16, 2, evt16, evd, evs, boxev, sw, l2)) return cudaErrorInvalidValue;
  }
  const size_t smem = sizeof(AttSmem) + 1024;
  static SmemOptIn opt;
  if (cudaError_t e = opt_in_smem(attention_tc_kernel, smem, opt)) return e;
  AttArgs a;
  a.len = len; a.qkv = reinterpret_cast<const __half*>(qkv16); a.ld = ld; a.out = reinterpret_cast<__half*>(out); a.T = T; a.n_heads = n_heads; a.window = window; a.H = n_heads * DKV;
  dim3 grid((T + BQ - 1) / BQ, n_heads, B);
  cudaError_t le = launch_pdl(attention_tc_kernel, grid, dim3(kThreadsAtt), smem, st, a, tmK, tmV, tmEk, tmEv);
  if (le != cudaSuccess) return le;
  launch_counter().n++;
  return cudaGetLastError();
}

}  // namespace rvc
