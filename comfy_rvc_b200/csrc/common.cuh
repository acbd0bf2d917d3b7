// Shared device/host helpers for the rvcb200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/rvcb200.h"

namespace rvc {

// Per-launch bookkeeping: launches are counted so bench.py can report gpu_launches.
struct LaunchCounter {
  long long n = 0;
};
LaunchCounter& launch_counter();

inline int cuda_ok(cudaError_t e, const char* what, char* errbuf, size_t errlen) {
  if (e == cudaSuccess) return 1;
  if (errbuf) snprintf(errbuf, errlen, "%s: %s", what, cudaGetErrorString(e));
  return 0;
}

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------------
// Kernels of the tensor path are launched with the programmatic-stream-serialization attribute: a kernel signals at its
// very start that its successor may be scheduled (pdl_trigger), so the successor's CTAs take over SMs as this grid's
// CTAs retire and run their prologue (barrier init, TMEM allocation, tensor-map fetch, constant weights -> smem) under
// this grid's tail; before touching anything a predecessor wrote -- or writing anything a predecessor may still read --
// every thread that accesses global memory executes pdl_wait(), which returns once all prerequisite grids have
// completed and their memory is visible.  Measured on B200: 60 s segment (181 launches) 12.20 ms with, 12.13 ms without --
// the step is the sum of its kernel times, there is no launch gap to hide; 1 s segment 1.89 ms with, 2.05 ms without.  So the
// engine turns it on for launch-bound sizes only (RVCB200_PDL=0/1 forces it; without the launch attribute both
// instructions are no-ops).
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
bool pdl_enabled();
void pdl_set_auto(bool on);      // per-call default when RVCB200_PDL is not set (engine.cu: launch-bound sizes)

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---- per-device launch state ---------------------------------------------------------------------------------------
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of a kernel and the SM count is a property of
// the current device, so both are cached per device ordinal (a process may run `SynthesizerB200.to("cuda:1")` after
// cuda:0).  Atomics only: a redundant cudaFuncSetAttribute from a racing thread is harmless.
constexpr int kMaxDevices = 64;
struct SmemOptIn {
  std::atomic<size_t> bytes[kMaxDevices];
  SmemOptIn() { for (auto& b : bytes) b.store(0); }
};
template <typename Kern>
inline cudaError_t opt_in_smem(Kern kern, size_t smem, SmemOptIn& cache) {
  if (smem <= 48 * 1024) return cudaSuccess;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const bool cached = dev >= 0 && dev < kMaxDevices;
  if (cached && cache.bytes[dev].load(std::memory_order_acquire) >= smem) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (cached) cache.bytes[dev].store(smem, std::memory_order_release);
  return cudaSuccess;
}
int current_num_sms();   // SM count of the current device (small_kernels.cu)

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }
__device__ __forceinline__ float sigmoidf_(float v) { return 1.f / (1.f + expf(-v)); }

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::); }

// ---- kernels implemented across the .cu files (host launchers) -----------------------------
typedef rvcb200_conv_desc ConvDesc;

cudaError_t launch_conv_f32(const ConvDesc& d, int B, cudaStream_t st);

cudaError_t launch_layernorm(const float* x, const float* gamma, const float* beta, float* y, long long rows, int C,
                             float eps, cudaStream_t st, void* y16 = nullptr, const int* len = nullptr, int T = 0);

cudaError_t launch_attention_f32(const float* qkv, const float* rel_k, const float* rel_v, const int* len, float* out,
                                 int B, int T, int n_heads, int dk, int window, cudaStream_t st);

size_t sine_scratch_bytes(int B, int T, int upp);
cudaError_t launch_sine_source(const float* f0, const float* noise, float* har, int B, int T, int upp, int sr,
                               float lin_w, float lin_b, void* scratch, cudaStream_t st);

// len32[b] = (int) len64[b]
cudaError_t launch_len_to_i32(const long long* len64, int* len32, int B, int T, cudaStream_t st);

// out[b][j] = bias[j] + sum_i W[j][i] * emb[sid[b]][i]   (all speaker-conditioning 1x1 convs at once)
cudaError_t launch_cond_gemv(const float* emb_g, const long long* sid, const float* W, const float* bias, float* out,
                             int B, int gin, int n_out, int n_spk, cudaStream_t st);

// z_p[b][t][c] = (m + exp(logs) * noise[b][c][t] * 0.66666) masked   (models.py:685/801)
cudaError_t launch_flow_x0_init(const void* z16, const int* len, void* abuf, int B, int T, int C, int in_off, int half, int xb, int aw,
                                cudaStream_t st);
cudaError_t launch_zp_sample(const float* stats, const float* noise_cf, const int* len, float* zp, int B, int T, int C,
                             cudaStream_t st, float* z = nullptr, void* z16 = nullptr);

// y[b][t][co] += nb[co] + sum_k har[b][t*s - pad + k] * wn[k][co]   (models.py:552-553)
cudaError_t launch_noise_conv_add(const float* har, const float* wn, const float* nb, float* y, int B, long long L_har,
                                  long long L_out, int C, int k, int s, int pad, cudaStream_t st);

// out[b][t] = tanh( sum_{k,ci} lrelu_{slope}(x[b][t+k-3][ci]) * w[k][ci] )   (models.py:561-563)
cudaError_t launch_conv_post_tanh(const float* x, const float* w, float* out, int B, long long L, int C, int k,
                                  float slope, cudaStream_t st);

// dst = src * scale, elementwise (row-strided copy): dst[r][c] = src[r][c] for c < C
cudaError_t launch_copy_rows(const float* src, int lds, float* dst, int ldd, long long rows, int C, cudaStream_t st);

// ---- segmented-driver pre/post steps (pipeline_kernels.cu) ----
cudaError_t launch_prepare_feats(const void* f, const void* f0, int dtype, const float* pitchf, float* out, int F, int T, int C,
                                 float protect, int use_protect, cudaStream_t st);
cudaError_t launch_absmax(const float* x, long long n, float* out, int reset, cudaStream_t st);
cudaError_t launch_to_int16(const float* x, long long n, const float* absmax, short* out, cudaStream_t st);
cudaError_t launch_rms_halfblock(const void* x, int x_f64, long long len, long long offset, int hop, double* out, cudaStream_t st);
cudaError_t launch_rms_fold(const double* table, int rows, long long n_hb, int frame_length, float* rms, cudaStream_t st);
cudaError_t launch_rms_gain(float* x, long long len, long long offset, long long N, const float* rms1, long long n1, const float* rms2,
                            long long n2, double rate, cudaStream_t st);
cudaError_t launch_resample_poly(const float* tab, int up, int down, int tpp, long long half_len, const float* left, long long n_left,
                                 const float* piece, long long n_piece, const float* right, long long n_right, long long piece_off,
                                 long long n_song, long long out_lo, long long out_hi, float* out, cudaStream_t st);
cudaError_t launch_quiet_point(const double* audio_pad, long long lo, long long hi, int window, double* best_v, long long* best_j,
                               int n_blocks, cudaStream_t st);

// ---- index blend of VC.vc, IVF-Flat nprobe 1 (index_kernels.cu) ----
long long ivf_scratch_bytes(int F, int nlist);
cudaError_t launch_ivf_assign(const void* x, int x_dtype, long long ldx, int F, int d, const float* cent, const float* cnorm, int nlist,
                              unsigned long long* coarse, cudaStream_t st);
cudaError_t launch_ivf_scan(const void* x, int x_dtype, long long ldx, int F, int d, const unsigned long long* coarse, int nlist,
                            const int* list_offsets, const float* vec, const long long* labels, void* scratch, long long scratch_bytes,
                            float* score, long long* ix, cudaStream_t st);
cudaError_t launch_index_blend(const void* feats, int feats_dtype, long long ldf, int F, int d, const float* score, const long long* ix,
                               const float* vec, const int* pos_of_label, long long ntotal, int is_half, double index_rate, void* out,
                               cudaStream_t st);

// ---- HuBERT / ContentVec front end, first layer (hubert_kernels.cu) ----
cudaError_t launch_hubert_conv0(const float* x, const float* w, const float* gn_w, const float* gn_b, double* stats, void* y16,
                                int B, long long n, int C, int K, int S, float eps, long long y_bstride, cudaStream_t st);


// ---- RMVPE f0 estimator: the non-contraction steps (rmvpe_kernels.cu) ----
cudaError_t launch_rmvpe_logmel(const float* audio, long long n, const float* window, const void* twiddle, const float* mel_basis,
                                const void* mel_range, float bn_scale, float bn_shift, float* mel_out, void* img, int n_frames,
                                int frames_out, int img_pitch, int img_c, cudaStream_t st);
cudaError_t launch_rmvpe_pool(const float* x, int ldx, void* y16, int H2, int W2, int C, int p_in, int p_out, cudaStream_t st);
cudaError_t launch_rmvpe_shuffle(const void* g16, void* out16, int H, int W, int Co, int ld, int p_in, int fp_out, int pack,
                                 cudaStream_t st);
cudaError_t launch_rmvpe_gru_pack(const float* y, int ldc, void* x16, long long T, int W, int pitch, cudaStream_t st);
cudaError_t launch_rmvpe_gru(const float* gi, const float* w_hh, const float* b_hh, void* out16, float* out32, int T, cudaStream_t st);
cudaError_t launch_rmvpe_decode(const float* in, int ld, int from_hidden, float* hidden, double* f0, double* cents, int T,
                                float thred, cudaStream_t st);
cudaError_t launch_rmvpe_mel_to_img(const float* mel, void* img, int n_frames, int frames_out, float bn_scale, float bn_shift,
                                    int img_pitch, int img_c, cudaStream_t st);

// ---- CREPE f0 estimator: the non-contraction steps (crepe_kernels.cu) ----
cudaError_t launch_crepe_frames(const float* audio, long long n, long long first, long long count, int hop, int pad, void* out,
                                cudaStream_t st);
cudaError_t launch_crepe_bn_pool(const void* x, const float* scale, const float* shift, void* out, long long frames, int C, int L,
                                 int p_in, int in_off, int p_out, int out_off, cudaStream_t st);
cudaError_t launch_crepe_decode(const float* in, int ld, int from_salience, long long T, int chunk, int lo, int hi, int mode,
                                const double* dither, const double* wcents, const double* ltab, double c_out, double log_init,
                                float* sal, double* logp, unsigned short* ptr, int* bins, double* f0, float* period, double* score,
                                cudaStream_t st);

}  // namespace rvc
