/*
 * rvcb200.h — C ABI of the B200-native RVC synthesis hot path.
 *
 * The reference has no native code and no FFI (SURVEY.md §2.2); its interface for this path
 * is the Python call
 *     net_g.infer(phone, phone_lengths, pitch, nsff0, sid, rate=None)
 *         -> (o, x_mask, (z, z_p, m_p, logs_p))
 * (/root/reference/lib/infer_pack/models.py:682-693 and :798-809), reached from
 * /root/reference/vc_infer_pipeline.py:100-101 after `get_vc` built the module and loaded
 * `cpt["weight"]` (:198-226).  This header is the thin boundary under the Python drop-in
 * (`comfy_rvc_b200.SynthesizerTrnMs{256,768}NSFsid`): plain pointers and sizes, device
 * memory owned by the caller (PyTorch tensors), status codes instead of exceptions, no
 * allocation inside the hot call.
 *
 * Layout convention on the device: activations are channels-last, `[B][rows][C]` fp32 with
 * the channel index contiguous; `phone` is therefore consumed as given by the reference
 * (`[B,T,C_f]`), `noise_zp` as drawn by the reference (`[B,192,T]`, torch.randn_like order),
 * and the waveform `out` is `[B][T*upp]`.
 */
#ifndef RVCB200_H
#define RVCB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RVCB200_ABI_VERSION 1

/* status codes (0 = ok) */
#define RVCB200_OK 0
#define RVCB200_ERR_ARG 1        /* bad argument / unsupported configuration      */
#define RVCB200_ERR_MISSING 2    /* a required packed tensor was never registered  */
#define RVCB200_ERR_WORKSPACE 3  /* workspace too small                            */
#define RVCB200_ERR_CUDA 4       /* a CUDA call or kernel launch failed            */
#define RVCB200_ERR_NO_DEVICE 5  /* no sm_100 device: there is no CPU fallback     */

/* arithmetic of the heavy contractions */
#define RVCB200_PREC_FP32 0 /* CUDA-core fp32 FMA everywhere (int16 +-1 LSB parity path)          */
#define RVCB200_PREC_FP16 1 /* tcgen05 kind::f16 with fp16 operands, fp32 accumulate/residuals     */
#define RVCB200_PREC_BF16 2 /* tcgen05 kind::f16 with bf16 operands, fp32 accumulate/residuals     */

#define RVCB200_MAX_UPS 8
#define RVCB200_MAX_RESK 4
#define RVCB200_MAX_DIL 4

typedef struct rvcb200_ctx rvcb200_ctx;

/* Mirrors the 18-element positional `cpt["config"]` list the reference constructors take
 * (models.py:573-603 / 696-719; process_ckpt.py:31-137) plus the class choice (feat_dim
 * 256 = SynthesizerTrnMs256NSFsid, 768 = SynthesizerTrnMs768NSFsid). */
typedef struct rvcb200_config {
  int32_t feat_dim;        /* 256 | 768 : TextEncoder256 / TextEncoder768 (models.py:33,80) */
  int32_t inter_channels;  /* 192 */
  int32_t hidden_channels; /* 192 */
  int32_t filter_channels; /* 768 */
  int32_t n_heads;         /* 2   */
  int32_t n_layers;        /* 6   */
  int32_t enc_kernel;      /* 3   (FFN kernel_size) */
  int32_t window_size;     /* 10  (attentions.py:18) */
  int32_t flow_kernel;     /* 5   (models.py:654-656) */
  int32_t flow_wn_layers;  /* 3   */
  int32_t n_flows;         /* 4   */
  int32_t resblock_kind;   /* 1 = ResBlock1, 2 = ResBlock2 (models.py:496) */
  int32_t n_res_kernels;
  int32_t res_kernels[RVCB200_MAX_RESK];
  int32_t n_res_dils[RVCB200_MAX_RESK];
  int32_t res_dils[RVCB200_MAX_RESK][RVCB200_MAX_DIL];
  int32_t n_ups;
  int32_t up_rates[RVCB200_MAX_UPS];
  int32_t up_kernels[RVCB200_MAX_UPS];
  int32_t up_init_channels; /* 512 */
  int32_t gin_channels;     /* 256 */
  int32_t n_speakers;       /* emb_g rows */
  int32_t sr;               /* 32000 | 40000 | 48000 */
  int32_t no_f0;            /* 0: NSF synthesizers with pitch (models.py:573-809); 1: the `_nono` classes (models.py:812-1021):
                             * no pitch embedding, plain `Generator` decoder (models.py:244-317) without harmonic source */
} rvcb200_config;

/* Optional copy-out of an intermediate (stage-level parity tests).  `name` is one of
 * "x_enc", "stats", "z_p", "z", "har_source", "dec.pre", "dec.ups.<i>", "dec.stage.<i>".
 * `dst` is a device buffer of at least `bytes` bytes; data is channels-last fp32. */
typedef struct rvcb200_tap {
  const char* name;
  void* dst;
  size_t bytes;
} rvcb200_tap;

/* Replaces: class construction `SynthesizerTrnMs768NSFsid(*cpt["config"], is_half=...)`
 * (vc_infer_pipeline.py:205-218). */
int rvcb200_create(const rvcb200_config* cfg, rvcb200_ctx** out);
void rvcb200_destroy(rvcb200_ctx* ctx);

/* Replaces: `net_g.load_state_dict(cpt["weight"], strict=False)` (vc_infer_pipeline.py:221).
 * The host folds weight-norm and re-lays-out each tensor (comfy_rvc_b200/weights.py) and
 * registers the resulting device buffers by name; the library keeps the pointers (the
 * caller keeps the memory alive).  dtype: 0 = fp32, 1 = fp16, 2 = bf16.  `finalize` resolves
 * every tensor the configuration needs and fails with RVCB200_ERR_MISSING otherwise. */
int rvcb200_set_tensor(rvcb200_ctx* ctx, const char* name, const void* dev_ptr, int64_t numel, int32_t dtype);
/* Host-side scalars of the checkpoint: "dec.src.lin_w", "dec.src.lin_b" (dec.m_source.l_linear, a 1->1
 * Linear, models.py:452,466). */
int rvcb200_set_scalar(rvcb200_ctx* ctx, const char* name, float value);
int rvcb200_finalize(rvcb200_ctx* ctx);

/* Bytes of scratch `rvcb200_infer` needs for a batch of B items of T frames. */
int64_t rvcb200_workspace_bytes(const rvcb200_ctx* ctx, int32_t B, int32_t T, int32_t precision);

/* Replaces: `net_g.infer(phone, phone_lengths, pitch, nsff0, sid)` (models.py:682-693 /
 * :798-809).  All pointers are device pointers.  The three RNG draws of the reference are
 * inputs (as in the reference's ONNX variant, models_onnx.py:634-648): `noise_zp`
 * [B][inter][T] and `noise_sine` [B][T*upp] as `torch.randn` lays them out; the reference's
 * `rand_ini` draw is zeroed for the fundamental (models.py:378-381) and needs no buffer.
 * Outputs: `out` [B][T*upp] fp32 waveform; optional `stats` [B][T][2*inter] (m_p | logs_p),
 * `z_p` [B][T][inter], `z` [B][T][inter], channels-last (NULL to skip).
 * With cfg.no_f0 (`net_g.infer(phone, phone_lengths, sid)`, models.py:905-915) pitch, nsff0 and noise_sine are
 * ignored and may be NULL.
 * Enqueues on `stream` (a cudaStream_t) and returns without synchronising. */
int rvcb200_infer(rvcb200_ctx* ctx, int32_t B, int32_t T,
                  const float* phone, const int64_t* phone_lengths, const int64_t* pitch,
                  const float* nsff0, const int64_t* sid,
                  const float* noise_zp, const float* noise_sine,
                  float* out, float* stats, float* z_p, float* z,
                  void* workspace, int64_t workspace_bytes, int32_t precision,
                  const rvcb200_tap* taps, int32_t n_taps, void* stream);

/* Second half of `net_g.infer(..., rate=r)` (models.py:802-806): reverse flow + source + decoder starting from a given masked
 * prior sample `z_p` [B][T][inter] (channels-last, the last int(T_full * r) frames of what rvcb200_infer returned), with
 * `lengths` / `nsff0` / `noise_sine` already cut to that tail.  Outputs `out` [B][T*upp], optional `z` [B][T][inter]. */
int rvcb200_infer_tail(rvcb200_ctx* ctx, int32_t B, int32_t T, const float* z_p, const int64_t* lengths, const float* nsff0,
                       const int64_t* sid, const float* noise_sine, float* out, float* z, void* workspace,
                       int64_t workspace_bytes, int32_t precision, void* stream);

/* Per-class device timing of the launches inside rvcb200_infer (CUDA events on the caller's stream,
 * accumulated until the next enable): class 0 = decoder resblock convolutions, 1 = attention,
 * 2 = NSF sine source, 3 = bandwidth-bound glue (LayerNorm, prior sample, source injection, conv_post,
 * layout conversion), 4 = decoder conv_pre + transposed-conv ladder, 5 = flow contractions,
 * 6 = text-encoder contractions (emb, qkv, o, FFN, proj), 7 = unused.  `collect` synchronises on the recorded events; ms/count have
 * RVCB200_PROF_CLASSES entries. */
#define RVCB200_PROF_CLASSES 8
int rvcb200_profile_enable(rvcb200_ctx* ctx, int32_t on);
int rvcb200_profile_collect(rvcb200_ctx* ctx, double* ms, int64_t* count);
/* Class (0..RVCB200_PROF_CLASSES-1), number of kernels and CUDA-event time of every timed scope recorded since `enable`, in
 * launch order (a scope is one launcher call; a few launchers enqueue several kernels): lets a profiler's per-launch
 * list (ncu) be joined with the classes above.  Call BEFORE `collect` (which resets the record); synchronises on the
 * events.  Returns the number of scopes recorded (may exceed `cap`; at most `cap` entries are written), < 0 on error.
 * `nkern` and `ms` may be NULL. */
int64_t rvcb200_profile_launches(rvcb200_ctx* ctx, int32_t* cls, int32_t* nkern, float* ms, int64_t cap);

/* Number of kernel launches the last `rvcb200_infer` enqueued (bench.py's gpu_launches). */
int64_t rvcb200_last_launch_count(const rvcb200_ctx* ctx);
const char* rvcb200_last_error(const rvcb200_ctx* ctx);
int32_t rvcb200_abi_version(void);
/* sizeof() of the structs that cross this boundary, as the library was compiled (0: rvcb200_config, 1: rvcb200_tap,
 * 2: rvcb200_conv_desc, 3: rvcb200_tc_conv_desc; -1 otherwise): a binding checks its own mirror against it. */
int64_t rvcb200_sizeof(int32_t which);

/* ---- op-level entry points (unit tests and micro-benchmarks; same kernels as infer) ---- */

/* Channels-last 1-D convolution / phase-decomposed transposed convolution, fp32 CUDA cores.
 * y[b][j*out_stride+g][co] = epilogue( bias[co] + sum_{tap,ci} act(x[b][j+g_off[g]+tap*dil][ci]) * w[g][tap][ci][co] ).
 * Replaces F.conv1d / F.conv_transpose1d call sites of modules.py:295-308, models.py:545-563. */
typedef struct rvcb200_conv_desc {
  const float* x; int64_t x_bstride; int32_t ldx; int32_t L_in; const int32_t* in_len; float in_slope;
  const float* w; const float* bias; int32_t Cin, Cout, ntaps, dil; int32_t G; int32_t g_off[16];
  int32_t Lj; int32_t out_stride;
  float* y; int64_t y_bstride; int32_t ldy;
  const float* cond; int32_t cond_bstride;
  const float* gather; const int64_t* gidx; int64_t gidx_bstride;
  float alpha; int32_t gate;
  int32_t mask_pre, mask_post; const int32_t* out_len;
  const float* res; int64_t res_bstride; int32_t ldr; int32_t res_mode;
  float out_slope; int32_t relu;
  int32_t accum; float div;
} rvcb200_conv_desc;
int rvcb200_op_conv_f32(const rvcb200_conv_desc* d, int32_t B, void* stream);

/* tcgen05/TMEM convolution (csrc/conv_tc.cu).  MMA operands: 16-bit channels-last activations
 * x16 [B][L_in][Cin] and packed weights w16 [G][C_out/N][taps][ceil(Cin/64)][N][64] (K zero-padded),
 * both staged by TMA into SWIZZLE_128B shared memory.  fp32 side (residual res32, output y32):
 * planar-vector [B][C/4][Lp_out][4] with `padf` rows in front; 16-bit output y16: channels-last
 * [B][Lj*out_stride][Cout_total] holding lrelu_{out_slope}(result).  a_mode 0 = one activation box per
 * k-block + per-tap descriptor offsets, 1 = one TMA box per (k-block, tap), 2 (2-D kernels, tap_w > 0) = one box per
 * (k-block, kernel row) whose tap_w taps are descriptor offsets. */
typedef struct rvcb200_tc_conv_desc {
  const void* x16; int32_t L_in; int32_t padf;
  const void* w16; const float* bias;
  int32_t Cin, ntaps, dil, G; int32_t g_off[16];
  int32_t N, Cout_total, tmem_cols;
  int32_t Lj, out_stride, Lp_out;
  float* y32; void* y16; const float* res32;
  const float* cond; int32_t cond_bstride;
  int32_t accum; float div; float out_slope;
  int32_t in_bf16, out_bf16;   /* operand format of x16/w16 and storage format of y16: 0 = fp16, 1 = bf16 */
  int32_t a_mode;
  int32_t batch, na_stages, nb_stages, b_stationary; /* filled in by the launcher */
  /* ---- generic epilogue (text encoder / flow); all zero = the lean decoder epilogue ---- */
  int32_t generic;             /* 1: use the fields below */
  int32_t ldx16;               /* row stride (elements) of x16 when it is a channel slice (0 = Cin) */
  int32_t f32_cl;              /* 1: y32 / res32 are channels-last with row strides ldy32 / ldr32 (floats) */
  int32_t ldy32, ldr32, ldy16; /* ldy16: row stride (elements) of y16 (0 = Cout_total, or Cout_total/2 with gate) */
  const float* gather; const int64_t* gidx; int64_t gidx_bstride;  /* += gather[gidx[b][row]][co] */
  float alpha;                 /* scale after bias/cond/gather */
  float pre_slope;             /* leaky slope applied to the value itself (1 = none) */
  int32_t relu, gate;          /* gate: interleaved (tanh, sigmoid) column pairs -> C_out/2 outputs */
  int32_t res_mode;            /* 1: v + res, 2: res - v */
  int32_t mask_pre, mask_post, mask16; const int32_t* out_len;    /* rows >= out_len[b] -> 0 */
  int32_t dbg_alt;             /* timing experiment only (wrong results): alternate accumulator regions */
  /* ---- fp16 activation stream of the decoder (lean epilogue) ---- */
  const void* res16;           /* residual, fp16 channels-last [B][Lj*out_stride][Cout_total] (exclusive with res32) */
  float res_neg_scale;         /* v += (r > 0 ? r : r * res_neg_scale); 0 or 1 = plain add.  The decoder keeps ONE fp16 copy
                                * of the stream, lrelu_{0.1}(x) -- the MMA operand of the next convolution -- and recovers the
                                * residual x from it with res_neg_scale = 10 (same relative precision as storing x itself) */
  int32_t a_fp16;              /* reserved, must be 0 (fp16 x bf16 mixed-format MMA: tcgen05 kind::f16 raises an illegal
                                * instruction on sm_100a) */
  int32_t acc_f16;             /* 1: y32 (output and `accum` input) is planar-vector fp16 [B][Cout/8][Lp_out][8] */
  int32_t tma_out;             /* filled in by the launcher: y16 leaves through swizzled staging boxes + TMA stores */
  /* ---- decoder tail on the specialised kernel (rvcb200_op_rbconv_tc only) ---- */
  float* tanh_out;             /* non-null: the ONLY output is tanh_out[b][row] = tanh(v[0]), fp32 [B][Lj] -- conv_post
                                * (/root/reference/lib/infer_pack/models.py:562-563) run as a C -> C convolution whose output
                                * channels 1.. are zero; y16 / y32 / res16 must be null */
  int32_t acc_nostore;         /* 1: y32 is read (accum) but not written back; only y16 leaves (the last pair of the last
                                * stage, whose branch sum is consumed once, by conv_post, as y16 = lrelu_{0.01}(.)) */
  /* Source injection x + noise_convs[i](har) (models.py:552-553) inside the epilogue of a stride-u transposed conv run
   * as a dense convolution (output columns = u phases x inj_cn channels, output row j = time rows j*u .. j*u+u-1):
   * v[ph*inj_cn + c] += inj_b[c] + sum_k har[b][(j*u + ph) * inj_s - inj_pad + k] * inj_w[k][c].  inj_k <= 4. */
  const float* inj_har; const float* inj_w; const float* inj_b;
  int32_t inj_k, inj_s, inj_pad, inj_cn; int64_t inj_Lhar;
  int32_t gelu;                /* generic epilogue: exact (erf) GELU right after bias / cond / gather / alpha, before the
                                * residual (the HuBERT front end: conv stack, positional conv, feed-forward) */
  /* 2-D kernels over an image stored row-major as lines of (W + 1) pixels, the last one a zero pad pixel (RMVPE's DeepUnet,
   * /root/reference/lib/rmvpe.py:232-267): tap t reads row offset (t / tap_w) * dil2 + (t % tap_w) * dil (tap_w = 0: 1-D,
   * t * dil).  Rows before 0 / past L_in are zero-filled by the tensor map, the pad pixel supplies the left / right border.
   * pad_period > 0 (generic epilogue): with mask_post, output rows whose (row % pad_period) >= pad_valid are written as 0. */
  int32_t tap_w, dil2, pad_period, pad_valid;
  int32_t b_group;             /* filled in by the launcher: weight tiles per ring stage (non-resident weights) */
  int32_t a_nt_stride;         /* grouped convolution (generic, G = 1): N tile nt reads input channels [nt * a_nt_stride, + Cin) of
                                * x16 (row stride ldx16); 0 = every N tile reads channels [0, Cin) */
  int32_t reserved1;           /* set by the launcher: 1 = pass-by-pass generic epilogue only (RVCB200_LEAN_EPI=0) */
} rvcb200_tc_conv_desc;
int rvcb200_op_conv_tc(const rvcb200_tc_conv_desc* d, int32_t B, void* stream);

/* Same contract, compile-time specialised kernel for the decoder ResBlock shapes (csrc/rbconv_tc.cu): Cin = Cout = N in
 * {32, 64, 128, 256}, ntaps in {3, 7, 11}, dil in {1, 3, 5}, "same" padding, G = 1, no cond, lean epilogue.  Returns
 * RVCB200_ERR_ARG for any other shape (the engine then uses rvcb200_op_conv_tc's kernel). */
int rvcb200_op_rbconv_tc(const rvcb200_tc_conv_desc* d, int32_t B, void* stream);

/* One ResBlock1 pair x' = x + c2(lrelu(c1(lrelu(x)))) (/root/reference/lib/infer_pack/modules.py:295-308) as ONE kernel
 * (csrc/rbpair_tc.cu): d1 / d2 are the descriptors the two rvcb200_op_rbconv_tc launches would take (d2->x16 == d1->y16,
 * d2->res16 == d1->x16, d2->y16 != d1->x16); h = lrelu(c1) stays in shared memory, so d1->y16 is NOT written.  Results
 * are bit-identical to the two launches.  Covers Cin in {32, 64}, ntaps in {3, 7}; RVCB200_ERR_ARG otherwise. */
int rvcb200_op_rbpair_tc(const rvcb200_tc_conv_desc* d1, const rvcb200_tc_conv_desc* d2, int32_t B, void* stream);

/* NSF harmonic source (SineGen + SourceModuleHnNSF, models.py:361-411,455-467):
 * f0 [B][T] -> har [B][T*upp]; scratch >= rvcb200_op_sine_scratch_bytes(B,T,upp). */
int64_t rvcb200_op_sine_scratch_bytes(int32_t B, int32_t T, int32_t upp);
int rvcb200_op_sine_source(const float* f0, const float* noise, float* har, int32_t B, int32_t T,
                           int32_t upp, int32_t sr, float lin_w, float lin_b, void* scratch, void* stream);

/* Windowed relative-position multi-head attention (attentions.py:212-270), fp32.
 * qkv [B][T][3*H] (q|k|v, head h at channels h*dk), out [B][T][H]. */
int rvcb200_op_attention_f32(const float* qkv, const float* rel_k, const float* rel_v, const int32_t* len,
                             float* out, int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t window,
                             void* stream);

/* tcgen05 attention (csrc/attention_tc.cu): qkv16 [B][T][3*heads*128] fp16 (q|k|v, 128 channels per head = dk + zero
 * pad, q pre-scaled by 1/sqrt(dk)), vt: unused since V is read in place as an MN-major operand (may be NULL), ek16 [32][128], evt16 [128][64] fp16
 * relative tables, out [B][T][heads*dk] fp16. */
int rvcb200_op_attention_tc(const void* qkv16, void* vt, const void* ek16, const void* evt16, const int32_t* len, void* out,
                            int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t window, void* stream);

/* Row LayerNorm over C contiguous channels (modules.py:25-28). */
int rvcb200_op_layernorm(const float* x, const float* gamma, const float* beta, float* y, int64_t rows,
                         int32_t C, float eps, void* stream);

/* ---- segmented-driver pre/post steps (csrc/pipeline_kernels.cu); replace the torch/numpy glue of VC.vc and the
 * tail of VC.pipeline so a whole song is converted without a host round trip per segment. ---- */

/* out[T][C] fp32 = x2 nearest interpolation of feats[F][C] (dtype 0 = fp32, 1 = fp16), optionally blended with
 * feats0 by the "protect" weight p = (pitchf[t] < 1 ? protect : 1): out = f*p + f0*(1-p)
 * (/root/reference/vc_infer_pipeline.py:77-95; T <= 2F). */
int rvcb200_op_prepare_feats(const void* feats, const void* feats0, int32_t dtype, const float* pitchf, float* out, int32_t F,
                             int32_t T, int32_t C, float protect, int32_t use_protect, void* stream);

/* *out = max(*out, max|x[0..n)|) on the device (reset != 0 zeroes *out first); x 16-byte aligned
 * (vc_infer_pipeline.py:188 `np.abs(audio_opt).max()`). */
int rvcb200_op_absmax(const float* x, int64_t n, float* out, int32_t reset, void* stream);

/* out[i] = (int16) trunc(x[i] * 32768 / (*absmax / 0.99)) in float32 arithmetic (vc_infer_pipeline.py:188-189,
 * NumPy >= 2 promotion). */
int rvcb200_op_to_int16(const float* x, int64_t n, const float* absmax, int16_t* out, void* stream);

/* Volume-envelope mix `change_rms` (/root/reference/lib/model_utils.py:39, called at vc_infer_pipeline.py:183):
 * librosa.feature.rms(frame_length = 2 * hop, hop) is built from half-block sums, half-block b = samples [b * hop, (b + 1) * hop)
 * of the song, so each segment's output contributes to the envelope on its own.  The three entries below return 1 on a bad
 * argument. */

/* Half-block power of one piece x[len] of a longer signal, starting at global sample `offset` (x_f64: 0 = float32,
 * 1 = float64): out[k] = sum of float32(x)^2 over the piece's samples in half-block offset / hop + k, k up to
 * (offset + len - 1) / hop - offset / hop.  Each square is rounded to float32 (numpy's `np.power(x, 2, dtype=np.float32)`),
 * the sum is accumulated in double in a fixed order that depends only on the samples' positions within their half-block. */
int rvcb200_op_rms_halfblock(const void* x, int32_t x_f64, int64_t len, int64_t offset, int32_t hop, double* out, void* stream);

/* Frame RMS from half-block sums split over `rows` rows (table[rows][n_hb], one row per segment): rows added in ascending
 * order from +0.0, frame f = hb[f - 1] + hb[f] (hb[-1] = 0), rms[f] = sqrt(float32(frame / frame_length)) for f < n_hb,
 * n_hb = 1 + len / hop (librosa's frame count with center=True). */
int rvcb200_op_rms_fold(const double* table, int32_t rows, int64_t n_hb, int32_t frame_length, float* rms, void* stream);

/* In place on samples [offset, offset + len) of an N-sample float32 song: x *= pow(e1, 1 - rate) * pow(max(e2, 1e-6), rate - 1),
 * e1 / e2 = rms1[n1] / rms2[n2] linearly interpolated to N samples with the float32 rounding of torch's CPU
 * F.interpolate(mode="linear", align_corners=False); exponents float32(1 - rate) / float32(rate - 1); the product and the
 * update are each one float32 rounding.  powf may differ from torch's CPU pow by an ulp or two. */
int rvcb200_op_rms_gain(float* x, int64_t len, int64_t offset, int64_t N, const float* rms1, int64_t n1, const float* rms2, int64_t n2,
                        double rate, void* stream);

/* Index blend of VC.vc (/root/reference/vc_infer_pipeline.py:59-75: `index.search(npy, k=1)`, the `1 / score` weight, the
 * `big_npy[ix]` gather and the `index_rate` blend) on the device, for a faiss IndexIVFFlat with METRIC_L2 and nprobe 1
 * (IndexFlatL2 = one list holding every vector in id order).  All distances are fp32 FMA on the CUDA cores; every result is the
 * same bits for every run.  Queries x: [F] rows of d values (x_dtype / feats_dtype 0 = fp32, 1 = fp16, promoted exactly), row
 * stride ldx >= d elements; d % 4 == 0.  The index: centroids fp32 [nlist][d], cnorm fp32 [nlist] = ||centroid||^2,
 * list_offsets int32 [nlist + 1] (CSR, list_offsets[0] = 0), vectors fp32 [ntotal][d] and labels int64 [ntotal] in list order,
 * pos_of_label int32 [ntotal] = position of label i in `vectors`.  The entries below return 1 on a bad argument and never
 * allocate: the caller passes the scratch. */

/* Bytes of scratch rvcb200_op_ivf_scan needs for F queries over nlist lists (-1 on a bad argument). */
int64_t rvcb200_op_ivf_scratch_bytes(int32_t F, int32_t nlist);

/* Coarse step: coarse[f] (uint64 [F]) = key(dist) << 32 | l for the l minimising ||c_l||^2 - 2 x_f . c_l, the lowest l on an
 * exact tie (key: the order-preserving unsigned image of the fp32 value). */
int rvcb200_op_ivf_assign(const void* x, int32_t x_dtype, int64_t ldx, int32_t F, int32_t d, const float* centroids, const float* cnorm,
                          int32_t nlist, uint64_t* coarse, void* stream);

/* Fine step: bucket the queries by the list rvcb200_op_ivf_assign chose, scan each list exhaustively with direct-form
 * sum_k (x - v)^2, and write score[f] (fp32) = the smallest distance and ix[f] (int64) = its label, the earliest list position
 * on an exact tie (faiss's heap replaces on a strict <).  A query whose list is empty gets score +inf, ix -1. */
int rvcb200_op_ivf_scan(const void* x, int32_t x_dtype, int64_t ldx, int32_t F, int32_t d, const uint64_t* coarse, int32_t nlist,
                        const int32_t* list_offsets, const float* vectors, const int64_t* labels, void* scratch, int64_t scratch_bytes,
                        float* score, int64_t* ix, void* stream);

/* Blend: out[f][:] (row-contiguous [F][d]) = round(round(g * r) + round(s * feats[f][:])), r = float(index_rate),
 * s = float(1.0 - index_rate) (the difference taken in double), g = big_npy[ix[f]] * (w / w) with w = float32(1 / score[f])^2
 * (1.0, or NaN when score is 0, +inf, or w over- / underflows), ix -1 = label ntotal - 1 (numpy's indexing), big_npy[i] =
 * vectors[pos_of_label[i]].  With is_half, g and g * r are rounded to fp16 (`astype("float16")`); s * f is rounded to the
 * dtype of feats; out is fp16 when is_half and feats is fp16 (torch's promotion), fp32 otherwise. */
int rvcb200_op_index_blend(const void* feats, int32_t feats_dtype, int64_t ldf, int32_t F, int32_t d, const float* score,
                           const int64_t* ix, const float* vectors, const int32_t* pos_of_label, int64_t ntotal, int32_t is_half,
                           double index_rate, void* out, void* stream);

/* Output resampling (`resample_sr`, /root/reference/vc_infer_pipeline.py:185-186) as a polyphase FIR:
 * y[j] = sum_{k < tpp} tab[r][k] * x[m0 - k], t = j * down + half_len, r = t % up, m0 = t / up, k ascending, one fp32 FMA each
 * from +0.0, so an output's bits depend only on j and the input values (any split of the output range gives the same bits).
 * tab: device [up][stride] float32, 16-byte aligned, stride = tpp rounded up to 4, row r = up * h[r + k * up]
 * (comfy_rvc_b200/resample.py `phase_table`).  Computes outputs [out_lo, out_hi) into out[out_hi - out_lo].  The input is the
 * virtual concatenation [left[n_left] | piece[n_piece] | right[n_right]] whose piece starts at global sample piece_off of an
 * n_song-sample song; samples outside the song read as zero, and every sample inside the song that the outputs reach must be
 * in the concatenation.  Returns 1 on a bad argument or an input window that does not cover the outputs. */
int rvcb200_op_resample_poly(const float* tab, int32_t up, int32_t down, int32_t tpp, int64_t half_len, const float* left, int64_t n_left,
                             const float* piece, int64_t n_piece, const float* right, int64_t n_right, int64_t piece_off, int64_t n_song,
                             int64_t out_lo, int64_t out_hi, float* out, void* stream);

/* Measurement aid: while `buf` (device, 16 x grid uint64) is set, every CTA of rvcb200_op_conv_tc launches records globaltimer
 * at 8 fixed points (start, prologue done, producer released, first slab landed, MMAs issued, accumulator complete,
 * epilogue done, exit); NULL switches it off.  tools/trace_generic.py. */
int rvcb200_debug_trace_conv_tc(void* buf);

/* ---- HuBERT / ContentVec front end (SURVEY.md §8f rank 3; host orchestration in comfy_rvc_b200/hubert.py) ----
 * Replaces transformers.HubertModel as reached from /root/reference/lib/infer_pack/loaders.py:52-61.  Every contraction
 * of the model runs through rvcb200_op_conv_tc (generic epilogue, `gelu`) and rvcb200_op_attention_tc; these two entries
 * are what is left: */

/* First feature-encoder layer: y16[b][t][c] = GELU(GroupNorm_c(sum_k w[c][k] x[b][t*S + k])) as fp16 channels-last,
 * t < L0 = (n - K) / S + 1; per-channel statistics over time, biased variance, affine gn_w / gn_b.  stats: scratch of
 * B * 2 * C doubles; y_bstride: elements between batch items of y16.  K <= 16.  Bitwise deterministic: the statistics are
 * summed in a fixed order (per-block partial sums are staged in y16 before the outputs overwrite them). */
int rvcb200_op_hubert_conv0(const float* x, const float* w, const float* gn_w, const float* gn_b, double* stats, void* y16,
                            int32_t B, int64_t n, int32_t C, int32_t K, int32_t S, float eps, int64_t y_bstride, void* stream);

/* LayerNorm over the last (contiguous) axis, C <= 1024: y (fp32) and, if y16 != NULL, an fp16 copy (the MMA operand of
 * the next contraction). */
int rvcb200_op_layernorm16(const float* x, const float* gamma, const float* beta, float* y, void* y16, int64_t rows, int32_t C,
                           float eps, void* stream);

/* Device form of the quiet-point search below (same sums, same order, one thread per candidate): block k of `n_blocks`
 * writes the first minimum of its contiguous share of [lo, hi) to best_v[k] / best_j[k] (absolute index, -1 if the share
 * is empty); the caller takes the first minimum over blocks in ascending order.  audio_pad: device float64. */
int rvcb200_op_quiet_point(const double* audio_pad, int64_t lo, int64_t hi, int32_t window, double* best_v, int64_t* best_j,
                           int32_t n_blocks, void* stream);

/* ---- RMVPE f0 estimator (SURVEY.md §8f rank 4; host orchestration in comfy_rvc_b200/rmvpe.py) ----
 * Replaces the torch modules of /root/reference/lib/rmvpe.py as reached from pitch_extraction.py:191-201.  The DeepUnet's
 * convolutions, the GRU input projection and the output Linear run through rvcb200_op_conv_tc (2-D taps); these entries are
 * what is left.  Images are fp16 channels-last, stored as lines of `pitch` >= W + 1 pixels; pixels [W, pitch) of a line are zero
 * (they are the left / right border of the 3 x 3 convolutions).  On the wide levels (C < 64) the host views `pack` = 64 / C pixels
 * as ONE 64-channel row (pitch = W + pack) and runs the convolutions with block-Toeplitz weights: 4x / 2x fewer TMA box rows. */

/* `MelSpectrogram.forward` (rmvpe.py:489-556; n_fft 1024, hop 160, 128 HTK mel filters 30-8000 Hz, log(clamp 1e-5)) of
 * audio[n] (16 kHz, n > 512), n_frames = n / 160 + 1.  window[1024]: periodic Hann; twiddle[512][2]: (cos, -sin)(2 pi i / 1024);
 * mel_basis[128][513]; mel_range[128][2]: first / one-past-last non-zero bin of each filter.  Outputs (either may be NULL):
 * mel_out fp32 [128][n_frames]; img16 fp16 [frames_out][img_pitch][img_c], channel 0 = mel * bn_scale + bn_shift (`Encoder.bn`,
 * rmvpe.py:299), frames n_frames.. = the reflect padding of `mel2hidden` (rmvpe.py:594-595); img16 must be zero-initialised. */
int rvcb200_op_rmvpe_logmel(const float* audio, int64_t n, const float* window, const float* twiddle, const float* mel_basis,
                            const int32_t* mel_range, float bn_scale, float bn_shift, float* mel_out, void* img16, int32_t n_frames,
                            int32_t frames_out, int32_t img_pitch, int32_t img_c, void* stream);

/* AvgPool2d((2, 2)) (rmvpe.py:318): x32 fp32 [2 H2][p_in][ldx] -> y16 fp16 [H2][p_out][C] (pixels [W2, p_out) zero). */
int rvcb200_op_rmvpe_pool(const float* x32, int32_t ldx, void* y16, int32_t H2, int32_t W2, int32_t C, int32_t p_in, int32_t p_out,
                          void* stream);

/* Scatter behind ConvTranspose2d(3 x 3, stride 2, padding 1, output_padding 1) (rmvpe.py:355-366) computed as a 2 x 2-tap GEMM
 * with (phase, channel) columns: g16 fp16 [H][p_in][4][Co] -> output pixel (oy, ox) = (2y + py, 2x + px) at row
 * oy * fp_out + ox / pack of out16 (row stride ld), columns (ox % pack) * Co .. + Co (the up-sampled half of the concat buffer). */
int rvcb200_op_rmvpe_shuffle(const void* g16, void* out16, int32_t H, int32_t W, int32_t Co, int32_t ld, int32_t p_in, int32_t fp_out,
                             int32_t pack, void* stream);

/* `x.transpose(1, 2).flatten(-2)` (rmvpe.py:468): y32 fp32 [T][pitch][ldc] (channels 0..2) -> x16 fp16 [T][3 W], column c W + w. */
int rvcb200_op_rmvpe_gru_pack(const float* y32, int32_t ldc, void* x16, int64_t T, int32_t W, int32_t pitch, void* stream);

/* Recurrence of nn.GRU(384, 256, bidirectional=True) (rmvpe.py:217-229): gi fp32 [T][2][3][256] = W_ih x + b_ih (gates r|z|n),
 * w_hh fp32 [2][768][256], b_hh fp32 [2][768] -> out16 fp16 [T][512] (forward | reverse), out32 the same in fp32 or NULL. */
int rvcb200_op_rmvpe_gru(const float* gi, const float* w_hh, const float* b_hh, void* out16, float* out32, int32_t T, void* stream);

/* Sigmoid (from_hidden = 0: `in` = logits [T][ld], `hidden` [T][360] receives the salience, may be NULL) and
 * `to_local_average_cents` + `decode` (rmvpe.py:610-615, 658-684) in float64 -> f0 [T] (Hz, 0 = unvoiced) and / or
 * cents [T] (the value `to_local_average_cents` returns); at least one of the two non-NULL. */
int rvcb200_op_rmvpe_decode(const float* in, int32_t ld, int32_t from_hidden, float* hidden, double* f0, double* cents, int32_t T,
                            float thred, void* stream);

/* `mel2hidden` called with a caller-supplied log-mel: mel fp32 [128][n_frames] -> the img16 of rvcb200_op_rmvpe_logmel. */
int rvcb200_op_rmvpe_mel_to_img(const float* mel, void* img16, int32_t n_frames, int32_t frames_out, float bn_scale, float bn_shift,
                                int32_t img_pitch, int32_t img_c, void* stream);

/* ---- CREPE f0 estimator (torchcrepe's model, framing and decoders; host orchestration in comfy_rvc_b200/crepe.py) ----
 * conv1..conv6 and the classifier run through rvcb200_op_conv_tc; these entries are what is left. */

/* Frames first .. first + count - 1 of 16 kHz audio[n] at `hop` (pad != 0: the audio is zero-padded by 512 on each side),
 * each mean-subtracted and divided by max(1e-10, unbiased std), written as conv1's operand: fp16 [count][368][64] with
 * row t, channel c = frame[4 t + c - 254] (0 outside the frame).  conv1 is then 8 taps at dilation 16 over these rows. */
int rvcb200_op_crepe_frames(const float* audio, int64_t n, int64_t first, int64_t count, int32_t hop, int32_t pad, void* frames16,
                            void* stream);

/* Eval-mode BatchNorm (y = x * scale + shift per channel) then max_pool (2, 1): x16 fp16 rows [frames * p_in][C], frame f's
 * L rows from row f * p_in + in_off -> y16 fp16 [frames][p_out][C], rows out_off .. out_off + L / 2 - 1 hold the pooled
 * values, every other row is written as 0 (the zero padding of the next convolution).  C % 8 == 0, L even. */
int rvcb200_op_crepe_bn_pool(const void* x16, const float* scale, const float* shift, void* y16, int64_t frames, int32_t C, int32_t L,
                             int32_t p_in, int32_t in_off, int32_t p_out, int32_t out_off, void* stream);

/* torchcrepe's postprocess for T frames: salience s = sigmoid(in) (from_salience != 0: in already is s) [T][ld >= 360], bins
 * outside [lo, hi) masked; mode 0 = argmax, 1 = weighted_argmax (wcents[360]: the dithered cents of each bin), 2 = Viterbi
 * over chunks of `chunk` frames (log_trans [360][23]: log(transition + tiny) of bin k to bin k + d - 11, log_out: the same outside
 * the band, log_init: log(1 / 360 + tiny); the observations log(softmax + tiny) in float64).  Outputs: bins int32 [T],
 * f0 float64 [T] (Hz; modes 0 / 2: from 20 bin + 1997.379... + dither[t] cents), periodicity fp32 [T] (the salience at the
 * bin, may be NULL).  salience fp32 [T][360] may be NULL except in mode 2; mode 2 also needs logp float64 [T][360],
 * ptr uint16 [T][360] and score float64 [chunks] (the log-probability of each chunk's best path). */
int rvcb200_op_crepe_decode(const float* in, int32_t ld, int32_t from_salience, int64_t T, int32_t chunk, int32_t lo, int32_t hi,
                            int32_t mode, const double* dither, const double* wcents, const double* log_trans, double log_out,
                            double log_init, float* salience, double* logp, uint16_t* ptr, int32_t* bins, double* f0, float* periodicity,
                            double* score, void* stream);

/* ---- host (CPU) side of the song-level driver (csrc/host_plan.cu) ---- */

/* Quiet-point search of /root/reference/vc_infer_pipeline.py:127-135: the first j in [lo, hi) (returned relative to lo)
 * that minimises |audio_pad[j] + audio_pad[j+1] + ... + audio_pad[j+window-1]|, each sum accumulated left to right in
 * double from +0.0 like the reference's `audio_sum += audio_pad[i : i - window]` loop (bit-identical sums).  audio_pad must
 * hold hi + window - 1 samples.  n_threads <= 0: all hardware threads.  -1 on bad arguments or if every sum is NaN. */
int64_t rvcb200_host_quiet_point(const double* audio_pad, int64_t lo, int64_t hi, int32_t window, int32_t n_threads);

/* Host (CPU) restatement of `audio = signal.filtfilt(bh, ah, audio)` (/root/reference/vc_infer_pipeline.py:122, scipy
 * defaults: odd padding of 3 * (order + 1) samples, transposed direct form II in double) followed by the reflect padding of
 * :141, bit-identical to scipy / numpy (sequential: see csrc/host_plan.cu for why it cannot be chunked).  b, a: order + 1
 * coefficients; zi: scipy.signal.lfilter_zi(b, a) (order values, contiguous); out: n + 2 * pad doubles (may be pinned
 * memory); scratch: n + 6 * (order + 1) doubles.  Returns 0, or 1 on a bad argument. */
int rvcb200_host_filtfilt_pad(const double* x, int64_t n, const double* b, const double* a, const double* zi, int32_t order,
                              int64_t pad, double* out, double* scratch);

#ifdef __cplusplus
}
#endif
#endif /* RVCB200_H */
