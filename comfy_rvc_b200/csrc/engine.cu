// Context, weight registry, workspace planning and the infer() orchestrator behind the C ABI
// (include/rvcb200.h).  Mirrors the call order of the reference
// `SynthesizerTrnMs{256,768}NSFsid.infer` (/root/reference/lib/infer_pack/models.py:682-693,
// :798-809): emb_g -> enc_p -> prior sample -> reverse flow -> NSF source -> GeneratorNSF.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "conv_tc.cuh"

using namespace rvc;

struct TensorRef {
  const void* ptr = nullptr;
  long long numel = 0;
  int dtype = 0;
};

struct rvcb200_ctx {
  rvcb200_config cfg;
  std::unordered_map<std::string, TensorRef> tensors;
  std::unordered_map<std::string, float> scalars;
  bool finalized = false;
  char err[512];
  long long last_launches = 0;
  // derived
  int upp = 1;
  int n_cond = 0;  // rows of the stacked conditioning matrix
  // optional per-class CUDA-event timing of the launches inside infer (bench.py roofline)
  bool prof = false;
  std::vector<cudaEvent_t> ev;   // pairs (start, stop)
  std::vector<int> ev_cls;
  std::vector<int> ev_nk;        // kernels launched inside the scope (a launcher may enqueue several)
  size_t ev_used = 0;
  double cls_ms[RVCB200_PROF_CLASSES] = {0};
  long long cls_n[RVCB200_PROF_CLASSES] = {0};
};

namespace {

int fail(rvcb200_ctx* c, int code, const char* fmt, const char* a = "", long long b = 0) {
  if (c) snprintf(c->err, sizeof(c->err), fmt, a, b);
  return code;
}

const float* T32(rvcb200_ctx* c, const std::string& name, long long expect, bool* ok) {
  auto it = c->tensors.find(name);
  if (it == c->tensors.end()) {
    if (*ok) snprintf(c->err, sizeof(c->err), "missing tensor '%s'", name.c_str());
    *ok = false;
    return nullptr;
  }
  if (it->second.dtype != 0 || (expect > 0 && it->second.numel != expect)) {
    if (*ok)
      snprintf(c->err, sizeof(c->err), "tensor '%s': numel %lld (expected %lld) dtype %d", name.c_str(),
               it->second.numel, expect, it->second.dtype);
    *ok = false;
    return nullptr;
  }
  return reinterpret_cast<const float*>(it->second.ptr);
}

const void* T16(rvcb200_ctx* c, const std::string& name, long long expect, int dtype, bool* ok) {
  auto it = c->tensors.find(name);
  if (it == c->tensors.end() || it->second.dtype != dtype || (expect > 0 && it->second.numel != expect)) {
    if (*ok)
      snprintf(c->err, sizeof(c->err), "missing/mismatched 16-bit tensor '%s' (dtype %d, numel %lld)", name.c_str(), dtype,
               expect);
    *ok = false;
    return nullptr;
  }
  return it->second.ptr;
}

std::string S(const char* fmt, int a = 0, int b = 0, int c = 0) {
  char buf[128];
  snprintf(buf, sizeof(buf), fmt, a, b, c);
  return std::string(buf);
}

struct Bump {
  char* base;
  size_t off = 0, cap;
  Bump(void* p, size_t c) : base(reinterpret_cast<char*>(p)), cap(c) {}
  template <typename T>
  T* take(size_t n) {
    size_t bytes = (n * sizeof(T) + 255) & ~(size_t)255;
    T* r = reinterpret_cast<T*>(base ? base + off : nullptr);
    off += bytes;
    return r;
  }
};

struct UpGeom {
  int k, u, pad, ntaps, cin, cout;
  int g_off[16];
};

UpGeom up_geom(const rvcb200_config& cfg, int i) {
  UpGeom g;
  g.k = cfg.up_kernels[i];
  g.u = cfg.up_rates[i];
  g.pad = (g.k - g.u) / 2;
  g.ntaps = (g.k + g.u - 1) / g.u;
  g.cin = cfg.up_init_channels >> i;
  g.cout = cfg.up_init_channels >> (i + 1);
  for (int p = 0; p < 16; ++p) g.g_off[p] = 0;
  for (int p = 0; p < g.u; ++p) g.g_off[p] = (p + g.pad) / g.u - (g.ntaps - 1);
  return g;
}

// Stage i's transposed conv as one ordinary 3-tap convolution C_in -> u*C_out = C_in on the specialised resblock kernel
// (weights.py ups_is_dense / pack_conv_transpose_dense): all phases side by side in N, output rows contiguous.
bool ups_dense(const rvcb200_config& cfg, int i) {
  const int u = cfg.up_rates[i], k = cfg.up_kernels[i], cin = cfg.up_init_channels >> i;
  return u == 2 && k == 2 * u && (cin == 32 || cin == 64 || cin == 128 || cin == 256);
}

void noise_geom(const rvcb200_config& cfg, int i, int* k, int* s, int* pad) {
  if (i + 1 < cfg.n_ups) {
    int st = 1;
    for (int j = i + 1; j < cfg.n_ups; ++j) st *= cfg.up_rates[j];
    *k = 2 * st; *s = st; *pad = st / 2;
  } else {
    *k = 1; *s = 1; *pad = 0;
  }
}

ConvDesc base_desc() {
  ConvDesc d;
  memset(&d, 0, sizeof(d));
  d.in_slope = 1.f; d.alpha = 1.f; d.out_slope = 1.f; d.div = 1.f;
  d.ntaps = 1; d.dil = 1; d.G = 1; d.out_stride = 1;
  return d;
}

struct Plan {  // workspace carve-up for (B, T)
  int* len32; int* len_head;
  float *cond, *x, *xt, *qkv, *att, *ffh, *stats, *zp, *z, *h, *acts, *skip, *har, *pre;
  void* sine_scratch;
  float* stage[5];
  // tensor-core path: planar-vector buffers
  void* z16; void* pv16[5]; float* pv32[2];
  void *phone16, *x16, *att16, *ffh16, *h16, *acts16, *skip16;   // fp16 MMA operands of enc_p / flow
  void *qkv16, *vt16;                                            // padded q|k|v and V^T for the tcgen05 attention
  size_t bytes;
};

Plan make_plan(const rvcb200_ctx* c, int B, int T, void* ws, int precision = RVCB200_PREC_FP32) {
  const rvcb200_config& cf = c->cfg;
  Plan p;
  Bump bp(ws, 0);
  const size_t BT = (size_t)B * T;
  const int H = cf.hidden_channels, C = cf.inter_channels;
  p.len32 = bp.take<int>(B);
  p.len_head = bp.take<int>(B);
  p.cond = bp.take<float>((size_t)B * c->n_cond);
  p.x = bp.take<float>(BT * H);
  p.xt = bp.take<float>(BT * H);
  p.qkv = bp.take<float>(BT * 3 * H);
  p.att = bp.take<float>(BT * H);
  p.ffh = bp.take<float>(BT * cf.filter_channels);
  p.stats = bp.take<float>(BT * 2 * C);
  p.zp = bp.take<float>(BT * C);
  p.z = bp.take<float>(BT * C);
  p.h = bp.take<float>(BT * H);
  p.acts = bp.take<float>(BT * H);
  p.skip = bp.take<float>(BT * H);
  p.har = bp.take<float>(BT * c->upp);
  p.sine_scratch = bp.take<char>(sine_scratch_bytes(B, T, c->upp));
  p.pre = bp.take<float>(BT * cf.up_init_channels);
  size_t mx = 0;
  long long L = T;
  for (int i = 0; i < cf.n_ups; ++i) {
    L *= cf.up_rates[i];
    size_t s = (size_t)B * L * (cf.up_init_channels >> (i + 1));
    if (s > mx) mx = s;
  }
  if (precision == RVCB200_PREC_FP32) {
    for (int i = 0; i < 5; ++i) p.stage[i] = bp.take<float>(mx);
    p.z16 = nullptr;
    for (int i = 0; i < 5; ++i) p.pv16[i] = nullptr;
    for (int i = 0; i < 2; ++i) p.pv32[i] = nullptr;
  } else {
    for (int i = 0; i < 5; ++i) p.stage[i] = nullptr;
    size_t mxe = (size_t)B * cf.up_init_channels * pv_pitch_rows(T);      // conv_pre output
    long long Ls = T;
    for (int i = 0; i < cf.n_ups; ++i) {
      Ls *= cf.up_rates[i];
      size_t e = (size_t)B * (cf.up_init_channels >> (i + 1)) * pv_pitch_rows(Ls);
      if (e > mxe) mxe = e;
    }
    p.z16 = bp.take<unsigned short>((size_t)B * C * pv_pitch_rows(T));
    p.phone16 = bp.take<unsigned short>(BT * cf.feat_dim);
    p.x16 = bp.take<unsigned short>(BT * H);
    p.att16 = bp.take<unsigned short>(BT * H);
    p.ffh16 = bp.take<unsigned short>(BT * cf.filter_channels);
    p.h16 = bp.take<unsigned short>(BT * H);
    // flow activation buffer [BT][xb + n H]: [x0 | mask | zeros] (xb columns) then every layer's gate output
    p.acts16 = bp.take<unsigned short>(BT * ((size_t)((C / 2 + 1 + 63) / 64 * 64) + (size_t)H * (cf.flow_wn_layers > 0 ? cf.flow_wn_layers : 1)));
    p.skip16 = bp.take<unsigned short>(BT * H);
    p.qkv16 = bp.take<unsigned short>(BT * 3 * cf.n_heads * 128);
    p.vt16 = bp.take<unsigned short>((size_t)B * cf.n_heads * 128 * ((T + 7) & ~7));
    for (int i = 0; i < 5; ++i) p.pv16[i] = bp.take<unsigned short>(mxe);
    for (int i = 0; i < 2; ++i) p.pv32[i] = bp.take<float>(mxe);
  }
  p.bytes = bp.off;
  return p;
}

struct TapSet {
  const rvcb200_tap* taps;
  int n;
  cudaStream_t st;
  const rvcb200_tap* find(const char* name) const {
    for (int i = 0; i < n; ++i)
      if (taps[i].name && strcmp(taps[i].name, name) == 0 && taps[i].dst) return &taps[i];
    return nullptr;
  }
  cudaError_t emit(const char* name, const void* src, size_t bytes) const {
    for (int i = 0; i < n; ++i)
      if (taps[i].name && strcmp(taps[i].name, name) == 0 && taps[i].dst) {
        size_t nb = bytes < taps[i].bytes ? bytes : taps[i].bytes;
        return cudaMemcpyAsync(taps[i].dst, src, nb, cudaMemcpyDeviceToDevice, st);
      }
    return cudaSuccess;
  }
};

#define CK(expr, what)                                                      \
  do {                                                                      \
    cudaError_t _e = (expr);                                                \
    if (_e != cudaSuccess) {                                                \
      snprintf(ctx->err, sizeof(ctx->err), "%s: %s", what, cudaGetErrorString(_e)); \
      return RVCB200_ERR_CUDA;                                              \
    }                                                                       \
  } while (0)

struct ProfScope {  // records an event pair around one launch when profiling is on
  rvcb200_ctx* c;
  cudaStream_t st;
  bool on;
  long long n0 = 0;
  ProfScope(rvcb200_ctx* c_, int cls, cudaStream_t st_) : c(c_), st(st_), on(c_->prof) {
    if (!on) return;
    if (c->ev_used + 2 > c->ev.size()) {
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) { on = false; return; }
      c->ev.push_back(a); c->ev.push_back(b);
    }
    c->ev_cls.resize(c->ev.size() / 2);
    c->ev_nk.resize(c->ev.size() / 2);
    c->ev_cls[c->ev_used / 2] = cls;
    n0 = launch_counter().n;
    cudaEventRecord(c->ev[c->ev_used], st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(c->ev[c->ev_used + 1], st);
    c->ev_nk[c->ev_used / 2] = (int)(launch_counter().n - n0);
    c->ev_used += 2;
  }
};

#define CKC(cls, expr, what)                 \
  do {                                       \
    ProfScope _ps(ctx, cls, st);             \
    CK(expr, what);                          \
  } while (0)

}  // namespace

extern "C" {

int32_t rvcb200_abi_version(void) { return RVCB200_ABI_VERSION; }

int64_t rvcb200_sizeof(int32_t which) {
  switch (which) {
    case 0: return (int64_t)sizeof(rvcb200_config);
    case 1: return (int64_t)sizeof(rvcb200_tap);
    case 2: return (int64_t)sizeof(rvcb200_conv_desc);
    case 3: return (int64_t)sizeof(rvcb200_tc_conv_desc);
    default: return -1;
  }
}

int rvcb200_create(const rvcb200_config* cfg, rvcb200_ctx** out) {
  if (!cfg || !out) return RVCB200_ERR_ARG;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return RVCB200_ERR_NO_DEVICE;
  rvcb200_ctx* c = new rvcb200_ctx();
  c->cfg = *cfg;
  c->err[0] = 0;
  const rvcb200_config& f = c->cfg;
  bool ok = f.n_heads > 0 && f.hidden_channels == f.n_heads * 96 && f.inter_channels == f.hidden_channels &&
            f.inter_channels % 2 == 0 && f.window_size <= 10 && f.n_ups >= 1 && f.n_ups <= RVCB200_MAX_UPS &&
            f.n_res_kernels >= 1 && f.n_res_kernels <= RVCB200_MAX_RESK && (f.resblock_kind == 1 || f.resblock_kind == 2) &&
            f.feat_dim % 8 == 0 && f.filter_channels % 64 == 0 && f.enc_kernel % 2 == 1 && f.flow_kernel % 2 == 1 &&
            f.gin_channels > 0 && f.n_flows % 2 == 0;
  c->upp = 1;
  for (int i = 0; ok && i < f.n_ups; ++i) {
    c->upp *= f.up_rates[i];
    if (f.up_rates[i] > 16 || f.up_rates[i] < 1 || (f.up_kernels[i] - f.up_rates[i]) % 2 != 0 || f.up_kernels[i] < f.up_rates[i])
      ok = false;
    if ((f.up_init_channels >> (i + 1)) % 16 != 0) ok = false;
  }
  for (int j = 0; ok && j < f.n_res_kernels; ++j) {
    if (f.res_kernels[j] % 2 != 1 || f.n_res_dils[j] < 1 || f.n_res_dils[j] > RVCB200_MAX_DIL) ok = false;
    // ResBlock2 has exactly two convs (modules.py:319-339); the fp32 decoder's XB/XT hand-over below relies on it
    if (f.resblock_kind == 2 && f.n_res_dils[j] != 2) ok = false;
    for (int d = 0; ok && d < f.n_res_dils[j]; ++d)
      if ((f.res_kernels[j] - 1) * f.res_dils[j][d] > 50) ok = false;
  }
  if (!ok) {
    delete c;
    return RVCB200_ERR_ARG;
  }
  c->n_cond = f.up_init_channels + f.n_flows * f.flow_wn_layers * 2 * f.hidden_channels;
  *out = c;
  return RVCB200_OK;
}

void rvcb200_destroy(rvcb200_ctx* ctx) {
  if (!ctx) return;
  for (cudaEvent_t e : ctx->ev) cudaEventDestroy(e);
  delete ctx;
}

int rvcb200_profile_enable(rvcb200_ctx* ctx, int32_t on) {
  if (!ctx) return RVCB200_ERR_ARG;
  ctx->prof = on != 0;
  ctx->ev_used = 0;
  for (int i = 0; i < RVCB200_PROF_CLASSES; ++i) { ctx->cls_ms[i] = 0; ctx->cls_n[i] = 0; }
  return RVCB200_OK;
}

int rvcb200_profile_collect(rvcb200_ctx* ctx, double* ms, int64_t* count) {
  if (!ctx || !ms || !count) return RVCB200_ERR_ARG;
  for (size_t i = 0; i + 1 < ctx->ev_used; i += 2) {
    if (cudaEventSynchronize(ctx->ev[i + 1]) != cudaSuccess) return RVCB200_ERR_CUDA;
    float t = 0.f;
    if (cudaEventElapsedTime(&t, ctx->ev[i], ctx->ev[i + 1]) != cudaSuccess) return RVCB200_ERR_CUDA;
    const int cls = ctx->ev_cls[i / 2];
    ctx->cls_ms[cls] += t;
    ctx->cls_n[cls] += 1;
  }
  ctx->ev_used = 0;
  for (int i = 0; i < RVCB200_PROF_CLASSES; ++i) { ms[i] = ctx->cls_ms[i]; count[i] = ctx->cls_n[i]; }
  return RVCB200_OK;
}

int64_t rvcb200_profile_launches(rvcb200_ctx* ctx, int32_t* cls, int32_t* nkern, float* ms, int64_t cap) {
  if (!ctx || !cls || cap < 0) return -1;
  const int64_t n = (int64_t)(ctx->ev_used / 2);
  for (int64_t i = 0; i < n && i < cap; ++i) {
    cls[i] = ctx->ev_cls[i];
    if (nkern) nkern[i] = ctx->ev_nk[i];
    if (ms) {
      if (cudaEventSynchronize(ctx->ev[2 * i + 1]) != cudaSuccess) return -1;
      if (cudaEventElapsedTime(&ms[i], ctx->ev[2 * i], ctx->ev[2 * i + 1]) != cudaSuccess) return -1;
    }
  }
  return n;
}

int rvcb200_set_tensor(rvcb200_ctx* ctx, const char* name, const void* dev_ptr, int64_t numel, int32_t dtype) {
  if (!ctx || !name || !dev_ptr || numel <= 0) return RVCB200_ERR_ARG;
  TensorRef t;
  t.ptr = dev_ptr; t.numel = numel; t.dtype = dtype;
  ctx->tensors[name] = t;
  ctx->finalized = false;
  return RVCB200_OK;
}

int rvcb200_set_scalar(rvcb200_ctx* ctx, const char* name, float value) {
  if (!ctx || !name) return RVCB200_ERR_ARG;
  ctx->scalars[name] = value;
  return RVCB200_OK;
}

int rvcb200_finalize(rvcb200_ctx* ctx) {
  if (!ctx) return RVCB200_ERR_ARG;
  const rvcb200_config& f = ctx->cfg;
  const int H = f.hidden_channels, C = f.inter_channels, F = f.filter_channels, half = C / 2;
  bool ok = true;
  T32(ctx, "emb_g", (long long)f.n_speakers * f.gin_channels, &ok);
  T32(ctx, "cond.w", (long long)ctx->n_cond * f.gin_channels, &ok);
  T32(ctx, "cond.b", ctx->n_cond, &ok);
  T32(ctx, "enc.emb.w", (long long)f.feat_dim * H, &ok);
  T32(ctx, "enc.emb.b", H, &ok);
  const bool f0 = f.no_f0 == 0;
  if (f0) T32(ctx, "enc.emb_pitch", 256LL * H, &ok);
  const int nrel = 2 * f.window_size + 1;
  for (int l = 0; l < f.n_layers; ++l) {
    T32(ctx, S("enc.%d.qkv.w", l), (long long)H * 3 * H, &ok);
    T32(ctx, S("enc.%d.qkv.b", l), 3 * H, &ok);
    T32(ctx, S("enc.%d.rel_k", l), (long long)nrel * 96, &ok);
    T32(ctx, S("enc.%d.rel_v", l), (long long)nrel * 96, &ok);
    T32(ctx, S("enc.%d.o.w", l), (long long)H * H, &ok);
    T32(ctx, S("enc.%d.o.b", l), H, &ok);
    T32(ctx, S("enc.%d.ln1.g", l), H, &ok);
    T32(ctx, S("enc.%d.ln1.b", l), H, &ok);
    T32(ctx, S("enc.%d.ffn1.w", l), (long long)f.enc_kernel * H * F, &ok);
    T32(ctx, S("enc.%d.ffn1.b", l), F, &ok);
    T32(ctx, S("enc.%d.ffn2.w", l), (long long)f.enc_kernel * F * H, &ok);
    T32(ctx, S("enc.%d.ffn2.b", l), H, &ok);
    T32(ctx, S("enc.%d.ln2.g", l), H, &ok);
    T32(ctx, S("enc.%d.ln2.b", l), H, &ok);
  }
  T32(ctx, "enc.proj.w", (long long)H * 2 * C, &ok);
  T32(ctx, "enc.proj.b", 2 * C, &ok);
  for (int i = 0; i < f.n_flows; ++i) {
    T32(ctx, S("flow.%d.pre.w", i), (long long)half * H, &ok);
    T32(ctx, S("flow.%d.pre.b", i), H, &ok);
    for (int j = 0; j < f.flow_wn_layers; ++j) {
      T32(ctx, S("flow.%d.in.%d.w", i, j), (long long)f.flow_kernel * H * 2 * H, &ok);
      T32(ctx, S("flow.%d.in.%d.b", i, j), 2 * H, &ok);
      if (j < f.flow_wn_layers - 1) {
        T32(ctx, S("flow.%d.rs.%d.res.w", i, j), (long long)H * H, &ok);
        T32(ctx, S("flow.%d.rs.%d.res.b", i, j), H, &ok);
      }
      T32(ctx, S("flow.%d.rs.%d.skip.w", i, j), (long long)H * H, &ok);
      T32(ctx, S("flow.%d.rs.%d.skip.b", i, j), H, &ok);
    }
    T32(ctx, S("flow.%d.post.w", i), (long long)H * half, &ok);
    T32(ctx, S("flow.%d.post.b", i), half, &ok);
  }
  T32(ctx, "dec.pre.w", 7LL * C * f.up_init_channels, &ok);
  T32(ctx, "dec.pre.b", f.up_init_channels, &ok);
  for (int i = 0; i < f.n_ups; ++i) {
    UpGeom g = up_geom(f, i);
    T32(ctx, S("dec.ups.%d.w", i), (long long)g.u * g.ntaps * g.cin * g.cout, &ok);
    T32(ctx, S("dec.ups.%d.b", i), g.cout, &ok);
    int nk, ns, np;
    noise_geom(f, i, &nk, &ns, &np);
    if (f0) {
      T32(ctx, S("dec.noise.%d.w", i), (long long)nk * g.cout, &ok);
      T32(ctx, S("dec.noise.%d.b", i), g.cout, &ok);
    }
    for (int j = 0; j < f.n_res_kernels; ++j) {
      const int n = i * f.n_res_kernels + j;
      for (int d = 0; d < f.n_res_dils[j]; ++d) {
        const long long wn = (long long)f.res_kernels[j] * g.cout * g.cout;
        if (f.resblock_kind == 1) {
          T32(ctx, S("dec.rb.%d.c1.%d.w", n, d), wn, &ok);
          T32(ctx, S("dec.rb.%d.c1.%d.b", n, d), g.cout, &ok);
          T32(ctx, S("dec.rb.%d.c2.%d.w", n, d), wn, &ok);
          T32(ctx, S("dec.rb.%d.c2.%d.b", n, d), g.cout, &ok);
        } else {
          T32(ctx, S("dec.rb.%d.c.%d.w", n, d), wn, &ok);
          T32(ctx, S("dec.rb.%d.c.%d.b", n, d), g.cout, &ok);
        }
      }
    }
  }
  T32(ctx, "dec.post.w", 7LL * (f.up_init_channels >> f.n_ups), &ok);
  if (f0 && (!ctx->scalars.count("dec.src.lin_w") || !ctx->scalars.count("dec.src.lin_b"))) {
    if (ok) snprintf(ctx->err, sizeof(ctx->err), "missing scalar 'dec.src.lin_w/lin_b'");
    ok = false;
  }
  if (!ok) return RVCB200_ERR_MISSING;
  ctx->finalized = true;
  return RVCB200_OK;
}

int64_t rvcb200_workspace_bytes(const rvcb200_ctx* ctx, int32_t B, int32_t T, int32_t precision) {
  if (!ctx || B <= 0 || T <= 0) return -1;
  Plan p = make_plan(ctx, B, T, nullptr, precision);
  return (int64_t)p.bytes + 256;
}

int64_t rvcb200_last_launch_count(const rvcb200_ctx* ctx) { return ctx ? ctx->last_launches : 0; }
const char* rvcb200_last_error(const rvcb200_ctx* ctx) { return ctx ? ctx->err : "null context"; }

}  // extern "C"

// `zp_in` != NULL: start from a given (masked) prior sample z_p [B][T][inter] instead of running the text encoder -- the
// second half of `infer(..., rate=r)` (models.py:802-806: flow and decoder on the last int(T * r) frames).
static int infer_impl(rvcb200_ctx* ctx, int32_t B, int32_t T, const float* phone, const int64_t* phone_lengths,
                      const int64_t* pitch, const float* nsff0, const int64_t* sid, const float* noise_zp,
                      const float* noise_sine, const float* zp_in, float* out, float* stats_out, float* zp_out, float* z_out,
                      void* workspace, int64_t workspace_bytes, int32_t precision, const rvcb200_tap* taps, int32_t n_taps,
                      void* stream) {
  if (!ctx) return RVCB200_ERR_ARG;
  if (!ctx->finalized) return fail(ctx, RVCB200_ERR_MISSING, "rvcb200_finalize() has not succeeded%s", "");
  const bool f0 = ctx->cfg.no_f0 == 0;
  if (B <= 0 || T <= 0 || !phone_lengths || !sid || !out || !workspace || (f0 && (!nsff0 || !noise_sine)) ||
      (!zp_in && (!phone || !noise_zp || (f0 && !pitch))))
    return fail(ctx, RVCB200_ERR_ARG, "null or empty argument%s", "");
  if (precision != RVCB200_PREC_FP32 && precision != RVCB200_PREC_FP16 && precision != RVCB200_PREC_BF16)
    return fail(ctx, RVCB200_ERR_ARG, "unknown precision %s%lld", "", precision);
  const bool tc = precision != RVCB200_PREC_FP32;
  const bool bf16 = precision == RVCB200_PREC_BF16;
  const rvcb200_config& f = ctx->cfg;
  // 256-byte align the workspace
  uintptr_t wsp = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
  const size_t slack = wsp - reinterpret_cast<uintptr_t>(workspace);
  Plan pl = make_plan(ctx, B, T, reinterpret_cast<void*>(wsp), precision);
  if ((int64_t)(pl.bytes + slack) > workspace_bytes)
    return fail(ctx, RVCB200_ERR_WORKSPACE, "workspace too small%s: need %lld bytes", "", (long long)(pl.bytes + 256));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  TapSet tp{taps, n_taps, st};
  struct PdlScope {            // programmatic dependent launch for launch-bound sizes (common.cuh), this call only
    explicit PdlScope(bool on) { pdl_set_auto(on); }
    ~PdlScope() { pdl_set_auto(false); }
  } pdl_scope((long long)B * T <= 2500 && n_taps == 0 && !ctx->prof);
  const long long launches0 = launch_counter().n;
  bool ok = true;
  auto W = [&](const std::string& n) { return T32(ctx, n, 0, &ok); };

  const int H = f.hidden_channels, C = f.inter_channels, F = f.filter_channels, half = C / 2;
  const long long BT = (long long)B * T;
  float* stats = stats_out ? stats_out : pl.stats;
  float* zp = zp_out ? zp_out : pl.zp;
  float* z = z_out ? z_out : pl.z;

  CKC(3, launch_len_to_i32(reinterpret_cast<const long long*>(phone_lengths), pl.len32, B, T, st), "len_to_i32");
  CKC(3, launch_cond_gemv(W("emb_g"), reinterpret_cast<const long long*>(sid), W("cond.w"), W("cond.b"), pl.cond, B,
                      f.gin_channels, ctx->n_cond, f.n_speakers, st),
     "cond_gemv");

  if (!tc) {
  if (zp_in) {
    CK(cudaMemcpyAsync(zp, zp_in, sizeof(float) * BT * C, cudaMemcpyDeviceToDevice, st), "z_p in");
  } else {
  // ---------------- TextEncoder (models.py:43-58 / 90-105) -----------------------------------
  {
    ConvDesc d = base_desc();
    d.x = phone; d.x_bstride = (long long)T * f.feat_dim; d.ldx = f.feat_dim; d.L_in = T;
    d.w = W("enc.emb.w"); d.bias = W("enc.emb.b"); d.Cin = f.feat_dim; d.Cout = H;
    d.Lj = T; d.y = pl.x; d.y_bstride = (long long)T * H; d.ldy = H;
    if (f0) { d.gather = W("enc.emb_pitch"); d.gidx = pitch; d.gidx_bstride = T; }
    d.alpha = sqrtf((float)H); d.out_slope = 0.1f; d.mask_post = 1; d.out_len = pl.len32;
    CKC(6, launch_conv_f32(d, B, st), "enc.emb");
  }
  const int kp = (f.enc_kernel - 1) / 2;
  for (int l = 0; l < f.n_layers; ++l) {
    {  // q|k|v = conv_{q,k,v}(x)   attentions.py:213-215
      ConvDesc d = base_desc();
      d.x = pl.x; d.x_bstride = (long long)T * H; d.ldx = H; d.L_in = T;
      d.w = W(S("enc.%d.qkv.w", l)); d.bias = W(S("enc.%d.qkv.b", l)); d.Cin = H; d.Cout = 3 * H;
      d.Lj = T; d.y = pl.qkv; d.y_bstride = (long long)T * 3 * H; d.ldy = 3 * H;
      CKC(6, launch_conv_f32(d, B, st), "enc.qkv");
    }
    CKC(1, launch_attention_f32(pl.qkv, W(S("enc.%d.rel_k", l)), W(S("enc.%d.rel_v", l)), pl.len32, pl.att, B, T,
                            f.n_heads, H / f.n_heads, f.window_size, st),
       "enc.attention");
    {  // x + conv_o(att)   attentions.py:219,63
      ConvDesc d = base_desc();
      d.x = pl.att; d.x_bstride = (long long)T * H; d.ldx = H; d.L_in = T;
      d.w = W(S("enc.%d.o.w", l)); d.bias = W(S("enc.%d.o.b", l)); d.Cin = H; d.Cout = H;
      d.Lj = T; d.y = pl.xt; d.y_bstride = (long long)T * H; d.ldy = H;
      d.res = pl.x; d.res_bstride = (long long)T * H; d.ldr = H; d.res_mode = 1;
      CKC(6, launch_conv_f32(d, B, st), "enc.o");
    }
    CKC(3, launch_layernorm(pl.xt, W(S("enc.%d.ln1.g", l)), W(S("enc.%d.ln1.b", l)), pl.x, BT, H, 1e-5f, st), "enc.ln1");
    {  // FFN conv_1 + ReLU   attentions.py:388-392
      ConvDesc d = base_desc();
      d.x = pl.x; d.x_bstride = (long long)T * H; d.ldx = H; d.L_in = T; d.in_len = pl.len32;
      d.w = W(S("enc.%d.ffn1.w", l)); d.bias = W(S("enc.%d.ffn1.b", l)); d.Cin = H; d.Cout = F;
      d.ntaps = f.enc_kernel; d.g_off[0] = -kp;
      d.Lj = T; d.y = pl.ffh; d.y_bstride = (long long)T * F; d.ldy = F; d.relu = 1;
      CKC(6, launch_conv_f32(d, B, st), "enc.ffn1");
    }
    {  // x + conv_2(h*mask)*mask   attentions.py:394-395,67
      ConvDesc d = base_desc();
      d.x = pl.ffh; d.x_bstride = (long long)T * F; d.ldx = F; d.L_in = T; d.in_len = pl.len32;
      d.w = W(S("enc.%d.ffn2.w", l)); d.bias = W(S("enc.%d.ffn2.b", l)); d.Cin = F; d.Cout = H;
      d.ntaps = f.enc_kernel; d.g_off[0] = -kp;
      d.Lj = T; d.y = pl.xt; d.y_bstride = (long long)T * H; d.ldy = H;
      d.mask_pre = 1; d.out_len = pl.len32;
      d.res = pl.x; d.res_bstride = (long long)T * H; d.ldr = H; d.res_mode = 1;
      CKC(6, launch_conv_f32(d, B, st), "enc.ffn2");
    }
    CKC(3, launch_layernorm(pl.xt, W(S("enc.%d.ln2.g", l)), W(S("enc.%d.ln2.b", l)), pl.x, BT, H, 1e-5f, st), "enc.ln2");
  }
  CK(tp.emit("x_enc", pl.x, sizeof(float) * BT * H), "tap");
  {  // stats = proj(x*mask)*mask   models.py:101-102
    ConvDesc d = base_desc();
    d.x = pl.x; d.x_bstride = (long long)T * H; d.ldx = H; d.L_in = T; d.in_len = pl.len32;
    d.w = W("enc.proj.w"); d.bias = W("enc.proj.b"); d.Cin = H; d.Cout = 2 * C;
    d.Lj = T; d.y = stats; d.y_bstride = (long long)T * 2 * C; d.ldy = 2 * C;
    d.mask_post = 1; d.out_len = pl.len32;
    CKC(6, launch_conv_f32(d, B, st), "enc.proj");
  }
  CK(tp.emit("stats", stats, sizeof(float) * BT * 2 * C), "tap");
  CKC(3, launch_zp_sample(stats, noise_zp, pl.len32, zp, B, T, C, st), "zp_sample");
  CK(tp.emit("z_p", zp, sizeof(float) * BT * C), "tap");
  }

  // ---------------- reverse flow (models.py:185-192; modules.py:436-455) ----------------------
  if (z != zp) CK(cudaMemcpyAsync(z, zp, sizeof(float) * BT * C, cudaMemcpyDeviceToDevice, st), "z copy");
  {
    bool flipped = false;
    for (int i = f.n_flows - 1; i >= 0; --i) {
      flipped = !flipped;  // the Flip that follows RCL_i in forward order
      const int in_off = flipped ? half : 0, out_off = half - in_off;
      {  // h = pre(x0)*mask
        ConvDesc d = base_desc();
        d.x = z + in_off; d.x_bstride = (long long)T * C; d.ldx = C; d.L_in = T;
        d.w = W(S("flow.%d.pre.w", i)); d.bias = W(S("flow.%d.pre.b", i)); d.Cin = half; d.Cout = H;
        d.Lj = T; d.y = pl.h; d.y_bstride = (long long)T * H; d.ldy = H; d.mask_post = 1; d.out_len = pl.len32;
        CKC(5, launch_conv_f32(d, B, st), "flow.pre");
      }
      for (int j = 0; j < f.flow_wn_layers; ++j) {
        {  // acts = tanh/sigmoid gate of in_layer(h) + cond   modules.py:192-199
          ConvDesc d = base_desc();
          d.x = pl.h; d.x_bstride = (long long)T * H; d.ldx = H; d.L_in = T;
          d.w = W(S("flow.%d.in.%d.w", i, j)); d.bias = W(S("flow.%d.in.%d.b", i, j)); d.Cin = H; d.Cout = 2 * H;
          d.ntaps = f.flow_kernel; d.g_off[0] = -(f.flow_kernel - 1) / 2;
          d.cond = pl.cond + f.up_init_channels + (i * f.flow_wn_layers + j) * 2 * H; d.cond_bstride = ctx->n_cond;
          d.gate = 1;
          d.Lj = T; d.y = pl.acts; d.y_bstride = (long long)T * H; d.ldy = H;
          CKC(5, launch_conv_f32(d, B, st), "flow.in");
        }
        if (j < f.flow_wn_layers - 1) {  // h = (h + res)*mask   modules.py:203-206
          ConvDesc d = base_desc();
          d.x = pl.acts; d.x_bstride = (long long)T * H; d.ldx = H; d.L_in = T;
          d.w = W(S("flow.%d.rs.%d.res.w", i, j)); d.bias = W(S("flow.%d.rs.%d.res.b", i, j)); d.Cin = H; d.Cout = H;
          d.Lj = T; d.y = pl.h; d.y_bstride = (long long)T * H; d.ldy = H;
          d.res = pl.h; d.res_bstride = (long long)T * H; d.ldr = H; d.res_mode = 1;
          d.mask_post = 1; d.out_len = pl.len32;
          CKC(5, launch_conv_f32(d, B, st), "flow.res");
        }
        {  // output += skip   modules.py:207-208
          ConvDesc d = base_desc();
          d.x = pl.acts; d.x_bstride = (long long)T * H; d.ldx = H; d.L_in = T;
          d.w = W(S("flow.%d.rs.%d.skip.w", i, j)); d.bias = W(S("flow.%d.rs.%d.skip.b", i, j)); d.Cin = H; d.Cout = H;
          d.Lj = T; d.y = pl.skip; d.y_bstride = (long long)T * H; d.ldy = H; d.accum = j > 0;
          CKC(5, launch_conv_f32(d, B, st), "flow.skip");
        }
      }
      {  // x1 = (x1 - post(out*mask)*mask)*mask   modules.py:441,453
        ConvDesc d = base_desc();
        d.x = pl.skip; d.x_bstride = (long long)T * H; d.ldx = H; d.L_in = T; d.in_len = pl.len32;
        d.w = W(S("flow.%d.post.w", i)); d.bias = W(S("flow.%d.post.b", i)); d.Cin = H; d.Cout = half;
        d.Lj = T; d.y = z + out_off; d.y_bstride = (long long)T * C; d.ldy = C;
        d.mask_pre = 1; d.mask_post = 1; d.out_len = pl.len32;
        d.res = z + out_off; d.res_bstride = (long long)T * C; d.ldr = C; d.res_mode = 2;
        CKC(5, launch_conv_f32(d, B, st), "flow.post");
      }
    }
  }
  CK(tp.emit("z", z, sizeof(float) * BT * C), "tap");


  } else {
    // ====== TextEncoder + reverse flow with every contraction on tcgen05 (fp16 operands, fp32 epilogues) ======
    auto W16h = [&](const std::string& n) { return T16(ctx, n + ".tc", 0, 1, &ok); };
    static const bool tc_attention = [] { const char* e = getenv("RVCB200_TC_ATTENTION"); return e ? atoi(e) != 0 : true; }();
    // N tile of the encoder/flow contractions: capped at 64 columns (weights.py tc_n_max_for_name): with only T/128
    // M tiles per launch, narrow N tiles occupy 3-12x more SMs and each CTA pulls 3-4x fewer weight bytes from L2
    auto n_for = [](int cout) { for (int n = 64; n >= 16; n -= 16) if (cout % n == 0) return n; return 16; };
    auto gen = [&](const void* x16, int Cin, const std::string& wname, const std::string& bname, int Cout) {
      TcConvDesc d;
      memset(&d, 0, sizeof(d));
      d.padf = kPadF; d.ntaps = 1; d.dil = 1; d.G = 1; d.out_stride = 1; d.div = 1.f; d.out_slope = 1.f;
      d.generic = 1; d.f32_cl = 1; d.alpha = 1.f; d.pre_slope = 1.f;
      d.x16 = x16; d.L_in = T; d.Cin = Cin; d.w16 = W16h(wname); d.bias = W(bname);
      d.N = n_for(Cout); d.Cout_total = Cout; d.Lj = T; d.Lp_out = pv_pitch_rows(T);
      d.out_len = pl.len32;
      return d;
    };
#define TCG(cls, d, what)                         \
  do {                                            \
    if (!ok) return RVCB200_ERR_MISSING;          \
    CKC(cls, launch_conv_tc(d, B, st), what);     \
  } while (0)
    if (zp_in) {
      CK(cudaMemcpyAsync(zp, zp_in, sizeof(float) * BT * C, cudaMemcpyDeviceToDevice, st), "z_p in");
      if (z != zp) CK(cudaMemcpyAsync(z, zp_in, sizeof(float) * BT * C, cudaMemcpyDeviceToDevice, st), "z in");
      CKC(3, launch_cl32_to_cl16(zp_in, pl.z16, (long long)BT * C, 1.f, false, st), "z_p->fp16");
    } else {
    CKC(3, launch_cl32_to_cl16(phone, pl.phone16, (long long)BT * f.feat_dim, 1.f, false, st), "phone->fp16");
    {  // x = lrelu((emb_phone(phone) + emb_pitch[pitch]) * sqrt(H)) * mask   models.py:92-100
      TcConvDesc d = gen(pl.phone16, f.feat_dim, "enc.emb.w", "enc.emb.b", H);
      if (f0) { d.gather = W("enc.emb_pitch"); d.gidx = pitch; d.gidx_bstride = T; }
      d.alpha = sqrtf((float)H); d.pre_slope = 0.1f; d.mask_post = 1; d.mask16 = 1;
      d.y32 = pl.x; d.ldy32 = H; d.y16 = pl.x16;
      TCG(6, d, "enc.emb(tc)");
    }
    const int kp = (f.enc_kernel - 1) / 2;
    for (int l = 0; l < f.n_layers; ++l) {
      if (tc_attention) {
        {  // q|k|v, 128 channels per head (96 + zero pad), q pre-scaled by 1/sqrt(dk): fp16 operands of the attention
          TcConvDesc d = gen(pl.x16, H, S("enc.%d.qkvp.w", l), S("enc.%d.qkvp.b", l), 3 * f.n_heads * 128);
          d.y16 = pl.qkv16;
          TCG(6, d, "enc.qkv(tc)");
        }
        if (!ok) return RVCB200_ERR_MISSING;
        CKC(1, launch_attention_tc(pl.qkv16, pl.vt16, T16(ctx, S("enc.%d.ek16", l), 32 * 128, 1, &ok),
                                   T16(ctx, S("enc.%d.evt16", l), 128 * 64, 1, &ok), pl.len32, pl.att16, B, T, f.n_heads,
                                   H / f.n_heads, f.window_size, st),
            "enc.attention(tc)");
      } else {
        {  // q|k|v (fp32, consumed by the CUDA-core banded attention kernel)
          TcConvDesc d = gen(pl.x16, H, S("enc.%d.qkv.w", l), S("enc.%d.qkv.b", l), 3 * H);
          d.y32 = pl.qkv; d.ldy32 = 3 * H;
          TCG(6, d, "enc.qkv(tc)");
        }
        CKC(1, launch_attention_f32(pl.qkv, W(S("enc.%d.rel_k", l)), W(S("enc.%d.rel_v", l)), pl.len32, pl.att, B, T,
                                    f.n_heads, H / f.n_heads, f.window_size, st),
            "enc.attention");
        CKC(3, launch_cl32_to_cl16(pl.att, pl.att16, (long long)BT * H, 1.f, false, st), "att->fp16");
      }
      {  // x + conv_o(att)
        TcConvDesc d = gen(pl.att16, H, S("enc.%d.o.w", l), S("enc.%d.o.b", l), H);
        d.res32 = pl.x; d.ldr32 = H; d.res_mode = 1; d.y32 = pl.xt; d.ldy32 = H;
        TCG(6, d, "enc.o(tc)");
      }
      CKC(3, launch_layernorm(pl.xt, W(S("enc.%d.ln1.g", l)), W(S("enc.%d.ln1.b", l)), pl.x, BT, H, 1e-5f, st, pl.x16,
                              pl.len32, T),
          "enc.ln1");
      {  // FFN conv_1 + ReLU; the fp16 copy is masked (it feeds conv_2(h * mask))
        TcConvDesc d = gen(pl.x16, H, S("enc.%d.ffn1.w", l), S("enc.%d.ffn1.b", l), F);
        d.ntaps = f.enc_kernel; d.g_off[0] = -kp; d.relu = 1; d.mask16 = 1; d.y16 = pl.ffh16;
        TCG(6, d, "enc.ffn1(tc)");
      }
      {  // x + conv_2(h*mask)*mask
        TcConvDesc d = gen(pl.ffh16, F, S("enc.%d.ffn2.w", l), S("enc.%d.ffn2.b", l), H);
        d.ntaps = f.enc_kernel; d.g_off[0] = -kp; d.mask_pre = 1;
        d.res32 = pl.x; d.ldr32 = H; d.res_mode = 1; d.y32 = pl.xt; d.ldy32 = H;
        TCG(6, d, "enc.ffn2(tc)");
      }
      CKC(3, launch_layernorm(pl.xt, W(S("enc.%d.ln2.g", l)), W(S("enc.%d.ln2.b", l)), pl.x, BT, H, 1e-5f, st, pl.x16,
                              pl.len32, T),
          "enc.ln2");
    }
    CK(tp.emit("x_enc", pl.x, sizeof(float) * BT * H), "tap");
    {  // stats = proj(x*mask)*mask
      TcConvDesc d = gen(pl.x16, H, "enc.proj.w", "enc.proj.b", 2 * C);
      d.mask_post = 1; d.y32 = stats; d.ldy32 = 2 * C;
      TCG(6, d, "enc.proj(tc)");
    }
    CK(tp.emit("stats", stats, sizeof(float) * BT * 2 * C), "tap");
    CKC(3, launch_zp_sample(stats, noise_zp, pl.len32, zp, B, T, C, st, z != zp ? z : nullptr, pl.z16), "zp_sample");
    CK(tp.emit("z_p", zp, sizeof(float) * BT * C), "tap");
    }
    {
      // Reverse coupling layers on folded weights (weights.py): per flow n in_layer launches + ONE skip/post launch, no h.
      // Activation buffer `acts` [BT][AW]: columns [0, xb) = [x0 | mask | zeros], then the n gate outputs (H columns each).
      // in_layer j reads columns [0, xb + j H) (x0, mask, acts_0..j-1: `pre` and the res convolutions are in its weights)
      // and writes acts_j (masked: its neighbours read it through a 5-tap window); the last launch contracts all gate
      // outputs with W_skip_j W_post, updates the other half of z in fp32 and writes its fp16 copy into columns [0, half):
      // after the Flip it is the next flow's x0.
      bool flipped = false;
      const int n_wn = f.flow_wn_layers;
      const int xb = (half + 1 + 63) / 64 * 64, AW = xb + n_wn * H;
      unsigned short* acts = reinterpret_cast<unsigned short*>(pl.acts16);
      CKC(3, launch_flow_x0_init(pl.z16, pl.len32, acts, B, T, C, /*in_off of the first flow*/ half, half, xb, AW, st), "flow.x0");
      for (int i = f.n_flows - 1; i >= 0; --i) {
        flipped = !flipped;
        const int in_off = flipped ? half : 0, out_off = half - in_off;
        (void)in_off;
        for (int j = 0; j < n_wn; ++j) {  // acts_j = gate(in_layer(h_j) + cond) * mask
          TcConvDesc d = gen(acts, xb + j * H, S("flow.%d.inf.%d.w", i, j), S("flow.%d.in.%d.b", i, j), 2 * H);
          d.ldx16 = AW;
          d.ntaps = f.flow_kernel; d.g_off[0] = -(f.flow_kernel - 1) / 2;
          d.cond = pl.cond + f.up_init_channels + (i * n_wn + j) * 2 * H; d.cond_bstride = ctx->n_cond;
          d.gate = 1; d.mask16 = 1; d.y16 = acts + xb + j * H; d.ldy16 = AW;
          TCG(5, d, "flow.in(tc)");
        }
        {  // x1 = (x1 - post(sum_j skip_j(acts_j))*mask)*mask, fp32 in place; fp16 copy = the next flow's x0
          TcConvDesc d = gen(acts + xb, n_wn * H, S("flow.%d.sp.w", i), S("flow.%d.sp.b", i), half);
          d.ldx16 = AW;
          d.mask_pre = 1; d.mask_post = 1;
          d.res32 = z + out_off; d.ldr32 = C; d.res_mode = 2; d.y32 = z + out_off; d.ldy32 = C;
          d.y16 = acts; d.ldy16 = AW;
          TCG(5, d, "flow.skip+post(tc)");
        }
      }
      // the decoder's fp16 operand: both halves of z as the flows left them
      CKC(3, launch_cl32_to_cl16(z, pl.z16, (long long)BT * C, 1.f, false, st), "z->fp16");
    }
    CK(tp.emit("z", z, sizeof(float) * BT * C), "tap");
#undef TCG
  }
  // ---------------- NSF source (models.py:361-411, 455-467) -----------------------------------
  const long long Lout = (long long)T * ctx->upp;
  if (f0) {
    CKC(2, launch_sine_source(nsff0, noise_sine, pl.har, B, T, ctx->upp, f.sr, ctx->scalars["dec.src.lin_w"],
                              ctx->scalars["dec.src.lin_b"], pl.sine_scratch, st),
        "sine_source");
    CK(tp.emit("har_source", pl.har, sizeof(float) * B * Lout), "tap");
  }

  if (!tc) {
  // ---------------- GeneratorNSF (models.py:542-564) -------------------------------------------
  {
    ConvDesc d = base_desc();
    d.x = z; d.x_bstride = (long long)T * C; d.ldx = C; d.L_in = T;
    d.w = W("dec.pre.w"); d.bias = W("dec.pre.b"); d.Cin = C; d.Cout = f.up_init_channels;
    d.ntaps = 7; d.g_off[0] = -3;
    d.cond = pl.cond; d.cond_bstride = ctx->n_cond;
    d.Lj = T; d.y = pl.pre; d.y_bstride = (long long)T * f.up_init_channels; d.ldy = f.up_init_channels;
    CKC(4, launch_conv_f32(d, B, st), "dec.conv_pre");
  }
  CK(tp.emit("dec.pre", pl.pre, sizeof(float) * BT * f.up_init_channels), "tap");
  const float* cur = pl.pre;
  long long Lc = T;
  int Cc = f.up_init_channels;
  float* X = pl.stage[0];
  float* XB = pl.stage[1];
  float* XT = pl.stage[2];
  float* ACC = pl.stage[3];
  float* ACC_next = pl.stage[4];
  for (int i = 0; i < f.n_ups; ++i) {
    UpGeom g = up_geom(f, i);
    const long long Ln = Lc * g.u;
    {  // x = ups[i](lrelu(x))   models.py:550-551 as g.u phase groups
      ConvDesc d = base_desc();
      d.x = cur; d.x_bstride = Lc * Cc; d.ldx = Cc; d.L_in = (int)Lc; d.in_slope = 0.1f;
      d.w = W(S("dec.ups.%d.w", i)); d.bias = W(S("dec.ups.%d.b", i)); d.Cin = g.cin; d.Cout = g.cout;
      d.ntaps = g.ntaps; d.dil = 1; d.G = g.u;
      for (int p = 0; p < g.u; ++p) d.g_off[p] = g.g_off[p];
      d.Lj = (int)Lc; d.out_stride = g.u;
      d.y = X; d.y_bstride = Ln * g.cout; d.ldy = g.cout;
      CKC(4, launch_conv_f32(d, B, st), "dec.ups");
    }
    if (f0) {
      int nk, ns, np;
      noise_geom(f, i, &nk, &ns, &np);
      CKC(3, launch_noise_conv_add(pl.har, W(S("dec.noise.%d.w", i)), W(S("dec.noise.%d.b", i)), X, B, Lout, Ln, g.cout, nk,
                               ns, np, st),
         "dec.noise_conv");
    }
    CK(tp.emit(S("dec.ups.%d", i).c_str(), X, sizeof(float) * B * Ln * g.cout), "tap");
    const int Cn = g.cout;
    for (int j = 0; j < f.n_res_kernels; ++j) {
      const int n = i * f.n_res_kernels + j;
      const int k = f.res_kernels[j];
      const float* src = X;
      const int nd = f.n_res_dils[j];
      for (int dd = 0; dd < nd; ++dd) {
        const bool last = dd == nd - 1;
        const int dil = f.res_dils[j][dd];
        ConvDesc o = base_desc();   // the conv that closes the residual pair / step
        if (f.resblock_kind == 1) {
          ConvDesc d = base_desc();  // xt = c1(lrelu(x))   modules.py:297-301
          d.x = src; d.x_bstride = Ln * Cn; d.ldx = Cn; d.L_in = (int)Ln; d.in_slope = 0.1f;
          d.w = W(S("dec.rb.%d.c1.%d.w", n, dd)); d.bias = W(S("dec.rb.%d.c1.%d.b", n, dd)); d.Cin = Cn; d.Cout = Cn;
          d.ntaps = k; d.dil = dil; d.g_off[0] = -((k - 1) / 2) * dil;
          d.Lj = (int)Ln; d.y = XT; d.y_bstride = Ln * Cn; d.ldy = Cn;
          CKC(0, launch_conv_f32(d, B, st), "dec.rb.c1");
          o.x = XT; o.dil = 1; o.g_off[0] = -((k - 1) / 2);   // x = c2(lrelu(xt)) + x   modules.py:302-305
          o.w = W(S("dec.rb.%d.c2.%d.w", n, dd)); o.bias = W(S("dec.rb.%d.c2.%d.b", n, dd));
        } else {                     // ResBlock2: x = c(lrelu(x)) + x   modules.py:347-352
          o.x = src; o.dil = dil; o.g_off[0] = -((k - 1) / 2) * dil;
          o.w = W(S("dec.rb.%d.c.%d.w", n, dd)); o.bias = W(S("dec.rb.%d.c.%d.b", n, dd));
        }
        o.x_bstride = Ln * Cn; o.ldx = Cn; o.L_in = (int)Ln; o.in_slope = 0.1f;
        o.Cin = Cn; o.Cout = Cn; o.ntaps = k;
        o.Lj = (int)Ln; o.y_bstride = Ln * Cn; o.ldy = Cn;
        o.res = src; o.res_bstride = Ln * Cn; o.ldr = Cn; o.res_mode = 1;
        if (last) {  // xs += resblock(x); x = xs / num_kernels   models.py:554-560
          o.y = ACC; o.accum = j > 0; o.div = (j == f.n_res_kernels - 1) ? (float)f.n_res_kernels : 1.f;
        } else {
          o.y = XB;
        }
        CKC(0, launch_conv_f32(o, B, st), "dec.rb.c2");
        src = XB;
      }
    }
    CK(tp.emit(S("dec.stage.%d", i).c_str(), ACC, sizeof(float) * B * Ln * Cn), "tap");
    cur = ACC;
    float* t = ACC; ACC = ACC_next; ACC_next = t;
    Lc = Ln; Cc = Cn;
  }
  CKC(3, launch_conv_post_tanh(cur, W("dec.post.w"), out, B, Lc, Cc, 7, 0.01f, st), "dec.conv_post");

  } else {
    // ------------- GeneratorNSF on tcgen05 (fp16/bf16 operands, fp32 accumulate + residual stream) -----------
    // Operand formats: resblock convolutions follow `precision`; the ladder on the main signal path
    // (conv_pre, ups) always runs on fp16 operands -- bf16 there costs ~9 dB of output SNR (SURVEY §7 H8).
    const int dt = bf16 ? 2 : 1;
    auto W16 = [&](const std::string& n) { return T16(ctx, n + ".tc", 0, dt, &ok); };
    auto W16h = [&](const std::string& n) { return T16(ctx, n + ".tc", 0, 1, &ok); };
    const int rb_bf16 = bf16 ? 1 : 0;
    static const int tc_a_mode = [] { const char* e = getenv("RVCB200_TC_AMODE"); return e ? atoi(e) : 0; }();
    // resblock convs run on the compile-time specialised kernel (rbconv_tc.cu) when it covers the shape;
    // RVCB200_RBCONV=0 forces the generic kernel (A/B measurements)
    static const int use_rb = [] { const char* e = getenv("RVCB200_RBCONV"); return e ? atoi(e) : 1; }();
    // ResBlock1 pairs the fused kernel covers (C <= 64, k <= 7) run as one launch; RVCB200_FUSE_PAIRS=0: two launches
    // (read per call so that a test can compare both forms in one process)
    const int fuse_pairs = [] { const char* e = getenv("RVCB200_FUSE_PAIRS"); return e ? atoi(e) : 1; }();
    auto launch_rb = [&](const TcConvDesc& d) -> cudaError_t {
      if (use_rb && rbconv_tc_supported(d)) return launch_rbconv_tc(d, B, st);
      return launch_conv_tc(d, B, st);
    };
    auto tmem_cols_for = [](int N) { int c = 32; while (c < N) c <<= 1; return c; };
    // conv_post on the specialised tcgen05 kernel (same rule as weights.post_is_tc); RVCB200_POST_TC=0: CUDA-core kernel
    const int c_last = f.up_init_channels >> f.n_ups;
    const bool post_tc = [] { const char* e = getenv("RVCB200_POST_TC"); return e ? atoi(e) != 0 : true; }() &&
                         f.resblock_kind == 1 && (c_last == 32 || c_last == 64 || c_last == 128) &&
                         ctx->tensors.count("dec.post.wt.tc") != 0 && ctx->tensors.count("dec.post.bt") != 0;
    auto tc_base = [&]() {
      TcConvDesc d;
      memset(&d, 0, sizeof(d));
      d.padf = kPadF; d.ntaps = 1; d.dil = 1; d.G = 1; d.out_stride = 1; d.div = 1.f; d.out_slope = 1.f;
      d.a_mode = tc_a_mode;
      return d;
    };
    const int LpT = pv_pitch_rows(T);
    // pl.z16 already holds z (fp16, masked) from the flow's `post` epilogues
    void* IN16 = pl.pv16[0];
    void* X16 = pl.pv16[1];
    void* XT16 = pl.pv16[2];
    void* XB16 = pl.pv16[3];
    void* N16 = pl.pv16[4];
    // The activation stream between convolutions lives in HBM ONCE, as fp16 lrelu_{0.1}(x), channels-last: it is the MMA
    // operand of the next convolution as it is, and the residual x is recovered from it in the pair-closing epilogue
    // (x = r > 0 ? r : 10 r -- the same relative precision as an fp16 copy of x itself; tools/emulate_precision.py: -2 dB
    // in fp16 mode, -0.2 dB in bf16 mode against an fp32 stream).  A pair moves 10 bytes per element instead of 16.
    // bf16 mode keeps the stream in fp16 (a bf16 stream costs 5 dB): convs1 (stream x weights) run on fp16 operands,
    // convs2 (h x weights, h never leaves the pair) on bf16 operands -- tcgen05 kind::f16 rejects mixed A/B formats.
    // The branch sum xs lives in planar-vector fp16 [B][C/8][Lp][8] (only epilogues touch it: 512 B per warp access).
    float* X32 = pl.pv32[0];
    float* ACC32 = pl.pv32[1];
    {
      const int U0 = f.up_init_channels;
      TcConvDesc d = tc_base();
      d.x16 = pl.z16; d.L_in = T; d.w16 = W16h("dec.pre.w"); d.bias = W("dec.pre.b");
      d.Cin = C; d.ntaps = 7; d.g_off[0] = -3;
      d.N = U0 < 256 ? U0 : 256; d.Cout_total = U0; d.tmem_cols = tmem_cols_for(d.N);
      d.Lj = T; d.Lp_out = LpT; d.y16 = IN16; d.out_slope = 0.1f;      // lrelu of models.py:550 folded into the store
      d.cond = pl.cond; d.cond_bstride = ctx->n_cond;
      if (!ok) return RVCB200_ERR_MISSING;
      d.in_bf16 = 0; d.out_bf16 = 0;
      CKC(4, launch_conv_tc(d, B, st), "dec.conv_pre(tc)");
    }
    long long Lc = T;
    int Cc = f.up_init_channels;
    int LpC = LpT;
    for (int i = 0; i < f.n_ups; ++i) {
      UpGeom g = up_geom(f, i);
      const long long Ln = Lc * g.u;
      const int Cn = g.cout;
      const int LpN = pv_pitch_rows(Ln);
      const bool last_stage = i == f.n_ups - 1;
      if (last_stage) CKC(3, launch_zero_pads(ACC32, (long long)B * (Cn / 8), LpN, kPadF, Ln, st), "zero_pads");
      int nk, ns, np;
      noise_geom(f, i, &nk, &ns, &np);
      const bool want_tap = tp.find(S("dec.ups.%d", i).c_str()) != nullptr;
      // x = ups[i](lrelu(x)) [+ noise_convs[i](har)]   (models.py:550-553; the input already holds lrelu(x) in 16 bit).
      // Default: the transposed conv writes its RAW result as fp16 straight into the stream buffer (2 B/elem) and the
      // source injection runs in place on it (2 + 2 B/elem) -- 6 B/elem per stage instead of the 10 of an fp32 planar
      // intermediate.  Stages with stride 2 run as ONE dense 3-tap convolution on the resblock kernel (ups_dense);
      // the others as phase groups on the generic kernel.  (Injecting the source inside the conv epilogue was measured
      // slower: 2-8 taps x 32 channels of FMAs per row chunk on the 8 epilogue warps, profiles/r1_ups_modes.jsonl.)
      // When a test taps x, the fp32 planar path of the first version is used.
      static const int dense_ok = [] { const char* e = getenv("RVCB200_UPS_DENSE"); return e ? atoi(e) : 1; }();
      const float first_slope = f0 ? 1.f : 0.1f;      // with f0 the lrelu is applied by the injection kernel
      bool injected = false;
      if (!want_tap && dense_ok && ups_dense(f, i)) {
        TcConvDesc d = tc_base();
        d.x16 = IN16; d.L_in = (int)Lc; d.w16 = W16h(S("dec.ups.%d.w3", i)); d.bias = W(S("dec.ups.%d.b3", i));
        d.Cin = Cc; d.ntaps = 3; d.dil = 1; d.g_off[0] = -1;
        d.N = Cc; d.Cout_total = Cc; d.tmem_cols = tmem_cols_for(d.N);
        d.Lj = (int)Lc; d.Lp_out = pv_pitch_rows(Lc); d.y16 = X16; d.out_slope = first_slope;   // [Lc][u*Cn] == [Ln][Cn]
        // late stages: the noise conv has <= 4 taps, cheap enough for the epilogue of this (HBM-bound) launch -- the
        // stream is then written once instead of written, re-read and re-written (RVCB200_INJECT_FUSED=0: separate)
        static const int inj_ok = [] { const char* e = getenv("RVCB200_INJECT_FUSED"); return e ? atoi(e) : 1; }();
        if (f0 && inj_ok && use_rb && nk <= 4 && (Cn == 32 || Cn == 64)) {
          d.inj_har = pl.har; d.inj_w = W(S("dec.noise.%d.w", i)); d.inj_b = W(S("dec.noise.%d.b", i));
          d.inj_k = nk; d.inj_s = ns; d.inj_pad = np; d.inj_cn = Cn; d.inj_Lhar = Lout;
          d.out_slope = 0.1f;
          injected = rbconv_tc_supported(d);
          if (!injected) { d.inj_har = nullptr; d.out_slope = first_slope; }
        }
        if (!ok) return RVCB200_ERR_MISSING;
        CKC(4, launch_rb(d), "dec.ups(dense)");
      } else {
        TcConvDesc d = tc_base();
        d.x16 = IN16; d.L_in = (int)Lc; d.w16 = W16h(S("dec.ups.%d.w", i)); d.bias = W(S("dec.ups.%d.b", i));
        d.Cin = Cc; d.ntaps = g.ntaps; d.G = g.u;
        for (int p = 0; p < g.u; ++p) d.g_off[p] = g.g_off[p];
        d.N = Cn < 256 ? Cn : 256; d.Cout_total = Cn; d.tmem_cols = tmem_cols_for(d.N);
        d.Lj = (int)Lc; d.out_stride = g.u; d.Lp_out = LpN;
        if (want_tap) d.y32 = X32;
        else { d.y16 = X16; d.out_slope = first_slope; }
        if (!ok) return RVCB200_ERR_MISSING;
        d.in_bf16 = 0; d.out_bf16 = 0;
        CKC(4, launch_conv_tc(d, B, st), "dec.ups(tc)");
      }
      if (want_tap) {
        if (f0)
          CKC(3, launch_noise_add_pv(pl.har, W(S("dec.noise.%d.w", i)), W(S("dec.noise.%d.b", i)), X32, X16, true, B,
                                     Lout, Ln, Cn, nk, ns, np, LpN, kPadF, 0.1f, false, st),
              "dec.noise_add(pv)");
        else    // plain Generator (models.py:298-300): only the fp32 planar -> fp16 stream conversion
          CKC(3, launch_noise_add_pv(nullptr, nullptr, nullptr, X32, X16, true, B, Lout, Ln, Cn, 0, 1, 0, LpN, kPadF, 0.1f,
                                     false, st),
              "dec.to_stream(pv)");
      } else if (f0 && !injected) {
        // (tried in round 2: the early stages' noise conv as an im2col GEMM on the tensor core with the stream as 16-bit
        //  residual -- 0.61 ms of glue instead of 0.53: the extra pass over the im2col rows and the generic kernel's
        //  thread-per-row residual reads cost more than the CUDA-core FMAs they replace)
        CKC(3, launch_noise_add16(pl.har, W(S("dec.noise.%d.w", i)), W(S("dec.noise.%d.b", i)), X16, B, Lout, Ln, Cn, nk, ns,
                                  np, 0.1f, st),
            "dec.noise_add16");
      }
      if (const rvcb200_tap* t = tp.find(S("dec.ups.%d", i).c_str()))
        CK(launch_pv32_to_cl(X32, reinterpret_cast<float*>(t->dst), B, Ln, Cn, LpN, kPadF, st), "tap");
      for (int j = 0; j < f.n_res_kernels; ++j) {
        const int n = i * f.n_res_kernels + j;
        const int k = f.res_kernels[j];
        const void* src16 = X16;
        const int nd = f.n_res_dils[j];
        for (int dd = 0; dd < nd; ++dd) {
          const bool last = dd == nd - 1;
          const int dil = f.res_dils[j][dd];
          TcConvDesc o = tc_base();
          const int c2_bf16 = f.resblock_kind == 1 ? rb_bf16 : 0;
          o.L_in = (int)Ln; o.Cin = Cn; o.ntaps = k;
          o.N = Cn < 256 ? Cn : 256; o.Cout_total = Cn; o.tmem_cols = tmem_cols_for(o.N);
          o.Lj = (int)Ln; o.Lp_out = LpN;
          // stream buffers: X16 (the stage input, shared by the three branches) stays intact; XT16 / XB16 alternate.
          // A convolution reads a halo of its input, so its 16-bit output never aliases it; only the pair-closing conv of
          // the two-launch form may update the stream in place (its input is h, the stream is a row-aligned residual).
          void* const hbuf = src16 == XT16 ? XB16 : XT16;                    // h = lrelu(c1(.)) of the two-launch form
          void* const ynew = src16 == XB16 ? XT16 : XB16;                    // output that aliases neither src16 nor X16
          TcConvDesc d = o;    // xt = c1(lrelu(x)); only lrelu(xt) is ever consumed -> 16-bit store only
          if (f.resblock_kind == 1) {
            d.x16 = src16; d.w16 = W16h(S("dec.rb.%d.c1.%d.w", n, dd)); d.bias = W(S("dec.rb.%d.c1.%d.b", n, dd));
            d.dil = dil; d.g_off[0] = -((k - 1) / 2) * dil;
            d.y16 = hbuf; d.out_slope = 0.1f;
            if (!ok) return RVCB200_ERR_MISSING;
            d.in_bf16 = 0; d.out_bf16 = rb_bf16;
            o.x16 = hbuf; o.dil = 1; o.g_off[0] = -((k - 1) / 2);
            o.w16 = W16(S("dec.rb.%d.c2.%d.w", n, dd)); o.bias = W(S("dec.rb.%d.c2.%d.b", n, dd));
          } else {
            o.x16 = src16; o.dil = dil; o.g_off[0] = -((k - 1) / 2) * dil;
            o.w16 = W16h(S("dec.rb.%d.c.%d.w", n, dd)); o.bias = W(S("dec.rb.%d.c.%d.b", n, dd));
          }
          o.res16 = src16; o.res_neg_scale = 10.f;
          o.in_bf16 = c2_bf16; o.out_bf16 = 0;           // the stream (and what the next ups consumes) is fp16
          if (last) {
            const bool final_branch = j == f.n_res_kernels - 1;
            o.y32 = ACC32; o.acc_f16 = 1; o.accum = j > 0; o.div = final_branch ? (float)f.n_res_kernels : 1.f;
            if (final_branch && !last_stage) { o.y16 = N16; o.out_slope = 0.1f; }
            if (final_branch && last_stage && post_tc) {
              // the decoder's last tensor is consumed once, by conv_post, as lrelu_{0.01}(x) (models.py:561): it leaves as
              // that 16-bit channels-last operand
              o.y16 = N16; o.out_slope = 0.01f;
            }
            // the stage's result leaves as the 16-bit stream N16 (the next ups / conv_post reads it) and the next stage's
            // first branch overwrites ACC32: the planar branch sum is not written back unless a test taps it
            if (final_branch && o.y16)
              o.acc_nostore = (o.accum && tp.find(S("dec.stage.%d", i).c_str()) == nullptr) ? 1 : 0;
          } else {
            o.y16 = ynew; o.out_slope = 0.1f;
          }
          if (!ok) return RVCB200_ERR_MISSING;
          if (f.resblock_kind == 1 && fuse_pairs && rbpair_tc_supported(d, o)) {
            // one kernel per pair, h stays in shared memory (rbpair_tc.cu): 4 B/element of HBM traffic instead of 10
            CKC(0, launch_rbpair_tc(d, o, B, st), "dec.rb.pair(tc)");
          } else {
            if (f.resblock_kind == 1) {
              CKC(0, launch_rb(d), "dec.rb.c1(tc)");
              if (!last && src16 != X16) o.y16 = const_cast<void*>(src16);   // in place: the third buffer holds h
            }
            CKC(0, launch_rb(o), "dec.rb.c2(tc)");
          }
          src16 = o.y16;
        }
      }
      if (const rvcb200_tap* t = tp.find(S("dec.stage.%d", i).c_str()))
        CK(launch_pv16_to_cl(ACC32, reinterpret_cast<float*>(t->dst), B, Ln, Cn, LpN, kPadF, st), "tap");
      void* tmp = IN16; IN16 = N16; N16 = tmp;
      Lc = Ln; Cc = Cn; LpC = LpN; (void)LpC;
    }
    if (post_tc) {
      // conv_post + tanh (models.py:562-563) on the tensor core: IN16 (after the swap) holds lrelu_{0.01}(x) in fp16
      TcConvDesc d = tc_base();
      d.x16 = IN16; d.L_in = (int)Lc; d.w16 = W16h("dec.post.wt"); d.bias = W("dec.post.bt");
      d.Cin = Cc; d.ntaps = 7; d.dil = 1; d.g_off[0] = -3;
      d.N = Cc; d.Cout_total = Cc; d.tmem_cols = tmem_cols_for(d.N);
      d.Lj = (int)Lc; d.Lp_out = LpC; d.tanh_out = out;
      if (!ok) return RVCB200_ERR_MISSING;
      CKC(3, launch_rbconv_tc(d, B, st), "dec.conv_post(tc)");
    } else {
      CKC(3, launch_conv_post_pv16(ACC32, W("dec.post.w"), out, B, Lc, Cc, 7, LpC, kPadF, 0.01f, st), "dec.conv_post(pv16)");
    }
  }
  if (!ok) return RVCB200_ERR_MISSING;
  ctx->last_launches = launch_counter().n - launches0;
  return RVCB200_OK;
}

extern "C" {

int rvcb200_infer(rvcb200_ctx* ctx, int32_t B, int32_t T, const float* phone, const int64_t* phone_lengths,
                  const int64_t* pitch, const float* nsff0, const int64_t* sid, const float* noise_zp,
                  const float* noise_sine, float* out, float* stats_out, float* zp_out, float* z_out, void* workspace,
                  int64_t workspace_bytes, int32_t precision, const rvcb200_tap* taps, int32_t n_taps, void* stream) {
  return infer_impl(ctx, B, T, phone, phone_lengths, pitch, nsff0, sid, noise_zp, noise_sine, nullptr, out, stats_out, zp_out,
                    z_out, workspace, workspace_bytes, precision, taps, n_taps, stream);
}

int rvcb200_infer_tail(rvcb200_ctx* ctx, int32_t B, int32_t T, const float* z_p, const int64_t* lengths, const float* nsff0,
                       const int64_t* sid, const float* noise_sine, float* out, float* z_out, void* workspace,
                       int64_t workspace_bytes, int32_t precision, void* stream) {
  if (!z_p) return RVCB200_ERR_ARG;
  return infer_impl(ctx, B, T, nullptr, lengths, nullptr, nsff0, sid, nullptr, noise_sine, z_p, out, nullptr, nullptr, z_out,
                    workspace, workspace_bytes, precision, nullptr, 0, stream);
}

// ---------------------------------- op-level entry points --------------------------------------
int rvcb200_op_conv_f32(const rvcb200_conv_desc* d, int32_t B, void* stream) {
  if (!d) return RVCB200_ERR_ARG;
  cudaError_t e = launch_conv_f32(*d, B, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_conv_tc(const rvcb200_tc_conv_desc* d, int32_t B, void* stream) {
  if (!d) return RVCB200_ERR_ARG;
  cudaError_t e = launch_conv_tc(*d, B, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_debug_trace_conv_tc(void* buf) {
  return conv_tc_set_trace(buf) == cudaSuccess ? RVCB200_OK : RVCB200_ERR_CUDA;
}

int rvcb200_op_rbconv_tc(const rvcb200_tc_conv_desc* d, int32_t B, void* stream) {
  if (!d) return RVCB200_ERR_ARG;
  cudaError_t e = launch_rbconv_tc(*d, B, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : ((e == cudaErrorInvalidValue || e == cudaErrorNotSupported) ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_rbpair_tc(const rvcb200_tc_conv_desc* d1, const rvcb200_tc_conv_desc* d2, int32_t B, void* stream) {
  if (!d1 || !d2) return RVCB200_ERR_ARG;
  cudaError_t e = launch_rbpair_tc(*d1, *d2, B, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : ((e == cudaErrorInvalidValue || e == cudaErrorNotSupported) ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int64_t rvcb200_op_sine_scratch_bytes(int32_t B, int32_t T, int32_t upp) { return (int64_t)sine_scratch_bytes(B, T, upp); }

int rvcb200_op_sine_source(const float* f0, const float* noise, float* har, int32_t B, int32_t T, int32_t upp,
                           int32_t sr, float lin_w, float lin_b, void* scratch, void* stream) {
  cudaError_t e = launch_sine_source(f0, noise, har, B, T, upp, sr, lin_w, lin_b, scratch,
                                     reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : RVCB200_ERR_CUDA;
}

int rvcb200_op_attention_f32(const float* qkv, const float* rel_k, const float* rel_v, const int32_t* len, float* out,
                             int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t window, void* stream) {
  cudaError_t e = launch_attention_f32(qkv, rel_k, rel_v, len, out, B, T, n_heads, dk, window,
                                       reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_attention_tc(const void* qkv16, void* vt, const void* ek16, const void* evt16, const int32_t* len, void* out,
                            int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t window, void* stream) {
  cudaError_t e = launch_attention_tc(qkv16, vt, ek16, evt16, len, out, B, T, n_heads, dk, window,
                                      reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_layernorm(const float* x, const float* gamma, const float* beta, float* y, int64_t rows, int32_t C,
                         float eps, void* stream) {
  cudaError_t e = launch_layernorm(x, gamma, beta, y, rows, C, eps, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : RVCB200_ERR_CUDA;
}

int rvcb200_op_prepare_feats(const void* feats, const void* feats0, int32_t dtype, const float* pitchf, float* out, int32_t F,
                             int32_t T, int32_t C, float protect, int32_t use_protect, void* stream) {
  cudaError_t e = launch_prepare_feats(feats, feats0, dtype, pitchf, out, F, T, C, protect, use_protect,
                                       reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_absmax(const float* x, int64_t n, float* out, int32_t reset, void* stream) {
  cudaError_t e = launch_absmax(x, n, out, reset, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_to_int16(const float* x, int64_t n, const float* absmax, int16_t* out, void* stream) {
  cudaError_t e = launch_to_int16(x, n, absmax, out, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

// change_rms (lib/model_utils.py:39, vc_infer_pipeline.py:183): float32 squares summed in double, in a grid-independent order.
int rvcb200_op_rms_halfblock(const void* x, int32_t x_f64, int64_t len, int64_t offset, int32_t hop, double* out, void* stream) {
  cudaError_t e = launch_rms_halfblock(x, x_f64, len, offset, hop, out, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

// change_rms (lib/model_utils.py:39, vc_infer_pipeline.py:183): rows folded in order in double, mean rounded once to float32.
int rvcb200_op_rms_fold(const double* table, int32_t rows, int64_t n_hb, int32_t frame_length, float* rms, void* stream) {
  cudaError_t e = launch_rms_fold(table, rows, n_hb, frame_length, rms, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

// change_rms (lib/model_utils.py:39, vc_infer_pipeline.py:183): torch's float32 linear interpolation, powf, two float32 products.
int rvcb200_op_rms_gain(float* x, int64_t len, int64_t offset, int64_t N, const float* rms1, int64_t n1, const float* rms2, int64_t n2,
                        double rate, void* stream) {
  cudaError_t e = launch_rms_gain(x, len, offset, N, rms1, n1, rms2, n2, rate, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

// Index blend (vc_infer_pipeline.py:59-75), IVF-Flat with nprobe 1: fp32 CUDA-core distances, packed-key atomicMin merges.
int64_t rvcb200_op_ivf_scratch_bytes(int32_t F, int32_t nlist) { return ivf_scratch_bytes(F, nlist); }

int rvcb200_op_ivf_assign(const void* x, int32_t x_dtype, int64_t ldx, int32_t F, int32_t d, const float* centroids, const float* cnorm,
                          int32_t nlist, uint64_t* coarse, void* stream) {
  cudaError_t e = launch_ivf_assign(x, x_dtype, ldx, F, d, centroids, cnorm, nlist, reinterpret_cast<unsigned long long*>(coarse),
                                    reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_ivf_scan(const void* x, int32_t x_dtype, int64_t ldx, int32_t F, int32_t d, const uint64_t* coarse, int32_t nlist,
                        const int32_t* list_offsets, const float* vectors, const int64_t* labels, void* scratch, int64_t scratch_bytes,
                        float* score, int64_t* ix, void* stream) {
  cudaError_t e = launch_ivf_scan(x, x_dtype, ldx, F, d, reinterpret_cast<const unsigned long long*>(coarse), nlist, list_offsets, vectors,
                                  reinterpret_cast<const long long*>(labels), scratch, scratch_bytes, score,
                                  reinterpret_cast<long long*>(ix), reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_index_blend(const void* feats, int32_t feats_dtype, int64_t ldf, int32_t F, int32_t d, const float* score,
                           const int64_t* ix, const float* vectors, const int32_t* pos_of_label, int64_t ntotal, int32_t is_half,
                           double index_rate, void* out, void* stream) {
  cudaError_t e = launch_index_blend(feats, feats_dtype, ldf, F, d, score, reinterpret_cast<const long long*>(ix), vectors, pos_of_label,
                                     ntotal, is_half, index_rate, out, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

// librosa.resample at vc_infer_pipeline.py:185-186, as resample_poly with the filter of comfy_rvc_b200/resample.py: one
// fixed-order fp32 FMA chain per output, so any split of the output range gives the same bits.
int rvcb200_op_resample_poly(const float* tab, int32_t up, int32_t down, int32_t tpp, int64_t half_len, const float* left, int64_t n_left,
                             const float* piece, int64_t n_piece, const float* right, int64_t n_right, int64_t piece_off, int64_t n_song,
                             int64_t out_lo, int64_t out_hi, float* out, void* stream) {
  cudaError_t e = launch_resample_poly(tab, up, down, tpp, half_len, left, n_left, piece, n_piece, right, n_right, piece_off, n_song,
                                       out_lo, out_hi, out, reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_hubert_conv0(const float* x, const float* w, const float* gn_w, const float* gn_b, double* stats, void* y16,
                            int32_t B, int64_t n, int32_t C, int32_t K, int32_t S, float eps, int64_t y_bstride, void* stream) {
  cudaError_t e = launch_hubert_conv0(x, w, gn_w, gn_b, stats, y16, B, n, C, K, S, eps, y_bstride,
                                      reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_layernorm16(const float* x, const float* gamma, const float* beta, float* y, void* y16, int64_t rows, int32_t C,
                           float eps, void* stream) {
  cudaError_t e = launch_layernorm(x, gamma, beta, y, rows, C, eps, reinterpret_cast<cudaStream_t>(stream), y16);
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

int rvcb200_op_quiet_point(const double* audio_pad, int64_t lo, int64_t hi, int32_t window, double* best_v, int64_t* best_j,
                           int32_t n_blocks, void* stream) {
  cudaError_t e = launch_quiet_point(audio_pad, lo, hi, window, best_v, reinterpret_cast<long long*>(best_j), n_blocks,
                                     reinterpret_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? RVCB200_OK : (e == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA);
}

#define RVC_RET(e) return (e) == cudaSuccess ? RVCB200_OK : ((e) == cudaErrorInvalidValue ? RVCB200_ERR_ARG : RVCB200_ERR_CUDA)

int rvcb200_op_rmvpe_logmel(const float* audio, int64_t n, const float* window, const float* twiddle, const float* mel_basis,
                            const int32_t* mel_range, float bn_scale, float bn_shift, float* mel_out, void* img16, int32_t n_frames,
                            int32_t frames_out, int32_t img_pitch, int32_t img_c, void* stream) {
  cudaError_t e = launch_rmvpe_logmel(audio, n, window, twiddle, mel_basis, mel_range, bn_scale, bn_shift, mel_out, img16, n_frames,
                                      frames_out, img_pitch, img_c, reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_rmvpe_pool(const float* x32, int32_t ldx, void* y16, int32_t H2, int32_t W2, int32_t C, int32_t p_in, int32_t p_out,
                          void* stream) {
  cudaError_t e = launch_rmvpe_pool(x32, ldx, y16, H2, W2, C, p_in, p_out, reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_rmvpe_shuffle(const void* g16, void* out16, int32_t H, int32_t W, int32_t Co, int32_t ld, int32_t p_in, int32_t fp_out,
                             int32_t pack, void* stream) {
  cudaError_t e = launch_rmvpe_shuffle(g16, out16, H, W, Co, ld, p_in, fp_out, pack, reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_rmvpe_gru_pack(const float* y32, int32_t ldc, void* x16, int64_t T, int32_t W, int32_t pitch, void* stream) {
  cudaError_t e = launch_rmvpe_gru_pack(y32, ldc, x16, T, W, pitch, reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_rmvpe_gru(const float* gi, const float* w_hh, const float* b_hh, void* out16, float* out32, int32_t T, void* stream) {
  cudaError_t e = launch_rmvpe_gru(gi, w_hh, b_hh, out16, out32, T, reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_rmvpe_decode(const float* in, int32_t ld, int32_t from_hidden, float* hidden, double* f0, double* cents, int32_t T,
                            float thred, void* stream) {
  cudaError_t e = launch_rmvpe_decode(in, ld, from_hidden, hidden, f0, cents, T, thred, reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_crepe_frames(const float* audio, int64_t n, int64_t first, int64_t count, int32_t hop, int32_t pad, void* frames16,
                            void* stream) {
  cudaError_t e = launch_crepe_frames(audio, n, first, count, hop, pad, frames16, reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_crepe_bn_pool(const void* x16, const float* scale, const float* shift, void* y16, int64_t frames, int32_t C, int32_t L,
                             int32_t p_in, int32_t in_off, int32_t p_out, int32_t out_off, void* stream) {
  cudaError_t e = launch_crepe_bn_pool(x16, scale, shift, y16, frames, C, L, p_in, in_off, p_out, out_off,
                                       reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_crepe_decode(const float* in, int32_t ld, int32_t from_salience, int64_t T, int32_t chunk, int32_t lo, int32_t hi,
                            int32_t mode, const double* dither, const double* wcents, const double* log_trans, double log_out,
                            double log_init, float* salience, double* logp, uint16_t* ptr, int32_t* bins, double* f0, float* periodicity,
                            double* score, void* stream) {
  cudaError_t e = launch_crepe_decode(in, ld, from_salience, T, chunk, lo, hi, mode, dither, wcents, log_trans, log_out, log_init,
                                      salience, logp, ptr, bins, f0, periodicity, score, reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

int rvcb200_op_rmvpe_mel_to_img(const float* mel, void* img16, int32_t n_frames, int32_t frames_out, float bn_scale, float bn_shift,
                                int32_t img_pitch, int32_t img_c, void* stream) {
  cudaError_t e = launch_rmvpe_mel_to_img(mel, img16, n_frames, frames_out, bn_scale, bn_shift, img_pitch, img_c,
                                          reinterpret_cast<cudaStream_t>(stream));
  RVC_RET(e);
}

}  // extern "C"
