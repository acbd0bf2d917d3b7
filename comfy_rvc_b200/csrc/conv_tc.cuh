// Descriptor + launchers of the tcgen05 convolution path (see conv_tc.cu).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/rvcb200.h"

namespace rvc {

typedef rvcb200_tc_conv_desc TcConvDesc;

// TMA tensor maps of the tcgen05 kernels, encoded by the driver's cuTensorMapEncodeTiled (looked up once through the
// runtime, so the library does not link libcuda).  False when the driver does not provide it.
bool tensor_map_encoder_available();
// One tiled tensor map with unit element strides, no interleave and the zero out-of-bounds fill (loads read elements
// outside `dims` as zero, stores skip them); false when encoding fails.
bool encode_tensor_map(CUtensorMap* tm, CUtensorMapDataType dt, int rank, const void* base, const cuuint64_t* dims,
                       const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle,
                       CUtensorMapL2promotion l2);

constexpr int kPadF = 32;                                   // zero rows in front of every PV plane
inline int pv_pitch_rows(long long L) { return (int)(((L + 127) / 128) * 128 + 128); }   // Lp
// epilogue divisors (the branch mean 1 / n_res_kernels) that tc::div_exact reproduces bit for bit
inline bool tc_div_exact(float d) { return d == 1.f || d == 2.f || d == 3.f || d == 4.f; }

cudaError_t launch_conv_tc(const TcConvDesc& d, int B, cudaStream_t st);
// debug: device buffer of 16 x grid uint64 that receives phase timestamps of the following launches (nullptr: off)
cudaError_t conv_tc_set_trace(void* buf);
// Compile-time specialised resblock convolution (rbconv_tc.cu); cudaErrorNotSupported if the shape is not covered.
bool rbconv_tc_supported(const TcConvDesc& d);
cudaError_t launch_rbconv_tc(const TcConvDesc& d, int B, cudaStream_t st);
// Fused ResBlock1 pair (rbpair_tc.cu): conv1 -> lrelu -> conv2 + residual in one kernel, h only in shared memory.
bool rbpair_tc_supported(const TcConvDesc& d1, const TcConvDesc& d2);
cudaError_t launch_rbpair_tc(const TcConvDesc& d1, const TcConvDesc& d2, int B, cudaStream_t st);
cudaError_t launch_zero_pads(void* base, long long planes, int Lp, int padf, long long L, cudaStream_t st);
cudaError_t launch_cl32_to_cl16(const float* x, void* y16, long long numel, float slope, bool bf16, cudaStream_t st);
// x = x32 (PV fp32, ups output) + noise_conv(har): x16 = lrelu(x) as 16-bit channels-last (the activation stream);
// x32 is written back only when write32 (stage taps)
cudaError_t launch_noise_add_pv(const float* har, const float* wn, const float* nb, void* x32, void* x16, bool write32, int B,
                                long long L_har, long long L, int C, int k, int s, int pad, int Lp, int padf, float slope,
                                bool bf16, cudaStream_t st);
// in place on the 16-bit stream: x16 <- lrelu(x16 + noise_conv(har)), x16 holding the transposed conv's raw fp16 output
cudaError_t launch_noise_add16(const float* har, const float* wn, const float* nb, void* x16, int B, long long L_har,
                               long long L, int C, int k, int s, int pad, float slope, cudaStream_t st);
cudaError_t launch_conv_post_pv(const void* x32, const float* w, float* out, int B, long long L, int C, int k, int Lp,
                                int padf, float slope, cudaStream_t st);
// same, x planar-vector fp16 [B][C/8][Lp][8] (k = 7)
cudaError_t launch_conv_post_pv16(const void* x16, const float* w, float* out, int B, long long L, int C, int k, int Lp,
                                  int padf, float slope, cudaStream_t st);
cudaError_t launch_pv16_to_cl(const void* src, float* y, int B, long long L, int C, int Lp, int padf, cudaStream_t st);
cudaError_t launch_pv32_to_cl(const void* src, float* y, int B, long long L, int C, int Lp, int padf, cudaStream_t st);

// tcgen05 flash attention with banded relative-position terms (attention_tc.cu)
cudaError_t launch_attention_tc(const void* qkv16, void* vt, const void* ek16, const void* evt16, const int* len, void* out,
                                int B, int T, int n_heads, int dk, int window, cudaStream_t st);

}  // namespace rvc
