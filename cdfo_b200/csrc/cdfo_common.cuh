// Shared helpers of the cdfo_b200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/cdfo_b200.h"

namespace cdfo {

// thread-local message of the last failing call (cdfo_last_error)
char *last_error_buf();
int fail(int code, const char *fmt, ...);

inline int check_launch(const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return CDFO_OK;
}

constexpr int kNumSMs = 148;  // B200

__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }

inline int conv_out_size(int in, int pad, int dil, int k, int stride) {
  return (in + 2 * pad - (dil * (k - 1) + 1)) / stride + 1;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// Source coordinate of flow_warp's normalise (python, arch/SIDECVSR_our.py:3093-3094) / un-normalise (ATen
// grid_sampler, align_corners=True) round trip, replayed with explicit round-to-nearest ops so that floor() indices are
// bit-exact against the reference arithmetic.
__device__ __forceinline__ float warp_src_coord(int pos, float flow, int size) {
  const float v = __fadd_rn((float)pos, flow);                                              // grid + flow
  const float g = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, v), (float)max(size - 1, 1)), 1.0f);  // 2*v/max(s-1,1) - 1
  return __fmul_rn(__fdiv_rn(__fadd_rn(g, 1.0f), 2.0f), (float)(size - 1));                 // ((g+1)/2)*(s-1)
}

// LLongRangAttention tap tables (csrc/lra.cu, csrc/lra_col_sm100.cu): device pointers, built on the host from directW1_conv / directH1_conv
struct LraTables {
  const float *kw;       // [9] taps along channels
  const float *kh;       // [9] taps along H
  const float *k1;       // [64]    K1[c]      = sum of in-range taps of a bump centred at channel c
  const float *r;        // [64*64] R[c1][c2]  = sum_c kw[c1-c+4] kw[c2-c+4] over in-range c
  float beta, bh;        // biases of directW1_conv / directH1_conv
};
// csrc/lra_col_sm100.cu: tcgen05 column pass; 1 = launched, 0 = shape outside its limits (caller falls back), < 0 = error
int lra_col_sm100_launch(const float *vrow_t, const uint8_t *midx, const float *qsel, float *long_out, const LraTables &t, int B, int H, int W,
                         cudaStream_t s);
// host-only: whether lra_col_sm100_launch takes H rows (no CUDA call)
bool lra_col_sm100_fits(int H);

// csrc/dcn_tex_sm100.cu, csrc/mv_dcn_fused_sm100.cu: the x samples of a texture DCN call are bound as pitch-2D textures of at most
// kTexRows rows (16 * (H + 3) rows per sample; fp32 texture coordinates keep >= 8 fractional bits below 65536 rows).  A call whose x batch
// does not fit is split into the fewest slices of `per` consecutive samples (the last one may be shorter), one launch per slice.
constexpr int kTexRows = 65000;
struct TexSlices { int count, per; };
TexSlices tex_slices(int x_batch, long long sample_rows);

// csrc/pointwise.cu: tensor-core 1x1 convolution (see cdfo_pointwise_conv_fwd in include/cdfo_b200.h)
int pointwise_conv(const float *in1, const float *in2, const float *w, const float *bias, const float *resid1, const float *resid2,
                   float *out, int B, int K, int Co, int HW, int act, int mode, cudaStream_t s, void *out_c8 = nullptr,
                   int out_channels = 0, int channel0 = 0);

// csrc/conv3x3_sm100.cu: weight [Cout][Cin][k][k] fp32 -> [n_tile][tap][Cin/8][NT][8] bf16 (streamed: [n_tile][K block][tap][8][NT][8])
int conv3x3_pack_weight_raw(const float *w, void *out, int Cout, int Cin, int NT, int n_tiles, int streamed, int taps, cudaStream_t s);

}  // namespace cdfo

#define CDFO_REQUIRE(cond, code, ...)                 \
  do {                                                \
    if (!(cond)) return cdfo::fail(code, __VA_ARGS__); \
  } while (0)
