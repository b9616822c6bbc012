// Bilinear x2 / x0.5 resampling (F.interpolate, align_corners=False) on channel-chunked bf16 activations, and the
// three-scale sum of the reconstruction trunk's cross-scale block:
//   Block_.forward  arch/SIDECVSR_our.py:401-406   out = x + body(x) + up(body(down(x))) + down(body(up(x)))
//   Interpolate     arch/SIDECVSR_our.py:324-333   bilinear, align_corners=False, scale 0.5 / 2.0
// scale 0.5 on an even size = the mean of each 2x2 block (source coordinate 2d + 0.5); scale 2: source = d/2 - 0.25
// clamped at 0 -> weights (0.25, 0.75) / (0.75, 0.25) with the edge pixel repeated.  One thread per output pixel and
// 8-channel chunk (16 bytes in, 16 bytes out, fp32 arithmetic): pure HBM-bound kernels.
#include "cdfo_common.cuh"
#include "up2_blend.cuh"

namespace cdfo {
namespace rs {

using up2::F8;
using up2::pack;
using up2::unpack;

__device__ __forceinline__ void axpy(F8 &acc, float w, const uint4 q) {
  const F8 t = unpack(q);
#pragma unroll
  for (int i = 0; i < 8; ++i) acc.v[i] = fmaf(w, t.v[i], acc.v[i]);
}

// mean of the 2x2 block at (2h, 2w) of a [H2][W2] plane (H2 = 2 Ho, W2 = 2 Wo)
__device__ __forceinline__ void avg2_acc(F8 &acc, const uint4 *plane, int h, int w, int W2) {
  const uint4 *p = plane + (size_t)(2 * h) * W2 + 2 * w;
  axpy(acc, 0.25f, __ldg(p));
  axpy(acc, 0.25f, __ldg(p + 1));
  axpy(acc, 0.25f, __ldg(p + W2));
  axpy(acc, 0.25f, __ldg(p + W2 + 1));
}
// bilinear x2 sample at output (h, w) of a [Hi][Wi] plane
__device__ __forceinline__ void up2_acc(F8 &acc, const uint4 *plane, int h, int w, int Hi, int Wi) {
  const int hk = h >> 1, wk = w >> 1;
  const int h0 = (h & 1) ? hk : max(hk - 1, 0), h1 = (h & 1) ? min(hk + 1, Hi - 1) : hk;
  const int w0 = (w & 1) ? wk : max(wk - 1, 0), w1 = (w & 1) ? min(wk + 1, Wi - 1) : wk;
  // weight of the first tap: odd output -> 0.75 on the nearer (first) pixel, even output -> 0.25 on the farther (first)
  const float ah = (h & 1) ? 0.75f : 0.25f, aw = (w & 1) ? 0.75f : 0.25f;
  axpy(acc, ah * aw, __ldg(plane + (size_t)h0 * Wi + w0));
  axpy(acc, ah * (1.f - aw), __ldg(plane + (size_t)h0 * Wi + w1));
  axpy(acc, (1.f - ah) * aw, __ldg(plane + (size_t)h1 * Wi + w0));
  axpy(acc, (1.f - ah) * (1.f - aw), __ldg(plane + (size_t)h1 * Wi + w1));
}

// mode 0: y[Ho,Wo] = avg2(a[2Ho,2Wo]);  mode 1: y[Ho,Wo] = up2(a[Ho/2,Wo/2]);
// mode 2: y[Ho,Wo] = base[Ho,Wo] + avg2(a[2Ho,2Wo]) + up2(b[Ho/2,Wo/2]);  mode 3: y = base + up2(b)   (planes = B * C/8)
__global__ void resample_c8_kernel(const uint4 *__restrict__ a, const uint4 *__restrict__ b, const uint4 *__restrict__ base,
                                   uint4 *__restrict__ y, int Ho, int Wo, int mode) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= Ho * Wo) return;
  const int plane = blockIdx.y;
  const int h = pix / Wo, w = pix - h * Wo;
  F8 acc;
#pragma unroll
  for (int i = 0; i < 8; ++i) acc.v[i] = 0.f;
  if (mode == 0) {
    avg2_acc(acc, a + (size_t)plane * 4 * Ho * Wo, h, w, 2 * Wo);
  } else if (mode == 1) {
    up2_acc(acc, a + (size_t)plane * (Ho / 2) * (Wo / 2), h, w, Ho / 2, Wo / 2);
  } else if (mode == 2) {
    axpy(acc, 1.f, __ldg(base + (size_t)plane * Ho * Wo + pix));
    avg2_acc(acc, a + (size_t)plane * 4 * Ho * Wo, h, w, 2 * Wo);
    up2_acc(acc, b + (size_t)plane * (Ho / 2) * (Wo / 2), h, w, Ho / 2, Wo / 2);
  } else {
    axpy(acc, 1.f, __ldg(base + (size_t)plane * Ho * Wo + pix));
    up2_acc(acc, b + (size_t)plane * (Ho / 2) * (Wo / 2), h, w, Ho / 2, Wo / 2);
  }
  y[(size_t)plane * Ho * Wo + pix] = pack(acc);
}


// Bilinear x2 with one thread per INPUT pixel and 8-channel chunk: its 3x3 neighbourhood (edge pixels repeated) gives the 2x2 outputs
// (2i .. 2i+1, 2j .. 2j+1) -- 2.25 loads per output instead of 4, each input unpacked once, separable blends (columns, then rows), and
// 32 contiguous bytes stored per thread and output row.  Same fp32 weights as up2_acc (products of 0.25 / 0.75 are exact), summed in a
// different order: results agree to one bf16 rounding of the output.
__global__ void upsample2_c8_kernel(const uint4 *__restrict__ a, uint4 *__restrict__ y, int Hi, int Wi) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= Hi * Wi) return;
  const int plane = blockIdx.y;
  const int i = pix / Wi, j = pix - i * Wi;
  const uint4 *src = a + (size_t)plane * Hi * Wi;
  const int jm = max(j - 1, 0), jp = min(j + 1, Wi - 1);
  const int rows[3] = {max(i - 1, 0), i, min(i + 1, Hi - 1)};
  F8 l[3], r[3];                       // per source row: output columns 2j (0.25 x[j-1] + 0.75 x[j]) and 2j+1 (0.75 x[j] + 0.25 x[j+1])
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const uint4 *row = src + (size_t)rows[k] * Wi;
    const F8 xm = unpack(__ldg(row + jm)), x0 = unpack(__ldg(row + j)), xp = unpack(__ldg(row + jp));
    l[k] = up2::blend(xm, x0);
    r[k] = up2::blend(xp, x0);
  }
  // rows 2i (0.25 row[i-1] + 0.75 row[i]) and 2i+1 (0.75 row[i] + 0.25 row[i+1])
  const F8 o00 = up2::blend(l[0], l[1]), o01 = up2::blend(r[0], r[1]), o10 = up2::blend(l[2], l[1]), o11 = up2::blend(r[2], r[1]);
  uint4 *d = y + (size_t)plane * 4 * Hi * Wi + (size_t)(2 * i) * (2 * Wi) + 2 * j;
  d[0] = pack(o00);
  d[1] = pack(o01);
  d[2 * Wi] = pack(o10);
  d[2 * Wi + 1] = pack(o11);
}

}  // namespace rs
}  // namespace cdfo

using namespace cdfo;

// mode 0: a [B,C/8,2Ho,2Wo,8] -> y [B,C/8,Ho,Wo,8] (bilinear x0.5); mode 1: a [B,C/8,Ho/2,Wo/2,8] -> y (bilinear x2);
// mode 2: y = base [Ho,Wo] + x0.5(a [2Ho,2Wo]) + x2(b [Ho/2,Wo/2]);  mode 3: y = base + x2(b) (a unused).  Ho, Wo even.
extern "C" int cdfo_resample_c8(const void *a, const void *b, const void *base, void *y, int B, int C, int Ho, int Wo, int mode,
                                void *stream) {
  CDFO_REQUIRE(y && (mode == 3 || a) && (mode < 2 || (b && base)), CDFO_ERR_NULL, "cdfo_resample_c8: NULL pointer");
  CDFO_REQUIRE(B > 0 && C > 0 && C % 8 == 0 && Ho > 0 && Wo > 0 && (long long)B * (C / 8) <= 65535, CDFO_ERR_SHAPE, "cdfo_resample_c8: bad shape");
  CDFO_REQUIRE(mode >= 0 && mode <= 3, CDFO_ERR_UNSUPPORTED, "cdfo_resample_c8: mode %d", mode);
  CDFO_REQUIRE(mode == 0 || (Ho % 2 == 0 && Wo % 2 == 0), CDFO_ERR_SHAPE, "cdfo_resample_c8: x2 output size must be even");
  if (mode == 1) {
    const int Hi = Ho / 2, Wi = Wo / 2;
    rs::upsample2_c8_kernel<<<dim3(ceil_div(Hi * Wi, 128), B * (C / 8)), 128, 0, (cudaStream_t)stream>>>((const uint4 *)a, (uint4 *)y, Hi, Wi);
    return check_launch("cdfo_resample_c8");
  }
  dim3 grid(ceil_div(Ho * Wo, 256), B * (C / 8));
  rs::resample_c8_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint4 *)a, (const uint4 *)b, (const uint4 *)base, (uint4 *)y, Ho, Wo, mode);
  return check_launch("cdfo_resample_c8");
}
