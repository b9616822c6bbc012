// Bilinear x2 (F.interpolate, align_corners=False) of c8 bf16 activations: the arithmetic shared by the stand-alone resampling kernel
// (resample.cu, upsample2_c8_kernel) and the A-operand builder of the 64 -> 256 convolution that reads the 1x image
// (conv3x3_pair_sm100.cu, UP2).  Both must produce the same bf16 values bit for bit, so both call these helpers and nothing else.
//   output 2i + d (d = 0 / 1) of source index i = blend(x[i - 1 + 2d], x[i]) with the source index clamped to the image,
//   evaluated on columns first, then on rows, in fp32, rounded to bf16 once.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace cdfo {
namespace up2 {

struct F8 { float v[8]; };

__device__ __forceinline__ F8 unpack(const uint4 q) {
  F8 r;
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    r.v[2 * i] = __uint_as_float(w[i] << 16);
    r.v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
  return r;
}
__device__ __forceinline__ uint32_t bf2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t *>(&v);
}
__device__ __forceinline__ uint4 pack(const F8 &a) {
  return make_uint4(bf2(a.v[0], a.v[1]), bf2(a.v[2], a.v[3]), bf2(a.v[4], a.v[5]), bf2(a.v[6], a.v[7]));
}
// one separable step: 0.75 on the source pixel the output lies in, 0.25 on its neighbour towards the output
__device__ __forceinline__ F8 blend(const F8 &nb, const F8 &x) {
  F8 r;
#pragma unroll
  for (int c = 0; c < 8; ++c) r.v[c] = fmaf(0.25f, nb.v[c], 0.75f * x.v[c]);
  return r;
}

}  // namespace up2
}  // namespace cdfo
