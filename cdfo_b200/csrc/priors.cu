// Coding-prior plumbing on the device: MV -> flow (A1), end-of-sequence fix-up (A2), flow_warp (A3),
// and the NCHW fp32 <-> c8 bf16 layout adapters used by the sm_100a kernels.
//
//   mv2mvs                     test_LD_37.py:83-105 (+ permute :160-161)
//   modify_mv_for_end_frames   test_LD_37.py:209-234
//   flow_warp                  arch/SIDECVSR_our.py:3068-3099 -> F.grid_sample(bilinear, zeros, align_corners=True)
//
// Every fp32 step that decides an integer index is written with explicit round-to-nearest intrinsics
// (__fadd_rn/__fmul_rn/__fdiv_rn) so that nvcc cannot contract or reassociate it: the floor() indices are
// bit-exact against the oracle's restatement of the reference arithmetic.
#include "cdfo_common.cuh"

namespace cdfo {

// ---------------------------------------------------------------- A1
template <typename MV>
__global__ void mv2mvs_kernel(const MV *__restrict__ mv, float *__restrict__ flows, int HW) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  // reference swaps channel 0 <-> 1 first: x-displacement = stored channel 1, y = stored channel 0
  const float a = (float)mv[p * 3 + 1];
  const float b = (float)mv[p * 3 + 0];
  const float den = __fmul_rn((float)mv[p * 3 + 2], -1.0f);
  float fx = __fdiv_rn(a, den), fy = __fdiv_rn(b, den);
  if (isnan(fx)) fx = 0.f;  // only NaN (0/0) is filtered; x/0 stays +-inf like the reference
  if (isnan(fy)) fy = 0.f;
  const float scale[7] = {3.0f, 2.0f, 1.0f, 0.0f, -1.0f, -2.0f, -3.0f};
#pragma unroll
  for (int f = 0; f < 7; ++f) {
    float vx, vy;
    if (f == 2) { vx = fx; vy = fy; }
    else if (f == 3) { vx = 0.f; vy = 0.f; }  // centre slot is never written by the reference: stays +0
    else { vx = __fmul_rn(fx, scale[f]); vy = __fmul_rn(fy, scale[f]); }
    flows[((size_t)f * 2 + 0) * HW + p] = __fdiv_rn(vx, 128.0f);
    flows[((size_t)f * 2 + 1) * HW + p] = __fdiv_rn(vy, 128.0f);
  }
}

// RA twin (opt/data_RA_bi.py:419-424,496-533 + the / 32 of train_RA_37.py:383-386): frame 2 = l0 / -refdist, frame 4 = l1 / refdist
// (no sign flip), NaN -> 0, refdist == -99 marks a missing list: frame 2 <- -frame 4 (raw), then frame 4 <- -frame 2 (already
// complemented), frames 1, 0 = 2x, 3x frame 2; 5, 6 = 2x, 3x frame 4; (/ 4) / 32.  Every step is one IEEE fp32 operation.
template <typename MV>
__global__ void mv2mvs_ra_kernel(const MV *__restrict__ l0, const MV *__restrict__ l1, float *__restrict__ flows, int HW) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const float d0 = (float)l0[p * 3 + 2], d1 = (float)l1[p * 3 + 2];
  const float n0 = __fmul_rn(d0, -1.0f);
  // channel swap first: x = stored channel 1, y = stored channel 0
  float x2 = __fdiv_rn((float)l0[p * 3 + 1], n0), y2 = __fdiv_rn((float)l0[p * 3 + 0], n0);
  float x4 = __fdiv_rn((float)l1[p * 3 + 1], d1), y4 = __fdiv_rn((float)l1[p * 3 + 0], d1);
  if (isnan(x2)) x2 = 0.f;
  if (isnan(y2)) y2 = 0.f;
  if (isnan(x4)) x4 = 0.f;
  if (isnan(y4)) y4 = 0.f;
  if (d0 == -99.f) { x2 = __fmul_rn(x4, -1.f); y2 = __fmul_rn(y4, -1.f); }
  if (d1 == -99.f) { x4 = __fmul_rn(x2, -1.f); y4 = __fmul_rn(y2, -1.f); }
  const float vx[7] = {__fmul_rn(x2, 3.f), __fmul_rn(x2, 2.f), x2, 0.f, x4, __fmul_rn(x4, 2.f), __fmul_rn(x4, 3.f)};
  const float vy[7] = {__fmul_rn(y2, 3.f), __fmul_rn(y2, 2.f), y2, 0.f, y4, __fmul_rn(y4, 2.f), __fmul_rn(y4, 3.f)};
#pragma unroll
  for (int f = 0; f < 7; ++f) {
    flows[((size_t)f * 2 + 0) * HW + p] = __fdiv_rn(__fdiv_rn(vx[f], 4.0f), 32.0f);
    flows[((size_t)f * 2 + 1) * HW + p] = __fdiv_rn(__fdiv_rn(vy[f], 4.0f), 32.0f);
  }
}

// ---------------------------------------------------------------- A2
// dst slot <- src slot (src >= 0) or 0 (src < 0) for every sample; slot = 2*H*W floats.
__global__ void mv_slot_kernel(float *__restrict__ flows, int B, int slot_elems, int dst, int src) {
  const size_t total = (size_t)B * slot_elems;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const size_t b = e / slot_elems, r = e % slot_elems;
    float *base = flows + b * 7 * (size_t)slot_elems;
    base[(size_t)dst * slot_elems + r] = src < 0 ? 0.f : base[(size_t)src * slot_elems + r];
  }
}

// A2 per sample: one thread per (pixel, sample) holds both flow components of the 7 frames in registers and applies the six
// conditional slot copies of modify_mv_for_end_frames in the reference's statement order (test_LD_37.py:209-234), with the
// sample's own (i, max_idx) from the device table i_max [B, 2].  Only the frame slots a condition rewrote are stored.
__global__ void mv_end_fix_batched_kernel(float *__restrict__ flows, int HW, const int *__restrict__ i_max) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (p >= HW) return;
  const int i = __ldg(i_max + 2 * b), m = __ldg(i_max + 2 * b + 1);
  const bool lo = i >= 0 && i <= 2, hi = i >= m - 3 && i <= m - 1;
  if (!lo && !hi) return;
  const size_t slot = 2 * (size_t)HW;
  float *base = flows + (size_t)b * 7 * slot + p;
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    float *f = base + (size_t)c * HW;
    float v[7];
#pragma unroll
    for (int t = 0; t < 7; ++t) v[t] = f[t * slot];
    if (i == 0) { v[0] = 0.f; v[1] = 0.f; v[2] = 0.f; }
    if (i == 1) { v[0] = v[2]; v[1] = v[2]; }
    if (i == 2) { v[0] = v[1]; }
    if (i == m - 1) { v[4] = 0.f; v[5] = 0.f; v[6] = 0.f; }
    if (i == m - 2) { v[5] = v[4]; v[6] = v[4]; }
    if (i == m - 3) { v[6] = v[5]; }
    if (lo) {
#pragma unroll
      for (int t = 0; t < 3; ++t) f[t * slot] = v[t];
    }
    if (hi) {
#pragma unroll
      for (int t = 4; t < 7; ++t) f[t * slot] = v[t];
    }
  }
}

// ---------------------------------------------------------------- A3
constexpr int kWarpCh = 8;  // channels per thread

__global__ void flow_warp_kernel(const float *__restrict__ x, const float *__restrict__ flow, float *__restrict__ y,
                                 int C, int H, int W, int32_t *__restrict__ idx) {
  const int HW = H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const int b = blockIdx.z, c0 = blockIdx.y * kWarpCh;
  const int h = p / W, w = p % W;
  const float ix = warp_src_coord(w, flow[((size_t)b * 2 + 0) * HW + p], W);
  const float iy = warp_src_coord(h, flow[((size_t)b * 2 + 1) * HW + p], H);
  const float fx = floorf(ix), fy = floorf(iy);
  const int x0 = (int)fx, y0 = (int)fy, x1 = x0 + 1, y1 = y0 + 1;
  const float tx1 = __fsub_rn((float)x1, ix), tx0 = __fsub_rn(ix, fx);
  const float ty1 = __fsub_rn((float)y1, iy), ty0 = __fsub_rn(iy, fy);
  const float nw = tx1 * ty1, ne = tx0 * ty1, sw = tx1 * ty0, se = tx0 * ty0;
  const bool ok_y0 = y0 >= 0 && y0 < H, ok_y1 = y1 >= 0 && y1 < H;
  const bool ok_x0 = x0 >= 0 && x0 < W, ok_x1 = x1 >= 0 && x1 < W;
  if (idx && blockIdx.y == 0) {
    idx[((size_t)b * HW + p) * 2 + 0] = y0;
    idx[((size_t)b * HW + p) * 2 + 1] = x0;
  }
#pragma unroll
  for (int cc = 0; cc < kWarpCh; ++cc) {
    const int c = c0 + cc;
    if (c >= C) break;
    const float *plane = x + ((size_t)b * C + c) * HW;
    float acc = 0.f;
    if (ok_y0 && ok_x0) acc += plane[y0 * W + x0] * nw;
    if (ok_y0 && ok_x1) acc += plane[y0 * W + x1] * ne;
    if (ok_y1 && ok_x0) acc += plane[y1 * W + x0] * sw;
    if (ok_y1 && ok_x1) acc += plane[y1 * W + x1] * se;
    y[((size_t)b * C + c) * HW + p] = acc;
  }
}

// ---------------------------------------------------------------- layout adapters
// out has out_chunks 8-channel chunks per sample; the C / 8 chunks of x go to [chunk0, chunk0 + C / 8) (a channel concatenation
// is then two packs into one tensor instead of a cat + pack)
__global__ void pack_c8_kernel(const float *__restrict__ x, uint4 *__restrict__ out, int C, int HW, int out_chunks, int chunk0) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const int c8 = blockIdx.y, b = blockIdx.z;
  const float *src = x + ((size_t)b * C + c8 * 8) * HW + p;
  __nv_bfloat162 v[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = __floats2bfloat162_rn(src[(size_t)(2 * i) * HW], src[(size_t)(2 * i + 1) * HW]);
  out[((size_t)b * out_chunks + chunk0 + c8) * HW + p] = *reinterpret_cast<uint4 *>(v);
}

__global__ void unpack_c8_kernel(const uint4 *__restrict__ in, float *__restrict__ y, int C, int HW) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const int c8 = blockIdx.y, b = blockIdx.z;
  uint4 raw = in[((size_t)b * (C / 8) + c8) * HW + p];
  const __nv_bfloat162 *v = reinterpret_cast<const __nv_bfloat162 *>(&raw);
  float *dst = y + ((size_t)b * C + c8 * 8) * HW + p;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __bfloat1622float2(v[i]);
    dst[(size_t)(2 * i) * HW] = f.x;
    dst[(size_t)(2 * i + 1) * HW] = f.y;
  }
}

// ---------------------------------------------------------------- A9: prior embedding convs
// conv_expand_ufs / conv_expand_rms (arch/SIDECVSR_our.py:4383-4384, :4446-4447): nn.Conv2d(1, Co, 3, 1, 1) on a one-channel
// prior map.  One thread per pixel holds its 3x3 neighbourhood in registers and writes Co channels (coalesced along the
// pixels of each channel plane): 4 * Co bytes written per pixel, HBM-bound.
__global__ void __launch_bounds__(128) prior_conv_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                                         const float *__restrict__ bias, float *__restrict__ y, int Co, int H, int W, int relu) {
  extern __shared__ float ws[];   // [Co][9] weights + [Co] bias
  for (int e = threadIdx.x; e < Co * 9; e += blockDim.x) ws[e] = w[e];
  for (int e = threadIdx.x; e < Co; e += blockDim.x) ws[Co * 9 + e] = bias ? bias[e] : 0.f;
  __syncthreads();
  const int HW = H * W, p = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (p >= HW) return;
  const int h = p / W, wq = p - h * W;
  const float *xp = x + (size_t)b * HW;
  float v[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int hh = h + i - 1, ww = wq + j - 1;
      v[i * 3 + j] = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? __ldg(xp + hh * W + ww) : 0.f;
    }
  float *yp = y + (size_t)b * Co * HW + p;
  for (int c = 0; c < Co; ++c) {
    float acc = ws[Co * 9 + c];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc = fmaf(ws[c * 9 + k], v[k], acc);   // same tap order as a direct fp32 convolution
    __stcs(yp + (size_t)c * HW, relu ? fmaxf(acc, 0.f) : acc);
  }
}

}  // namespace cdfo

using namespace cdfo;

extern "C" int cdfo_prior_conv_act_fwd(const float *x, const float *w, const float *bias, float *y, int B, int Co, int H, int W, int relu,
                                       void *stream) {
  CDFO_REQUIRE(x && w && y, CDFO_ERR_NULL, "cdfo_prior_conv_fwd: NULL pointer");
  CDFO_REQUIRE(B > 0 && B <= 65535 && Co > 0 && Co <= 1024 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_prior_conv_fwd: bad shape");
  prior_conv_kernel<<<dim3(ceil_div(H * W, 128), B), 128, (size_t)Co * 10 * 4, (cudaStream_t)stream>>>(x, w, bias, y, Co, H, W, relu ? 1 : 0);
  return check_launch("cdfo_prior_conv_fwd");
}

extern "C" int cdfo_prior_conv_fwd(const float *x, const float *w, const float *bias, float *y, int B, int Co, int H, int W, void *stream) {
  return cdfo_prior_conv_act_fwd(x, w, bias, y, B, Co, H, W, 0, stream);
}

extern "C" int cdfo_mv2mvs(const void *mv, int mv_is_int32, float *flows, int H, int W, void *stream) {
  CDFO_REQUIRE(mv && flows, CDFO_ERR_NULL, "cdfo_mv2mvs: NULL pointer");
  CDFO_REQUIRE(H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_mv2mvs: bad size %d x %d", H, W);
  const int HW = H * W;
  cudaStream_t s = (cudaStream_t)stream;
  if (mv_is_int32) mv2mvs_kernel<int32_t><<<ceil_div(HW, 256), 256, 0, s>>>((const int32_t *)mv, flows, HW);
  else mv2mvs_kernel<int8_t><<<ceil_div(HW, 256), 256, 0, s>>>((const int8_t *)mv, flows, HW);
  return check_launch("cdfo_mv2mvs");
}

extern "C" int cdfo_mv2mvs_ra(const void *mv_l0, const void *mv_l1, int mv_is_int32, float *flows, int H, int W, void *stream) {
  CDFO_REQUIRE(mv_l0 && mv_l1 && flows, CDFO_ERR_NULL, "cdfo_mv2mvs_ra: NULL pointer");
  CDFO_REQUIRE(H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_mv2mvs_ra: bad size %d x %d", H, W);
  const int HW = H * W;
  cudaStream_t s = (cudaStream_t)stream;
  if (mv_is_int32) mv2mvs_ra_kernel<int32_t><<<ceil_div(HW, 256), 256, 0, s>>>((const int32_t *)mv_l0, (const int32_t *)mv_l1, flows, HW);
  else mv2mvs_ra_kernel<int8_t><<<ceil_div(HW, 256), 256, 0, s>>>((const int8_t *)mv_l0, (const int8_t *)mv_l1, flows, HW);
  return check_launch("cdfo_mv2mvs_ra");
}

extern "C" int cdfo_mv_end_fix(float *flows, int B, int H, int W, int i, int max_idx, void *stream) {
  CDFO_REQUIRE(flows, CDFO_ERR_NULL, "cdfo_mv_end_fix: NULL pointer");
  CDFO_REQUIRE(B > 0 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_mv_end_fix: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  const int slot = 2 * H * W;
  const int blocks = min(kNumSMs * 4, ceil_div(B * slot, 256));
  auto op = [&](int dst, int src) { mv_slot_kernel<<<blocks, 256, 0, s>>>(flows, B, slot, dst, src); };
  // same statement order as the reference (several conditions can hold at once on short sequences)
  if (i == 0) { op(0, -1); op(1, -1); op(2, -1); }
  if (i == 1) { op(0, 2); op(1, 2); }
  if (i == 2) { op(0, 1); }
  if (i == max_idx - 1) { op(4, -1); op(5, -1); op(6, -1); }
  if (i == max_idx - 2) { op(5, 4); op(6, 4); }
  if (i == max_idx - 3) { op(6, 5); }
  return check_launch("cdfo_mv_end_fix");
}

extern "C" int cdfo_mv_end_fix_batched(float *flows, int B, int H, int W, const int *i_max, void *stream) {
  CDFO_REQUIRE(flows && i_max, CDFO_ERR_NULL, "cdfo_mv_end_fix_batched: NULL pointer");
  CDFO_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0 && (long long)H * W <= INT_MAX / 2, CDFO_ERR_SHAPE,
               "cdfo_mv_end_fix_batched: bad shape B=%d H=%d W=%d", B, H, W);
  const int HW = H * W;
  mv_end_fix_batched_kernel<<<dim3(ceil_div(HW, 256), B), 256, 0, (cudaStream_t)stream>>>(flows, HW, i_max);
  return check_launch("cdfo_mv_end_fix_batched");
}

extern "C" int cdfo_flow_warp_fwd(const float *x, const float *flow, float *y, int B, int C, int H, int W,
                                  int32_t *idx, void *stream) {
  CDFO_REQUIRE(x && flow && y, CDFO_ERR_NULL, "cdfo_flow_warp_fwd: NULL pointer");
  CDFO_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && B <= 65535, CDFO_ERR_SHAPE, "cdfo_flow_warp_fwd: bad shape");
  dim3 grid(ceil_div(H * W, 128), ceil_div(C, kWarpCh), B);
  flow_warp_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(x, flow, y, C, H, W, idx);
  return check_launch("cdfo_flow_warp_fwd");
}

extern "C" int cdfo_pack_c8(const float *x_nchw, void *x_c8, int B, int C, int H, int W, void *stream) {
  CDFO_REQUIRE(x_nchw && x_c8, CDFO_ERR_NULL, "cdfo_pack_c8: NULL pointer");
  CDFO_REQUIRE(B > 0 && C > 0 && C % 8 == 0 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_pack_c8: C %% 8 != 0 or bad shape");
  dim3 grid(ceil_div(H * W, 128), C / 8, B);
  pack_c8_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(x_nchw, (uint4 *)x_c8, C, H * W, C / 8, 0);
  return check_launch("cdfo_pack_c8");
}

extern "C" int cdfo_pack_c8_into(const float *x_nchw, void *x_c8, int B, int C, int H, int W, int out_channels, int channel0, void *stream) {
  CDFO_REQUIRE(x_nchw && x_c8, CDFO_ERR_NULL, "cdfo_pack_c8_into: NULL pointer");
  CDFO_REQUIRE(B > 0 && B <= 65535 && C > 0 && C % 8 == 0 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_pack_c8_into: C %% 8 != 0 or bad shape");
  CDFO_REQUIRE(out_channels % 8 == 0 && channel0 % 8 == 0 && channel0 >= 0 && channel0 + C <= out_channels, CDFO_ERR_SHAPE,
               "cdfo_pack_c8_into: channels [%d, %d) do not fit %d output channels (multiples of 8)", channel0, channel0 + C, out_channels);
  dim3 grid(ceil_div(H * W, 128), C / 8, B);
  pack_c8_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(x_nchw, (uint4 *)x_c8, C, H * W, out_channels / 8, channel0 / 8);
  return check_launch("cdfo_pack_c8_into");
}

extern "C" int cdfo_unpack_c8(const void *x_c8, float *x_nchw, int B, int C, int H, int W, void *stream) {
  CDFO_REQUIRE(x_nchw && x_c8, CDFO_ERR_NULL, "cdfo_unpack_c8: NULL pointer");
  CDFO_REQUIRE(B > 0 && C > 0 && C % 8 == 0 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_unpack_c8: C %% 8 != 0 or bad shape");
  dim3 grid(ceil_div(H * W, 128), C / 8, B);
  unpack_c8_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>((const uint4 *)x_c8, x_nchw, C, H * W);
  return check_launch("cdfo_unpack_c8");
}
