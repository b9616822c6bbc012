// Modulated deformable convolution (DCNv2) forward at the model's hot shape, third generation of the sm_100a kernel:
// the bilinear gather runs on the TEXTURE UNITS.
//
// Semantics: ops/dcn/src/deform_conv_cuda_kernel.cu:467-496,570-632 + deform_conv_cuda.cpp:486-564
// (= torchvision.ops.deform_conv2d at arch/SIDECVSR_our.py:3352) with offset = learned residual + decoded MV prior
// (arch/SIDECVSR_our.py:3347), C = Co = 64, 3x3, stride = pad = dil = 1, groups = 1, dg | 16.
//
// Why textures: ncu on the LSU-gather kernel (dcn_sm100.cu, profiles/r01_dcn_sm100_v2_ncu.md) and on the gather probe
// (tools/gather_probe.cu, profiles/r01_gather_probe.md) shows that the binding resource of this op is neither HBM nor
// the issue slots but the L1TEX data stage (~1 wavefront / clk / SM, shared by LDG, LDS/STS and TEX): an LDG gather of
// the 2x2 footprint costs 16-20 wavefronts per 32 samples and ~50 instructions per sample; one hardware-filtered
// fetch of an fp16x4 texel costs 15 wavefronts and ~20 instructions, independent of how scattered the offsets are.
//   * x lives in HBM as "q4t": [xB][16 quads][H+3][Wpt] texels of 4 fp16 channels with the same zero border as q4p
//     (1 before, 2 after; Wpt = W+3 rounded up to 4 texels so that the row pitch is 32-byte aligned); every sample
//     the whole tensor is ONE pitch-linear 2-D texture whose row axis folds (sample, quad plane, row).  The reference's inside test and its
//     per-corner zero padding become: clamp the sample position to [-1, H] x [-1, W], read the zero border.
//   * offsets / mask arrive as packed fields [B][9 taps][dg/gp][H*W][gp] x fp16x4 (dy, dx, mask, 0), gp = 2 for dg = 16
//     (a warp's 32 pixels x 2 groups = 512 contiguous bytes per 16-byte load), else 1 -- what the fused head
//     (conv3x3_sm100.cu) writes; the MV prior is added here, in the reference's fp32 order (residual + flow, then
//     base + offset).
//   * the filter weights are the texture unit's (8 fractional bits): the blended value deviates from the fp32
//     bilinear by <= 2^-9 of the local texel differences, the same order as the bf16/fp16 rounding of the A operand;
//     the exact-arithmetic gather (bit-exact floor indices, cdfo_dcn_sample_index) stays available in dcn_sm100.cu.
//   * implicit GEMM: producers write the fp16 A operand of a tap (128 px x 64 ci) with tcgen05.st into a 4-stage ring in
//     TENSOR MEMORY (32 columns per stage, two K elements per column) -- the operand never touches shared memory, whose
//     data stage is the bottleneck -- one thread issues tcgen05.mma with A in TMEM (M128 N64 K16, fp16 -> fp32), 4 warps
//     drain the accumulator (+ bias) to NCHW fp32 or c8 bf16.  Producers are software-pipelined two taps deep
//     (fields of tap t+2 and the texture fetches of tap t+1 are in flight while tap t is packed).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "cdfo_common.cuh"
#include "sm100_ptx.cuh"

namespace cdfo {
namespace dtex {

constexpr int kTileM = 128;
constexpr int kTileH = 4, kTileW = 32;
constexpr int kStages = 4;
constexpr int kEpiWarps = 4;
constexpr int kProdWarps = 16;
constexpr int kProdThreads = kProdWarps * 32;
constexpr int kWBytes = 9 * 64 * 64 * 2;
constexpr int kABytes = kTileM * 64 * 2;
constexpr int kALbo = kTileM * 16;
constexpr int kBLbo = 64 * 16;
constexpr int kSbo = 128;
constexpr int kTapWBytes = 64 * 64 * 2;
constexpr int kTmemCols = 256;        // [0,64) accumulator, [64,192) A operand ring: 4 stages x 32 columns (128 rows x 64 fp16)
constexpr int kAColBase = 64, kAColsPerStage = 32;

struct Params {
  cudaTextureObject_t tex;           // ONE pitch-2D texture over the x samples [x0, x0 + xn): rows = ((sample - x0) * 16 + quad) * (H + 3) + row
  const uint2 *fields;               // [B][9 taps][dg/gp][H*W][gp] (dy, dx, m, 0) fp16, gp = 2 when dg = 16, else 1
  const float *mv;                   // [B][2][H*W] (x, y) or nullptr
  const uint8_t *wpk;                // [9][8][64][8] fp16
  const float *bias;
  void *y;
  int B, H, W, dg, out_mode, gshift, x_batch;
  int x0, xn;                        // this launch's x slice: the tiles enumerate samples b = k * x_batch + j, j in [x0, x0 + xn)
  long long f_bstride;               // uint2 elements between samples of fields
  // c8 output placement: sample s goes to 8-channel chunks [(s % y_nb) * y_cs + y_grp[s / y_nb], +8) of y
  // (dense: y_nb = B, y_cs = 8, y_grp[0] = 0; stacked for tsa_fusion: y_nb = sequences, y_cs = 56, y_grp = frame slot * 8)
  int y_nb, y_cs, y_grp[8];
  int tiles_x, tiles_per_img, num_tiles;
};

// Mode 2 (dg = 16, dense fields): the fields of a (tile, tap) = 8 group-pair planes x 4 rows x 512 bytes arrive as ONE tiled TMA
// box in a 6-stage shared-memory ring, issued by a dedicated warp; producers read them with two conflict-free LDS.128.  An
// L1-missing LDG.128 costs the L1TEX data stage ~11 wavefronts per 512-byte warp request (fill + read-out), an LDS.128 costs 4,
// and that stage is what bounds this kernel (profiles/r01_dcn_tex_ncu.md).
constexpr int kFStages = 6;
constexpr int kFStageBytes = 8 * kTileH * kTileW * 16;      // 16 KB
constexpr int kFRingOff = (kWBytes + 256 + 32 * 8 + 16 + 1023) & ~1023;
constexpr int kBarFFull = 16, kBarFEmpty = 24;
constexpr size_t smem_bytes(int mode) { return mode == 2 ? (size_t)kFRingOff + kFStages * kFStageBytes : (size_t)kWBytes + 256 + 32 * 8 + 16; }

__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t *>(&v);
}
__device__ __forceinline__ uint32_t h2_as_u32(__half2 v) { return *reinterpret_cast<uint32_t *>(&v); }
// streaming 8-byte load that does not allocate in L1: the fields are read exactly once, and an allocating miss costs
// the L1TEX data stage ~6.6 wavefronts per 256-byte warp request (fill + read-out) instead of the 2 of the payload.
__device__ __forceinline__ uint4 ld_stream_u4(const uint4 *p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ uint2 ld_stream_u2(const uint2 *p) {
  uint2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}

struct TileCoord { int b, h0, w0; };
__device__ __forceinline__ TileCoord tile_coord(const Params &p, int tile) {
  TileCoord t;
  const int bl = tile / p.tiles_per_img;               // sample within this launch's x slice
  const int r = tile - bl * p.tiles_per_img;
  t.b = bl + (bl / p.xn) * (p.x_batch - p.xn) + p.x0;  // = bl when the slice is the whole x batch
  const int ty = r / p.tiles_x;
  t.h0 = ty * kTileH;
  t.w0 = (r - ty * p.tiles_x) * kTileW;
  return t;
}

// instruction descriptor: fp16 x fp16 -> fp32, both K-major
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// kMode 0: dg < 16 (per-group LDG of the fields); 1: dg = 16, two coalesced LDG.128 per tap; 2: dg = 16, fields staged by TMA
template <int kMode>
__global__ void __launch_bounds__((kEpiWarps + kProdWarps) * 32, 1)
dcn_tex_sm100_kernel(const __grid_constant__ Params p, const __grid_constant__ CUtensorMap ftm) {
  constexpr bool kDG16 = kMode != 0;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *wsm = smem;
  float *bias_s = reinterpret_cast<float *>(smem + kWBytes);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kWBytes + 256);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 32);
  // barrier map: [0,4) A stage full, [4,8) A stage empty, 8 accumulator full, 12 weights, [16,22) fields full, [24,30) fields empty
  const uint32_t bar0 = ptx::smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int P = p.H * p.W;

  if (tid < 64) bias_s[tid] = p.bias ? p.bias[tid] : 0.f;
  if (warp == 0) {
    if (lane == 0) {
      for (int s = 0; s < kStages; ++s) {
        ptx::mbar_init(BAR(s), kProdThreads);
        ptx::mbar_init(BAR(4 + s), 1);
      }
      ptx::mbar_init(BAR(8), 1);
      ptx::mbar_init(BAR(12), 1);
      if (kMode == 2)
        for (int s = 0; s < kFStages; ++s) {
          ptx::mbar_init(BAR(kBarFFull + s), 1);
          ptx::mbar_init(BAR(kBarFEmpty + s), kProdWarps);
        }
      ptx::fence_mbar_init();
      ptx::mbar_arrive_expect_tx(BAR(12), kWBytes);
      for (int t = 0; t < 9; ++t)
        ptx::bulk_g2s(ptx::smem_u32(wsm) + t * kTapWBytes, p.wpk + t * kTapWBytes, kTapWBytes, BAR(12));
    }
    __syncwarp();
    ptx::tmem_alloc(ptx::smem_u32(tmem_slot), kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kEpiWarps) {
    // ============ warp 0 lane 0 issues the MMAs of a tile, then all 4 warps drain TMEM ============
    const uint32_t idesc = make_idesc_f16(kTileM, 64);
    if (warp == 0) ptx::mbar_wait(BAR(12), 0);
    int stage = 0, phase = 0, acc_phase = 0;
    // mode 2: lane 0 of warp 1 streams the fields of every (tile, tap) of this CTA into the shared-memory ring while the warp
    // waits for the accumulator (non-blocking probes on both sides, so the pump can never be starved by its own wait)
    int ftile = blockIdx.x, ftap = 0, fs = 0, fph = 0;
    const uint32_t ring = ptx::smem_u32(smem + kFRingOff);
    auto pump_fields = [&]() {
      while (ftile < p.num_tiles && ptx::mbar_test_wait(BAR(kBarFEmpty + fs), fph ^ 1)) {
        const TileCoord fc = tile_coord(p, ftile);
        ptx::mbar_arrive_expect_tx(BAR(kBarFFull + fs), kFStageBytes);
        // box = (32 px x 2 groups x 2 words, 4 rows, 8 pair planes); rows / columns outside the frame arrive as zeros
        ptx::tma_load_3d(ring + fs * kFStageBytes, &ftm, BAR(kBarFFull + fs), fc.w0 * 4, fc.h0, (fc.b * 9 + ftap) * 8);
        if (++fs == kFStages) { fs = 0; fph ^= 1; }
        if (++ftap == 9) { ftap = 0; ftile += gridDim.x; }
      }
    };
    if (kMode == 2 && warp == 1 && lane == 0) ptx::prefetch_tmap(&ftm);
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      if (warp == 0) {
        for (int tap = 0; tap < 9; ++tap) {
          ptx::mbar_wait(BAR(stage), phase);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t a0 = tmem_base + kAColBase + stage * kAColsPerStage;   // A operand of this tap lives in TMEM
            const uint32_t b0 = ptx::smem_u32(wsm) + tap * kTapWBytes;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint64_t bd = ptx::make_smem_desc(b0 + j * 2 * kBLbo, kBLbo, kSbo);
              ptx::umma_f16_ts(tmem_base, a0 + j * 8, bd, idesc, (tap | j) != 0);
            }
            ptx::umma_commit(BAR(4 + stage));
            if (tap == 8) ptx::umma_commit(BAR(8));
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      const TileCoord tc = tile_coord(p, tile);
      const int h = tc.h0 + warp, w = tc.w0 + lane;
      const bool live = h < p.H && w < p.W;
      const int pix = h * p.W + w;
      if (kMode == 2 && warp == 1) {
        bool done = false;
        uint32_t spins = 0;
        while (!done) {
          uint32_t d = 0;
          if (lane == 0) {
            pump_fields();
            d = ptx::mbar_test_wait(BAR(8), acc_phase) ? 1u : 0u;
          }
          done = __shfl_sync(0xffffffffu, d, 0) != 0;      // warp-uniform exit: lanes must not leave this loop one by one
          if (!done) {
            __nanosleep(64);
            if (++spins > (1u << 26)) __trap();
          }
        }
      } else {
        ptx::mbar_wait(BAR(8), acc_phase);
      }
      acc_phase ^= 1;
      ptx::tc_fence_after();
      uint32_t r[32];
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        ptx::tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + half * 32, r);
        ptx::tmem_ld_wait();
        if (half == 1) {
          ptx::tc_fence_before();
          asm volatile("bar.sync 1, 128;" ::: "memory");
        }
        if (live) {
          if (p.out_mode == 0) {
            float *y = reinterpret_cast<float *>(p.y) + ((size_t)tc.b * 64 + half * 32) * P + pix;
#pragma unroll
            for (int n = 0; n < 32; ++n) __stcs(y + (size_t)n * P, __uint_as_float(r[n]) + bias_s[half * 32 + n]);
          } else {
            uint4 *y = reinterpret_cast<uint4 *>(p.y) + ((size_t)(tc.b % p.y_nb) * p.y_cs + p.y_grp[tc.b / p.y_nb] + half * 4) * P + pix;
#pragma unroll
            for (int kc = 0; kc < 4; ++kc) {
              uint4 v;
              const float *bs = bias_s + half * 32 + kc * 8;
              v.x = pack_bf2(__uint_as_float(r[kc * 8 + 0]) + bs[0], __uint_as_float(r[kc * 8 + 1]) + bs[1]);
              v.y = pack_bf2(__uint_as_float(r[kc * 8 + 2]) + bs[2], __uint_as_float(r[kc * 8 + 3]) + bs[3]);
              v.z = pack_bf2(__uint_as_float(r[kc * 8 + 4]) + bs[4], __uint_as_float(r[kc * 8 + 5]) + bs[5]);
              v.w = pack_bf2(__uint_as_float(r[kc * 8 + 6]) + bs[6], __uint_as_float(r[kc * 8 + 7]) + bs[7]);
              y[(size_t)kc * P] = v;
            }
          }
        }
      }
    }
  } else {
    // =========================== producers: fields -> texture fetch -> x mask -> A operand ===========================
    // The loop is bound by instruction issue (ncu: removing the texture fetches altogether changes nothing), so it is
    // written for instruction count: taps fully unrolled (18 steps = 2 tiles per trip, so that the tap index, the tap's
    // base coordinates and the double-buffer index are compile-time), one 64-bit pointer per thread for the fields
    // (two coalesced 16-byte loads per tap when dg = 16), no liveness handling (rows of ragged tiles compute finite garbage that
    // the epilogue never stores; MMA rows are independent), no w clamp (border addressing returns 0 outside the frame).
    const int ptid = tid - kEpiWarps * 32;
    const int row = ptid & (kTileM - 1);
    const int ty = row >> 5, tx = row & 31;
    const int quad0 = (ptid / kTileM) * 4;
    const float Hf = (float)p.H;
    const int dg = p.dg;
    int goff[4];        // this thread's deformable groups (dg < 16 only)
#pragma unroll
    for (int qi = 0; qi < 4; ++qi) goff[qi] = (quad0 + qi) >> p.gshift;
    const cudaTextureObject_t tex = p.tex;   // kernel parameter: provably warp-uniform (a per-tile handle made ptxas wrap
                                             // every fetch in a divergence loop: ~12 extra instructions per sample)
    const size_t tap_stride = (size_t)P * dg;   // uint2 elements between taps of one sample
    const size_t pair_stride = (size_t)P * 2;   // dg = 16: between consecutive group pairs

    struct Pix {   // per-tile state of the pixel this thread owns
      const uint2 *f;                 // fields of tap 0 (dg = 16: already at this thread's first group pair)
      float py;                       // texture row of image row -1.5 of this thread's first quad plane (+1 border, +0.5 centre)
      float hb[3], wb[3], mvx, mvy;   // hb[i] = h - 1 + i;  wb[j] = w - 1 + j + 1.5 (border shift + texel centre)
    };
    auto pix_state = [&](int tile) {
      Pix s;
      const TileCoord tc = tile_coord(p, tile);
      const int h = tc.h0 + ty, w = tc.w0 + tx;
      const int pixc = min(h, p.H - 1) * p.W + min(w, p.W - 1);
      s.f = p.fields + (size_t)tc.b * p.f_bstride + (kDG16 ? ((size_t)(quad0 >> 1) * P + pixc) * 2 : (size_t)pixc);
      s.py = (float)(((tc.b % p.x_batch - p.x0) * 16 + quad0) * (p.H + 3)) + 1.5f;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        s.hb[i] = (float)(h - 1 + i);
        s.wb[i] = (float)(w - 1 + i) + 1.5f;
      }
      s.mvx = p.mv ? __ldg(p.mv + ((size_t)tc.b * 2 + 0) * P + pixc) : 0.f;
      s.mvy = p.mv ? __ldg(p.mv + ((size_t)tc.b * 2 + 1) * P + pixc) : 0.f;
      return s;
    };
    struct Buf { float4 v[4]; uint32_t m2[4]; };

    const int my_tiles = blockIdx.x < p.num_tiles ? (p.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int total = my_tiles * 9;
    if (total > 0) {
      // F: field-fetch cursor (two steps ahead of the consumer), I: texture-issue cursor (one step ahead)
      Pix fpix = pix_state(blockIdx.x), ipix = fpix;
      int ftile = blockIdx.x;
      uint2 f[4];
      int fstage = 0, fphase = 0;
      const uint8_t *fring = smem + kFRingOff + ((quad0 >> 1) * kTileH + ty) * (kTileW * 16) + tx * 16;
      auto fetch_fields = [&](int tap) {
        const uint2 *src = fpix.f + (size_t)tap * tap_stride;
        if (kMode == 2) {
          // this thread's two group pairs of the tap the TMA warp staged: a warp reads 512 contiguous bytes per load
          ptx::mbar_wait(BAR(kBarFFull + fstage), fphase);
          const uint4 *q = reinterpret_cast<const uint4 *>(fring + fstage * kFStageBytes);
          const uint4 a = q[0], c = q[kTileH * kTileW];        // next pair plane: + 4 rows x 512 bytes
          f[0] = make_uint2(a.x, a.y); f[1] = make_uint2(a.z, a.w); f[2] = make_uint2(c.x, c.y); f[3] = make_uint2(c.z, c.w);
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(BAR(kBarFEmpty + fstage));   // LSU order: the loads above read before this arrive lands
          if (++fstage == kFStages) { fstage = 0; fphase ^= 1; }
        } else if (kDG16) {
          // lanes = consecutive pixels, 16 bytes (two groups) each: 512 contiguous bytes per warp request
          const uint4 a = ld_stream_u4(reinterpret_cast<const uint4 *>(src)), c = ld_stream_u4(reinterpret_cast<const uint4 *>(src + pair_stride));
          f[0] = make_uint2(a.x, a.y); f[1] = make_uint2(a.z, a.w); f[2] = make_uint2(c.x, c.y); f[3] = make_uint2(c.z, c.w);
        } else {
#pragma unroll
          for (int qi = 0; qi < 4; ++qi) f[qi] = ld_stream_u2(src + (size_t)goff[qi] * P);
        }
      };
      auto issue = [&](Buf &b, int ti, int tj) {
#pragma unroll
        for (int qi = 0; qi < 4; ++qi) {
          const float2 d = __half22float2(*reinterpret_cast<const __half2 *>(&f[qi].x));
          // reference order: offset = residual + flow (arch :3347), then h_im = base + offset (.cu:614-615)
          const float h_im = __fadd_rn(ipix.hb[ti], __fadd_rn(d.x, ipix.mvy));
          const float w_t = __fadd_rn(ipix.wb[tj], __fadd_rn(d.y, ipix.mvx));
          const float hc = fminf(fmaxf(h_im, -1.f), Hf);   // stay inside this quad's plane (+ zero border); NaN -> -1 -> 0
          b.v[qi] = tex2D<float4>(tex, w_t, hc + (ipix.py + (float)(qi * (p.H + 3))));
          b.m2[qi] = __byte_perm(f[qi].y, 0, 0x1010);      // (m, m) fp16x2
        }
      };
      int stage = 0, phase = 0;
      auto consume = [&](const Buf &b) {
        ptx::mbar_wait(BAR(4 + stage), phase ^ 1);
        ptx::tc_fence_after();
        uint32_t o[8];
#pragma unroll
        for (int qi = 0; qi < 4; ++qi) {
          const __half2 m2 = *reinterpret_cast<const __half2 *>(&b.m2[qi]);
          o[qi * 2 + 0] = h2_as_u32(__hmul2(m2, __floats2half2_rn(b.v[qi].x, b.v[qi].y)));
          o[qi * 2 + 1] = h2_as_u32(__hmul2(m2, __floats2half2_rn(b.v[qi].z, b.v[qi].w)));
        }
        // row = TMEM lane (this warp's quarter is (warp % 4) = row / 32), K elements quad0*4 .. +15 = columns quad0*2 .. +7
        ptx::tmem_st8(tmem_base + ((uint32_t)(row & ~31) << 16) + kAColBase + stage * kAColsPerStage + quad0 * 2, o);
        ptx::tmem_st_wait();
        ptx::tc_fence_before();
        ptx::mbar_arrive(BAR(stage));
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      };

      Buf buf[2];
      fetch_fields(0);         // fields of step 0
      issue(buf[0], 0, 0);     // textures of step 0
      fetch_fields(1);         // fields of step 1 (every tile has 9 steps)
      bool running = true;
      for (int s0 = 0; running; s0 += 18) {
#pragma unroll
        for (int u = 0; u < 18; ++u) {
          const int s = s0 + u;
          if (s >= total) { running = false; break; }
          const int tap_i = (u + 1) % 9, tap_f = (u + 2) % 9;
          if (s + 1 < total) {
            if (tap_i == 0) ipix = fpix;        // the F cursor entered this tile one step ago
            issue(buf[(u + 1) & 1], tap_i / 3, tap_i % 3);
          }
          if (s + 2 < total) {
            if (tap_f == 0) {
              ftile += gridDim.x;
              fpix = pix_state(ftile);
            }
            fetch_fields(tap_f);
          }
          consume(buf[u & 1]);
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) ptx::tmem_dealloc(tmem_base, kTmemCols);
}

// W [64 co][64 ci][3][3] fp32 -> [tap][kc][co][8] fp16
__global__ void pack_weight_f16_kernel(const float *__restrict__ w, __half *__restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= 9 * 64 * 64) return;
  const int j = e % 8, co = (e / 8) % 64, kc = (e / 512) % 8, tap = e / 4096;
  out[e] = __float2half_rn(fminf(fmaxf(w[((size_t)co * 64 + kc * 8 + j) * 9 + tap], -65504.f), 65504.f));
}

// NCHW fp32 -> [B][C/4][H+3][Wpt] texels of 4 fp16 (saturated), zero border 1 before / 2 after, zero pitch padding
__global__ void pack_q4t_kernel(const float *__restrict__ x, uint2 *__restrict__ out, int C, int H, int W, int Wpt) {
  const int Hp = H + 3;
  const int pp = blockIdx.x * blockDim.x + threadIdx.x;
  if (pp >= Hp * Wpt) return;
  const int q = blockIdx.y, b = blockIdx.z;
  const int h = pp / Wpt - 1, w = pp % Wpt - 1;
  uint2 v = make_uint2(0, 0);
  if (h >= 0 && h < H && w >= 0 && w < W) {
    const float *src = x + (((size_t)b * C + q * 4) * H + h) * W + w;
    const size_t HW = (size_t)H * W;
    auto sat = [](float a) { return fminf(fmaxf(a, -65504.f), 65504.f); };
    v.x = h2_as_u32(__floats2half2_rn(sat(src[0]), sat(src[HW])));
    v.y = h2_as_u32(__floats2half2_rn(sat(src[2 * HW]), sat(src[3 * HW])));
  }
  out[((size_t)b * (C / 4) + q) * Hp * Wpt + pp] = v;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}
static bool g_no_tma_fields = false;   // cdfo_dcn_tex_sm100_set_fields_path: A/B switch for tools/bench_dcn.py

// ---- texture objects over caller-owned linear memory, cached by (device, pointer, rows, W, pitch) ----
// A handle is a descriptor only (it owns no memory), but it may be baked into a captured CUDA graph or be in use by kernels still
// queued on any stream, so it is never destroyed behind the caller's back: handles created while the launching stream is being
// captured are pinned for the life of the process, and the cache only evicts (oldest unpinned entry first) once it holds
// kTexCacheMax descriptors, and then only after cudaDeviceSynchronize() -- never while a capture is in progress, in which case
// the cache simply grows.
struct TexEntry { int dev; const void *ptr; int rows, W, Wpt; cudaTextureObject_t tex; unsigned long long stamp; bool pinned; };
static std::mutex g_mu;
static std::vector<TexEntry> g_cache;
static unsigned long long g_stamp = 0;
constexpr size_t kTexCacheMax = 1024;

static cudaError_t get_texture(const void *ptr, int rows, int W, int Wpt, cudaStream_t stream, cudaTextureObject_t *out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &cap) != cudaSuccess) {
    cudaGetLastError();
    cap = cudaStreamCaptureStatusNone;
  }
  const bool capturing = cap != cudaStreamCaptureStatusNone;
  std::lock_guard<std::mutex> lock(g_mu);
  for (TexEntry &t : g_cache)
    if (t.dev == dev && t.ptr == ptr && t.rows == rows && t.W == W && t.Wpt == Wpt) {
      t.stamp = ++g_stamp;
      t.pinned = t.pinned || capturing;
      *out = t.tex;
      return cudaSuccess;
    }
  cudaResourceDesc rd = {};
  rd.resType = cudaResourceTypePitch2D;
  rd.res.pitch2D.devPtr = const_cast<void *>(ptr);
  rd.res.pitch2D.desc = cudaCreateChannelDescHalf4();
  rd.res.pitch2D.width = (size_t)W + 3;
  rd.res.pitch2D.height = (size_t)rows;
  rd.res.pitch2D.pitchInBytes = (size_t)Wpt * 8;
  cudaTextureDesc td = {};
  td.addressMode[0] = td.addressMode[1] = cudaAddressModeBorder;
  td.filterMode = cudaFilterModeLinear;
  td.readMode = cudaReadModeElementType;
  td.normalizedCoords = 0;
  cudaTextureObject_t t = 0;
  e = cudaCreateTextureObject(&t, &rd, &td, nullptr);
  if (e != cudaSuccess) return e;
  if (g_cache.size() >= kTexCacheMax && !capturing) {
    size_t victim = g_cache.size();
    for (size_t i = 0; i < g_cache.size(); ++i)
      if (!g_cache[i].pinned && (victim == g_cache.size() || g_cache[i].stamp < g_cache[victim].stamp)) victim = i;
    if (victim != g_cache.size() && cudaDeviceSynchronize() == cudaSuccess) {   // nothing queued can still sample through it
      cudaDestroyTextureObject(g_cache[victim].tex);
      g_cache.erase(g_cache.begin() + (long)victim);
    }
  }
  g_cache.push_back(TexEntry{dev, ptr, rows, W, Wpt, t, ++g_stamp, capturing});
  *out = t;
  return cudaSuccess;
}

}  // namespace dtex

// shared with csrc/mv_dcn_fused_sm100.cu
TexSlices tex_slices(int x_batch, long long sample_rows) {
  const int fit = (int)(kTexRows / sample_rows);        // >= 1: the callers reject taller frames
  const int n = (x_batch + fit - 1) / fit;              // fewest slices that fit; equal sizes up to one sample
  return TexSlices{n, (x_batch + n - 1) / n};
}
cudaError_t dcn_tex_get_texture(const void *ptr, int rows, int W, int Wpt, cudaStream_t stream, cudaTextureObject_t *out) {
  return dtex::get_texture(ptr, rows, W, Wpt, stream, out);
}
}  // namespace cdfo

using namespace cdfo;

extern "C" int cdfo_dcn_tex_sm100_set_fields_path(int use_tma) {
  dtex::g_no_tma_fields = use_tma == 0;
  return CDFO_OK;
}

extern "C" int cdfo_q4t_pitch(int W) { return (W + 3 + 3) & ~3; }

extern "C" size_t cdfo_q4t_bytes(int B, int C, int H, int W) {
  if (B <= 0 || C <= 0 || C % 4 || H <= 0 || W <= 0) return 0;
  return (size_t)B * (C / 4) * (H + 3) * cdfo_q4t_pitch(W) * 8;
}

extern "C" int cdfo_pack_q4t(const float *x_nchw, void *x_q4t, int B, int C, int H, int W, void *stream) {
  CDFO_REQUIRE(x_nchw && x_q4t, CDFO_ERR_NULL, "cdfo_pack_q4t: NULL pointer");
  CDFO_REQUIRE(B > 0 && B <= 65535 && C > 0 && C % 4 == 0 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_pack_q4t: bad shape");
  const int Wpt = cdfo_q4t_pitch(W);
  dim3 grid(ceil_div((H + 3) * Wpt, 128), C / 4, B);
  dtex::pack_q4t_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(x_nchw, (uint2 *)x_q4t, C, H, W, Wpt);
  return check_launch("cdfo_pack_q4t");
}

extern "C" int cdfo_dcn_tex_sm100_pack_weight(const float *w, void *wpk, void *stream) {
  CDFO_REQUIRE(w && wpk, CDFO_ERR_NULL, "cdfo_dcn_tex_sm100_pack_weight: NULL pointer");
  dtex::pack_weight_f16_kernel<<<ceil_div(9 * 64 * 64, 256), 256, 0, (cudaStream_t)stream>>>(w, (__half *)wpk);
  return check_launch("cdfo_dcn_tex_sm100_pack_weight");
}

static int dcn_tex_run(const void *x_q4t, const void *fields, const float *mv, const void *wpk, const float *bias, void *y, int B,
                       int H, int W, int dg, int out_mode, int num_ctas, int x_batch, long long fields_bstride, int y_nb, int y_cs,
                       const int *y_grp, void *stream);

extern "C" int cdfo_dcn_tex_sm100_fwd(const void *x_q4t, const void *fields, const float *mv, const void *wpk,
                                      const float *bias, void *y, int B, int H, int W, int dg, int out_mode,
                                      int num_ctas, int x_batch, long long fields_bstride, void *stream) {
  const int grp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  return dcn_tex_run(x_q4t, fields, mv, wpk, bias, y, B, H, W, dg, out_mode, num_ctas, x_batch, fields_bstride, B, 8, grp, stream);
}

extern "C" int cdfo_dcn_tex_sm100_stacked_fwd(const void *x_q4t, const void *fields, const float *mv, const void *wpk,
                                              const float *bias, void *y_stack, int n_seq, int n_groups, int stack_chunks,
                                              const int *group_chunk, int H, int W, int dg, int x_batch, void *stream) {
  CDFO_REQUIRE(n_seq > 0 && n_groups > 0 && n_groups <= 8 && group_chunk, CDFO_ERR_SHAPE, "cdfo_dcn_tex_sm100_stacked_fwd: 1..8 groups");
  for (int g = 0; g < n_groups; ++g)
    CDFO_REQUIRE(group_chunk[g] >= 0 && group_chunk[g] + 8 <= stack_chunks, CDFO_ERR_SHAPE, "cdfo_dcn_tex_sm100_stacked_fwd: chunk slot out of range");
  return dcn_tex_run(x_q4t, fields, mv, wpk, bias, y_stack, n_seq * n_groups, H, W, dg, 1, 0, x_batch, 0, n_seq, stack_chunks, group_chunk, stream);
}

static int dcn_tex_run(const void *x_q4t, const void *fields, const float *mv, const void *wpk, const float *bias, void *y, int B,
                       int H, int W, int dg, int out_mode, int num_ctas, int x_batch, long long fields_bstride, int y_nb, int y_cs,
                       const int *y_grp, void *stream) {
  CDFO_REQUIRE(x_q4t && fields && wpk && y, CDFO_ERR_NULL, "cdfo_dcn_tex_sm100_fwd: NULL pointer");
  CDFO_REQUIRE(B > 0 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_dcn_tex_sm100_fwd: bad shape");
  CDFO_REQUIRE(dg == 1 || dg == 2 || dg == 4 || dg == 8 || dg == 16, CDFO_ERR_UNSUPPORTED,
               "cdfo_dcn_tex_sm100_fwd: deformable groups must divide 16 (got %d)", dg);
  CDFO_REQUIRE(out_mode == 0 || out_mode == 1, CDFO_ERR_UNSUPPORTED, "cdfo_dcn_tex_sm100_fwd: out_mode %d", out_mode);
  CDFO_REQUIRE(((uintptr_t)wpk & 15) == 0 && ((uintptr_t)x_q4t & 511) == 0 && ((uintptr_t)y & 15) == 0 && ((uintptr_t)fields & 15) == 0,
               CDFO_ERR_SHAPE, "cdfo_dcn_tex_sm100_fwd: x_q4t must be 512-byte aligned (texture base), wpk / y / fields 16-byte");
  CDFO_REQUIRE(W + 3 <= 131072, CDFO_ERR_UNSUPPORTED, "cdfo_dcn_tex_sm100_fwd: frame width %d exceeds the 2-D linear texture limit", W);
  dtex::Params p;
  p.x_batch = x_batch > 0 ? x_batch : B;
  CDFO_REQUIRE(B % p.x_batch == 0, CDFO_ERR_SHAPE, "cdfo_dcn_tex_sm100_fwd: B (%d) must be a multiple of x_batch (%d)", B, p.x_batch);
  // one texture per x slice; fp32 texture coordinates keep >= 8 fractional bits (the filter's resolution) below 65536 rows
  const long long sample_rows = 16ll * (H + 3);
  CDFO_REQUIRE(sample_rows <= kTexRows, CDFO_ERR_UNSUPPORTED,
               "cdfo_dcn_tex_sm100_fwd: frame height %d exceeds the 2-D linear texture limit (16 * (H + 3) <= %d rows)", H, kTexRows);
  const int Wpt = cdfo_q4t_pitch(W);
  p.fields = (const uint2 *)fields; p.mv = mv; p.wpk = (const uint8_t *)wpk; p.bias = bias; p.y = y;
  p.B = B; p.H = H; p.W = W; p.dg = dg; p.out_mode = out_mode;
  p.y_nb = y_nb; p.y_cs = y_cs;
  for (int g = 0; g < 8; ++g) p.y_grp[g] = y_grp[g];
  p.f_bstride = fields_bstride > 0 ? fields_bstride : (long long)dg * 9 * H * W;
  p.gshift = 0;
  while ((16 >> p.gshift) > dg) ++p.gshift;
  p.tiles_x = ceil_div(W, dtex::kTileW);
  p.tiles_per_img = p.tiles_x * ceil_div(H, dtex::kTileH);
  CDFO_REQUIRE((long long)dg * 9 * H * W < (1ll << 31), CDFO_ERR_UNSUPPORTED, "cdfo_dcn_tex_sm100_fwd: field planes too large for 32-bit indexing");
  const long long nt = (long long)p.tiles_per_img * B;
  CDFO_REQUIRE(nt < (1ll << 31), CDFO_ERR_UNSUPPORTED, "cdfo_dcn_tex_sm100_fwd: too many tiles");
  // mode 2 (fields through TMA) needs the dense [B][9][8][H][W][2] layout; tiny frames keep the LDG path
  const bool dense = p.f_bstride == (long long)dg * 9 * H * W;
  int mode = dg != 16 ? 0 : (dense && W >= dtex::kTileW && H >= dtex::kTileH && !dtex::g_no_tma_fields ? 2 : 1);
  CUtensorMap ftm;
  memset(&ftm, 0, sizeof(ftm));
  if (mode == 2) {
    dtex::EncodeTiledFn enc = dtex::encode_tiled_fn();
    if (!enc) {
      mode = 1;
    } else {
      const cuuint64_t gdim[3] = {(cuuint64_t)W * 4, (cuuint64_t)H, (cuuint64_t)B * 72};
      const cuuint64_t gstr[2] = {(cuuint64_t)W * 16, (cuuint64_t)H * W * 16};
      const cuuint32_t box[3] = {(cuuint32_t)dtex::kTileW * 4, (cuuint32_t)dtex::kTileH, 8};
      const cuuint32_t estr[3] = {1, 1, 1};
      CUresult cr = enc(&ftm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<void *>(fields), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      CDFO_REQUIRE(cr == CUDA_SUCCESS, CDFO_ERR_CUDA, "cdfo_dcn_tex_sm100_fwd: cuTensorMapEncodeTiled(fields) failed with CUresult %d", (int)cr);
    }
  }
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(dtex::dcn_tex_sm100_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dtex::smem_bytes(0));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dtex::dcn_tex_sm100_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dtex::smem_bytes(1));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dtex::dcn_tex_sm100_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dtex::smem_bytes(2));
    if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "cudaFuncSetAttribute(dcn_tex_sm100): %s", cudaGetErrorString(e));
    attr_done = true;
  }
  const int threads = (dtex::kEpiWarps + dtex::kProdWarps) * 32;
  cudaStream_t st = (cudaStream_t)stream;
  const TexSlices sl = tex_slices(p.x_batch, sample_rows);
  for (int x0 = 0; x0 < p.x_batch; x0 += sl.per) {
    p.x0 = x0;
    p.xn = p.x_batch - x0 < sl.per ? p.x_batch - x0 : sl.per;
    const uint8_t *base = (const uint8_t *)x_q4t + (size_t)x0 * (size_t)sample_rows * Wpt * 8;   // a multiple of 512 bytes
    cudaError_t e = dtex::get_texture(base, (int)(p.xn * sample_rows), W, Wpt, st, &p.tex);
    if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "cdfo_dcn_tex_sm100_fwd: cudaCreateTextureObject: %s", cudaGetErrorString(e));
    p.num_tiles = p.tiles_per_img * (B / p.x_batch) * p.xn;
    int grid = num_ctas > 0 ? num_ctas : kNumSMs;
    if (grid > p.num_tiles) grid = p.num_tiles;
    if (mode == 2) dtex::dcn_tex_sm100_kernel<2><<<grid, threads, dtex::smem_bytes(2), st>>>(p, ftm);
    else if (mode == 1) dtex::dcn_tex_sm100_kernel<1><<<grid, threads, dtex::smem_bytes(1), st>>>(p, ftm);
    else dtex::dcn_tex_sm100_kernel<0><<<grid, threads, dtex::smem_bytes(0), st>>>(p, ftm);
    if (int rc = check_launch("cdfo_dcn_tex_sm100_fwd")) return rc;
  }
  return CDFO_OK;
}
