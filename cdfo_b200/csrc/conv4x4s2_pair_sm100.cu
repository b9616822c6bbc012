// 4x4 / stride 2 / padding 1 convolution 256 -> 64 on a CTA pair: the trunk's "conv 3x3 at twice the resolution, then bilinear x0.5".
//
// Block_.forward (arch/SIDECVSR_our.py:401-406) contains down(body(up(x))): the body's second convolution (256 -> 64, composed with
// the 1x1 of `down`) runs at 2H x 2W and is followed by Interpolate(0.5) = the mean of each 2x2 block (align_corners=False on an even
// size).  Both are linear, so the pair is ONE convolution with a 4x4 kernel and stride 2 on the 2x grid,
//     W4[u][v] = 1/4 * sum over (dy, i): dy + i - 1 = u, (dx, j): dx + j - 1 = v of W3[i][j],   u, v in {-1, 0, 1, 2},
// evaluated directly at H x W: 16 taps per output pixel instead of 9 taps on 4 pixels (2.25x fewer FLOPs on the most expensive
// convolution of the block) and no 2x-resolution intermediate in HBM (the reference writes and re-reads it).
//
// Implicit GEMM as in conv3x3_pair_sm100.cu (tcgen05.mma cta_group::2, M = 256 pixels over the two SMs of a TPC, N = 64, each CTA
// supplying the weights of 32 output channels).  The stride-2 access becomes dense by splitting the input into its four parity
// phases: tap u = 2 m' - a reads phase a (rows 2q - a ... ) at row offset m' in {0, 1}, so every tap's A operand is a (16+1) x (8+1)
// window of ONE phase image at a byte offset.  TMA loads a phase directly from the c8 tensor with elementStrides = 2 (box 18 x 34
// traversed -> 9 x 17 pixels landed), zero-filling outside the frame = the convolution's padding.  Per pipeline stage (32 input
// channels): 4 phase boxes (4 x 9.8 KB) + this CTA's 16 x 32 x 32 weights (32 KB) by one 3-D tensor-map load; the completion bytes of
// both CTAs are credited to the leader's barrier.  Weights cannot be resident here (16 taps x 256 x 32 x 2 B = 262 KB per CTA).
#include <cuda.h>

#include "cdfo_common.cuh"
#include "sm100_pair.cuh"
#include "sm100_ptx.cuh"

namespace cdfo {
namespace c4 {

using namespace pairptx;

constexpr int kTileH = 16, kTileW = 8;
constexpr int kPH = kTileH + 1, kPW = kTileW + 1;        // window of one parity phase
constexpr int kPlane = kPH * kPW * 16;                    // one 8-channel chunk of one phase: 2448 B
constexpr int kSbo = kPW * 16;
constexpr int kChunks = 4;                                // 32 input channels per stage
constexpr int kPhaseBytes = kChunks * kPlane;             // 9792 B landed per phase
constexpr int kPhaseStride = (kPhaseBytes + 127) & ~127;  // TMA destinations are 128-byte aligned
constexpr int kAStage = 4 * kPhaseStride;
constexpr int kNH = 32;
constexpr int kTapBytes = kNH * 32 * 2;                   // weights of one tap, stage and CTA: [4 chunks][32 co][8]
constexpr int kWStage = 16 * kTapBytes;                   // 32 KB
constexpr int kStageBytes = kAStage + kWStage;
constexpr int kTxBytes = 4 * kPhaseBytes + kWStage;       // per CTA and stage
constexpr int kStages = 3;
constexpr int kThreads = 320, kEpiWarps = 8;
constexpr int kAccCols = 64, kTmemCols = 128;

struct Params {
  const float *bias;    // [64] or nullptr
  const uint4 *resid;   // c8 bf16 [B][8][H][W][8] or nullptr
  const uint4 *up;      // c8 bf16 [B][8][H/2][W/2][8] or nullptr: its bilinear x2 (align_corners=False) is added (Block_'s up(body(down(x))))
  uint4 *y;             // c8 bf16 [B][8][H][W][8]
  uint4 *half_out;      // c8 bf16 [B][8][H/2][W/2][8] or nullptr: bilinear x0.5 (2x2 mean) of the fp32 result = the next block's down input
  int B, Cin, H, W;     // H, W = OUTPUT size (input is 2H x 2W)
  int tiles_x, tiles_y, m_tiles;
  int x_planes;         // 1: x is stored as parity planes [B][Cin/8][2][2][H][W][8] (what cdfo_conv3x3_pair_sm100_planes_fwd writes):
                        // every phase window is a DENSE box.  0: plain c8, loaded with elementStrides = 2 -- each 16-byte pixel chunk
                        // is then a separate L2 request that drags a 32-byte sector, the kernel's bottleneck in that mode.
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
conv4x4s2_pair_sm100_kernel(const __grid_constant__ CUtensorMap xmap, const __grid_constant__ CUtensorMap wmap, const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int KB = p.Cin / 32;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kStages * kStageBytes);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 16);
  float *bias_s = reinterpret_cast<float *>(bars + 18);
  // barrier map: [0,3) stage full (leader's is used), [4,7) stage empty, 8/9 accumulator full, 10/11 accumulator empty (leader's)
  const uint32_t bar0 = ptx::smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  for (int i = tid; i < 64; i += kThreads) bias_s[i] = p.bias ? p.bias[i] : 0.f;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(BAR(s), 1);
      ptx::mbar_init(BAR(4 + s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(BAR(8 + a), 1);
      ptx::mbar_init(BAR(10 + a), 2 * kEpiWarps);
    }
    ptx::fence_mbar_init();
    ptx::prefetch_tmap(&xmap);
    ptx::prefetch_tmap(&wmap);
  }
  if (warp == 1) {
    tmem_alloc2(ptx::smem_u32(tmem_slot), kTmemCols);
    tmem_relinquish2();
  }
  ptx::tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // every barrier of the pair is initialised before any remote arrival / transaction
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const uint32_t stage0 = ptx::smem_u32(smem);

  if (warp == 0) {
    // =========================== TMA producer (both CTAs: own pixel tile, own half of the weights) ===========================
    if (lane == 0) {
      int stage = 0, phase = 0;
      for (int it = 0;; ++it) {
        const int t0 = (it * num_pairs + pair) * 2;
        if (t0 >= p.m_tiles) break;
        const int mt = t0 + (int)rank;
        int b = 0, h0 = 0, w0 = 0;          // a pair's odd tile past the end recomputes tile 0 and stores nothing
        if (mt < p.m_tiles) {
          b = mt / tiles_per_img;
          const int r = mt - b * tiles_per_img;
          h0 = (r / p.tiles_x) * kTileH;
          w0 = (r % p.tiles_x) * kTileW;
        }
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(BAR(4 + stage), phase ^ 1);
          if (leader) ptx::mbar_arrive_expect_tx(BAR(stage), 2 * kTxBytes);
          const uint32_t dst = stage0 + stage * kStageBytes;
#pragma unroll
          for (int ph = 0; ph < 4; ++ph) {   // phase (a, b) = (ph >> 1, ph & 1): input rows 2 h0 - a + 2 r, columns 2 w0 - b + 2 c
            if (p.x_planes)                  // = rows h0 - a + r of the plane of parity a (odd rows start one plane row earlier);
                                             // innermost dimension = a whole window row (9 pixels x 8 channels = 144 contiguous bytes)
              tma_load_5d_pair(dst + ph * kPhaseStride, &xmap, BAR(stage), (w0 - (ph & 1)) * 8, h0 - (ph >> 1), ph, b * (p.Cin / 8) + kb * kChunks, 0);
            else
              tma_load_5d_pair(dst + ph * kPhaseStride, &xmap, BAR(stage), 0, 2 * w0 - (ph & 1), 2 * h0 - (ph >> 1), kb * kChunks, b);
          }
          tma_load_3d_pair(dst + kAStage, &wmap, BAR(stage), 0, 0, (int)rank * KB + kb);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      for (int s = 0; s < kStages; ++s) {    // producer tail (see conv3x3_pair_sm100.cu)
        ptx::mbar_wait(BAR(4 + stage), phase ^ 1);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (leader CTA only) ===========================
    if (leader) {
      const uint32_t idesc = ptx::make_idesc_bf16(256, 64);
      int stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (int it = 0;; ++it) {
        if ((it * num_pairs + pair) * 2 >= p.m_tiles) break;
        ptx::mbar_wait(BAR(10 + acc), acc_phase ^ 1);
        ptx::tc_fence_after();
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(BAR(stage), phase);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {       // one elected lane: no per-thread waterfall around the uniform-operand MMAs
            const uint32_t a0 = stage0 + stage * kStageBytes, b0 = a0 + kAStage;
            // descriptors once per stage; every MMA adds compile-time constants to the low words (the issuing thread is the critical path)
            const uint64_t ad0 = ptx::make_smem_desc(a0, kPlane, kSbo), bd0 = ptx::make_smem_desc(b0, kNH * 16, 128);
            const uint32_t a_lo0 = (uint32_t)ad0, a_hi = (uint32_t)(ad0 >> 32), b_lo0 = (uint32_t)bd0, b_hi = (uint32_t)(bd0 >> 32);
            const uint32_t tmem_d = tmem_base + acc * kAccCols;
#pragma unroll
            for (int tap = 0; tap < 16; ++tap) {
              // tap (ui, vi), u = ui - 1: parity a = u & 1, window row offset m' = (u + a) / 2 (same for columns)
              const int ui = tap >> 2, vi = tap & 3;
              const int pa = (ui + 1) & 1, pb = (vi + 1) & 1;
              const int mr = (ui - 1 + pa) >> 1, mc = (vi - 1 + pb) >> 1;
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const uint32_t a_lo = a_lo0 + (((pa * 2 + pb) * kPhaseStride + (mr * kPW + mc) * 16 + j * 2 * kPlane) >> 4);
                const uint32_t b_lo = b_lo0 + ((tap * kTapBytes + j * 2 * (kNH * 16)) >> 4);
                umma_f16_2sm_w(tmem_d, a_lo, a_hi, b_lo, b_hi, idesc, (tap | j) != 0 ? 1u : (uint32_t)(kb != 0));
              }
            }
            umma_commit_pair(BAR(4 + stage));
            if (kb == KB - 1) umma_commit_pair(BAR(8 + acc));
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
      for (int k = 0; k < 2; ++k) {          // accumulator tail (see conv3x3_pair_sm100.cu)
        ptx::mbar_wait(BAR(10 + acc), acc_phase ^ 1);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    // =========================== epilogue (both CTAs, own 128 pixels x 64 channels) ===========================
    const int quarter = warp & 3;
    const int ehalf = (warp - 2) >> 2;
    const int row = quarter * 32 + lane;
    const int ty = row >> 3, tx = row & 7;
    const size_t HW = (size_t)p.H * p.W;
    int acc = 0, acc_phase = 0;
    for (int it = 0;; ++it) {
      const int t0 = (it * num_pairs + pair) * 2;
      if (t0 >= p.m_tiles) break;
      const int mt = t0 + (int)rank;
      const bool valid = mt < p.m_tiles;
      const int b = valid ? mt / tiles_per_img : 0;
      const int r = valid ? mt - b * tiles_per_img : 0;
      const int h = (r / p.tiles_x) * kTileH + ty, w = (r % p.tiles_x) * kTileW + tx;
      const bool live = valid && h < p.H && w < p.W;
      const size_t pix = (size_t)h * p.W + w;
      ptx::mbar_wait(BAR(8 + acc), acc_phase);
      ptx::tc_fence_after();
#pragma unroll 1
      for (int c0 = ehalf * 16; c0 < 64; c0 += 32) {
        uint32_t rr[16];
        tmem_ld16(tmem_base + acc * kAccCols + ((uint32_t)(quarter * 32) << 16) + c0, rr);
        ptx::tmem_ld_wait();
        if (c0 + 32 >= 64) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (leader) ptx::mbar_arrive(BAR(10 + acc));
            else mbar_arrive_cluster(BAR(10 + acc), 0);
          }
        }
        // all global loads of the pass first (residual: 2, bilinear x2 source: 2 chunks x 4 taps), then the arithmetic
        float v[16];
        if (live) {
          uint4 rq[2] = {}, uq[8] = {};
          float wq[4] = {0.f, 0.f, 0.f, 0.f};
          if (p.resid) {
            rq[0] = __ldg(p.resid + ((size_t)b * 8 + c0 / 8) * HW + pix);
            rq[1] = __ldg(p.resid + ((size_t)b * 8 + c0 / 8 + 1) * HW + pix);
          }
          if (p.up) {
            // bilinear x2, align_corners=False: source d / 2 - 0.25 clamped at 0 -> taps (0.25, 0.75) / (0.75, 0.25), edge pixel repeated
            const int Hh = p.H >> 1, Wh = p.W >> 1, hk = h >> 1, wk = w >> 1;
            const int r0 = (h & 1) ? hk : max(hk - 1, 0), r1 = (h & 1) ? min(hk + 1, Hh - 1) : hk;
            const int q0 = (w & 1) ? wk : max(wk - 1, 0), q1 = (w & 1) ? min(wk + 1, Wh - 1) : wk;
            const float ah = (h & 1) ? 0.75f : 0.25f, aw = (w & 1) ? 0.75f : 0.25f;
            wq[0] = ah * aw; wq[1] = ah * (1.f - aw); wq[2] = (1.f - ah) * aw; wq[3] = (1.f - ah) * (1.f - aw);
            const size_t HWh = (size_t)Hh * Wh;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              const uint4 *src = p.up + ((size_t)b * 8 + c0 / 8 + half) * HWh;
              uq[half * 4 + 0] = __ldg(src + (size_t)r0 * Wh + q0);
              uq[half * 4 + 1] = __ldg(src + (size_t)r0 * Wh + q1);
              uq[half * 4 + 2] = __ldg(src + (size_t)r1 * Wh + q0);
              uq[half * 4 + 3] = __ldg(src + (size_t)r1 * Wh + q1);
            }
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(rr[i]) + bias_s[c0 + i];
          if (p.resid) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              const uint32_t qq[4] = {rq[half].x, rq[half].y, rq[half].z, rq[half].w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                v[half * 8 + 2 * i] += __uint_as_float(qq[i] << 16);
                v[half * 8 + 2 * i + 1] += __uint_as_float(qq[i] & 0xffff0000u);
              }
            }
          }
          if (p.up) {
#pragma unroll
            for (int half = 0; half < 2; ++half)
#pragma unroll
              for (int tp = 0; tp < 4; ++tp) {
                const uint4 q = uq[half * 4 + tp];
                const uint32_t qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  v[half * 8 + 2 * i] = fmaf(wq[tp], __uint_as_float(qq[i] << 16), v[half * 8 + 2 * i]);
                  v[half * 8 + 2 * i + 1] = fmaf(wq[tp], __uint_as_float(qq[i] & 0xffff0000u), v[half * 8 + 2 * i + 1]);
                }
              }
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0.f;
        }
        if (p.half_out) {
          // 2x2 mean of the fp32 result: the quad of pixel (ty, tx) is lanes ^1 (column) and ^8 (row); tiles start at even (h, w) and
          // H, W are even, so a quad is live or dead as a whole.  Every lane of the warp takes part in the shuffles.
          float m[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float t = v[i] + __shfl_xor_sync(0xffffffffu, v[i], 1);
            t += __shfl_xor_sync(0xffffffffu, t, 8);
            m[i] = 0.25f * t;
          }
          if (live && (lane & 9) == 0) {
            uint4 *d = p.half_out + ((size_t)b * 8 + c0 / 8) * ((size_t)(p.H >> 1) * (p.W >> 1)) + (size_t)(h >> 1) * (p.W >> 1) + (w >> 1);
            d[0] = make_uint4(pack_bf2(m[0], m[1]), pack_bf2(m[2], m[3]), pack_bf2(m[4], m[5]), pack_bf2(m[6], m[7]));
            d[(size_t)(p.H >> 1) * (p.W >> 1)] = make_uint4(pack_bf2(m[8], m[9]), pack_bf2(m[10], m[11]), pack_bf2(m[12], m[13]), pack_bf2(m[14], m[15]));
          }
        }
        if (live) {
          uint4 *y = p.y + ((size_t)b * 8 + c0 / 8) * HW + pix;
          y[0] = make_uint4(pack_bf2(v[0], v[1]), pack_bf2(v[2], v[3]), pack_bf2(v[4], v[5]), pack_bf2(v[6], v[7]));
          y[HW] = make_uint4(pack_bf2(v[8], v[9]), pack_bf2(v[10], v[11]), pack_bf2(v[12], v[13]), pack_bf2(v[14], v[15]));
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc2(tmem_base, kTmemCols);
  cluster_sync_all();
}

// w3 [64][Cin][3][3] fp32 -> W4 = (x0.5 bilinear) o (3x3 conv) as a 4x4 stride-2 kernel, packed [half][Cin/32][tap = ui*4+vi][4 chunks][32 co][8] bf16
__global__ void pack_weight_4x4_kernel(const float *__restrict__ w3, __nv_bfloat16 *__restrict__ out, int Cin) {
  const size_t total = (size_t)64 * Cin * 16;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int j = e % 8, n = (e / 8) % 32, c = (e / 256) % 4, tap = (e / 1024) % 16;
    const int kb = (int)((e / 16384) % (Cin / 32)), half = (int)(e / 16384 / (Cin / 32));
    const int co = half * 32 + n, ci = kb * 32 + c * 8 + j;
    const int u = (tap >> 2) - 1, v = (tap & 3) - 1;
    float s = 0.f;
    for (int dy = 0; dy < 2; ++dy)
      for (int dx = 0; dx < 2; ++dx) {
        const int i = u + 1 - dy, jj = v + 1 - dx;
        if (i >= 0 && i < 3 && jj >= 0 && jj < 3) s += w3[((size_t)co * Cin + ci) * 9 + i * 3 + jj];
      }
    out[e] = __float2bfloat16_rn(0.25f * s);
  }
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

constexpr size_t kSmem = (size_t)kStages * kStageBytes + 18 * 8 + 64 * 4 + 64;

}  // namespace c4
}  // namespace cdfo

using namespace cdfo;

extern "C" int cdfo_conv4x4s2_pair_sm100_supported(int Cout, int Cin) { return Cout == 64 && Cin % 32 == 0 && Cin >= 32 && Cin <= 1024 ? 1 : 0; }

extern "C" size_t cdfo_conv4x4s2_pair_sm100_weight_bytes(int Cin) {
  return cdfo_conv4x4s2_pair_sm100_supported(64, Cin) ? (size_t)16 * Cin * 64 * 2 : 0;
}

extern "C" int cdfo_conv4x4s2_pair_sm100_pack_weight(const float *w3, void *wpk, int Cin, void *stream) {
  CDFO_REQUIRE(w3 && wpk, CDFO_ERR_NULL, "cdfo_conv4x4s2_pair_sm100_pack_weight: NULL pointer");
  CDFO_REQUIRE(cdfo_conv4x4s2_pair_sm100_supported(64, Cin), CDFO_ERR_UNSUPPORTED, "cdfo_conv4x4s2_pair_sm100: unsupported input channels %d", Cin);
  c4::pack_weight_4x4_kernel<<<kNumSMs * 2, 256, 0, (cudaStream_t)stream>>>(w3, (__nv_bfloat16 *)wpk, Cin);
  return check_launch("cdfo_conv4x4s2_pair_sm100_pack_weight");
}

extern "C" int cdfo_conv4x4s2_pair_sm100_block_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, const void *up_c8,
                                                   void *y_c8, void *half_c8, int B, int Cin, int H_in, int W_in, int x_planes, void *stream) {
  CDFO_REQUIRE(x_c8 && wpk && y_c8, CDFO_ERR_NULL, "cdfo_conv4x4s2_pair_sm100_block_fwd: NULL pointer");
  CDFO_REQUIRE((!up_c8 && !half_c8) || (H_in % 4 == 0 && W_in % 4 == 0), CDFO_ERR_SHAPE,
               "cdfo_conv4x4s2_pair_sm100_block_fwd: up_c8 / half_c8 need an even output size (input %d x %d)", H_in, W_in);
  CDFO_REQUIRE(((uintptr_t)up_c8 & 15) == 0 && ((uintptr_t)half_c8 & 15) == 0, CDFO_ERR_SHAPE,
               "cdfo_conv4x4s2_pair_sm100_block_fwd: pointers must be 16-byte aligned");
  CDFO_REQUIRE(x_planes == 0 || x_planes == 1, CDFO_ERR_UNSUPPORTED, "cdfo_conv4x4s2_pair_sm100_block_fwd: x_planes %d", x_planes);
  CDFO_REQUIRE(B > 0 && H_in > 0 && W_in > 0 && H_in % 2 == 0 && W_in % 2 == 0, CDFO_ERR_SHAPE,
               "cdfo_conv4x4s2_pair_sm100_block_fwd: the input size must be even (got %d x %d)", H_in, W_in);
  CDFO_REQUIRE(cdfo_conv4x4s2_pair_sm100_supported(64, Cin), CDFO_ERR_UNSUPPORTED, "cdfo_conv4x4s2_pair_sm100_block_fwd: unsupported input channels %d", Cin);
  CDFO_REQUIRE(((uintptr_t)x_c8 & 15) == 0 && ((uintptr_t)wpk & 15) == 0 && ((uintptr_t)y_c8 & 15) == 0 && ((uintptr_t)resid_c8 & 15) == 0,
               CDFO_ERR_SHAPE, "cdfo_conv4x4s2_pair_sm100_block_fwd: pointers must be 16-byte aligned");
  c4::EncodeTiledFn enc = c4::encode_tiled_fn();
  CDFO_REQUIRE(enc, CDFO_ERR_CUDA, "cdfo_conv4x4s2_pair_sm100_block_fwd: cuTensorMapEncodeTiled not available from the driver");
  CUtensorMap xm, wm;
  if (x_planes) {
    // [B * Cin/8][4 planes][H][W][8]: a box of 4 channel chunks starts at a multiple of 4 and never crosses a sample
    const cuuint64_t Ho = H_in / 2, Wo = W_in / 2;
    CDFO_REQUIRE((long long)B * (Cin / 8) < (1ll << 31), CDFO_ERR_UNSUPPORTED, "cdfo_conv4x4s2_pair_sm100_block_fwd: too many chunks");
    // the pixel and channel axes are merged (a window row of 9 pixels = 72 contiguous elements): 17 x 4 requests of 144 bytes per
    // box instead of 9 x 17 x 4 of 16 bytes
    const cuuint64_t gdim[5] = {Wo * 8, Ho, 4, (cuuint64_t)B * (Cin / 8), 1};
    const cuuint64_t gstr[4] = {Wo * 16, Ho * Wo * 16, 4 * Ho * Wo * 16, (cuuint64_t)B * (Cin / 8) * 4 * Ho * Wo * 16};
    const cuuint32_t box[5] = {8 * c4::kPW, c4::kPH, 1, c4::kChunks, 1};
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult cr = enc(&xm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void *>(x_c8), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CDFO_REQUIRE(cr == CUDA_SUCCESS, CDFO_ERR_CUDA, "cuTensorMapEncodeTiled(x, parity planes) failed with CUresult %d", (int)cr);
  } else {
    const cuuint64_t gdim[5] = {8, (cuuint64_t)W_in, (cuuint64_t)H_in, (cuuint64_t)(Cin / 8), (cuuint64_t)B};
    const cuuint64_t gstr[4] = {16, (cuuint64_t)W_in * 16, (cuuint64_t)H_in * W_in * 16, (cuuint64_t)(Cin / 8) * H_in * W_in * 16};
    const cuuint32_t box[5] = {8, 2 * c4::kPW, 2 * c4::kPH, c4::kChunks, 1};      // traversed with stride 2 -> 9 x 17 pixels landed
    const cuuint32_t estr[5] = {1, 2, 2, 1, 1};
    CUresult cr = enc(&xm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void *>(x_c8), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CDFO_REQUIRE(cr == CUDA_SUCCESS, CDFO_ERR_CUDA, "cuTensorMapEncodeTiled(x, stride 2) failed with CUresult %d", (int)cr);
  }
  {
    // one (half, K block) = 32 KB contiguous = 64 rows of 256 elements (512-byte requests)
    const cuuint64_t gdim[3] = {256, 64, (cuuint64_t)2 * (Cin / 32)};
    const cuuint64_t gstr[2] = {512, 32768};
    const cuuint32_t box[3] = {256, 64, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult cr = enc(&wm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(wpk), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CDFO_REQUIRE(cr == CUDA_SUCCESS, CDFO_ERR_CUDA, "cuTensorMapEncodeTiled(weights) failed with CUresult %d", (int)cr);
  }
  c4::Params p;
  p.bias = bias; p.resid = (const uint4 *)resid_c8; p.y = (uint4 *)y_c8;
  p.up = (const uint4 *)up_c8; p.half_out = (uint4 *)half_c8;
  p.B = B; p.Cin = Cin; p.H = H_in / 2; p.W = W_in / 2; p.x_planes = x_planes;
  p.tiles_x = ceil_div(p.W, c4::kTileW); p.tiles_y = ceil_div(p.H, c4::kTileH);
  const long long mt = (long long)B * p.tiles_x * p.tiles_y;
  CDFO_REQUIRE(mt < (1ll << 30), CDFO_ERR_UNSUPPORTED, "cdfo_conv4x4s2_pair_sm100_block_fwd: too many tiles");
  p.m_tiles = (int)mt;
  static bool attr_done = false;
  static int max_pairs = kNumSMs / 2;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(c4::conv4x4s2_pair_sm100_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c4::kSmem);
    if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "cudaFuncSetAttribute(conv4x4s2_pair_sm100, %zu): %s", c4::kSmem, cudaGetErrorString(e));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs & ~1);
    cfg.blockDim = dim3(c4::kThreads);
    cfg.dynamicSmemBytes = c4::kSmem;
    int n = 0;
    e = cudaOccupancyMaxActiveClusters(&n, c4::conv4x4s2_pair_sm100_kernel, &cfg);
    if (e == cudaSuccess && n > 0 && n < max_pairs) max_pairs = n;
    (void)cudaGetLastError();
    attr_done = true;
  }
  int pairs = (p.m_tiles + 1) / 2;
  if (pairs > max_pairs) pairs = max_pairs;
  c4::conv4x4s2_pair_sm100_kernel<<<pairs * 2, c4::kThreads, c4::kSmem, (cudaStream_t)stream>>>(xm, wm, p);
  return check_launch("cdfo_conv4x4s2_pair_sm100_block_fwd");
}
