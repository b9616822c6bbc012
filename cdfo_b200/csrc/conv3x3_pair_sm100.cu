// 3x3 / stride 1 / padding 1 convolutions of the reconstruction trunk (256 -> 64 and 64 -> 256, arch/SIDECVSR_our.py:378-406) and other
// Cin -> 64 layers as a TWO-SM tcgen05 implicit GEMM: a cluster of 2 CTAs (one TPC) issues tcgen05.mma.cta_group::2 with M = 256 and
// N = 64 or 256; each CTA holds the weights of HALF the output channels (template NH = 32 or 128) resident in shared memory.
//
// Why a CTA pair: at N = 64 the single-SM kernel (conv3x3_sm100.cu) cannot keep 9 x 256 x 64 weights (295 KB) in shared memory, so it
// streams them from L2 with every pixel tile: 387 KB per 128 pixels and SM, i.e. 84 B/clk at tensor peak against an L2 that sustains
// ~43 B/clk per SM (6300 B/clk chip-wide, B300_MICROARCH.md) -- measured 714 TFLOP/s = 87 % of that cap.  In a pair each CTA supplies
// HALF of the B operand (its 32 output channels: 147 KB, resident for the lifetime of the persistent CTA) and its own 128-pixel A
// tile; the tensor cores of both SMs read both halves.  L2 traffic drops to the A halos (92 KB per tile) and the shared-memory
// operand read per MMA from 6 KB to 5 KB.
//
// Layouts are the single-SM kernel's: activations "c8" = [B][C/8][H][W][8] bf16, the (16+2) x (8+2) halo of 64 channels lands by one
// TMA 5-D box per (tile, K block) in the tcgen05 canonical K-major layout, tap (i, j) = the same shared memory at +(i*10 + j)*16 bytes;
// weights [half][tap][Cin/8][32][8] bf16.  Pipeline: warp 0 = TMA producer (both CTAs; completion bytes of both land on the LEADER's
// full barrier), warp 1 of the leader = MMA issuer (commits are multicast to both CTAs' barriers), warps 2..9 = epilogue of the
// CTA's own 128 pixels (bias -> act -> +residual -> c8 bf16), accumulator double-buffered in TMEM (2 x 64 columns per CTA).
//
// UP2 (64 -> 256 only, body.0 of Block_'s down(body(up(x))) branch): the input is the 1x image and the A stage is BUILT instead of
// loaded -- the 18 x 10 halo of bilinear_x2(x) -- by four builder warps (warps 10..13) from a 10 x 6 x 64-channel raw tile of the 1x
// image in shared memory (7.7 KB instead of 23 KB of L2 -> SM traffic, and no 2x tensor written to and read back from HBM).  The
// values are those of resample.cu's upsample2_c8_kernel bit for bit (same helpers, up2_blend.cuh), so the convolution's result is too.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "cdfo_common.cuh"
#include "sm100_pair.cuh"
#include "sm100_ptx.cuh"
#include "up2_blend.cuh"

namespace cdfo {
namespace cpair {

constexpr int kTileH = 16, kTileW = 8, kHaloH = 18, kHaloW = 10;
constexpr int kPlane = kHaloH * kHaloW * 16;      // bytes of one 8-channel chunk of the halo
constexpr int kSbo = kHaloW * 16;
constexpr int kChunks = 8;                        // 64 channels per pipeline stage
constexpr int kABytes = kChunks * kPlane;         // 23 040
constexpr int kStages = 3;
constexpr int kEpiWarps = 8;
// UP2: the 1x source of one A stage = source rows h0/2 - 1 .. h0/2 + 8 and columns w0/2 - 1 .. w0/2 + 4 (edge-clamped) of 8 chunks
constexpr int kRawH = kTileH / 2 + 2, kRawW = kTileW / 2 + 2, kRawPix = kChunks * kRawH * kRawW, kRawBytes = kRawPix * 16;   // 7 680
constexpr int kBuildWarps = 4, kBuildThreads = kBuildWarps * 32;
constexpr int threads_of(bool up2) { return (2 + kEpiWarps + (up2 ? kBuildWarps : 0)) * 32; }   // 320 / 448

struct Params {
  const uint8_t *wpk;   // [2 halves][9 taps][Cin/8][NH][8] bf16
  const float *bias;    // [2 NH] or nullptr
  const float *bias_edge;  // [9][2 NH] or nullptr: the bias of border pixels by class (row top / middle / bottom) * 3 + (column left / middle /
                           // right) -- a 1x1 convolution composed INTO this 3x3 one has its own bias under the taps inside the frame only
  const uint4 *resid;   // c8 bf16 [B][2 NH / 8][H][W][8] or nullptr (added after the activation)
  const uint4 *x1;      // UP2: the 1x input c8 bf16 [B][8][H/2][W/2][8]; H, W below are the 2x (output) size
  uint4 *y;             // c8 bf16 [B][2 NH / 8][H][W][8]
  int B, Cin, H, W, act;
  int tiles_x, tiles_y, m_tiles;
  int tma_wide;         // 1: the tensor map merges the pixel and channel axes (a halo row = 80 contiguous elements = one 160-byte request)
  int y_planes;         // 2: y is NCHW fp32 [B][2 NH][H][W].  1: y is stored as its four parity planes [B][2 NH / 8][row parity][column parity][H/2][W/2][8] (H, W even) --
                        // the layout from which the 4x4 / stride-2 convolution (conv4x4s2_pair_sm100.cu) loads dense TMA boxes
};

using namespace pairptx;

// NH = output channels whose weights one CTA holds (N = 2 NH over the pair); UP2: A built from the 1x image (NH = 128, Cin = 64)
template <int NH, bool UP2>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(threads_of(UP2), 1)
conv3x3_pair_sm100_kernel(const __grid_constant__ CUtensorMap tmap, const Params p) {
  static_assert(!UP2 || NH == 128, "UP2 is instantiated for 64 -> 256 only");
  constexpr int kThreads = threads_of(UP2);
  constexpr int kNH = NH, kN = 2 * NH;
  constexpr int kPiece = kNH * 64 * 2;              // weights of one (tap, K block) and CTA
  constexpr int kAccCols = kN, kTmemCols = 2 * kN;  // accumulator double-buffered: 128 or 512 columns
  extern __shared__ __align__(1024) uint8_t smem[];
  const int KB = p.Cin / 64;
  const int w_bytes = 9 * p.Cin * kNH * 2;                // this CTA's half of the weights
  uint8_t *wsm = smem;
  uint8_t *asmem = smem + ((w_bytes + 1023) & ~1023);
  uint4 *raw = reinterpret_cast<uint4 *>(asmem + kStages * kABytes);         // UP2 only
  uint64_t *bars = reinterpret_cast<uint64_t *>(asmem + kStages * kABytes + (UP2 ? kRawBytes : 0));
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 16);
  float *bias_s = reinterpret_cast<float *>(bars + 18);
  // barrier map: [0,3) A full (leader's is used; UP2: one arrival per builder warp of both CTAs), [4,7) A empty, 8/9 accumulator full, 10/11 accumulator empty (leader's), 12 weights
  const uint32_t bar0 = ptx::smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  for (int i = tid; i < kN; i += kThreads) bias_s[i] = p.bias ? p.bias[i] : 0.f;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(BAR(s), UP2 ? 2 * kBuildWarps : 1);
      ptx::mbar_init(BAR(4 + s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(BAR(8 + a), 1);
      ptx::mbar_init(BAR(10 + a), 2 * kEpiWarps);         // one arrival per epilogue warp of BOTH CTAs
    }
    ptx::mbar_init(BAR(12), 1);
    ptx::fence_mbar_init();
    if (!UP2) ptx::prefetch_tmap(&tmap);
    ptx::mbar_arrive_expect_tx(BAR(12), w_bytes);
    const uint8_t *src = p.wpk + (size_t)rank * w_bytes;
    for (int i = 0; i < 9 * KB; ++i) ptx::bulk_g2s(ptx::smem_u32(wsm) + i * kPiece, src + (size_t)i * kPiece, kPiece, BAR(12));
  }
  if (warp == 1) {
    tmem_alloc2(ptx::smem_u32(tmem_slot), kTmemCols);
    tmem_relinquish2();
  }
  ptx::tc_fence_before();
  __syncthreads();                                        // barriers initialised (a wait before this point would probe stale memory)
  if (warp == 1) ptx::mbar_wait(BAR(12), 0);              // this CTA's weights have landed ...
  cluster_sync_all();                                     // ... and so have the peer's; every barrier of the pair is initialised
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles_per_img = p.tiles_x * p.tiles_y;

  if (warp == 0) {
    // =========================== TMA producer (both CTAs, own tile) ===========================
    if (!UP2 && lane == 0) {
      int stage = 0, phase = 0;
      for (int it = 0;; ++it) {
        const int t0 = (it * num_pairs + pair) * 2;
        if (t0 >= p.m_tiles) break;
        const int mt = t0 + (int)rank;
        int b = 0, h0 = 0, w0 = 0;                        // a pair's odd tile past the end: recompute tile 0, never stored (a box
        if (mt < p.m_tiles) {                             // beyond the batch would make TMA touch addresses past the allocation)
          b = mt / tiles_per_img;
          const int r = mt - b * tiles_per_img;
          h0 = (r / p.tiles_x) * kTileH;
          w0 = (r % p.tiles_x) * kTileW;
        }
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(BAR(4 + stage), phase ^ 1);
          if (leader) ptx::mbar_arrive_expect_tx(BAR(stage), 2 * kABytes);
          if (p.tma_wide) tma_load_5d_pair(ptx::smem_u32(asmem) + stage * kABytes, &tmap, BAR(stage), (w0 - 1) * 8, h0 - 1, kb * kChunks, b, 0);
          else tma_load_5d_pair(ptx::smem_u32(asmem) + stage * kABytes, &tmap, BAR(stage), 0, w0 - 1, h0 - 1, kb * kChunks, b);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      // producer tail: the multicast commits that release the last stages are asynchronous arrivals on THIS CTA's barriers; the CTA
      // must not retire (and have its shared memory reassigned) before they have landed
      for (int s = 0; s < kStages; ++s) {
        ptx::mbar_wait(BAR(4 + stage), phase ^ 1);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (leader CTA only) ===========================
    if (leader) {
      const uint32_t idesc = ptx::make_idesc_bf16(256, kN);
      int stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (int it = 0;; ++it) {
        if ((it * num_pairs + pair) * 2 >= p.m_tiles) break;
        ptx::mbar_wait(BAR(10 + acc), acc_phase ^ 1);
        ptx::tc_fence_after();
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(BAR(stage), phase);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {       // one elected lane: no per-thread waterfall around the uniform-operand MMAs
            // descriptors of (tap 0, K step 0) once per stage; every MMA then adds compile-time constants to the low words
            const uint64_t ad0 = ptx::make_smem_desc(ptx::smem_u32(asmem) + stage * kABytes, kPlane, kSbo);
            const uint64_t bd0 = ptx::make_smem_desc(ptx::smem_u32(wsm) + kb * kPiece, kNH * 16, 128);
            const uint32_t a_lo0 = (uint32_t)ad0, a_hi = (uint32_t)(ad0 >> 32), b_lo0 = (uint32_t)bd0, b_hi = (uint32_t)(bd0 >> 32);
            const uint32_t b_tap_step = (uint32_t)(KB * kPiece) >> 4;
            const uint32_t tmem_d = tmem_base + acc * kAccCols;
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint32_t a_lo = a_lo0 + ((((tap / 3) * kHaloW + (tap % 3)) * 16 + j * 2 * kPlane) >> 4);
                const uint32_t b_lo = b_lo0 + tap * b_tap_step + ((j * 2 * (kNH * 16)) >> 4);
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
      // accumulator tail: the peer's epilogue warps signal "drained" with REMOTE arrivals on this CTA's barriers; consume the
      // last ones too, so that none is still in flight towards this SM when the CTA retires
      for (int k = 0; k < 2; ++k) {
        ptx::mbar_wait(BAR(10 + acc), acc_phase ^ 1);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp < 2 + kEpiWarps) {
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
      // parity planes: pixel (h, w) -> plane (h & 1, w & 1), position (h / 2, w / 2); a chunk still spans H * W pixels
      const size_t opix = p.y_planes == 1 ? (size_t)((h & 1) * 2 + (w & 1)) * (HW >> 2) + (size_t)(h >> 1) * (p.W >> 1) + (w >> 1) : pix;
      ptx::mbar_wait(BAR(8 + acc), acc_phase);
      ptx::tc_fence_after();
      // the two warps of a TMEM lane quarter take alternate 16-column chunks; 16 channels = two c8 chunks of 16 bytes per pixel
#pragma unroll 1
      for (int c0 = ehalf * 16; c0 < kN; c0 += 32) {
        uint32_t rr[16];
        tmem_ld16(tmem_base + acc * kAccCols + ((uint32_t)(quarter * 32) << 16) + c0, rr);
        ptx::tmem_ld_wait();
        if (c0 + 32 >= kN) {                               // this warp has drained its part of the buffer: tell the leader's issuer
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (leader) ptx::mbar_arrive(BAR(10 + acc));
            else mbar_arrive_cluster(BAR(10 + acc), 0);
          }
        }
        if (!live) continue;
        float v[16];
        const int cls = (h == 0 ? 0 : (h == p.H - 1 ? 2 : 1)) * 3 + (w == 0 ? 0 : (w == p.W - 1 ? 2 : 1));
        float bb[16];
        if (p.bias_edge != nullptr && cls != 4) {             // border pixels only (< 1 %): ONE branch per pass, not one per channel
          const float4 *be = reinterpret_cast<const float4 *>(p.bias_edge + cls * kN + c0);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 q = __ldg(be + i);
            bb[4 * i] = q.x; bb[4 * i + 1] = q.y; bb[4 * i + 2] = q.z; bb[4 * i + 3] = q.w;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) bb[i] = bias_s[c0 + i];
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float t = __uint_as_float(rr[i]) + bb[i];
          if (p.act == 1) t = fmaxf(t, 0.f);
          else if (p.act == 2) t = t > 0.f ? t : 0.1f * t;
          v[i] = t;
        }
        if (p.resid) {
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const uint4 q = __ldg(p.resid + ((size_t)b * (kN / 8) + c0 / 8 + half) * HW + pix);
            const uint32_t qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              v[half * 8 + 2 * i] += __uint_as_float(qq[i] << 16);
              v[half * 8 + 2 * i + 1] += __uint_as_float(qq[i] & 0xffff0000u);
            }
          }
        }
        if (p.y_planes == 2) {               // NCHW fp32 (consumers that still read fp32 planes: the MDTA statistics kernel)
          float *yf = reinterpret_cast<float *>(p.y) + ((size_t)b * kN + c0) * HW + pix;
#pragma unroll
          for (int i = 0; i < 16; ++i) yf[(size_t)i * HW] = v[i];
          continue;
        }
        uint4 *y = p.y + ((size_t)b * (kN / 8) + c0 / 8) * HW + opix;
        y[0] = make_uint4(pack_bf2(v[0], v[1]), pack_bf2(v[2], v[3]), pack_bf2(v[4], v[5]), pack_bf2(v[6], v[7]));
        y[HW] = make_uint4(pack_bf2(v[8], v[9]), pack_bf2(v[10], v[11]), pack_bf2(v[12], v[13]), pack_bf2(v[14], v[15]));
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (UP2) {
    // =========================== A builders (UP2: both CTAs, own tile) ===========================
    const int bt = tid - (2 + kEpiWarps) * 32;
    const int Hi = p.H >> 1, Wi = p.W >> 1;
    constexpr int kFetch = (kRawPix + kBuildThreads - 1) / kBuildThreads;     // 4 raw blocks per thread
    // the stage's 8 chunks x 10 halo columns, 20 per builder warp (one warp per SM sub-partition, the same issue load on each)
    constexpr int kColsPerWarp = kChunks * kHaloW / kBuildWarps;
    const bool col_live = lane < kColsPerWarp;
    const int bcol = (bt >> 5) * kColsPerWarp + lane, bc = bcol / kHaloW, bj = bcol % kHaloW;
    // the tile of iteration `it`; a pair's odd tile past the end builds tile 0, which is never stored (as the TMA producer loads it)
    auto tile_of = [&](int it, int &b, int &h0, int &w0) {
      const int t0 = (it * num_pairs + pair) * 2;
      if (t0 >= p.m_tiles) return false;
      const int mt = t0 + (int)rank;
      b = h0 = w0 = 0;
      if (mt < p.m_tiles) {
        b = mt / tiles_per_img;
        const int r = mt - b * tiles_per_img;
        h0 = (r / p.tiles_x) * kTileH;
        w0 = (r % p.tiles_x) * kTileW;
      }
      return true;
    };
    // raw block (chunk, row, column) of the 10 x 6 source window holds the EDGE-CLAMPED source pixel: bilinear x2 repeats the edge pixel
    auto fetch = [&](int b, int h0, int w0, uint4 (&v)[kFetch]) {
#pragma unroll
      for (int k = 0; k < kFetch; ++k) {
        const int q = bt + k * kBuildThreads;
        if (q < kRawPix) {
          const int c = q / (kRawH * kRawW), rr = (q / kRawW) % kRawH, cc = q % kRawW;
          const int si = min(max((h0 >> 1) - 1 + rr, 0), Hi - 1), sj = min(max((w0 >> 1) - 1 + cc, 0), Wi - 1);
          v[k] = __ldg(p.x1 + (((size_t)b * kChunks + c) * Hi + si) * Wi + sj);
        }
      }
    };
    int b = 0, h0 = 0, w0 = 0, stage = 0, phase = 0;
    uint4 v[kFetch];
    bool more = tile_of(0, b, h0, w0);
    if (more) fetch(b, h0, w0, v);
    for (int it = 0; more; ++it) {
#pragma unroll
      for (int k = 0; k < kFetch; ++k)
        if (bt + k * kBuildThreads < kRawPix) raw[bt + k * kBuildThreads] = v[k];
      asm volatile("bar.sync 1, %0;" ::"n"(kBuildThreads) : "memory");      // the raw tile is complete
      int nb = 0, nh0 = 0, nw0 = 0;
      more = tile_of(it + 1, nb, nh0, nw0);
      if (more) fetch(nb, nh0, nw0, v);                   // the next tile's loads are in flight while this one is built
      ptx::mbar_wait(BAR(4 + stage), phase ^ 1);
      if (col_live) {
        // one (chunk, halo column) per lane, walked down the raw rows: each column blend feeds the two 2x rows around its source row
        uint4 *d = reinterpret_cast<uint4 *>(asmem + stage * kABytes) + bc * (kHaloH * kHaloW) + bj;   // the TMA box's canonical layout
        const int C = w0 - 1 + bj;                        // 2x column
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);    // the convolution's zero padding outside the 2x frame
        if (C < 0 || C >= p.W) {
#pragma unroll
          for (int i = 0; i < kHaloH; ++i) d[i * kHaloW] = zero;
        } else {
          // source column C/2 and its neighbour towards the output, as raw-tile indices (the clamped copies do the edge clamp)
          const int c0 = (C >> 1) - (w0 >> 1) + 1, cn = c0 + ((C & 1) ? 1 : -1);
          const uint4 *rp = raw + bc * (kRawH * kRawW);
          up2::F8 prev = up2::blend(up2::unpack(rp[cn]), up2::unpack(rp[c0]));                                    // columns first
#pragma unroll
          for (int rr = 1; rr < kRawH; ++rr) {
            const up2::F8 cur = up2::blend(up2::unpack(rp[rr * kRawW + cn]), up2::unpack(rp[rr * kRawW + c0]));
            // halo row 2 rr - 2 = odd 2x row R (source row rr - 1, neighbour rr), halo row 2 rr - 1 = even row R + 1 (source rr,
            // neighbour rr - 1); then rows
            const int R = h0 + 2 * rr - 3;
            d[(2 * rr - 2) * kHaloW] = R >= 0 && R < p.H ? up2::pack(up2::blend(cur, prev)) : zero;
            d[(2 * rr - 1) * kHaloW] = R + 1 < p.H ? up2::pack(up2::blend(prev, cur)) : zero;
            prev = cur;
          }
        }
      }
      ptx::fence_proxy_async_smem();                      // generic-proxy stores -> visible to the tensor cores (async proxy)
      __syncwarp();
      if (lane == 0) {
        if (leader) ptx::mbar_arrive(BAR(stage));
        else mbar_arrive_cluster(BAR(stage), 0);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kBuildThreads) : "memory");      // every builder is done reading the raw tile
      if (++stage == kStages) { stage = 0; phase ^= 1; }
      b = nb; h0 = nh0; w0 = nw0;
    }
    // the producer's tail: the multicast commits that release the last stages must land before the CTA retires
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_wait(BAR(4 + stage), phase ^ 1);
      if (++stage == kStages) { stage = 0; phase ^= 1; }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  cluster_sync_all();            // neither CTA may free TMEM / leave while the pair's MMAs or remote arrivals are in flight
  if (warp == 1) tmem_dealloc2(tmem_base, kTmemCols);
  cluster_sync_all();            // the pair-wide deallocation is complete in both CTAs before either SM is handed to the next kernel
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

static int half_channels(int Cout, int Cin) {
  if (Cout == 64 && Cin % 64 == 0 && Cin >= 64 && Cin <= 256) return 32;
  if (Cout == 256 && Cin == 64) return 128;
  return 0;
}
static size_t smem_bytes(int Cin, int NH, bool up2 = false) {
  return (size_t)((9 * Cin * NH * 2 + 1023) & ~1023) + kStages * kABytes + (up2 ? kRawBytes : 0) + 18 * 8 + 2 * NH * 4 + 64;
}

template <int NH, bool UP2>
static int launch(const CUtensorMap &tm, const Params &p, cudaStream_t stream) {
  constexpr int kThreads = threads_of(UP2);
  const size_t smem = smem_bytes(p.Cin, NH, UP2);
  static size_t attr_smem = 0;
  static int max_pairs = 0;
  auto kern = conv3x3_pair_sm100_kernel<NH, UP2>;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "cudaFuncSetAttribute(conv3x3_pair_sm100<%d>, %zu): %s", NH, smem, cudaGetErrorString(e));
    attr_smem = smem;
    // how many CTA pairs are co-resident (one CTA per SM; a GPC with an odd SM count leaves one SM out)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs & ~1);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    int n = 0;
    e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
    max_pairs = (e == cudaSuccess && n > 0) ? n : kNumSMs / 2;
    if (max_pairs > kNumSMs / 2) max_pairs = kNumSMs / 2;
    (void)cudaGetLastError();
  }
  int pairs = (p.m_tiles + 1) / 2;
  if (pairs > max_pairs) pairs = max_pairs;
  kern<<<pairs * 2, kThreads, smem, stream>>>(tm, p);
  return check_launch(UP2 ? "cdfo_conv3x3_pair_sm100_up2_fwd" : "cdfo_conv3x3_pair_sm100_fwd");
}

}  // namespace cpair
}  // namespace cdfo

using namespace cdfo;

extern "C" int cdfo_conv3x3_pair_sm100_supported(int Cout, int Cin) {
  const int nh = cpair::half_channels(Cout, Cin);
  return nh && cpair::smem_bytes(Cin, nh) <= 227 * 1024 ? 1 : 0;
}

extern "C" size_t cdfo_conv3x3_pair_sm100_weight_bytes(int Cout, int Cin) {
  return cdfo_conv3x3_pair_sm100_supported(Cout, Cin) ? (size_t)9 * Cin * Cout * 2 : 0;
}

extern "C" int cdfo_conv3x3_pair_sm100_pack_weight(const float *w, void *wpk, int Cout, int Cin, void *stream) {
  CDFO_REQUIRE(w && wpk, CDFO_ERR_NULL, "cdfo_conv3x3_pair_sm100_pack_weight: NULL pointer");
  CDFO_REQUIRE(cdfo_conv3x3_pair_sm100_supported(Cout, Cin), CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100: unsupported channels %d -> %d", Cin, Cout);
  return conv3x3_pack_weight_raw(w, wpk, Cout, Cin, cpair::half_channels(Cout, Cin), 2, 0, 9, (cudaStream_t)stream);
}

extern "C" int cdfo_conv3x3_pair_sm100_edge_fwd(const void *x_c8, const void *wpk, const float *bias, const float *bias_edge, const void *resid_c8,
                                               void *y, int B, int Cin, int Cout, int H, int W, int act, int y_planes, void *stream);
extern "C" int cdfo_conv3x3_pair_sm100_planes_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, void *y,
                                                  int B, int Cin, int Cout, int H, int W, int act, int y_planes, void *stream);

extern "C" int cdfo_conv3x3_pair_sm100_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, void *y_c8, int B,
                                           int Cin, int Cout, int H, int W, int act, void *stream) {
  return cdfo_conv3x3_pair_sm100_planes_fwd(x_c8, wpk, bias, resid_c8, y_c8, B, Cin, Cout, H, W, act, 0, stream);
}

extern "C" int cdfo_conv3x3_pair_sm100_planes_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, void *y_c8,
                                                  int B, int Cin, int Cout, int H, int W, int act, int y_planes, void *stream) {
  return cdfo_conv3x3_pair_sm100_edge_fwd(x_c8, wpk, bias, nullptr, resid_c8, y_c8, B, Cin, Cout, H, W, act, y_planes, stream);
}

extern "C" int cdfo_conv3x3_pair_sm100_edge_fwd(const void *x_c8, const void *wpk, const float *bias, const float *bias_edge, const void *resid_c8,
                                               void *y_c8, int B, int Cin, int Cout, int H, int W, int act, int y_planes, void *stream) {
  CDFO_REQUIRE(x_c8 && wpk && y_c8, CDFO_ERR_NULL, "cdfo_conv3x3_pair_sm100_fwd: NULL pointer");
  CDFO_REQUIRE(y_planes == 0 || y_planes == 2 || (y_planes == 1 && H % 2 == 0 && W % 2 == 0), CDFO_ERR_SHAPE,
               "cdfo_conv3x3_pair_sm100_planes_fwd: the parity-plane output needs an even size (got %d x %d)", H, W);
  CDFO_REQUIRE(B > 0 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_conv3x3_pair_sm100_fwd: bad shape");
  CDFO_REQUIRE(cdfo_conv3x3_pair_sm100_supported(Cout, Cin), CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100_fwd: unsupported channels %d -> %d", Cin, Cout);
  CDFO_REQUIRE(act >= 0 && act <= 2, CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100_fwd: act %d", act);
  CDFO_REQUIRE(((uintptr_t)x_c8 & 15) == 0 && ((uintptr_t)wpk & 15) == 0 && ((uintptr_t)y_c8 & 15) == 0 && ((uintptr_t)resid_c8 & 15) == 0,
               CDFO_ERR_SHAPE, "cdfo_conv3x3_pair_sm100_fwd: pointers must be 16-byte aligned");
  cpair::EncodeTiledFn enc = cpair::encode_tiled_fn();
  CDFO_REQUIRE(enc, CDFO_ERR_CUDA, "cdfo_conv3x3_pair_sm100_fwd: cuTensorMapEncodeTiled not available from the driver");
  CUtensorMap tm;
  static const bool wide128 = getenv("CDFO_TMA_WIDE") == nullptr || getenv("CDFO_TMA_WIDE")[0] != '0';
  static const bool wide32 = getenv("CDFO_TMA_WIDE32") == nullptr || getenv("CDFO_TMA_WIDE32")[0] != '0';
  const bool wide = cpair::half_channels(Cout, Cin) == 128 ? wide128 : wide32;
  cuuint64_t gdim[5] = {8, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)(Cin / 8), (cuuint64_t)B};
  cuuint64_t gstr[4] = {16, (cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)(Cin / 8) * H * W * 16};
  cuuint32_t box[5] = {8, (cuuint32_t)cpair::kHaloW, (cuuint32_t)cpair::kHaloH, 8, 1};
  if (wide) {   // same bytes, same landing order, one request per halo row instead of one per pixel chunk
    gdim[0] = (cuuint64_t)W * 8; gdim[1] = H; gdim[2] = Cin / 8; gdim[3] = B; gdim[4] = 1;
    gstr[0] = (cuuint64_t)W * 16; gstr[1] = (cuuint64_t)H * W * 16; gstr[2] = (cuuint64_t)(Cin / 8) * H * W * 16; gstr[3] = gstr[2] * B;
    box[0] = 8 * cpair::kHaloW; box[1] = cpair::kHaloH; box[2] = 8; box[3] = 1; box[4] = 1;
  }
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult cr = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void *>(x_c8), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CDFO_REQUIRE(cr == CUDA_SUCCESS, CDFO_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)cr);
  cpair::Params p;
  p.wpk = (const uint8_t *)wpk; p.bias = bias; p.bias_edge = bias_edge; p.resid = (const uint4 *)resid_c8; p.x1 = nullptr; p.y = (uint4 *)y_c8;
  p.B = B; p.Cin = Cin; p.H = H; p.W = W; p.act = act; p.y_planes = y_planes; p.tma_wide = wide ? 1 : 0;
  p.tiles_x = ceil_div(W, cpair::kTileW); p.tiles_y = ceil_div(H, cpair::kTileH);
  const long long mt = (long long)B * p.tiles_x * p.tiles_y;
  CDFO_REQUIRE(mt < (1ll << 30), CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100_fwd: too many tiles");
  p.m_tiles = (int)mt;
  if (cpair::half_channels(Cout, Cin) == 32) return cpair::launch<32, false>(tm, p, (cudaStream_t)stream);
  return cpair::launch<128, false>(tm, p, (cudaStream_t)stream);
}

extern "C" int cdfo_conv3x3_pair_sm100_up2_fwd(const void *x8_1x, const void *wpk, const float *bias, const float *bias_edge, void *y,
                                               int B, int Cin, int Cout, int H2, int W2, int act, int y_planes, void *stream) {
  CDFO_REQUIRE(x8_1x && wpk && y, CDFO_ERR_NULL, "cdfo_conv3x3_pair_sm100_up2_fwd: NULL pointer");
  CDFO_REQUIRE(Cin == 64 && Cout == 256, CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100_up2_fwd: unsupported channels %d -> %d (64 -> 256 only)",
               Cin, Cout);
  CDFO_REQUIRE(B > 0 && H2 > 0 && W2 > 0 && H2 % 2 == 0 && W2 % 2 == 0, CDFO_ERR_SHAPE,
               "cdfo_conv3x3_pair_sm100_up2_fwd: the 2x size must be positive and even (got %d x %d)", H2, W2);
  CDFO_REQUIRE(y_planes == 0 || y_planes == 1, CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100_up2_fwd: y_planes %d", y_planes);
  CDFO_REQUIRE(act >= 0 && act <= 2, CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100_up2_fwd: act %d", act);
  CDFO_REQUIRE(((uintptr_t)x8_1x & 15) == 0 && ((uintptr_t)wpk & 15) == 0 && ((uintptr_t)y & 15) == 0, CDFO_ERR_SHAPE,
               "cdfo_conv3x3_pair_sm100_up2_fwd: pointers must be 16-byte aligned");
  CDFO_REQUIRE(cpair::smem_bytes(Cin, 128, true) <= 227 * 1024, CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100_up2_fwd: shared memory");
  CUtensorMap tm;                // unused: the A operand is built from x8_1x, not loaded by TMA
  memset(&tm, 0, sizeof(tm));
  cpair::Params p;
  p.wpk = (const uint8_t *)wpk; p.bias = bias; p.bias_edge = bias_edge; p.resid = nullptr; p.x1 = (const uint4 *)x8_1x; p.y = (uint4 *)y;
  p.B = B; p.Cin = Cin; p.H = H2; p.W = W2; p.act = act; p.y_planes = y_planes; p.tma_wide = 0;
  p.tiles_x = ceil_div(W2, cpair::kTileW); p.tiles_y = ceil_div(H2, cpair::kTileH);
  const long long mt = (long long)B * p.tiles_x * p.tiles_y;
  CDFO_REQUIRE(mt < (1ll << 30), CDFO_ERR_UNSUPPORTED, "cdfo_conv3x3_pair_sm100_up2_fwd: too many tiles");
  p.m_tiles = (int)mt;
  return cpair::launch<128, true>(tm, p, (cudaStream_t)stream);
}
