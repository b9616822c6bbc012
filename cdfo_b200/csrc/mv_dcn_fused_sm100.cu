// Offset / mask head + MV prior + modulated deformable convolution of MVDualAttAlignment as ONE sm_100a kernel.
//
// Reference chain (arch/SIDECVSR_our.py:3339-3352):
//   out_k  = conv_offset[-1](hidden_k), k = 1, 2                (64 -> 432, 3x3; hidden_k = lrelu(conv_offset[0](mdta_k)))
//   offset = 10 tanh(cat(o1_1, o2_1)) + 10 tanh(cat(o1_2, o2_2)) + flow.flip(1).repeat(...)
//   mask   = sigmoid(mask_1 + mask_2)
//   y      = deform_conv2d(x, offset, weight[64,64,3,3], bias, 1, 1, 1, mask)     (= ops/dcn .cu:570-632 semantics)
// The two-kernel path (conv3x3_sm100.cu DUAL head -> dcn_tex_sm100.cu) writes the 288 + 144 offset / mask values of every pixel
// to HBM as fp16 fields (1152 B / px) and reads them back; here they never leave the SM (SURVEY 8d row 3: the fused op is
// tensor-bound, 1 069 056 FLOP and 516 B per pixel).
//
// One persistent CTA per SM walks 16 x 8-pixel tiles.  Per tile, for each of the three tap-triples T (DCN taps 3T .. 3T+2):
//   MMA warp     head GEMM  D_e[128 px, 144] = sum over the 9 head taps, 64 ci:  hidden_e(halo) * W_T,  e = 1, 2  (tcgen05.mma
//                kind::f16, bf16, A = the TMA-staged 18 x 10 halo of the hidden map at a byte offset per tap, B = an 18 KB piece of
//                the permuted head weights streamed once per tile through a 3-stage ring and used for BOTH hidden maps)
//   16 producer  tcgen05.ld of their 2 x 36 accumulator columns -> bias, tanh / sigmoid (mv_head_math.cuh: bit-identical to
//   warps        the unfused head), + decoded MV prior in the reference's fp32 order -> 12 texture fetches (hardware bilinear of
//                the fp16x4 texel of one deformable group, dcn_tex_sm100.cu) -> x mask -> fp16 A operand of 3 DCN taps written
//                with tcgen05.st into a 4-stage ring in TENSOR MEMORY
//   MMA warp     DCN GEMM  Y[128 px, 64] += A_tap(TMEM) * Wd_tap   (TS form, fp16; issued one triple late, so that the gather of
//                triple T overlaps the head GEMM of triple T+1)
// and the producers drain Y (+ bias) to c8 bf16 / NCHW fp32 one triple into the next tile.
// TMEM (512 columns): head accumulators [0,144) and [160,304), DCN accumulator [320,384), A ring [384,512).
// Shared memory (218 KB): DCN weights 72 KB (resident), 2 x 2 hidden-map halos 90 KB, head weight ring 54 KB, biases, barriers.
// 18 warps: MMA issuer, one TMA pump thread (weight pieces + halos, non-blocking probes), 16 producers.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "cdfo_common.cuh"
#include "mv_head_math.cuh"
#include "sm100_ptx.cuh"

namespace cdfo {

// csrc/dcn_tex_sm100.cu: texture object over a q4t tensor (cached, never destroyed while it may be in use)
cudaError_t dcn_tex_get_texture(const void *ptr, int rows, int W, int Wpt, cudaStream_t stream, cudaTextureObject_t *out);

namespace fdcn {

constexpr int kTileH = 16, kTileW = 8;                  // 128 pixels: row m = ty * 8 + tx = TMEM lane
constexpr int kHaloH = kTileH + 2, kHaloW = kTileW + 2;
constexpr int kPlane = kHaloH * kHaloW * 16;            // one 8-channel chunk of the halo: 2880 B
constexpr int kZBytes = 8 * kPlane;                     // halo of one hidden map: 23040 B
constexpr int kNT = 144;                                // head output channels per triple: 3 taps x 16 groups x (dy, dx, m)
constexpr int kPiece = kNT * 64 * 2;                    // head weights of one (triple, head tap): 18432 B
constexpr int kWStages = 3, kAStages = 4;
constexpr int kDcnWBytes = 9 * 64 * 64 * 2, kTapWBytes = 64 * 64 * 2, kBLbo = 64 * 16;
constexpr int kWarps = 18, kThreads = kWarps * 32;      // warp 0 MMA issuer, 1 TMA pump (weights + hidden maps), 2..17 producers
constexpr int kProdWarp0 = 2, kProdThreads = 16 * 32;   // (576 threads: 112 registers per thread, no spills in the producers)
constexpr int kColH0 = 0, kColH1 = 160, kColD = 320, kColA = 384, kAColsPerStage = 32, kTmemCols = 512;

constexpr int kOffZ = kDcnWBytes;                       // 73728
constexpr int kOffRing = kOffZ + 4 * kZBytes;           // 165888
constexpr int kOffHBias = kOffRing + kWStages * kPiece; // 221184
constexpr int kOffDBias = kOffHBias + 432 * 4;
constexpr int kOffBars = kOffDBias + 64 * 4;
constexpr int kOffSlot = kOffBars + 32 * 8;
constexpr int kSmemBytes = kOffSlot + 16;
static_assert(kSmemBytes <= 232448, "shared memory budget");
static_assert(kOffZ % 128 == 0 && kZBytes % 128 == 0 && kOffRing % 128 == 0 && kPiece % 128 == 0 && kOffBars % 8 == 0, "alignment");

// barriers
constexpr int kBarZFull = 0, kBarZEmpty = 2, kBarWFull = 4, kBarWEmpty = 7, kBarHFull = 10, kBarHEmpty = 11, kBarAFull = 12,
              kBarAEmpty = 16, kBarDFull = 20, kBarDEmpty = 21, kBarDcnW = 22;

struct Params {
  cudaTextureObject_t tex;   // pitch-2D texture over the x samples [x0, x0 + xn) (q4t), rows = ((sample - x0) * 16 + quad) * (H + 3) + row
  const uint8_t *hw;         // head weights [3 triples][9 head taps][8 chunks][144][8] bf16, channels permuted (see host side)
  const float *hbias;        // [432] permuted the same way
  const float *mv;           // [B][2][H*W] (x, y) or nullptr
  const uint8_t *dw;         // DCN weights [9][8][64][8] fp16
  const float *dbias;        // [64] or nullptr
  void *y;
  uint2 *fields_out;         // debug tap: the fields this kernel computed, [B][9][8][H*W][2] x (dy, dx | m, 0) fp16, or nullptr
  float mag;
  int B, H, W, out_mode, x_batch;
  int x0, xn;                // this launch's x slice (csrc/dcn_tex_sm100.cu)
  int y_nb, y_cs, y_grp[8];  // c8 placement, as in dcn_tex_sm100.cu
  int tiles_x, tiles_per_img, num_tiles;
  int poll_ns;               // back-off between failed probes of the producers' long waits (0: none)
};

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

__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {   // fp16 x fp16 -> fp32, both K-major
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t *r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t *>(&v);
}
__device__ __forceinline__ uint32_t h2_as_u32(__half2 v) { return *reinterpret_cast<uint32_t *>(&v); }

// Long waits of the producer warps (a head GEMM or a DCN tap away): probe, then sleep -- every probe of an mbarrier is a wavefront in
// the L1TEX data stage, the resource this kernel saturates (ncu: tensor-core operand reads 45 % + texture 34 % + LSU 19 %).
__device__ __forceinline__ void wait_backoff(uint32_t bar, uint32_t parity, int ns) {
  uint32_t spins = 0;
  while (!ptx::mbar_try_wait_hint(bar, parity, 20000u)) {
    if (ns) __nanosleep(ns);
    if (++spins > (1u << 24)) __trap();
  }
}

__global__ void __launch_bounds__(kThreads, 1)
mv_head_dcn_fused_sm100_kernel(const __grid_constant__ Params p, const __grid_constant__ CUtensorMap ztm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  float *hbias_s = reinterpret_cast<float *>(smem + kOffHBias);
  float *dbias_s = reinterpret_cast<float *>(smem + kOffDBias);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kOffBars);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + kOffSlot);
  const uint32_t bar0 = ptx::smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  const uint32_t s_dw = ptx::smem_u32(smem), s_z = ptx::smem_u32(smem + kOffZ), s_ring = ptx::smem_u32(smem + kOffRing);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int P = p.H * p.W;
  const int my_tiles = blockIdx.x < p.num_tiles ? (p.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  for (int i = tid; i < 432; i += kThreads) hbias_s[i] = p.hbias[i];
  if (tid < 64) dbias_s[tid] = p.dbias ? p.dbias[tid] : 0.f;
  if (warp == 0) {
    if (lane == 0) {
      for (int s = 0; s < 2; ++s) {
        ptx::mbar_init(BAR(kBarZFull + s), 1);
        ptx::mbar_init(BAR(kBarZEmpty + s), 1);
      }
      for (int s = 0; s < kWStages; ++s) {
        ptx::mbar_init(BAR(kBarWFull + s), 1);
        ptx::mbar_init(BAR(kBarWEmpty + s), 1);
      }
      ptx::mbar_init(BAR(kBarHFull), 1);
      ptx::mbar_init(BAR(kBarHEmpty), kProdThreads);
      for (int s = 0; s < kAStages; ++s) {
        ptx::mbar_init(BAR(kBarAFull + s), kProdThreads);
        ptx::mbar_init(BAR(kBarAEmpty + s), 1);
      }
      ptx::mbar_init(BAR(kBarDFull), 1);
      ptx::mbar_init(BAR(kBarDEmpty), kProdThreads);
      ptx::mbar_init(BAR(kBarDcnW), 1);
      ptx::fence_mbar_init();
    }
    __syncwarp();
    ptx::tmem_alloc(ptx::smem_u32(tmem_slot), kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ======================================= MMA issuer =======================================
    const uint32_t idesc_h = ptx::make_idesc_bf16(128, kNT), idesc_d = make_idesc_f16(128, 64);
    ptx::mbar_wait_parked(BAR(kBarDcnW), 0);
    int wst = 0, wph = 0, ast = 0, aph = 0;
    uint32_t q = 0;                        // triples issued by this CTA so far (3 per tile)
    auto issue_dcn = [&](uint32_t qq) {    // the three DCN taps of triple qq: A operand from the TMEM ring, weights resident
      const int T = (int)(qq % 3u);
      if (T == 0) {                        // first tap of a tile overwrites the accumulator: the previous tile must be drained
        ptx::mbar_wait_parked(BAR(kBarDEmpty), ((qq / 3u) & 1u) ^ 1u);
        ptx::tc_fence_after();
      }
      for (int tl = 0; tl < 3; ++tl) {
        const int tap = T * 3 + tl;
        ptx::mbar_wait_parked(BAR(kBarAFull + ast), aph);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const uint32_t a0 = tmem_base + kColA + ast * kAColsPerStage;
          const uint32_t b0 = s_dw + tap * kTapWBytes;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint64_t bd = ptx::make_smem_desc(b0 + j * 2 * kBLbo, kBLbo, 128);
            ptx::umma_f16_ts(tmem_base + kColD, a0 + j * 8, bd, idesc_d, (tap | j) != 0 ? 1u : 0u);
          }
          ptx::umma_commit(BAR(kBarAEmpty + ast));
          if (tap == 8) ptx::umma_commit(BAR(kBarDFull));
        }
        __syncwarp();
        if (++ast == kAStages) { ast = 0; aph ^= 1; }
      }
    };
    for (int it = 0; it < my_tiles; ++it) {
      const int zb = it & 1;
      ptx::mbar_wait_parked(BAR(kBarZFull + zb), (it >> 1) & 1);
      ptx::tc_fence_after();
      for (int T = 0; T < 3; ++T) {
        ptx::mbar_wait_parked(BAR(kBarHEmpty), (q & 1u) ^ 1u);      // the producers hold the previous triple's accumulators in registers
        ptx::tc_fence_after();
        for (int ht = 0; ht < 9; ++ht) {
          ptx::mbar_wait_parked(BAR(kBarWFull + wst), wph);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t za = s_z + zb * 2 * kZBytes + ((ht / 3) * kHaloW + (ht % 3)) * 16;
            const uint32_t b0 = s_ring + wst * kPiece;
#pragma unroll
            for (int ev = 0; ev < 2; ++ev) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint64_t ad = ptx::make_smem_desc(za + ev * kZBytes + j * 2 * kPlane, kPlane, kHaloW * 16);
                const uint64_t bd = ptx::make_smem_desc(b0 + j * 2 * (kNT * 16), kNT * 16, 128);
                ptx::umma_f16(tmem_base + (ev ? kColH1 : kColH0), ad, bd, idesc_h, (ht | j) != 0 ? 1u : 0u);
              }
            }
            ptx::umma_commit(BAR(kBarWEmpty + wst));
            if (ht == 8) {
              ptx::umma_commit(BAR(kBarHFull));
              if (T == 2) ptx::umma_commit(BAR(kBarZEmpty + zb));
            }
          }
          __syncwarp();
          if (++wst == kWStages) { wst = 0; wph ^= 1; }
        }
        if (q > 0) issue_dcn(q - 1);       // one triple late: its gather ran underneath the head GEMM just issued
        ++q;
      }
    }
    if (q > 0) issue_dcn(q - 1);
  } else if (warp == 1) {
    // ======================================= TMA pump: DCN weights (once), head weight pieces (ring), hidden-map halos =======================================
    // One thread feeds both queues with non-blocking probes, so that a full weight ring never delays a halo load or vice versa.
    if (lane == 0) {
      ptx::prefetch_tmap(&ztm);
      ptx::mbar_arrive_expect_tx(BAR(kBarDcnW), kDcnWBytes);
      for (int t = 0; t < 9; ++t) ptx::bulk_g2s(s_dw + t * kTapWBytes, p.dw + t * kTapWBytes, kTapWBytes, BAR(kBarDcnW));
      int wst = 0, wph = 0, piece = 0, pit = 0, zit = 0;
      uint32_t idle = 0;
      while (pit < my_tiles || zit < my_tiles) {
        bool progress = false;
        if (zit < my_tiles && ptx::mbar_test_wait(BAR(kBarZEmpty + (zit & 1)), ((zit >> 1) & 1) ^ 1)) {
          const int zb = zit & 1;
          const TileCoord tc = tile_coord(p, blockIdx.x + zit * gridDim.x);
          ptx::mbar_arrive_expect_tx(BAR(kBarZFull + zb), 2 * kZBytes);
          // box = (10 px x 8 ch, 18 rows, 8 chunks): lands as [chunk][18][10][8] = the canonical K-major operand; out-of-frame
          // rows / columns arrive as zeros = the convolution's zero padding
          ptx::tma_load_5d(s_z + zb * 2 * kZBytes, &ztm, BAR(kBarZFull + zb), (tc.w0 - 1) * 8, tc.h0 - 1, 0, tc.b, 0);
          ptx::tma_load_5d(s_z + zb * 2 * kZBytes + kZBytes, &ztm, BAR(kBarZFull + zb), (tc.w0 - 1) * 8, tc.h0 - 1, 0, tc.b + p.B, 0);
          ++zit;
          progress = true;
        }
        if (pit < my_tiles && ptx::mbar_test_wait(BAR(kBarWEmpty + wst), wph ^ 1)) {
          // (triple, head tap) in issue order: [3][9] pieces, contiguous in HBM, the same 27 for every tile (L2-resident)
          ptx::mbar_arrive_expect_tx(BAR(kBarWFull + wst), kPiece);
          ptx::bulk_g2s(s_ring + wst * kPiece, p.hw + (size_t)piece * kPiece, kPiece, BAR(kBarWFull + wst));
          if (++wst == kWStages) { wst = 0; wph ^= 1; }
          if (++piece == 27) { piece = 0; ++pit; }
          progress = true;
        }
        if (progress) {
          idle = 0;
        } else {
          __nanosleep(250);
          if (++idle > (1u << 28)) __trap();     // a protocol bug must fault, not hang
        }
      }
    }
    __syncwarp();
  } else {
    // ======================================= producers: fields -> gather -> A operand; epilogue =======================================
    const int quarter = warp & 3;                    // TMEM lane quarter this warp may touch
    const int qs = (warp - kProdWarp0) >> 2;         // this thread's deformable groups 4 qs .. 4 qs + 3 (= channel quads)
    const int row = quarter * 32 + lane;             // tile pixel = TMEM lane
    const int ty = row >> 3, tx = row & 7;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const float Hf = (float)p.H;
    const cudaTextureObject_t tex = p.tex;
    const int plane_rows = p.H + 3;
    int ast = 0, aph = 0;
    uint32_t q = 0;

    auto epilogue = [&](int it) {                    // drain columns [16 qs, 16 qs + 16) of the DCN accumulator of tile `it`
      const TileCoord tc = tile_coord(p, blockIdx.x + it * gridDim.x);
      const int h = tc.h0 + ty, w = tc.w0 + tx;
      wait_backoff(BAR(kBarDFull), it & 1, p.poll_ns);
      ptx::tc_fence_after();
      uint32_t r[16];
      tmem_ld16(lane_base + kColD + qs * 16, r);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(BAR(kBarDEmpty));
      if (h < p.H && w < p.W) {
        const int pix = h * p.W + w;
        const float *bs = dbias_s + qs * 16;
        if (p.out_mode == 0) {
          float *y = reinterpret_cast<float *>(p.y) + ((size_t)tc.b * 64 + qs * 16) * P + pix;
#pragma unroll
          for (int n = 0; n < 16; ++n) __stcs(y + (size_t)n * P, __uint_as_float(r[n]) + bs[n]);
        } else {
          uint4 *y = reinterpret_cast<uint4 *>(p.y) + ((size_t)(tc.b % p.y_nb) * p.y_cs + p.y_grp[tc.b / p.y_nb] + qs * 2) * P + pix;
#pragma unroll
          for (int kc = 0; kc < 2; ++kc) {
            uint4 v;
            v.x = pack_bf2(__uint_as_float(r[kc * 8 + 0]) + bs[kc * 8 + 0], __uint_as_float(r[kc * 8 + 1]) + bs[kc * 8 + 1]);
            v.y = pack_bf2(__uint_as_float(r[kc * 8 + 2]) + bs[kc * 8 + 2], __uint_as_float(r[kc * 8 + 3]) + bs[kc * 8 + 3]);
            v.z = pack_bf2(__uint_as_float(r[kc * 8 + 4]) + bs[kc * 8 + 4], __uint_as_float(r[kc * 8 + 5]) + bs[kc * 8 + 5]);
            v.w = pack_bf2(__uint_as_float(r[kc * 8 + 6]) + bs[kc * 8 + 6], __uint_as_float(r[kc * 8 + 7]) + bs[kc * 8 + 7]);
            y[(size_t)kc * P] = v;
          }
        }
      }
    };

    for (int it = 0; it < my_tiles; ++it) {
      const TileCoord tc = tile_coord(p, blockIdx.x + it * gridDim.x);
      const int h = tc.h0 + ty, w = tc.w0 + tx;
      const bool live = h < p.H && w < p.W;
      const int pixc = min(h, p.H - 1) * p.W + min(w, p.W - 1);
      const float mvx = p.mv ? __ldg(p.mv + ((size_t)tc.b * 2 + 0) * P + pixc) : 0.f;
      const float mvy = p.mv ? __ldg(p.mv + ((size_t)tc.b * 2 + 1) * P + pixc) : 0.f;
      const float py = (float)(((tc.b % p.x_batch - p.x0) * 16 + qs * 4) * plane_rows) + 1.5f;   // texture row of image row -1.5, first quad
      const float wb0 = (float)(w - 1) + 1.5f;                                              // border shift + texel centre
#pragma unroll
      for (int T = 0; T < 3; ++T) {
        // ---- this thread's 2 x 36 head outputs of triple T: columns qs * 36 + (tl * 12 + gi * 3 + {dy, dx, m})
        uint32_t a0[36], a1[36];
        wait_backoff(BAR(kBarHFull), q & 1u, p.poll_ns);
        ptx::tc_fence_after();
#pragma unroll
        for (int c = 0; c < 9; ++c) {
          tmem_ld4(lane_base + kColH0 + qs * 36 + c * 4, a0 + c * 4);
          tmem_ld4(lane_base + kColH1 + qs * 36 + c * 4, a1 + c * 4);
        }
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        ptx::mbar_arrive(BAR(kBarHEmpty));             // the head GEMM of the next triple may overwrite both accumulators
        float hb[36];                                  // this thread's 36 biases: 9 broadcast LDS.128 (144-byte aligned rows)
        {
          const float4 *hb4 = reinterpret_cast<const float4 *>(hbias_s + T * kNT + qs * 36);
#pragma unroll
          for (int c = 0; c < 9; ++c) {
            const float4 v = hb4[c];
            hb[4 * c] = v.x; hb[4 * c + 1] = v.y; hb[4 * c + 2] = v.z; hb[4 * c + 3] = v.w;
          }
        }
        uint2 fld[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) {
          const float b0 = hb[3 * k], b1 = hb[3 * k + 1], b2 = hb[3 * k + 2];
          const uint2 f1 = head::first(__fadd_rn(__uint_as_float(a0[3 * k]), b0), __fadd_rn(__uint_as_float(a0[3 * k + 1]), b1),
                                       __fadd_rn(__uint_as_float(a0[3 * k + 2]), b2), p.mag);
          fld[k] = head::second(f1, __fadd_rn(__uint_as_float(a1[3 * k]), b0), __fadd_rn(__uint_as_float(a1[3 * k + 1]), b1),
                                __fadd_rn(__uint_as_float(a1[3 * k + 2]), b2), p.mag);
        }
        if (p.fields_out && live) {
          // same layout as the unfused head writes: [B][9 taps][8 group pairs][H*W][2 groups] x 8 bytes
          const int pix = h * p.W + w;
#pragma unroll
          for (int tl = 0; tl < 3; ++tl) {
            uint2 *dst = p.fields_out + ((((size_t)tc.b * 9 + T * 3 + tl) * 8 + qs * 2) * P + pix) * 2;
            *reinterpret_cast<uint4 *>(dst) = make_uint4(fld[tl * 4].x, fld[tl * 4].y, fld[tl * 4 + 1].x, fld[tl * 4 + 1].y);
            *reinterpret_cast<uint4 *>(dst + (size_t)P * 2) = make_uint4(fld[tl * 4 + 2].x, fld[tl * 4 + 2].y, fld[tl * 4 + 3].x, fld[tl * 4 + 3].y);
          }
        }
        // ---- texture fetches, two taps (8 fetches) in flight: reference order offset = residual + flow (arch:3347), then
        //      h_im = base + offset (.cu:614-615); x mask -> fp16 A operand (row = TMEM lane, K elements 16 qs .. +15 = columns 8 qs .. +7)
        const float hbT = (float)(h - 1 + T);
        float4 tv[3][4];
        auto fetch = [&](int tl) {
#pragma unroll
          for (int gi = 0; gi < 4; ++gi) {
            const float2 d = __half22float2(*reinterpret_cast<const __half2 *>(&fld[tl * 4 + gi].x));
            const float h_im = __fadd_rn(hbT, __fadd_rn(d.x, mvy));
            const float w_t = __fadd_rn(wb0 + (float)tl, __fadd_rn(d.y, mvx));
            const float hc = fminf(fmaxf(h_im, -1.f), Hf);      // stay inside this quad's plane (+ zero border); NaN -> -1 -> 0
            tv[tl][gi] = tex2D<float4>(tex, w_t, hc + (py + (float)(gi * plane_rows)));
          }
        };
        fetch(0);
        fetch(1);
#pragma unroll
        for (int tl = 0; tl < 3; ++tl) {
          uint32_t o[8];
#pragma unroll
          for (int gi = 0; gi < 4; ++gi) {
            const uint32_t mm = __byte_perm(fld[tl * 4 + gi].y, 0, 0x1010);      // (m, m) fp16x2
            const __half2 m2 = *reinterpret_cast<const __half2 *>(&mm);
            const float4 v = tv[tl][gi];
            o[gi * 2 + 0] = h2_as_u32(__hmul2(m2, __floats2half2_rn(v.x, v.y)));
            o[gi * 2 + 1] = h2_as_u32(__hmul2(m2, __floats2half2_rn(v.z, v.w)));
          }
          if (tl == 0) fetch(2);                       // its latency hides under the pack / store of taps 0 and 1
          wait_backoff(BAR(kBarAEmpty + ast), aph ^ 1, p.poll_ns);
          ptx::tc_fence_after();
          ptx::tmem_st8(lane_base + kColA + ast * kAColsPerStage + qs * 8, o);
          ptx::tmem_st_wait();
          ptx::tc_fence_before();
          ptx::mbar_arrive(BAR(kBarAFull + ast));
          if (++ast == kAStages) { ast = 0; aph ^= 1; }
        }
        if (T == 0 && it > 0) epilogue(it - 1);        // its last DCN taps were issued behind the head GEMM we just consumed
        ++q;
      }
    }
    if (my_tiles > 0) epilogue(my_tiles - 1);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) ptx::tmem_dealloc(tmem_base, kTmemCols);
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

static int run(const void *z_c8, const void *head_wpk, const float *head_bias, float magnitude, const void *x_q4t, const float *mv,
               const void *dcn_wpk, const float *dcn_bias, void *y, void *fields_out, int B, int H, int W, int out_mode, int x_batch,
               int y_nb, int y_cs, const int *y_grp, int num_ctas, void *stream) {
  CDFO_REQUIRE(z_c8 && head_wpk && head_bias && x_q4t && dcn_wpk && y, CDFO_ERR_NULL, "cdfo_mv_head_dcn_fused_sm100_fwd: NULL pointer");
  CDFO_REQUIRE(B > 0 && H > 0 && W > 0, CDFO_ERR_SHAPE, "cdfo_mv_head_dcn_fused_sm100_fwd: bad shape");
  CDFO_REQUIRE(out_mode == 0 || out_mode == 1, CDFO_ERR_UNSUPPORTED, "cdfo_mv_head_dcn_fused_sm100_fwd: out_mode %d", out_mode);
  CDFO_REQUIRE(((uintptr_t)z_c8 & 15) == 0 && ((uintptr_t)head_wpk & 15) == 0 && ((uintptr_t)dcn_wpk & 15) == 0 && ((uintptr_t)y & 15) == 0 &&
                   ((uintptr_t)x_q4t & 511) == 0 && ((uintptr_t)fields_out & 15) == 0,
               CDFO_ERR_SHAPE, "cdfo_mv_head_dcn_fused_sm100_fwd: x_q4t must be 512-byte aligned (texture base), the other pointers 16-byte");
  CDFO_REQUIRE(W + 3 <= 131072, CDFO_ERR_UNSUPPORTED, "cdfo_mv_head_dcn_fused_sm100_fwd: frame width %d exceeds the 2-D linear texture limit", W);
  fdcn::Params p;
  memset(&p, 0, sizeof(p));
  p.x_batch = x_batch > 0 ? x_batch : B;
  CDFO_REQUIRE(B % p.x_batch == 0, CDFO_ERR_SHAPE, "cdfo_mv_head_dcn_fused_sm100_fwd: B (%d) must be a multiple of x_batch (%d)", B, p.x_batch);
  const long long sample_rows = 16ll * (H + 3);
  CDFO_REQUIRE(sample_rows <= kTexRows, CDFO_ERR_UNSUPPORTED,
               "cdfo_mv_head_dcn_fused_sm100_fwd: frame height %d exceeds the 2-D linear texture limit (16 * (H + 3) <= %d rows)", H, kTexRows);
  CDFO_REQUIRE((long long)9 * 16 * H * W < (1ll << 31), CDFO_ERR_UNSUPPORTED, "cdfo_mv_head_dcn_fused_sm100_fwd: frame too large for 32-bit indexing");
  const int Wpt = cdfo_q4t_pitch(W);
  fdcn::EncodeTiledFn enc = fdcn::encode_tiled_fn();
  CDFO_REQUIRE(enc, CDFO_ERR_CUDA, "cdfo_mv_head_dcn_fused_sm100_fwd: cuTensorMapEncodeTiled not available from the driver");
  // hidden maps: c8 bf16 [2 B][8][H][W][8]; pixel and channel axes merged so that TMA issues one request per halo row
  CUtensorMap ztm;
  const cuuint64_t gdim[5] = {(cuuint64_t)W * 8, (cuuint64_t)H, 8, (cuuint64_t)2 * B, 1};
  const cuuint64_t gstr[4] = {(cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)8 * H * W * 16, (cuuint64_t)8 * H * W * 16 * 2 * B};
  const cuuint32_t box[5] = {8 * fdcn::kHaloW, fdcn::kHaloH, 8, 1, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult cr = enc(&ztm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void *>(z_c8), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CDFO_REQUIRE(cr == CUDA_SUCCESS, CDFO_ERR_CUDA, "cdfo_mv_head_dcn_fused_sm100_fwd: cuTensorMapEncodeTiled failed with CUresult %d", (int)cr);
  p.hw = (const uint8_t *)head_wpk; p.hbias = head_bias; p.mv = mv; p.dw = (const uint8_t *)dcn_wpk; p.dbias = dcn_bias; p.y = y;
  p.fields_out = (uint2 *)fields_out; p.mag = magnitude;
  p.B = B; p.H = H; p.W = W; p.out_mode = out_mode;
  p.y_nb = y_nb; p.y_cs = y_cs;
  for (int g = 0; g < 8; ++g) p.y_grp[g] = y_grp[g];
  p.tiles_x = ceil_div(W, fdcn::kTileW);
  p.tiles_per_img = p.tiles_x * ceil_div(H, fdcn::kTileH);
  const long long nt = (long long)p.tiles_per_img * B;
  CDFO_REQUIRE(nt < (1ll << 31), CDFO_ERR_UNSUPPORTED, "cdfo_mv_head_dcn_fused_sm100_fwd: too many tiles");
  {
    static const int poll = getenv("CDFO_FUSED_POLL_NS") ? atoi(getenv("CDFO_FUSED_POLL_NS")) : 0;
    p.poll_ns = poll;
  }
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(fdcn::mv_head_dcn_fused_sm100_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fdcn::kSmemBytes);
    if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "cudaFuncSetAttribute(mv_head_dcn_fused_sm100): %s", cudaGetErrorString(e));
    attr_done = true;
  }
  const TexSlices sl = tex_slices(p.x_batch, sample_rows);
  for (int x0 = 0; x0 < p.x_batch; x0 += sl.per) {
    p.x0 = x0;
    p.xn = p.x_batch - x0 < sl.per ? p.x_batch - x0 : sl.per;
    const uint8_t *base = (const uint8_t *)x_q4t + (size_t)x0 * (size_t)sample_rows * Wpt * 8;   // a multiple of 512 bytes
    cudaError_t e = dcn_tex_get_texture(base, (int)(p.xn * sample_rows), W, Wpt, (cudaStream_t)stream, &p.tex);
    if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "cdfo_mv_head_dcn_fused_sm100_fwd: cudaCreateTextureObject: %s", cudaGetErrorString(e));
    p.num_tiles = p.tiles_per_img * (B / p.x_batch) * p.xn;
    int grid = num_ctas > 0 ? num_ctas : kNumSMs;
    if (grid > p.num_tiles) grid = p.num_tiles;
    fdcn::mv_head_dcn_fused_sm100_kernel<<<grid, fdcn::kThreads, fdcn::kSmemBytes, (cudaStream_t)stream>>>(p, ztm);
    if (int rc = check_launch("cdfo_mv_head_dcn_fused_sm100_fwd")) return rc;
  }
  return CDFO_OK;
}

}  // namespace fdcn
}  // namespace cdfo

using namespace cdfo;

extern "C" int cdfo_mv_head_dcn_fused_sm100_fwd(const void *z_c8, const void *head_wpk, const float *head_bias, float magnitude,
                                                const void *x_q4t, const float *mv, const void *dcn_wpk, const float *dcn_bias, void *y,
                                                void *fields_out, int B, int H, int W, int out_mode, int x_batch, int num_ctas,
                                                void *stream) {
  const int grp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  return fdcn::run(z_c8, head_wpk, head_bias, magnitude, x_q4t, mv, dcn_wpk, dcn_bias, y, fields_out, B, H, W, out_mode, x_batch, B, 8, grp,
                   num_ctas, stream);
}

extern "C" int cdfo_mv_head_dcn_fused_sm100_stacked_fwd(const void *z_c8, const void *head_wpk, const float *head_bias, float magnitude,
                                                        const void *x_q4t, const float *mv, const void *dcn_wpk, const float *dcn_bias,
                                                        void *y_stack, int n_seq, int n_groups, int stack_chunks, const int *group_chunk,
                                                        int H, int W, int x_batch, void *stream) {
  CDFO_REQUIRE(n_seq > 0 && n_groups > 0 && n_groups <= 8 && group_chunk, CDFO_ERR_SHAPE, "cdfo_mv_head_dcn_fused_sm100_stacked_fwd: 1..8 groups");
  int grp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int g = 0; g < n_groups; ++g) {
    CDFO_REQUIRE(group_chunk[g] >= 0 && group_chunk[g] + 8 <= stack_chunks, CDFO_ERR_SHAPE,
                 "cdfo_mv_head_dcn_fused_sm100_stacked_fwd: chunk slot out of range");
    grp[g] = group_chunk[g];
  }
  return fdcn::run(z_c8, head_wpk, head_bias, magnitude, x_q4t, mv, dcn_wpk, dcn_bias, y_stack, nullptr, n_seq * n_groups, H, W, 1, x_batch,
                   n_seq, stack_chunks, grp, 0, stream);
}
