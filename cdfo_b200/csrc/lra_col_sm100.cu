// Column pass of LLongRangAttention (arch/SIDECVSR_our.py:2225-2231) on the 5th-generation tensor cores:
//   per image column (b, w), H tokens of 64 channels:   long[h] = softmax_h'( q_c[h] . q_c[h'] ) . vrow[h']
//   q_c = conv9x1 along H of sq (built from the compact mask info exactly as lra_col_bf16_kernel does), vrow = the row pass's output.
// Round 1 ran it as warp-level mma.sync flash passes (1.2 ms per 12 calls at 272x480, tensor pipe 19 %); here one persistent CTA per SM
// keeps the whole H x H score tile of 128 queries in TENSOR MEMORY:
//   8 builder warps   next column's operands into the other shared-memory buffer, in the tcgen05 canonical K-major layout: Q [Mp rows][64]
//                     bf16 (queries AND keys: the scores are q_c q_c^T) and V^T [64 dims][Hp keys] bf16 (fp32 -> bf16 on the fly)
//   MMA warp          per 128-query tile: S[128, Hp] = Q_tile Q^T (tcgen05.mma kind::f16, bf16, N <= 256 per instruction), then
//                     O[128, 64] = P V with P read from tensor memory (TS form)
//   4 softmax warps   thread = query row: two passes over its S row with tcgen05.ld (max, then exp2 / sum), probabilities written
//                     back as bf16 with tcgen05.st OVER the scores they came from (column c of P covers keys 2c, 2c+1, already consumed),
//                     then the O tile * 1/sum -> long_out (NHWC fp32, 256 contiguous bytes per thread)
// TMEM: S / P columns [0, Hp), O columns [448, 512).  Hp = H rounded up to 16 <= 448; taller frames keep the mma.sync kernel.
#include "cdfo_common.cuh"
#include "sm100_ptx.cuh"

namespace cdfo {

namespace lct {

constexpr int kWarps = 13, kThreads = kWarps * 32;      // warp 0 MMA issuer, 1..4 softmax / epilogue, 5..12 builders
constexpr int kBuildWarp0 = 5, kBuildThreads = 8 * 32;
constexpr int kColO = 448, kTmemCols = 512;
constexpr int kBarQvFull = 0, kBarQvEmpty = 2, kBarSFull = 4, kBarPFull = 5, kBarOFull = 6, kBarOEmpty = 7;

struct Params {
  const float *vrow_t;     // [B][W][H][64]
  const uint8_t *midx;     // [B][H][W]
  const float *qsel;       // [B][H][W]
  float *long_out;         // [B][H][W][64]
  LraTables t;
  int B, H, W, Hp, n_mt, Mp, ncols;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&v);
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
      "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(kThreads, 1) lra_col_sm100_kernel(const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int H = p.H, W = p.W, Hp = p.Hp, Mp = p.Mp, HW = H * W;
  const uint32_t q_bytes = (uint32_t)Mp * 128u, v_bytes = (uint32_t)Hp * 128u, buf_bytes = q_bytes + v_bytes;
  uint8_t *scratch = smem + 2 * buf_bytes;                 // builders: cq [H + 8] | cm [H + 8] | kws [9]
  float *cq = reinterpret_cast<float *>(scratch);
  int *cm = reinterpret_cast<int *>(cq + H + 8);
  float *kws = reinterpret_cast<float *>(cm + H + 8);
  uint64_t *bars = reinterpret_cast<uint64_t *>(scratch + (((size_t)(2 * (H + 8) + 16) * 4 + 15) & ~(size_t)15));
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 8);
  const uint32_t bar0 = ptx::smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  const uint32_t s_buf0 = ptx::smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int my_cols = blockIdx.x < p.ncols ? (p.ncols - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp == 0) {
    if (lane == 0) {
      for (int s = 0; s < 2; ++s) {
        ptx::mbar_init(BAR(kBarQvFull + s), kBuildThreads);
        ptx::mbar_init(BAR(kBarQvEmpty + s), 1);
      }
      ptx::mbar_init(BAR(kBarSFull), 1);
      ptx::mbar_init(BAR(kBarPFull), 128);
      ptx::mbar_init(BAR(kBarOFull), 1);
      ptx::mbar_init(BAR(kBarOEmpty), 128);
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

  // score MMAs: keys in chunks of N <= 256 (multiples of 16)
  const int n_chunks = Hp > 256 ? 2 : 1;
  const int n_first = n_chunks == 2 ? (((Hp / 2) + 15) & ~15) : Hp;

  if (warp == 0) {
    // ======================================= MMA issuer =======================================
    const uint32_t idesc_o = ptx::make_idesc_bf16(128, 64);
    uint32_t gt = 0;
    for (int ci = 0; ci < my_cols; ++ci) {
      const int buf = ci & 1;
      const uint32_t qb = s_buf0 + buf * buf_bytes, vb = qb + q_bytes;
      ptx::mbar_wait_parked(BAR(kBarQvFull + buf), (ci >> 1) & 1);
      ptx::tc_fence_after();
      for (int mt = 0; mt < p.n_mt; ++mt) {
        if (ptx::elect_one()) {
          // S = Q_tile Q^T.  (In order behind the previous tile's P V, which was the last reader of these columns.)
          for (int c = 0; c < n_chunks; ++c) {
            const int n0 = c ? n_first : 0, nn = c ? Hp - n_first : n_first;
            const uint32_t idesc_s = ptx::make_idesc_bf16(128, nn);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t ad = ptx::make_smem_desc(qb + (uint32_t)mt * 2048u + (uint32_t)k * 2u * (uint32_t)Mp * 16u, (uint32_t)Mp * 16u, 128);
              const uint64_t bd = ptx::make_smem_desc(qb + (uint32_t)(n0 >> 3) * 128u + (uint32_t)k * 2u * (uint32_t)Mp * 16u, (uint32_t)Mp * 16u, 128);
              ptx::umma_f16(tmem_base + n0, ad, bd, idesc_s, k != 0 ? 1u : 0u);
            }
          }
          ptx::umma_commit(BAR(kBarSFull));
        }
        __syncwarp();
        ptx::mbar_wait_parked(BAR(kBarPFull), gt & 1u);                // probabilities are in tensor memory
        ptx::tc_fence_after();
        ptx::mbar_wait_parked(BAR(kBarOEmpty), (gt & 1u) ^ 1u);        // the previous tile's O has been read
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          for (int ks = 0; ks < Hp / 16; ++ks) {                        // O = P V: A = 16 keys of P (8 TMEM columns), B = V^T
            const uint64_t bd = ptx::make_smem_desc(vb + (uint32_t)ks * 2048u, 1024, 128);
            ptx::umma_f16_ts(tmem_base + kColO, tmem_base + ks * 8, bd, idesc_o, ks != 0 ? 1u : 0u);
          }
          ptx::umma_commit(BAR(kBarOFull));
          if (mt == p.n_mt - 1) ptx::umma_commit(BAR(kBarQvEmpty + buf));
        }
        __syncwarp();
        ++gt;
      }
    }
  } else if (warp < kBuildWarp0) {
    // ======================================= softmax + epilogue: thread = query row =======================================
    const int quarter = warp & 3, row = quarter * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int n32 = (Hp + 31) >> 5;
    uint32_t gt = 0;
    for (int ci = 0; ci < my_cols; ++ci) {
      const int col = blockIdx.x + ci * gridDim.x, b = col / W, w = col - b * W;
      for (int mt = 0; mt < p.n_mt; ++mt) {
        ptx::mbar_wait_parked(BAR(kBarSFull), gt & 1u);
        ptx::tc_fence_after();
        // pass 1: row maximum over the live keys.  The tcgen05.ld of chunk c + 1 is in flight while chunk c is reduced (two register
        // buffers); only the last chunk can hold keys >= H (stale columns), so only it pays the bounds checks.
        float mx = -INFINITY;
        uint32_t ra[32], rb[32];
        auto max_chunk = [&](const uint32_t (&r)[32], int c) {
          if (c * 32 + 32 <= H) {
#pragma unroll
            for (int i = 0; i < 32; i += 2) mx = fmaxf(mx, fmaxf(__uint_as_float(r[i]), __uint_as_float(r[i + 1])));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c * 32 + i < H) mx = fmaxf(mx, __uint_as_float(r[i]));
          }
        };
        ptx::tmem_ld32(lane_base, ra);
        for (int c = 0; c < n32; c += 2) {
          ptx::tmem_ld_wait();
          if (c + 1 < n32) ptx::tmem_ld32(lane_base + (c + 1) * 32, rb);
          max_chunk(ra, c);
          if (c + 1 < n32) {
            ptx::tmem_ld_wait();
            if (c + 2 < n32) ptx::tmem_ld32(lane_base + (c + 2) * 32, ra);
            max_chunk(rb, c + 1);
          }
        }
        // pass 2: p = exp(s - max) as bf16 back into tensor memory (over the consumed scores: chunk c writes columns [16 c, 16 c + 16), which
        // belong to score chunk c / 2 <= c, already in registers or consumed; the prefetched chunk c + 1 starts at column 32 c + 32), row
        // sum in fp32
        const float mneg = -mx * 1.4426950408889634f;
        float sum = 0.f;
        auto exp_chunk = [&](const uint32_t (&r)[32], int c) {
          uint32_t o[16];
          if (c * 32 + 32 <= H) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float e0 = ex2(fmaf(__uint_as_float(r[2 * i]), 1.4426950408889634f, mneg));
              const float e1 = ex2(fmaf(__uint_as_float(r[2 * i + 1]), 1.4426950408889634f, mneg));
              sum += e0 + e1;
              o[i] = pack_bf16x2(e0, e1);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int k0 = c * 32 + 2 * i;
              const float e0 = k0 < H ? ex2(fmaf(__uint_as_float(r[2 * i]), 1.4426950408889634f, mneg)) : 0.f;
              const float e1 = k0 + 1 < H ? ex2(fmaf(__uint_as_float(r[2 * i + 1]), 1.4426950408889634f, mneg)) : 0.f;
              sum += e0 + e1;
              o[i] = pack_bf16x2(e0, e1);
            }
          }
          if (c * 16 < Hp / 2) tmem_st16(lane_base + c * 16, o);      // warp-uniform condition
        };
        ptx::tmem_ld32(lane_base, ra);
        for (int c = 0; c < n32; c += 2) {
          ptx::tmem_ld_wait();
          if (c + 1 < n32) ptx::tmem_ld32(lane_base + (c + 1) * 32, rb);
          exp_chunk(ra, c);
          if (c + 1 < n32) {
            ptx::tmem_ld_wait();
            if (c + 2 < n32) ptx::tmem_ld32(lane_base + (c + 2) * 32, ra);
            exp_chunk(rb, c + 1);
          }
        }
        ptx::tmem_st_wait();
        ptx::tc_fence_before();
        ptx::mbar_arrive(BAR(kBarPFull));
        const float inv = 1.f / sum;
        // epilogue: O * 1/sum -> long_out[b][h][w][0..63]
        ptx::mbar_wait_parked(BAR(kBarOFull), gt & 1u);
        ptx::tc_fence_after();
        uint32_t a0[32], a1[32];
        ptx::tmem_ld32(lane_base + kColO, a0);
        ptx::tmem_ld32(lane_base + kColO + 32, a1);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        ptx::mbar_arrive(BAR(kBarOEmpty));
        const int h = mt * 128 + row;
        if (h < H) {
          float4 *dst = reinterpret_cast<float4 *>(p.long_out + (((size_t)b * H + h) * W + w) * 64);
#pragma unroll
          for (int i = 0; i < 8; ++i)
            dst[i] = make_float4(__uint_as_float(a0[4 * i]) * inv, __uint_as_float(a0[4 * i + 1]) * inv, __uint_as_float(a0[4 * i + 2]) * inv,
                                 __uint_as_float(a0[4 * i + 3]) * inv);
#pragma unroll
          for (int i = 0; i < 8; ++i)
            dst[8 + i] = make_float4(__uint_as_float(a1[4 * i]) * inv, __uint_as_float(a1[4 * i + 1]) * inv, __uint_as_float(a1[4 * i + 2]) * inv,
                                     __uint_as_float(a1[4 * i + 3]) * inv);
        }
        ++gt;
      }
    }
  } else {
    // ======================================= builders: Q and V^T of a column, canonical K-major =======================================
    const int bt = tid - kBuildWarp0 * 32, bl = bt & 31, bw = bt >> 5;
    float kh[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) kh[i] = p.t.kh[i];
    if (bt < 9) kws[bt] = p.t.kw[bt];
    // query / key rows >= H (up to Mp) are zero in both buffers for the whole launch: no column ever writes them
    for (int bsel = 0; bsel < 2; ++bsel) {
      uint4 *q4 = reinterpret_cast<uint4 *>(smem + (size_t)bsel * buf_bytes);
      for (uint32_t e = bt; e < q_bytes / 16; e += kBuildThreads) q4[e] = make_uint4(0u, 0u, 0u, 0u);
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kBuildThreads) : "memory");
    const float beta = p.t.beta, bh = p.t.bh;
    for (int ci = 0; ci < my_cols; ++ci) {
      const int buf = ci & 1;
      const int col = blockIdx.x + ci * gridDim.x, b = col / W, w = col - b * W;
      uint8_t *Qs = smem + (size_t)buf * buf_bytes, *Vs = Qs + q_bytes;
      ptx::mbar_wait_parked(BAR(kBarQvEmpty + buf), ((ci >> 1) & 1) ^ 1);
      // compact mask info of the column, rows -4 .. H + 3
      for (int e = bt; e < H + 8; e += kBuildThreads) {
        const int h = e - 4;
        int c = -1;
        float q = 0.f;
        if (h >= 0 && h < H) {
          c = p.midx[(size_t)b * HW + h * W + w];
          q = p.qsel[(size_t)b * HW + h * W + w];
        }
        cm[e] = c;
        cq[e] = q;
      }
      // V^T[d][k] <- vrow[k][d] (bf16): element (d, k) at (k / 8) * 1024 + (d / 8) * 128 + (d % 8) * 16 + (k % 8) * 2; keys >= H are zero.
      // A thread takes two consecutive keys x four channels; lanes = (key pair & 3) x (channel quad & 7), stores rotated per thread so
      // that a warp's 32 words of one store instruction fall into 32 different banks.
      {
        const float *vsrc = p.vrow_t + ((size_t)b * W + w) * H * 64;
        const int n_tasks = (Hp / 2) * 16;
        for (int e0 = bt; e0 < n_tasks; e0 += 4 * kBuildThreads) {          // four tasks' loads in flight per thread
          float4 v0[4], v1[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * kBuildThreads;
            v0[u] = v1[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (e < n_tasks) {
              const int kp = (e >> 6) * 4 + (e & 3), c4 = ((e >> 2) & 7) + ((e >> 5) & 1) * 8;      // e = [kp_hi | c4_hi | c4_lo(3) | kp_lo(2)]
              if (2 * kp < H) v0[u] = __ldg(reinterpret_cast<const float4 *>(vsrc + (size_t)(2 * kp) * 64 + c4 * 4));
              if (2 * kp + 1 < H) v1[u] = __ldg(reinterpret_cast<const float4 *>(vsrc + (size_t)(2 * kp + 1) * 64 + c4 * 4));
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * kBuildThreads;
            if (e < n_tasks) {
              const int kp = (e >> 6) * 4 + (e & 3), c4 = ((e >> 2) & 7) + ((e >> 5) & 1) * 8;
              const uint32_t wv[4] = {pack_bf16x2(v0[u].x, v1[u].x), pack_bf16x2(v0[u].y, v1[u].y), pack_bf16x2(v0[u].z, v1[u].z),
                                      pack_bf16x2(v0[u].w, v1[u].w)};
              uint32_t *base = reinterpret_cast<uint32_t *>(Vs + (size_t)(kp >> 2) * 1024) + (kp & 3);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int j = (i + (c4 >> 1)) & 3, d = c4 * 4 + j;
                base[(d >> 3) * 32 + (d & 7) * 4] = j == 0 ? wv[0] : (j == 1 ? wv[1] : (j == 2 ? wv[2] : wv[3]));
              }
            }
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kBuildThreads) : "memory");      // cm / cq complete
      // Q[h][c] = bh + sum_i kh[i] sq[h + i - 4][c],  sq[h'][c] = beta + kw[cm - c + 4] q inside the frame, 0 outside.
      // A warp owns a run of ceil(H / 8) consecutive rows, a lane two channels: the nine sq rows a query row needs slide through
      // registers (one new sq row per output row instead of nine; the window index is static after unrolling by 9), same fp32 operation
      // order as lra_col_bf16_kernel.  The 4-byte stores of a warp fall on four banks (eight channel chunks Mp * 16 bytes apart):
      // 8 wavefronts per row, negligible next to the arithmetic.
      {
        const int L = (H + 7) >> 3, r0 = bw * L, r1 = min(r0 + L, H);
        const int c0 = 2 * bl;
        auto sq_row = [&](int e, float &s0, float &s1) {       // e = row + 4
          const int c = cm[e];
          s0 = s1 = 0.f;
          if (c >= 0) {
            s0 = s1 = beta;
            if (c != 255) {
              const int t0 = c - c0 + 4, t1 = t0 - 1;
              const float q = cq[e];
              if (t0 >= 0 && t0 <= 8) s0 = fmaf(kws[t0], q, s0);
              if (t1 >= 0 && t1 <= 8) s1 = fmaf(kws[t1], q, s1);
            }
          }
        };
        if (r0 < r1) {
          float w0[9], w1[9];
#pragma unroll
          for (int i = 0; i < 8; ++i) sq_row(r0 + i, w0[i], w1[i]);
          uint32_t *qdst = reinterpret_cast<uint32_t *>(Qs + (size_t)(bl >> 2) * Mp * 16) + (bl & 3);
          for (int hb = r0; hb < r1; hb += 9) {
#pragma unroll
            for (int j = 0; j < 9; ++j) {
              const int h = hb + j;
              if (h < r1) {
                sq_row(h + 8, w0[(8 + j) % 9], w1[(8 + j) % 9]);
                float a0 = bh, a1 = bh;
#pragma unroll
                for (int i = 0; i < 9; ++i) {
                  a0 = fmaf(kh[i], w0[(i + j) % 9], a0);
                  a1 = fmaf(kh[i], w1[(i + j) % 9], a1);
                }
                qdst[(h >> 3) * 32 + (h & 7) * 4] = pack_bf16x2(a0, a1);
              }
            }
          }
        }
      }
      ptx::fence_proxy_async_smem();            // generic-proxy stores -> visible to tcgen05.mma's operand reads
      ptx::mbar_arrive(BAR(kBarQvFull + buf));
      asm volatile("bar.sync 1, %0;" ::"n"(kBuildThreads) : "memory");      // cm / cq may be overwritten
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) ptx::tmem_dealloc(tmem_base, kTmemCols);
}

}  // namespace lct

// dynamic shared memory of the kernel for H rows, 0 if the shape is outside its limits
static size_t lra_col_sm100_smem(int H) {
  const int Hp = (H + 15) & ~15;
  if (Hp > 448) return 0;
  const int Mp = ceil_div(H, 128) * 128 > Hp ? ceil_div(H, 128) * 128 : Hp;
  const size_t smem = 2 * ((size_t)Mp * 128 + (size_t)Hp * 128) + (((size_t)(2 * (H + 8) + 16) * 4 + 15) & ~(size_t)15) + 8 * 8 + 16;
  return smem > 227 * 1024 ? 0 : smem;
}

bool lra_col_sm100_fits(int H) { return lra_col_sm100_smem(H) != 0; }

// returns 1 if the kernel was launched, 0 if the shape is outside its limits (the caller falls back to the mma.sync kernel), < 0 on error
int lra_col_sm100_launch(const float *vrow_t, const uint8_t *midx, const float *qsel, float *long_out, const LraTables &t, int B, int H, int W,
                         cudaStream_t s) {
  const size_t smem = lra_col_sm100_smem(H);
  if (!smem) return 0;
  const int Hp = (H + 15) & ~15;
  lct::Params p;
  p.vrow_t = vrow_t; p.midx = midx; p.qsel = qsel; p.long_out = long_out; p.t = t;
  p.B = B; p.H = H; p.W = W; p.Hp = Hp;
  p.n_mt = ceil_div(H, 128);
  p.Mp = p.n_mt * 128 > Hp ? p.n_mt * 128 : Hp;
  p.ncols = B * W;
  static size_t attr_smem = 0;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(lct::lra_col_sm100_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "cudaFuncSetAttribute(lra_col_sm100): %s", cudaGetErrorString(e));
    attr_smem = smem;
  }
  const int grid = p.ncols < kNumSMs ? p.ncols : kNumSMs;
  lct::lra_col_sm100_kernel<<<grid, lct::kThreads, smem, s>>>(p);
  return check_launch("lra_col_sm100") == CDFO_OK ? 1 : CDFO_ERR_CUDA;
}

}  // namespace cdfo
