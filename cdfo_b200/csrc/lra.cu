// Prior-guided long-range attention (LLongRangAttention.forward, arch/SIDECVSR_our.py:2179-2249) without ever
// materialising a score tensor (the reference writes [B*H,W,W] + [B*W,H,H] + [B*H*W/64,64,64] fp32 scores).
//
// Observation that shapes the kernels: the residual mask is 1[softmax_c(v_c + gumbel_c) >= 0.5] (arch:2188-2195), so
// at most ONE channel per pixel is set.  The row-attention query/key  sq = conv1x9_channels(mask * q) + beta  is then
// "beta everywhere + one 9-tap bump", and the row score  sq_w . sq_w'  has the closed form
//     64 beta^2 + beta (s_w + s_w') + q_w q_w' R[c_w][c_w'],   s_w = q_w * K1[c_w]
// (K1 / R: 64 / 64x64 tables of tap sums, built on the host from directW1_conv).  Terms that do not depend on w'
// cancel in the softmax, so all unmasked queries of a row share ONE softmax distribution; masked queries get their own.
// Column attention has dense 64-d queries (9-tap mix along H of those rows) and is done as a flash-style pass per column.
//
//   lra_mask_kernel   u (uniform noise), v_max, q      -> per pixel: masked channel index (or 255) + its q value
//   lra_row_kernel    per (b, h): v -> conv1x9 over channels -> softmax(W) -> vrow, stored column-major for the next pass
//   lra_col_kernel    per (b, w): Q from the compact mask info (9-tap along H), softmax(H) . vrow -> long_out (NHWC)
//   lra_win_kernel    per 8x8 window: q with the masked channel zeroed, softmax(64) . v -> loc_out (NHWC)
//   fuse              1x1 conv(128 -> 64) over [long_out, loc_out] + bias + x -> NCHW fp32 (csrc/pointwise.cu, tensor cores)
// All arithmetic fp32 (the 0.5 threshold makes the mask discontinuous: keep it and the softmax exponents exact).
#include <cuda.h>
#include <cstring>

#include "cdfo_common.cuh"
#include "sm100_ptx.cuh"

namespace cdfo {

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------ mask
// u [B,64,H,W], vmax [B,64], q = qv[:, :64] of input_conv's output [B,128,H,W] -> midx [B,H,W] uint8, qsel [B,H,W] fp32
__global__ void lra_mask_kernel(const float *__restrict__ u, const float *__restrict__ vmax, const float *__restrict__ qv,
                                uint8_t *__restrict__ midx, float *__restrict__ qsel, int HW) {
  __shared__ float vm[64];
  const int b = blockIdx.y;
  if (threadIdx.x < 64) vm[threadIdx.x] = vmax[b * 64 + threadIdx.x];
  __syncthreads();
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const float *up = u + (size_t)b * 64 * HW + p;
  float lmax = -INFINITY, second_sum = 0.f;
  int cmax = 0;
  float l[64];
#pragma unroll
  for (int c = 0; c < 64; ++c) {
    const float g = -logf(-logf(up[(size_t)c * HW]));   // gumbel_softmax, arch:2173
    l[c] = vm[c] + g;
    if (l[c] > lmax) { lmax = l[c]; cmax = c; }
  }
#pragma unroll
  for (int c = 0; c < 64; ++c) second_sum += expf(l[c] - lmax);   // includes exp(0) = 1 of the max channel
  const bool on = (1.0f / second_sum) >= 0.5f;                    // softmax of the max channel >= 0.5 (arch:2194-2195)
  midx[(size_t)b * HW + p] = on ? (uint8_t)cmax : (uint8_t)255;
  qsel[(size_t)b * HW + p] = on ? qv[((size_t)b * 128 + cmax) * HW + p] : 0.f;
}

constexpr int kLd = 68;   // 68 % 32 == 4: eight consecutive rows hit distinct 16-byte bank groups
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}


// One 64-key block of a flash pass for a 16-query tile held by one warp (mma.sync m16n8k8 TF32 fragments):
// sc = raw scores in C-fragment layout ([n][0..1] = row g, keys 8n + 2tq, +1; [n][2..3] = row g + 8); keys >= n_keys are
// masked here.  Updates the running max / sum and O += P V with V rows [key0, key0 + 64) of Vu (TF32 bits, stride kLd).
// The probabilities feed the MMA from registers: C-fragment columns (2tq, 2tq+1) are used as A-fragment key positions
// (tq, tq+4) and the V fragment is loaded with the same permutation of the 8 keys.
__device__ __forceinline__ void flash_tile_block(float (&sc)[8][4], float (&m_run)[2], float (&l_run)[2], float (&o)[8][4],
                                                 const uint32_t *__restrict__ Vu, int key0, int n_keys, int g, int tq) {
  float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    const int key = key0 + 8 * n + 2 * tq;
    if (key >= n_keys) { sc[n][0] = -INFINITY; sc[n][2] = -INFINITY; }
    if (key + 1 >= n_keys) { sc[n][1] = -INFINITY; sc[n][3] = -INFINITY; }
    mx[0] = fmaxf(mx[0], fmaxf(sc[n][0], sc[n][1]));
    mx[1] = fmaxf(mx[1], fmaxf(sc[n][2], sc[n][3]));
  }
  float scale[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
    const float m_new = fmaxf(m_run[r], mx[r]);    // every block holds at least one live key (key0 < n_keys)
    scale[r] = expf(m_run[r] - m_new);
    m_run[r] = m_new;
    l_run[r] *= scale[r];
  }
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    sc[n][0] = expf(sc[n][0] - m_run[0]); sc[n][1] = expf(sc[n][1] - m_run[0]);
    sc[n][2] = expf(sc[n][2] - m_run[1]); sc[n][3] = expf(sc[n][3] - m_run[1]);
    l_run[0] += sc[n][0] + sc[n][1];
    l_run[1] += sc[n][2] + sc[n][3];
    o[n][0] *= scale[0]; o[n][1] *= scale[0]; o[n][2] *= scale[1]; o[n][3] *= scale[1];
  }
#pragma unroll
  for (int s = 0; s < 8; ++s) {
    const uint32_t ap[4] = {to_tf32(sc[s][0]), to_tf32(sc[s][2]), to_tf32(sc[s][1]), to_tf32(sc[s][3])};
    const uint32_t *vr = Vu + (key0 + 8 * s + 2 * tq) * kLd + g;
#pragma unroll
    for (int n = 0; n < 8; ++n) mma_tf32(o[n], ap, vr[8 * n], vr[kLd + 8 * n]);
  }
}

// ------------------------------------------------------------------------------------------------ rows
// CTA per (b, h).  v = qv[:, 64:]; output vrow_t [B][W][H][64] (token-major per column for the column pass).
// Unmasked queries share one softmax distribution (see the header): one weighted sum N0 for all of them.  Masked
// queries (~20 % of the tokens) get their own softmax over the row: their scores come from the closed form (tables,
// no dot products), and the P V products run on the tensor cores in 16-query tiles (flash_tile_block above).
constexpr int kRowWarps = 9, kRowThreads = kRowWarps * 32;
// TMA = true (W % 4 == 0): the raw v row arrives as 64-pixel pieces [64 channels][64 pixels] by tiled TMA (one box per piece from the NCHW
// map, zero-filled past W) through a two-stage mbarrier ring issued by warp 8, and warps 0-7 run the channel convolution from the piece
// (thread = pixel x 16 channels) straight into vr[w][c] -- the 4-byte cp.async copies of the other variant cost the LSU one request per
// element (32 768 per row: two thirds of the kernel, ncu + the same finding as csrc/lra_mask_logits.cu).  Same fp32 operation order.
constexpr int kRowPiece = 64;
constexpr int kRowRawBytes = 2 * 64 * kRowPiece * 4 + 64;      // two pieces + four mbarriers (128-byte aligned in front of vr)
// NCTA > 1 (rows too wide for one CTA's shared memory): the row is split over a cluster of NCTA CTAs (NCTA, 1, 1).  CTA rank r holds vr
// only for its slice [r * Ws, r * Ws + Ws) of the keys (whole 64-key blocks) and owns the queries of the same columns; the small per-key
// arrays, m0 and d0 cover the whole row in every CTA.  The N0 partials over each slice are exchanged through distributed shared memory and
// summed in rank order; a masked query's flash tile reads the key blocks of other slices from the holder's shared memory (generic loads
// through mapa addresses).  NCTA = 1 is the single-CTA kernel: every NCTA branch below folds away at compile time.
__host__ __device__ constexpr int lra_row_slice(int Wk, int ncta) { return ((Wk / 64 + ncta - 1) / ncta) * 64; }

template <typename T>
__device__ __forceinline__ const T *peer_smem(const T *p, int rank) {   // generic address of the same shared-memory offset in CTA `rank`
  uint64_t r;
  asm volatile("mapa.u64 %0, %1, %2;" : "=l"(r) : "l"(p), "r"(rank));
  return reinterpret_cast<const T *>(r);
}
__device__ __forceinline__ void row_cluster_sync() {
  __syncwarp();
  asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
}

template <int NCTA, bool TMA>
__global__ void __launch_bounds__(kRowThreads, 1) lra_row_kernel(const __grid_constant__ CUtensorMap qvmap, const float *__restrict__ qv,
                                                                const uint8_t *__restrict__ midx, const float *__restrict__ qsel,
                                                                float *__restrict__ vrow_t, LraTables t, int H, int W) {
  extern __shared__ __align__(1024) float sm_all[];
  float *sm = TMA ? sm_all + kRowRawBytes / 4 : sm_all;
  const int b = blockIdx.y, h = blockIdx.x / NCTA;
  const int rank = NCTA == 1 ? 0 : (int)(blockIdx.x % NCTA);   // = %cluster_ctarank for cluster dims (NCTA, 1, 1)
  const int HW = H * W;
  const int Wk = (W + 63) & ~63;      // keys padded to whole 64-key blocks
  const int Ws = NCTA == 1 ? Wk : lra_row_slice(Wk, NCTA);
  const int k_lo = rank * Ws;                                  // this CTA's keys [k_lo, k_hi) and queries [k_lo, w_end)
  const int k_hi = NCTA == 1 ? Wk : min(k_lo + Ws, Wk);
  const int w_end = NCTA == 1 ? W : min(W, k_hi);
  float *vr = sm;                     // [Ws][kLd] conv1x9(v) of keys k_lo + row as TF32 bits (keys >= W zero)
  float *Rs = vr + Ws * kLd;          // [64*64] R table
  float *sw = Rs + 4096;              // [Wk]  beta * s_w
  float *e0 = sw + Wk;                // [Wk]  exp(beta s_w - m0)
  float *qs = e0 + Wk;                // [Wk]  q of the masked channel
  float *n0 = qs + Wk;                // [64] common numerator
  float *red = n0 + 64;               // [kRowThreads] reduction scratch
  int *cs = reinterpret_cast<int *>(red + kRowThreads);  // [Wk] masked channel or -1
  int *mlist = cs + Wk;               // [Wk] indices of masked tokens
  __shared__ int mcount;
  __shared__ float m0_s, d0_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, tq = lane & 3;
  float kw[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) kw[i] = t.kw[i];
  for (int e = tid; e < 4096; e += kRowThreads) Rs[e] = t.r[e];

  // v_r[w][c] = beta + sum_t kw[t] v[c + t - 4][w]   (conv along the channel axis, arch:2219)
  if (TMA) {
    float *raw = sm_all;                                                    // [2][64 c][64 px]
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm_all + 2 * 64 * kRowPiece);
    const uint32_t bar0 = ptx::smem_u32(bars);                              // full 0, 1 | empty 0, 1
    if (tid == 0) {
      ptx::mbar_init(bar0, 1);
      ptx::mbar_init(bar0 + 8, 1);
      ptx::mbar_init(bar0 + 16, 8);
      ptx::mbar_init(bar0 + 24, 8);
      ptx::fence_mbar_init();
    }
    __syncthreads();
    const int n_pieces = (k_hi - k_lo) / kRowPiece;
    if (warp == 8) {
      if (lane == 0) {
        for (int pc = 0; pc < n_pieces; ++pc) {
          const int st = pc & 1;
          ptx::mbar_wait_parked(bar0 + 16 + 8 * st, ((pc >> 1) & 1) ^ 1);
          ptx::mbar_arrive_expect_tx(bar0 + 8 * st, 64 * kRowPiece * 4);
          ptx::tma_load_3d(ptx::smem_u32(raw) + st * 64 * kRowPiece * 4, &qvmap, bar0 + 8 * st, k_lo + pc * kRowPiece, h, b * 128 + 64);
        }
      }
    } else {
      const int px = tid & 63, c0 = (tid >> 6) * 16;                        // 256 threads: pixel x quarter of the channels
      for (int pc = 0; pc < n_pieces; ++pc) {
        const int st = pc & 1, w = k_lo + pc * kRowPiece + px;
        ptx::mbar_wait_parked(bar0 + 8 * st, (pc >> 1) & 1);
        const float *rp = raw + st * 64 * kRowPiece + px;
        float win[24];                                                      // channels c0 - 4 .. c0 + 19 (zero outside 0 .. 63)
#pragma unroll
        for (int i = 0; i < 24; ++i) {
          const int c = c0 - 4 + i;
          win[i] = (c >= 0 && c < 64) ? rp[c * kRowPiece] : 0.f;
        }
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bar0 + 16 + 8 * st);                // the piece is in registers
        float *row = vr + (w - k_lo) * kLd + c0;
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          float o[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float acc = t.beta;
#pragma unroll
            for (int i = 0; i < 9; ++i) acc = fmaf(kw[i], win[4 * c4 + j + i], acc);
            o[j] = w < W ? acc : 0.f;                                       // key rows past the frame stay zero
          }
          *reinterpret_cast<float4 *>(row + 4 * c4) = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
  } else {
  // the raw row is read from
  // global once (coalesced along w) into vr[w][c]; then one thread per pixel slides the 9 taps over its 64 channels in place
  const float *vbase = qv + ((size_t)b * 128 + 64) * HW + (size_t)h * W;
  // (4-byte cp.async: the ~107 copies of a thread are all in flight at once -- with one CTA of 9 warps per SM a load -> store loop
  // through registers leaves the SM waiting on one DRAM round trip per iteration)
  const int Wn = k_hi - k_lo;
  for (int e = tid; e < 64 * Wn; e += kRowThreads) {
    const int c = e / Wn, wl = e - c * Wn, w = k_lo + wl;
    const bool ok = w < W;
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(vr + wl * kLd + c);
    const float *src = vbase + (size_t)c * HW + (ok ? w : 0);
    const int nb = ok ? 4 : 0;            // src-size 0: zero fill
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(nb) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  for (int w = tid; w < w_end - k_lo; w += kRowThreads) {
    float *row = vr + w * kLd;
    float win[72];                         // channels -4 .. 67 of this pixel (zero outside 0 .. 63)
#pragma unroll
    for (int i = 0; i < 4; ++i) { win[i] = 0.f; win[68 + i] = 0.f; }
#pragma unroll
    for (int c4 = 0; c4 < 16; ++c4) {
      const float4 v = *reinterpret_cast<const float4 *>(row + 4 * c4);
      win[4 + 4 * c4] = v.x; win[5 + 4 * c4] = v.y; win[6 + 4 * c4] = v.z; win[7 + 4 * c4] = v.w;
    }
#pragma unroll
    for (int c4 = 0; c4 < 16; ++c4) {
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float acc = t.beta;
#pragma unroll
        for (int i = 0; i < 9; ++i) acc = fmaf(kw[i], win[4 * c4 + j + i], acc);
        o[j] = acc;
      }
      *reinterpret_cast<float4 *>(row + 4 * c4) = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
  }
  if (tid == 0) mcount = 0;
  __syncthreads();
  for (int w = tid; w < Wk; w += kRowThreads) {
    int c = 255;
    float q = 0.f;
    if (w < W) {
      c = midx[(size_t)b * HW + h * W + w];
      q = qsel[(size_t)b * HW + h * W + w];
    }
    const bool on = c != 255;
    cs[w] = on ? c : -1;
    qs[w] = q;
    sw[w] = on ? t.beta * q * t.k1[c] : 0.f;
    if (on && (NCTA == 1 || (w >= k_lo && w < k_hi))) mlist[atomicAdd(&mcount, 1)] = w;
  }
  __syncthreads();
  // common distribution of every unmasked query: softmax_w'(beta * s_w')
  float m = -INFINITY;
  for (int w = tid; w < W; w += kRowThreads) m = fmaxf(m, sw[w]);
  m = warp_max(m);
  if (lane == 0) red[warp] = m;
  __syncthreads();
  if (tid == 0) {
    float mm = red[0];
    for (int i = 1; i < kRowWarps; ++i) mm = fmaxf(mm, red[i]);
    m0_s = mm;
  }
  __syncthreads();
  const float m0 = m0_s;
  float d = 0.f;
  for (int w = tid; w < W; w += kRowThreads) {
    const float e = expf(sw[w] - m0);
    e0[w] = e;
    d += e;
  }
  d = warp_sum(d);
  __syncthreads();
  if (lane == 0) red[warp] = d;
  __syncthreads();
  if (tid == 0) {
    float dd = 0.f;
    for (int i = 0; i < kRowWarps; ++i) dd += red[i];
    d0_s = dd;
  }
  {  // N0[c] = sum_w' e0[w'] v_r[w'][c]: thread = (c, quarter of the row); exact fp32 (v_r is rounded to TF32 only afterwards)
    const int c = tid & 63, part = tid >> 6;
    float acc = 0.f;
    if (part < 4)
      for (int w = k_lo + part; w < w_end; w += 4) acc = fmaf(e0[w], vr[(w - k_lo) * kLd + c], acc);
    __syncthreads();
    red[tid] = acc;
    __syncthreads();
    if (NCTA == 1) {
      if (tid < 64) n0[tid] = (red[tid] + red[tid + 64] + red[tid + 128] + red[tid + 192]) / d0_s;
    } else {
      if (tid < 64) red[tid] = red[tid] + red[tid + 64] + red[tid + 128] + red[tid + 192];   // this slice's partial, read by every peer
    }
  }
  if (NCTA > 1) {
    // round this slice's v_r to TF32 here: the cluster barrier below then publishes both the partials and the finished key blocks
    for (int e = tid; e < (k_hi - k_lo) * 64; e += kRowThreads) {
      float *p = vr + (e >> 6) * kLd + (e & 63);
      *p = __uint_as_float(to_tf32(*p));
    }
    row_cluster_sync();
    if (tid < 64) {
      float s = 0.f;
      for (int r = 0; r < NCTA; ++r) s += r == rank ? red[tid] : peer_smem(red, r)[tid];   // rank order: the same sum in every CTA
      n0[tid] = s / d0_s;
    }
  }
  __syncthreads();
  // unmasked queries: the common vector
  for (int e = k_lo * 64 + tid; e < w_end * 64; e += kRowThreads) {
    const int w = e >> 6, c = e & 63;
    if (cs[w] < 0) vrow_t[(((size_t)b * W + w) * H + h) * 64 + c] = n0[c];
  }
  if (NCTA == 1) {
    // round v_r to TF32 in place for the tensor-core pass
    for (int e = tid; e < Wk * 64; e += kRowThreads) {
      float *p = vr + (e >> 6) * kLd + (e & 63);
      *p = __uint_as_float(to_tf32(*p));
    }
  }
  __syncthreads();
  // masked queries: own softmax over w'; one warp per tile of 16 masked queries
  const int nm = mcount;
  const uint32_t *Vu = reinterpret_cast<const uint32_t *>(vr);
  for (int q0 = warp * 16; q0 < nm; q0 += kRowWarps * 16) {
    int wq[2], c1[2];
    float q1[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int qi = q0 + g + 8 * r;
      wq[r] = qi < nm ? mlist[qi] : -1;
      c1[r] = wq[r] >= 0 ? cs[wq[r]] : 0;
      q1[r] = wq[r] >= 0 ? qs[wq[r]] : 0.f;
    }
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) o[n][i] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
    for (int key0 = 0; key0 < Wk; key0 += 64) {
      float sc[8][4];
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        const int k = key0 + 8 * n + 2 * tq;      // this thread's two keys of the group (C-fragment columns 2tq, 2tq + 1)
        const float2 s2 = *reinterpret_cast<const float2 *>(sw + k), q2 = *reinterpret_cast<const float2 *>(qs + k);
        const int2 c2 = *reinterpret_cast<const int2 *>(cs + k);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          sc[n][2 * r] = c2.x >= 0 ? fmaf(q1[r] * q2.x, Rs[c1[r] * 64 + c2.x], s2.x) : s2.x;
          sc[n][2 * r + 1] = c2.y >= 0 ? fmaf(q1[r] * q2.y, Rs[c1[r] * 64 + c2.y], s2.y) : s2.y;
        }
      }
      if (NCTA == 1) {
        flash_tile_block(sc, m_run, l_run, o, Vu, key0, W, g, tq);
      } else {   // the block's holder, with keys counted from the start of its slice
        const int r = key0 / Ws, lo = r * Ws;
        flash_tile_block(sc, m_run, l_run, o, r == rank ? Vu : peer_smem(Vu, r), key0 - lo, W - lo, g, tq);
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
      l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      if (wq[r] < 0) continue;
      const float inv = 1.f / l_run[r];
      float *dst = vrow_t + (((size_t)b * W + wq[r]) * H + h) * 64 + 2 * tq;
#pragma unroll
      for (int n = 0; n < 8; ++n) *reinterpret_cast<float2 *>(dst + 8 * n) = make_float2(o[n][2 * r] * inv, o[n][2 * r + 1] * inv);
    }
  }
  if (NCTA > 1) row_cluster_sync();   // no CTA retires while a peer may still read its key blocks
}

// ------------------------------------------------------------------------------------------------ flash-style block
// 256 threads compute, for a block of 64 queries against n_keys keys, softmax(Q K^T) V with an online softmax, fp32.
// Q / K / V rows have 64 features, row stride kLd floats in shared memory.  Register tile 4 x 4 per thread:
// thread (ty, tx) owns query rows {ty + 16 i} and key columns {tx + 16 j} of every 64 x 64 score tile, and query rows
// {ty + 16 i} x channels {4 tx .. 4 tx + 3} of the output: 8 LDS.128 feed 64 FMAs (the v1 kernels were LDS-bound at 2:1).

// key_chunk(kb) must make *Kptr point at keys kb*64 .. kb*64+63 and rows [0, 64) of Vs hold their values (rows beyond
// n_keys may hold anything finite: their probabilities are forced to 0), ending with a __syncthreads() if it wrote.
template <typename LoadKV, typename Store>
__device__ __forceinline__ void flash_block_fp32_kptr(const float *Qs, const float *const *Kptr, const float *Vs, float *Ps,
                                                      int n_keys, LoadKV key_chunk, Store store) {
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  float m_run[4], l_run[4], o[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m_run[i] = -INFINITY;
    l_run[i] = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) o[i][c] = 0.f;
  }
  const int n_chunks = (n_keys + 63) >> 6;
  for (int kb = 0; kb < n_chunks; ++kb) {
    key_chunk(kb);
    const float *Ks = *Kptr;
    float sacc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) sacc[i][j] = 0.f;
#pragma unroll 4
    for (int k = 0; k < 64; k += 4) {
      float4 a[4], bq[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4 *>(Qs + (ty + 16 * i) * kLd + k);
#pragma unroll
      for (int j = 0; j < 4; ++j) bq[j] = *reinterpret_cast<const float4 *>(Ks + (tx + 16 * j) * kLd + k);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          sacc[i][j] = fmaf(a[i].x, bq[j].x, sacc[i][j]);
          sacc[i][j] = fmaf(a[i].y, bq[j].y, sacc[i][j]);
          sacc[i][j] = fmaf(a[i].z, bq[j].z, sacc[i][j]);
          sacc[i][j] = fmaf(a[i].w, bq[j].w, sacc[i][j]);
        }
    }
    // online softmax: rows are shared by the 16 lanes with equal ty
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (kb * 64 + tx + 16 * j >= n_keys) sacc[i][j] = -INFINITY;
        mx = fmaxf(mx, sacc[i][j]);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float m_new = fmaxf(m_run[i], mx);
      const float scale = expf(m_run[i] - m_new);   // exp(-inf) = 0 on the first chunk
      m_run[i] = m_new;
      float ps = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float pv = expf(sacc[i][j] - m_new);
        Ps[(ty + 16 * i) * kLd + tx + 16 * j] = pv;
        ps += pv;
      }
      l_run[i] = l_run[i] * scale + ps;
#pragma unroll
      for (int c = 0; c < 4; ++c) o[i][c] *= scale;
    }
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < 64; j += 4) {
      float4 pr[4], vv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) pr[i] = *reinterpret_cast<const float4 *>(Ps + (ty + 16 * i) * kLd + j);
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) vv[jj] = *reinterpret_cast<const float4 *>(Vs + (j + jj) * kLd + 4 * tx);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float pe[4] = {pr[i].x, pr[i].y, pr[i].z, pr[i].w};
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          o[i][0] = fmaf(pe[jj], vv[jj].x, o[i][0]);
          o[i][1] = fmaf(pe[jj], vv[jj].y, o[i][1]);
          o[i][2] = fmaf(pe[jj], vv[jj].z, o[i][2]);
          o[i][3] = fmaf(pe[jj], vv[jj].w, o[i][3]);
        }
      }
    }
    __syncthreads();   // Ps / Ks / Vs are rewritten by the next chunk
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float l = l_run[i];
#pragma unroll
    for (int off = 8; off > 0; off >>= 1) l += __shfl_xor_sync(0xffffffffu, l, off);
    const float inv = 1.f / l;
    store(ty + 16 * i, 4 * tx, make_float4(o[i][0] * inv, o[i][1] * inv, o[i][2] * inv, o[i][3] * inv));
  }
}

// ------------------------------------------------------------------------------------------------ columns
// CTA per (b, w): q_c[h] = bh + sum_t kh[t] sq[h+t-4] (zero rows outside the frame), sq[h'] = beta + bump(h').
// The contraction is dense here (64-d queries, H x H scores per column), so it runs on the tensor cores: warp-level
// mma.sync m16n8k8 TF32 with fp32 accumulation, flash-style (online softmax over 64-key blocks, scores never leave
// registers).  Each of the 9 warps owns 16-query tiles; Q (also the keys: scores are q_c q_c^T, arch:2228) and V sit in
// shared memory as TF32-rounded fp32 with a row stride of 68 floats, which makes every fragment load conflict-free.
// The probabilities feed the second MMA straight from the accumulator registers: the C-fragment column pair (2t, 2t+1)
// is used as A-fragment key positions (t, t+4), and the V fragment is loaded with the same permutation of the 8 keys.
// TF32 (10-bit mantissa) on logits of magnitude <~ 1 (q_c is a 9-tap mix of beta + sparse bumps) changes the softmax
// weights by < 1e-3 relative; the window attention, whose logits reach +-40, stays in fp32 below.
constexpr int kColWarps = 9, kColThreads = kColWarps * 32;

__global__ void __launch_bounds__(kColThreads, 1) lra_col_kernel(const float *__restrict__ vrow_t, const uint8_t *__restrict__ midx,
                                                                const float *__restrict__ qsel, float *__restrict__ long_out,
                                                                LraTables t, int H, int W) {
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.y, w = blockIdx.x;
  const int HW = H * W;
  const int Hk = (H + 63) & ~63;          // keys padded to whole 64-key blocks (rows >= H are zero and masked)
  float *Q = sm;                          // [Hk][kLd] tf32 bit patterns
  float *V = Q + Hk * kLd;                // [Hk][kLd]; first used as scratch for sq [H + 8][64]
  float *sq = V;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, tq = lane & 3;
  float kh[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) kh[i] = t.kh[i];

  for (int e = tid; e < (H + 8) * 64; e += kColThreads) {   // sq[h][c] = beta + bump, zero padding rows
    const int h = (e >> 6) - 4, c = e & 63;
    float v = 0.f;
    if (h >= 0 && h < H) {
      v = t.beta;
      const int cm = midx[(size_t)b * HW + h * W + w];
      if (cm != 255) {
        const int ti = cm - c + 4;
        if (ti >= 0 && ti <= 8) v = fmaf(__ldg(t.kw + ti), qsel[(size_t)b * HW + h * W + w], v);
      }
    }
    sq[e] = v;
  }
  __syncthreads();
  for (int e = tid; e < Hk * 64; e += kColThreads) {   // Q = conv9 along H (rows >= H: zero)
    const int h = e >> 6, c = e & 63;
    float acc = 0.f;
    if (h < H) {
      acc = t.bh;
#pragma unroll
      for (int i = 0; i < 9; ++i) acc = fmaf(kh[i], sq[(h + i) * 64 + c], acc);
    }
    Q[h * kLd + c] = __uint_as_float(to_tf32(acc));
  }
  __syncthreads();   // sq is dead: V overwrites it
  const float *vsrc = vrow_t + ((size_t)b * W + w) * H * 64;   // contiguous [H][64]
  for (int e = tid; e < Hk * 16; e += kColThreads) {
    const int r = e >> 4, c4 = (e & 15) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < H) v = *reinterpret_cast<const float4 *>(vsrc + (size_t)r * 64 + c4);
    v.x = __uint_as_float(to_tf32(v.x)); v.y = __uint_as_float(to_tf32(v.y));
    v.z = __uint_as_float(to_tf32(v.z)); v.w = __uint_as_float(to_tf32(v.w));
    *reinterpret_cast<float4 *>(V + r * kLd + c4) = v;
  }
  __syncthreads();

  const uint32_t *Qu = reinterpret_cast<const uint32_t *>(Q), *Vu = reinterpret_cast<const uint32_t *>(V);
  const int n_qt = (H + 15) >> 4, n_kb = Hk >> 6;
  for (int qt = warp; qt < n_qt; qt += kColWarps) {
    const int q0 = qt * 16;
    uint32_t aq[8][4];   // A fragments of the 16 x 64 query tile
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      aq[s][0] = Qu[(q0 + g) * kLd + 8 * s + tq];
      aq[s][1] = Qu[(q0 + g + 8) * kLd + 8 * s + tq];
      aq[s][2] = Qu[(q0 + g) * kLd + 8 * s + tq + 4];
      aq[s][3] = Qu[(q0 + g + 8) * kLd + 8 * s + tq + 4];
    }
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) o[n][i] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};   // rows g and g + 8
    for (int kb = 0; kb < n_kb; ++kb) {
      const int key0 = kb * 64;
      float sc[8][4];
#pragma unroll
      for (int n = 0; n < 8; ++n) {
#pragma unroll
        for (int i = 0; i < 4; ++i) sc[n][i] = 0.f;
        const uint32_t *kr = Qu + (key0 + 8 * n + g) * kLd + tq;
#pragma unroll
        for (int s = 0; s < 8; ++s) mma_tf32(sc[n], aq[s], kr[8 * s], kr[8 * s + 4]);
      }
      flash_tile_block(sc, m_run, l_run, o, Vu, key0, H, g, tq);
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
      l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
    }
    const float inv0 = 1.f / l_run[0], inv1 = 1.f / l_run[1];
    const int h0 = q0 + g, h1 = q0 + g + 8;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      if (h0 < H) *reinterpret_cast<float2 *>(long_out + (((size_t)b * H + h0) * W + w) * 64 + 8 * n + 2 * tq) = make_float2(o[n][0] * inv0, o[n][1] * inv0);
      if (h1 < H) *reinterpret_cast<float2 *>(long_out + (((size_t)b * H + h1) * W + w) * 64 + 8 * n + 2 * tq) = make_float2(o[n][2] * inv1, o[n][3] * inv1);
    }
  }
}

// ---- bf16 variant of the column pass (the one cdfo_lra_fwd launches) ----
// Same flash pass on mma.sync m16n8k16 bf16 (fp32 accumulate): half the MMA and fragment-load count of the TF32 kernel, and the
// operands take half the shared memory (Q [Hk][64] bf16 with 72-element rows, V TRANSPOSED [64][Hk] bf16 with Hk + 8 element rows:
// both strides are 4 mod 32 words, every fragment load conflict-free), so two CTAs fit an SM and one column's load phase hides
// behind the other's MMAs.  Q is built straight from the compact mask info (no fp32 sq scratch).  With V transposed the
// probabilities feed the second MMA in their natural C-fragment order (keys 2t, 2t+1 of n-tiles 2s and 2s+1 are exactly the A
// fragment of key step s).  bf16 keeps 8 mantissa bits: logits are O(1), so softmax weights move by < 4e-3 relative, the same
// order as the bf16 rounding the consumer (conv_expand_fea_r, c8 bf16 input) applies to the result anyway.
constexpr int kQw = 36;   // Q row stride in 32-bit words

__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&v);
}

__global__ void __launch_bounds__(kColThreads, 2) lra_col_bf16_kernel(const float *__restrict__ vrow_t, const uint8_t *__restrict__ midx,
                                                                     const float *__restrict__ qsel, float *__restrict__ long_out,
                                                                     LraTables t, int H, int W) {
  extern __shared__ __align__(16) uint32_t smu[];
  const int b = blockIdx.y, w = blockIdx.x;
  const int HW = H * W;
  const int Hk = (H + 63) & ~63;          // keys padded to whole 64-key blocks (rows >= H are zero and masked)
  const int SW = Hk / 2 + 4;              // V^T row stride in words
  uint32_t *Qw = smu;                     // [Hk][kQw]
  uint32_t *Vt = Qw + Hk * kQw;           // [64][SW]
  float *cq = reinterpret_cast<float *>(Vt + 64 * SW);      // [H + 8] q value of the masked channel (rows -4 .. H + 3)
  int *cm = reinterpret_cast<int *>(cq + H + 8);            // [H + 8] masked channel, 255 = none, -1 = outside the frame
  float *kws = reinterpret_cast<float *>(cm + H + 8);       // [9]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, tq = lane & 3;
  float kh[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) kh[i] = t.kh[i];
  if (tid < 9) kws[tid] = t.kw[tid];
  for (int e = tid; e < H + 8; e += kColThreads) {
    const int h = e - 4;
    int c = -1;
    float q = 0.f;
    if (h >= 0 && h < H) {
      c = midx[(size_t)b * HW + h * W + w];
      q = qsel[(size_t)b * HW + h * W + w];
    }
    cm[e] = c;
    cq[e] = q;
  }
  {  // V^T: a thread takes two consecutive keys x four channels; store order rotated per thread so that a warp's 32 words of one
     // store instruction fall into 32 different banks
    const float *vsrc = vrow_t + ((size_t)b * W + w) * H * 64;   // contiguous [H][64]
    for (int e = tid; e < (Hk / 2) * 16; e += kColThreads) {
      const int kp = (e >> 6) * 4 + (e & 3), c4 = (e >> 2) & 15;
      float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
      if (2 * kp < H) v0 = __ldg(reinterpret_cast<const float4 *>(vsrc + (size_t)(2 * kp) * 64 + c4 * 4));
      if (2 * kp + 1 < H) v1 = __ldg(reinterpret_cast<const float4 *>(vsrc + (size_t)(2 * kp + 1) * 64 + c4 * 4));
      const uint32_t wv[4] = {pack_bf16x2(v0.x, v1.x), pack_bf16x2(v0.y, v1.y), pack_bf16x2(v0.z, v1.z), pack_bf16x2(v0.w, v1.w)};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int j = (i + (c4 >> 1)) & 3;
        Vt[(c4 * 4 + j) * SW + kp] = j == 0 ? wv[0] : (j == 1 ? wv[1] : (j == 2 ? wv[2] : wv[3]));
      }
    }
  }
  __syncthreads();
  // Q[h][c] = bh + sum_i kh[i] sq[h + i - 4][c],  sq[h'][c] = beta + kw[cm - c + 4] q (inside the frame), 0 outside; rows >= H: zero
  for (int e = tid; e < Hk * 32; e += kColThreads) {
    const int h = e >> 5, c0 = (e & 31) * 2;
    float a0 = 0.f, a1 = 0.f;
    if (h < H) {
      a0 = a1 = t.bh;
#pragma unroll
      for (int i = 0; i < 9; ++i) {
        const int c = cm[h + i];
        if (c < 0) continue;
        float s0 = t.beta, s1 = t.beta;
        if (c != 255) {
          const int t0 = c - c0 + 4, t1 = t0 - 1;
          const float q = cq[h + i];
          if (t0 >= 0 && t0 <= 8) s0 = fmaf(kws[t0], q, s0);
          if (t1 >= 0 && t1 <= 8) s1 = fmaf(kws[t1], q, s1);
        }
        a0 = fmaf(kh[i], s0, a0);
        a1 = fmaf(kh[i], s1, a1);
      }
    }
    Qw[h * kQw + (e & 31)] = pack_bf16x2(a0, a1);
  }
  __syncthreads();

  const int n_qt = (H + 15) >> 4, n_kb = Hk >> 6;
  for (int qt = warp; qt < n_qt; qt += kColWarps) {
    const int q0 = qt * 16;
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) o[n][i] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};   // rows g and g + 8
    for (int kb = 0; kb < n_kb; ++kb) {
      const int key0 = kb * 64;
      float sc[8][4];
      {
        uint32_t aq[4][4];   // A fragments of the 16 x 64 query tile (four 16-channel steps), re-read per key block: 16 conflict-free
                             // loads against 64 MMAs, and 16 registers less across the softmax / P V part (two CTAs per SM: 112 regs)
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          aq[s][0] = Qw[(q0 + g) * kQw + 8 * s + tq];
          aq[s][1] = Qw[(q0 + g + 8) * kQw + 8 * s + tq];
          aq[s][2] = Qw[(q0 + g) * kQw + 8 * s + tq + 4];
          aq[s][3] = Qw[(q0 + g + 8) * kQw + 8 * s + tq + 4];
        }
#pragma unroll
        for (int n = 0; n < 8; ++n) {
#pragma unroll
          for (int i = 0; i < 4; ++i) sc[n][i] = 0.f;
          const uint32_t *kr = Qw + (key0 + 8 * n + g) * kQw + tq;
#pragma unroll
          for (int s = 0; s < 4; ++s) mma_bf16(sc[n], aq[s], kr[8 * s], kr[8 * s + 4]);
        }
      }
      float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        const int key = key0 + 8 * n + 2 * tq;
        if (key >= H) { sc[n][0] = -INFINITY; sc[n][2] = -INFINITY; }
        if (key + 1 >= H) { sc[n][1] = -INFINITY; sc[n][3] = -INFINITY; }
        mx[0] = fmaxf(mx[0], fmaxf(sc[n][0], sc[n][1]));
        mx[1] = fmaxf(mx[1], fmaxf(sc[n][2], sc[n][3]));
      }
      float scale[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
        const float m_new = fmaxf(m_run[r], mx[r]);    // every block holds at least one live key (key0 < H)
        scale[r] = expf(m_run[r] - m_new);
        m_run[r] = m_new;
        l_run[r] *= scale[r];
      }
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        sc[n][0] = expf(sc[n][0] - m_run[0]); sc[n][1] = expf(sc[n][1] - m_run[0]);
        sc[n][2] = expf(sc[n][2] - m_run[1]); sc[n][3] = expf(sc[n][3] - m_run[1]);
        l_run[0] += sc[n][0] + sc[n][1];
        l_run[1] += sc[n][2] + sc[n][3];
        o[n][0] *= scale[0]; o[n][1] *= scale[0]; o[n][2] *= scale[1]; o[n][3] *= scale[1];
      }
#pragma unroll
      for (int s = 0; s < 4; ++s) {      // 16 keys per step: A = probabilities of n-tiles 2s (keys +0..7) and 2s + 1 (keys +8..15)
        const uint32_t ap[4] = {pack_bf16x2(sc[2 * s][0], sc[2 * s][1]), pack_bf16x2(sc[2 * s][2], sc[2 * s][3]),
                                pack_bf16x2(sc[2 * s + 1][0], sc[2 * s + 1][1]), pack_bf16x2(sc[2 * s + 1][2], sc[2 * s + 1][3])};
        const uint32_t *vr = Vt + g * SW + (key0 >> 1) + 8 * s + tq;
#pragma unroll
        for (int n = 0; n < 8; ++n) mma_bf16(o[n], ap, vr[8 * n * SW], vr[8 * n * SW + 4]);
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
      l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
    }
    const float inv0 = 1.f / l_run[0], inv1 = 1.f / l_run[1];
    const int h0 = q0 + g, h1 = q0 + g + 8;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      if (h0 < H) *reinterpret_cast<float2 *>(long_out + (((size_t)b * H + h0) * W + w) * 64 + 8 * n + 2 * tq) = make_float2(o[n][0] * inv0, o[n][1] * inv0);
      if (h1 < H) *reinterpret_cast<float2 *>(long_out + (((size_t)b * H + h1) * W + w) * 64 + 8 * n + 2 * tq) = make_float2(o[n][2] * inv1, o[n][3] * inv1);
    }
  }
}

// ------------------------------------------------------------------------------------------------ 8x8 windows
// CTA per window; tokens = 64 pixels, sq = q with the masked channel zeroed ((1 - mask) * q, arch:2236-2239).
constexpr int kWinThreads = 256;
__global__ void __launch_bounds__(kWinThreads) lra_win_kernel(const float *__restrict__ qv, const uint8_t *__restrict__ midx,
                                                             float *__restrict__ loc_out, int H, int W) {
  extern __shared__ __align__(16) float sm[];
  float *q = sm;                 // [64][kLd]
  float *v = q + 64 * kLd;
  float *Ps = v + 64 * kLd;
  const int b = blockIdx.z, wy = blockIdx.y, wx = blockIdx.x;
  const int HW = H * W;
  const int tid = threadIdx.x;
  static_assert(kWinThreads == 256, "one token and 16 + 16 channels per thread");
  {
    // a thread owns one token (tok = dh*8 + dw) and channels cg, cg + 4, ...: its 32 loads are issued back to back, then stored
    const int tok = tid & 63, cg = tid >> 6;
    const int h = wy * 8 + (tok >> 3), w = wx * 8 + (tok & 7);
    const size_t pix = (size_t)h * W + w;
    const int cm = midx[(size_t)b * HW + pix];
    const float *qp = qv + ((size_t)b * 128 + cg) * HW + pix;
    float qr[16], vv[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      qr[k] = __ldg(qp + (size_t)(4 * k) * HW);
      vv[k] = __ldg(qp + (size_t)(64 + 4 * k) * HW);
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const int c = 4 * k + cg;
      q[tok * kLd + c] = cm == c ? 0.f : qr[k];
      v[tok * kLd + c] = vv[k];
    }
  }
  __syncthreads();
  const float *Kcur = q;
  flash_block_fp32_kptr(q, &Kcur, v, Ps, 64, [&](int) {}, [&](int tok, int c4, float4 val) {
    const int h = wy * 8 + (tok >> 3), w = wx * 8 + (tok & 7);
    *reinterpret_cast<float4 *>(loc_out + (((size_t)b * H + h) * W + w) * 64 + c4) = val;
  });
}

// ---- tensor-core variant of the 8x8 window pass (the one cdfo_lra_fwd launches) ----
// One CTA (4 warps) per window, a warp per 16 query tokens; S = q q^T and O = P V on warp-level mma.sync m16n8k16 bf16 (fp32 accumulate).
// The window logits reach +-40 (dense 64-d dot products of unnormalised q), where one bf16 rounding of q would move the softmax weights by
// percents, so q is split into bf16 hi + lo parts and the scores are the three-term product hi.hi + hi.lo + lo.hi (error ~2^-16 |q|^2, the
// same order as the TF32 rounding of the other passes); P and V are split the same way (a peaked softmax copies a value row to the output).  The
// probabilities feed the second MMA straight from the score accumulators (C fragments of key tiles 2s, 2s+1 = A fragment of key step s),
// V is held transposed.  Shared memory 36.9 KB per CTA: six windows per SM hide each other's load phase.
constexpr int kWinTcThreads = 128, kWinLd = 36;     // row stride in 32-bit words (72 bf16): 36 = 4 (mod 32), conflict-free fragment loads
__global__ void __launch_bounds__(kWinTcThreads, 6) lra_win_tc_kernel(const float *__restrict__ qv, const uint8_t *__restrict__ midx,
                                                                      float *__restrict__ loc_out, int H, int W) {
  __shared__ uint32_t Qh[64 * kWinLd], Ql[64 * kWinLd], Vt[64 * kWinLd], Vl[64 * kWinLd];   // [token][channel pairs] x 2, [channel][key pairs] x 2 (hi, lo)
  const int b = blockIdx.z, wy = blockIdx.y, wx = blockIdx.x;
  const int HW = H * W;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, tq = lane & 3;
  {
    // thread = (token pair for V / token for Q, channel group): loads are 32-byte runs of 8 consecutive pixels per (channel, window row)
    const int tok = tid & 63, half = tid >> 6;            // half 0: channels 0..31, half 1: 32..63
    const int h = wy * 8 + (tok >> 3), w = wx * 8 + (tok & 7);
    const size_t pix = (size_t)h * W + w;
    const int cm = midx[(size_t)b * HW + pix];
    const float *qp = qv + ((size_t)b * 128 + half * 32) * HW + pix;
#pragma unroll 4
    for (int k = 0; k < 16; ++k) {
      const int c = half * 32 + 2 * k;
      float q0 = __ldg(qp + (size_t)(2 * k) * HW), q1 = __ldg(qp + (size_t)(2 * k + 1) * HW);
      if (cm == c) q0 = 0.f;                              // (1 - mask) * q, arch:2236-2239
      if (cm == c + 1) q1 = 0.f;
      const __nv_bfloat16 h0 = __float2bfloat16_rn(q0), h1 = __float2bfloat16_rn(q1);
      Qh[tok * kWinLd + (c >> 1)] = pack_bf16x2(__bfloat162float(h0), __bfloat162float(h1));
      Ql[tok * kWinLd + (c >> 1)] = pack_bf16x2(q0 - __bfloat162float(h0), q1 - __bfloat162float(h1));
      // V transposed: element (channel, key = tok) -- 16-bit stores, two tokens share a word
      const float v0 = __ldg(qp + (size_t)(64 + 2 * k) * HW), v1 = __ldg(qp + (size_t)(64 + 2 * k + 1) * HW);
      const __nv_bfloat16 vh0 = __float2bfloat16_rn(v0), vh1 = __float2bfloat16_rn(v1);
      reinterpret_cast<__nv_bfloat16 *>(Vt)[(c * kWinLd) * 2 + tok] = vh0;
      reinterpret_cast<__nv_bfloat16 *>(Vt)[((c + 1) * kWinLd) * 2 + tok] = vh1;
      reinterpret_cast<__nv_bfloat16 *>(Vl)[(c * kWinLd) * 2 + tok] = __float2bfloat16_rn(v0 - __bfloat162float(vh0));
      reinterpret_cast<__nv_bfloat16 *>(Vl)[((c + 1) * kWinLd) * 2 + tok] = __float2bfloat16_rn(v1 - __bfloat162float(vh1));
    }
  }
  __syncthreads();
  const int q0r = warp * 16;
  uint32_t ah[4][4], al[4][4];                            // A fragments of this warp's 16 queries, hi and lo parts
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    ah[s][0] = Qh[(q0r + g) * kWinLd + 8 * s + tq];      ah[s][1] = Qh[(q0r + g + 8) * kWinLd + 8 * s + tq];
    ah[s][2] = Qh[(q0r + g) * kWinLd + 8 * s + tq + 4];  ah[s][3] = Qh[(q0r + g + 8) * kWinLd + 8 * s + tq + 4];
    al[s][0] = Ql[(q0r + g) * kWinLd + 8 * s + tq];      al[s][1] = Ql[(q0r + g + 8) * kWinLd + 8 * s + tq];
    al[s][2] = Ql[(q0r + g) * kWinLd + 8 * s + tq + 4];  al[s][3] = Ql[(q0r + g + 8) * kWinLd + 8 * s + tq + 4];
  }
  float sc[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) {
#pragma unroll
    for (int i = 0; i < 4; ++i) sc[n][i] = 0.f;
    const uint32_t *kh_ = Qh + (8 * n + g) * kWinLd + tq, *kl_ = Ql + (8 * n + g) * kWinLd + tq;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      const uint32_t bh0 = kh_[8 * s], bh1 = kh_[8 * s + 4];
      mma_bf16(sc[n], al[s], bh0, bh1);                   // small terms first
      mma_bf16(sc[n], ah[s], kl_[8 * s], kl_[8 * s + 4]);
      mma_bf16(sc[n], ah[s], bh0, bh1);
    }
  }
  float mx[2] = {-INFINITY, -INFINITY}, sum[2] = {0.f, 0.f};
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    mx[0] = fmaxf(mx[0], fmaxf(sc[n][0], sc[n][1]));
    mx[1] = fmaxf(mx[1], fmaxf(sc[n][2], sc[n][3]));
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
  }
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    sc[n][0] = expf(sc[n][0] - mx[0]); sc[n][1] = expf(sc[n][1] - mx[0]);
    sc[n][2] = expf(sc[n][2] - mx[1]); sc[n][3] = expf(sc[n][3] - mx[1]);
    sum[0] += sc[n][0] + sc[n][1];
    sum[1] += sc[n][2] + sc[n][3];
  }
  float o[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n)
#pragma unroll
    for (int i = 0; i < 4; ++i) o[n][i] = 0.f;
#pragma unroll
  for (int s = 0; s < 4; ++s) {        // 16 keys per step
    // probabilities and values as bf16 hi + lo parts as well (P V = Ph Vh + Pl Vh + Ph Vl): a sharply peaked softmax copies one value
    // row to the output, and a single bf16 rounding of it (2^-9 relative) would be the largest error of the whole module
    uint32_t ap[4], apl[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float p0 = sc[2 * s + (i >> 1)][2 * (i & 1)], p1 = sc[2 * s + (i >> 1)][2 * (i & 1) + 1];
      const float h0 = __bfloat162float(__float2bfloat16_rn(p0)), h1 = __bfloat162float(__float2bfloat16_rn(p1));
      ap[i] = pack_bf16x2(h0, h1);
      apl[i] = pack_bf16x2(p0 - h0, p1 - h1);
    }
    const uint32_t *vr = Vt + g * kWinLd + 8 * s + tq, *vl = Vl + g * kWinLd + 8 * s + tq;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      const uint32_t b0 = vr[8 * n * kWinLd], b1 = vr[8 * n * kWinLd + 4];
      mma_bf16(o[n], apl, b0, b1);
      mma_bf16(o[n], ap, vl[8 * n * kWinLd], vl[8 * n * kWinLd + 4]);
      mma_bf16(o[n], ap, b0, b1);
    }
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 1);
    sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 2);
  }
  const float inv0 = 1.f / sum[0], inv1 = 1.f / sum[1];
  const int t0 = q0r + g, t1 = t0 + 8;
  float *d0 = loc_out + (((size_t)b * H + wy * 8 + (t0 >> 3)) * W + wx * 8 + (t0 & 7)) * 64 + 2 * tq;
  float *d1 = loc_out + (((size_t)b * H + wy * 8 + (t1 >> 3)) * W + wx * 8 + (t1 & 7)) * 64 + 2 * tq;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    *reinterpret_cast<float2 *>(d0 + 8 * n) = make_float2(o[n][0] * inv0, o[n][1] * inv0);
    *reinterpret_cast<float2 *>(d1 + 8 * n) = make_float2(o[n][2] * inv1, o[n][3] * inv1);
  }
}

}  // namespace cdfo

using namespace cdfo;

typedef CUresult (*LraEncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                     const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static LraEncodeTiledFn lra_encode_tiled_fn() {
  static LraEncodeTiledFn fn = nullptr;
  if (!fn) {
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<LraEncodeTiledFn>(ptr);
  }
  return fn;
}

static bool g_lra_row_tma = true;     // cdfo_lra_set_row_tma: the TMA-fed load phase of the row kernel (default) vs 4-byte cp.async
extern "C" int cdfo_lra_set_row_tma(int on) {
  g_lra_row_tma = on != 0;
  return CDFO_OK;
}
static bool g_lra_col_tf32 = false;   // cdfo_lra_set_col_precision: A/B switch (tests, tools)
static bool g_lra_col_tc = true;      // cdfo_lra_set_col_tcgen05: the tcgen05 column kernel (default) vs the warp-level mma.sync kernels
static bool g_lra_win_tc = true;      // cdfo_lra_set_win_tensor_core: the bf16 split tensor-core window kernel (default) vs the fp32 SIMT one
extern "C" int cdfo_lra_set_col_precision(int tf32) {
  g_lra_col_tf32 = tf32 != 0;
  return CDFO_OK;
}
extern "C" int cdfo_lra_set_col_tcgen05(int on) {
  g_lra_col_tc = on != 0;
  return CDFO_OK;
}
extern "C" int cdfo_lra_set_win_tensor_core(int on) {
  g_lra_win_tc = on != 0;
  return CDFO_OK;
}

// tables: float[9 kw | 9 kh | 64 k1 | 4096 r] on the device; scratch sizes are the caller's (see cdfo_lra_workspace_bytes).
extern "C" size_t cdfo_lra_workspace_bytes(int B, int H, int W) {
  const size_t P = (size_t)B * H * W;
  return P * (1 + 4) + 3 * P * 64 * 4 + 256;   // midx + qsel + vrow_t + long_out + loc_out
}

static int lra_run(const float *qv, const float *u, const float *vmax, const float *x, const float *x2, const float *tables,
                   float beta, float bh, const float *fuse_w, const float *fuse_b, float *out, void *out_c8, int out_channels,
                   int channel0, void *workspace, int B, int H, int W, void *stream);

extern "C" int cdfo_lra_fwd(const float *qv, const float *u, const float *vmax, const float *x, const float *x2, const float *tables,
                            float beta, float bh, const float *fuse_w, const float *fuse_b, float *out, void *workspace, int B,
                            int H, int W, void *stream) {
  return lra_run(qv, u, vmax, x, x2, tables, beta, bh, fuse_w, fuse_b, out, nullptr, 0, 0, workspace, B, H, W, stream);
}

extern "C" int cdfo_lra_c8_fwd(const float *qv, const float *u, const float *vmax, const float *x, const float *x2, const float *tables,
                               float beta, float bh, const float *fuse_w, const float *fuse_b, void *out_c8, int out_channels,
                               int channel0, void *workspace, int B, int H, int W, void *stream) {
  CDFO_REQUIRE(out_c8 && ((uintptr_t)out_c8 & 15) == 0, CDFO_ERR_NULL, "cdfo_lra_c8_fwd: out_c8 must be a 16-byte aligned pointer");
  CDFO_REQUIRE(out_channels % 8 == 0 && channel0 % 8 == 0 && channel0 >= 0 && channel0 + 64 <= out_channels, CDFO_ERR_SHAPE,
               "cdfo_lra_c8_fwd: channels [%d, %d) do not fit %d output channels (multiples of 8)", channel0, channel0 + 64, out_channels);
  return lra_run(qv, u, vmax, x, x2, tables, beta, bh, fuse_w, fuse_b, nullptr, out_c8, out_channels, channel0, workspace, B, H, W, stream);
}

static int lra_run(const float *qv, const float *u, const float *vmax, const float *x, const float *x2, const float *tables,
                   float beta, float bh, const float *fuse_w, const float *fuse_b, float *out, void *out_c8, int out_channels,
                   int channel0, void *workspace, int B, int H, int W, void *stream) {
  CDFO_REQUIRE(qv && u && vmax && x && tables && fuse_w && fuse_b && (out || out_c8) && workspace, CDFO_ERR_NULL, "cdfo_lra_fwd: NULL pointer");
  CDFO_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0 && H % 8 == 0 && W % 8 == 0, CDFO_ERR_SHAPE,
               "cdfo_lra_fwd: H and W must be multiples of the window size 8 (got %d x %d)", H, W);
  // every shape check comes before the first launch: a rejected call leaves the workspace untouched
  const int kDynMax = 224 * 1024;  // 227 KB opt-in limit minus the kernels' small static shared memory
  const int Wk = (W + 63) & ~63;
  auto row_bytes = [&](int ncta) {   // the row kernel's dynamic shared memory (without the TMA ring) when ncta CTAs share a row
    const size_t Ws = ncta == 1 ? (size_t)Wk : (size_t)lra_row_slice(Wk, ncta);
    return (Ws * kLd + 4096 + 3 * (size_t)Wk + 64 + kRowThreads + 2 * (size_t)Wk) * 4;
  };
  const int row_ncta = row_bytes(1) <= (size_t)kDynMax ? 1 : 2;   // by width alone: W <= 704 runs on one CTA
  const size_t row_smem = row_bytes(row_ncta);
  const int Hk = (H + 63) & ~63;
  const size_t col_v = (size_t)Hk * kLd > (size_t)(H + 8) * 64 ? (size_t)Hk * kLd : (size_t)(H + 8) * 64;
  const size_t col_smem = ((size_t)Hk * kLd + col_v) * 4;
  const size_t col16_smem = ((size_t)Hk * kQw + 64 * ((size_t)Hk / 2 + 4) + 2 * (size_t)(H + 8) + 16) * 4;
  const size_t win_smem = (size_t)3 * 64 * kLd * 4;
  CDFO_REQUIRE(row_smem <= (size_t)kDynMax, CDFO_ERR_UNSUPPORTED,
               "cdfo_lra_fwd: frame width %d exceeds the row pass's shared memory over a 2-CTA cluster (W <= 1280)", W);
  // the column kernel that will run: tcgen05 when it takes the shape, else the bf16 mma.sync kernel; the TF32 one only on request
  const bool col_tc = !g_lra_col_tf32 && g_lra_col_tc && lra_col_sm100_fits(H);
  if (!col_tc) {
    if (g_lra_col_tf32)
      CDFO_REQUIRE(col_smem <= (size_t)kDynMax, CDFO_ERR_UNSUPPORTED,
                   "cdfo_lra_fwd: frame height %d exceeds the TF32 column pass's shared memory (H <= 384)", H);
    else
      CDFO_REQUIRE(col16_smem <= (size_t)kDynMax, CDFO_ERR_UNSUPPORTED,
                   "cdfo_lra_fwd: frame height %d exceeds the bf16 column pass's shared memory (H <= 768)", H);
  }
  cudaStream_t s = (cudaStream_t)stream;
  const size_t P = (size_t)B * H * W;
  const int HW = H * W;
  uint8_t *ws = (uint8_t *)workspace;
  float *qsel = (float *)ws;
  float *vrow_t = qsel + P;
  float *long_out = vrow_t + P * 64;
  float *loc_out = long_out + P * 64;
  uint8_t *midx = (uint8_t *)(loc_out + P * 64);
  LraTables t{tables, tables + 9, tables + 18, tables + 82, beta, bh};
  static bool attr = false;
  if (!attr) {
    cudaError_t e1 = cudaFuncSetAttribute(lra_row_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kDynMax);
    if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(lra_row_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kDynMax);
    if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(lra_row_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kDynMax);
    if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(lra_row_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kDynMax);
    cudaError_t e2 = cudaFuncSetAttribute(lra_col_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDynMax);
    if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(lra_col_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDynMax);
    cudaError_t e3 = cudaFuncSetAttribute(lra_win_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)win_smem);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)
      return fail(CDFO_ERR_CUDA, "cdfo_lra_fwd: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
    attr = true;
  }

  lra_mask_kernel<<<dim3(ceil_div(HW, 128), B), 128, 0, s>>>(u, vmax, qv, midx, qsel, HW);

  {
    CUtensorMap qm;
    memset(&qm, 0, sizeof(qm));
    bool row_tma = g_lra_row_tma && W % 4 == 0 && ((uintptr_t)qv & 15) == 0 && row_smem + kRowRawBytes <= (size_t)kDynMax;
    if (row_tma) {
      static LraEncodeTiledFn enc = lra_encode_tiled_fn();
      if (enc) {
        const cuuint64_t gdim[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B * 128};
        const cuuint64_t gstr[2] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4};
        const cuuint32_t box[3] = {kRowPiece, 1, 64};
        const cuuint32_t estr[3] = {1, 1, 1};
        CUresult cr = enc(&qm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(qv), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        CDFO_REQUIRE(cr == CUDA_SUCCESS, CDFO_ERR_CUDA, "cuTensorMapEncodeTiled(qv rows) failed with CUresult %d", (int)cr);
      } else {
        row_tma = false;
      }
    }
    const size_t row_dyn = row_smem + (row_tma ? kRowRawBytes : 0);
    if (row_ncta == 1) {
      if (row_tma) lra_row_kernel<1, true><<<dim3(H, B), kRowThreads, row_dyn, s>>>(qm, qv, midx, qsel, vrow_t, t, H, W);
      else lra_row_kernel<1, false><<<dim3(H, B), kRowThreads, row_dyn, s>>>(qm, qv, midx, qsel, vrow_t, t, H, W);
    } else {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(2 * H, B);
      cfg.blockDim = dim3(kRowThreads);
      cfg.dynamicSmemBytes = row_dyn;
      cfg.stream = s;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = 2;
      at[0].val.clusterDim.y = 1;
      at[0].val.clusterDim.z = 1;
      cfg.attrs = at;
      cfg.numAttrs = 1;
      const cudaError_t e = row_tma ? cudaLaunchKernelEx(&cfg, lra_row_kernel<2, true>, qm, qv, midx, qsel, vrow_t, t, H, W)
                                    : cudaLaunchKernelEx(&cfg, lra_row_kernel<2, false>, qm, qv, midx, qsel, vrow_t, t, H, W);
      if (e != cudaSuccess) return fail(CDFO_ERR_CUDA, "cdfo_lra_fwd: cluster launch of the row pass: %s", cudaGetErrorString(e));
    }
  }
  if (col_tc) {     // csrc/lra_col_sm100.cu: whole score tile in tensor memory (H <= 384)
    const int rc = lra_col_sm100_launch(vrow_t, midx, qsel, long_out, t, B, H, W, s);
    if (rc < 0) return rc;
  } else if (g_lra_col_tf32) {
    lra_col_kernel<<<dim3(W, B), kColThreads, col_smem, s>>>(vrow_t, midx, qsel, long_out, t, H, W);
  } else {
    lra_col_bf16_kernel<<<dim3(W, B), kColThreads, col16_smem, s>>>(vrow_t, midx, qsel, long_out, t, H, W);
  }
  if (g_lra_win_tc) lra_win_tc_kernel<<<dim3(W / 8, H / 8, B), kWinTcThreads, 0, s>>>(qv, midx, loc_out, H, W);
  else lra_win_kernel<<<dim3(W / 8, H / 8, B), kWinThreads, win_smem, s>>>(qv, midx, loc_out, H, W);
  if (int rc = check_launch("cdfo_lra_fwd")) return rc;
  // fuse: 1x1 conv(128 -> 64) over cat[long, local] (pixel-major) + bias + x (+ x2): tensor-core pointwise kernel
  return pointwise_conv(long_out, loc_out, fuse_w, fuse_b, x, x2, out, B, 128, 64, HW, 0, 1, s, out_c8, out_channels, channel0);
}
