/*
 * cdfo_b200 -- C ABI of the B200 (sm_100a) hot path of CDFO's CVSR_V8 forward.
 *
 * Every entry point takes plain device pointers + sizes + a CUDA stream
 * (cudaStream_t passed as void*), allocates nothing, never throws, returns
 * CDFO_OK (0) or a negative cdfo_status and leaves a message retrievable with
 * cdfo_last_error().  Tensors are contiguous; "NCHW" = the reference's layout.
 *
 * Reference interfaces replaced (paths relative to the reference tree):
 *   cdfo_dcn_fwd            ops/dcn/src/deform_conv_cuda.cpp:486-564  modulated_deform_conv_cuda_forward
 *                           ops/dcn/src/deform_conv_cuda.cpp:151-258  deform_conv_forward_cuda  (mask == NULL)
 *                           bound by ops/dcn/deform_conv.py:52-57,144-148; also the semantics of
 *                           torchvision.ops.deform_conv2d at arch/SIDECVSR_our.py:3352
 *   cdfo_dcn_sample_index   floor() indices of deform_conv_cuda_kernel.cu:614-615 + :470-471 (parity probe)
 *   cdfo_flow_warp_fwd      arch/SIDECVSR_our.py:3068-3099  flow_warp (bilinear, zeros, align_corners=True)
 *   cdfo_mv2mvs             test_LD_37.py:83-105  mv2mvs  (+ permute at :160-161);  cdfo_mv2mvs_ra: opt/data_RA_bi.py:496-533
 *   cdfo_mv_end_fix         test_LD_37.py:209-234 modify_mv_for_end_frames
 *   cdfo_pack_c8 / unpack   layout adapters NCHW fp32 <-> channel-chunked bf16 used by the sm_100a kernels
 *   cdfo_dcn_sm100_fwd      same contraction as cdfo_dcn_fwd at the model's hot shape (C=Co=64, 3x3, s=p=d=1,
 *                           groups=1), tcgen05 implicit GEMM, bf16 operands, fp32 accumulate
 *   cdfo_dcn_tex_sm100_fwd  the same contraction with the bilinear gather on the texture units (fields input, fp16 operands)
 *   cdfo_mv_offset_assemble arch/SIDECVSR_our.py:3341-3350 (chunk/cat/tanh/x10/+flow.flip/sigmoid)
 *   cdfo_conv3x3_sm100_fwd  3x3 s1 p1 convolutions on the path (arch/SIDECVSR_our.py:3271-3275 conv_offset,
 *                           :254-271 ResidualBlock_noBN, :4382 conv_expand_fea_r), tcgen05 implicit GEMM
 *   cdfo_mdta_*             arch/SIDECVSR_our.py:3303-3337 / :3455-3492 (warp + fusion + dual MDTA)
 *   cdfo_lra_*              arch/SIDECVSR_our.py:2179-2249 LLongRangAttention.forward
 *   cdfo_tail_fwd           arch/SIDECVSR_our.py:4473-4480 (upconv/PixelShuffle/lrelu x2, conv_last, bilinear x4 skip)
 *   cdfo_planes_to_unit_f32 / cdfo_sr_to_u8   test_LD_37.py:19-29,172-180 (frame I/O of eval_seq)
 *   cdfo_psnr_ssim_u8       metric/psnr_ssim.py:278-399,446-484 (calculate_psnr / calculate_ssim, Y channel, border 4)
 */
#ifndef CDFO_B200_H_
#define CDFO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum cdfo_status {
  CDFO_OK = 0,
  CDFO_ERR_SHAPE = -1,       /* inconsistent sizes (the reference raises AT_ERROR / TORCH_CHECK) */
  CDFO_ERR_NULL = -2,        /* required pointer is NULL */
  CDFO_ERR_CUDA = -3,        /* CUDA runtime / launch error (reference only printf()s these) */
  CDFO_ERR_UNSUPPORTED = -4, /* valid request outside what this build implements */
  CDFO_ERR_NO_DEVICE = -5    /* no sm_100 device visible */
} cdfo_status;

typedef enum cdfo_dtype { CDFO_F32 = 0, CDFO_F16 = 1, CDFO_BF16 = 2 } cdfo_dtype;
/* offset/mask given to cdfo_dcn_sm100_fwd as packed fields [B, 9 taps, dg/gp, H, W, gp] x fp16x4 (dy, dx, mask, 0), gp = 2 when
 * dg = 16 and 1 otherwise: `offset` points at them, `mask` is ignored. */
#define CDFO_FIELDS_F16X4 16

/* Message of the last failing call on this thread ("" if none). */
const char *cdfo_last_error(void);
/* ABI version: major*1000 + minor. */
int cdfo_version(void);
/* 1 if device `dev` is compute capability 10.x, 0 otherwise, <0 on CUDA error. */
int cdfo_device_ok(int dev);

/* ---- A6/A7: deformable convolution forward, reference semantics, any shape ----
 * x [B,C,H,W], offset [B,dg*2*kh*kw,Ho,Wo], mask [B,dg*kh*kw,Ho,Wo] or NULL (DCNv1),
 * weight [Co,C/groups,kh,kw], bias [Co] or NULL, y [B,Co,Ho,Wo] (overwritten).
 * dtype applies to x/offset/mask/weight/bias/y alike (fp32 accumulate). */
int cdfo_dcn_fwd(const void *x, const void *offset, const void *mask, const void *weight,
                 const void *bias, void *y, int B, int C, int H, int W, int Co, int kh, int kw,
                 int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                 int groups, int dg, int dtype, void *stream);

/* Integer sample indices (floor(h_im), floor(w_im)) per (b, g*kh*kw+tap, ho, wo): idx int32 [B,dg*kh*kw,Ho,Wo,2].
 * offset fp32. */
int cdfo_dcn_sample_index(const float *offset, int32_t *idx, int B, int H, int W, int kh, int kw,
                          int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                          int dg, void *stream);

/* ---- A3: flow_warp. x [B,C,H,W] fp32, flow [B,2,H,W] fp32 (channel 0 = x, 1 = y: the layout the model holds
 * before its permute, arch/SIDECVSR_our.py:3304,3456), y [B,C,H,W]; idx int32 [B,H,W,2]=(iy_nw,ix_nw) or NULL. */
int cdfo_flow_warp_fwd(const float *x, const float *flow, float *y, int B, int C, int H, int W,
                       int32_t *idx, void *stream);

/* ---- A1: mv [H,W,3] (mv_a, mv_b, refdist) int8 or int32 -> flows fp32 [7,2,H,W] (already permuted). ---- */
int cdfo_mv2mvs(const void *mv, int mv_is_int32, float *flows, int H, int W, void *stream);
/* RA twin (opt/data_RA_bi.py:419-424,496-533 and the / 32 of train_RA_37.py:383-386): an (l0, l1) pair of MV fields [H,W,3] with
 * refdist == -99 marking a missing list -> flows fp32 [7,2,H,W]: frames 0-2 from l0, 4-6 from l1 (no sign flip), complemented. */
int cdfo_mv2mvs_ra(const void *mv_l0, const void *mv_l1, int mv_is_int32, float *flows, int H, int W, void *stream);
/* ---- A2: in-place end-of-sequence fix-up on flows [B,7,2,H,W]; frame index i, max_idx as the caller passes. */
int cdfo_mv_end_fix(float *flows, int B, int H, int W, int i, int max_idx, void *stream);

/* ---- A9: prior embedding convs conv_expand_ufs / conv_expand_rms = nn.Conv2d(1, Co, 3, 1, 1) (arch/SIDECVSR_our.py:4383-4384,
 * :4446-4447).  x [B,1,H,W] fp32, w [Co,1,3,3], bias [Co] or NULL -> y [B,Co,H,W] fp32. */
int cdfo_prior_conv_fwd(const float *x, const float *w, const float *bias, float *y, int B, int Co, int H, int W, void *stream);
/* Same with an optional ReLU: a 1x1 convolution + ReLU that follows the prior convolution (LLongRangAttention.conv_du_re.0 on the residual
 * prior, arch/SIDECVSR_our.py:2183 after :4447) composes into its weights exactly (w' = W1 w, b' = W1 b + b1: the 1x1 comes after). */
int cdfo_prior_conv_act_fwd(const float *x, const float *w, const float *bias, float *y, int B, int Co, int H, int W, int relu, void *stream);

/* ---- layout adapters: NCHW fp32 <-> "c8" = [B, C/8, H, W, 8] bf16 (C % 8 == 0). ---- */
int cdfo_pack_c8(const float *x_nchw, void *x_c8, int B, int C, int H, int W, void *stream);
/* Same, into channels [channel0, channel0 + C) of a c8 tensor with out_channels channels (both multiples of 8): the channel
 * concatenations of the model (arch/SIDECVSR_our.py:4454 cat([fea, x_n])) become two packs into one tensor. */
int cdfo_pack_c8_into(const float *x_nchw, void *x_c8, int B, int C, int H, int W, int out_channels, int channel0, void *stream);
int cdfo_unpack_c8(const void *x_c8, float *x_nchw, int B, int C, int H, int W, void *stream);

/* ---- A6 at the model's hot shape on the 5th-generation tensor cores (tcgen05, TMEM) ----
 * C = Co = 64, 3x3, stride = pad = dil = 1, groups = 1, dg in {1,2,4,8,16}; bf16 operands, fp32 accumulate.
 *   x_q4p  [B, 16, H+3, W+3, 4] bf16 : quad-planar input (4 channels = 8 bytes per pixel per plane) with a zero
 *           border of 1 pixel before and 2 after in H and W (cdfo_pack_q4p)
 *   offset [B, dg*18, H, W], mask [B, dg*9, H, W] : fp32 (off_dtype = CDFO_F32) or fp16 (CDFO_F16), reference layout
 *   mv     [B, 2, H, W] fp32 (x, y) or NULL : decoded MV prior added to every offset pair inside the kernel
 *           (dy += mv_y, dx += mv_x), i.e. offset + flow.flip(1).repeat(...) of arch/SIDECVSR_our.py:3347
 *   wpk    73728 bytes from cdfo_dcn_sm100_pack_weight; bias [64] fp32 or NULL
 *   y      out_mode 0: [B, 64, H, W] fp32 (reference layout); out_mode 1: [B, 8, H, W, 8] bf16
 *   num_ctas <= 0: one persistent CTA per SM.
 *   x_batch: x_q4p holds x_batch samples and output sample b samples x[b % x_batch] (<= 0: x_batch = B); the model's six
 *           neighbour calls of a frame all sample the SAME centre-frame feature (arch/SIDECVSR_our.py:4456).
 *   off_bstride / msk_bstride: elements between consecutive samples of offset / mask (<= 0: dense), so that both
 *           can live in one [B, dg*27, H, W] buffer as cdfo_mv_offset_head_sm100_fwd writes them. */
int cdfo_dcn_sm100_fwd(const void *x_q4p, const void *offset, const void *mask, const float *mv,
                       const void *wpk, const float *bias, void *y, int B, int H, int W, int dg,
                       int off_dtype, int out_mode, int num_ctas, int x_batch, long long off_bstride,
                       long long msk_bstride, void *stream);
/* weight [64, 64, 3, 3] fp32 (reference layout) -> bf16 B operand [tap, ci/8, co, 8]. */
int cdfo_dcn_sm100_pack_weight(const float *w, void *wpk, void *stream);
/* NCHW fp32 -> [B, C/4, H+3, W+3, 4] bf16 with the zero border described above (C % 4 == 0). */
int cdfo_pack_q4p(const float *x_nchw, void *x_q4p, int B, int C, int H, int W, void *stream);
/* ---- A6 at the model's hot shape, gather on the texture units (csrc/dcn_tex_sm100.cu) ----
 * Same contraction and shape limits as cdfo_dcn_sm100_fwd; fp16 operands, fp32 accumulate.  The 2x2 bilinear footprint
 * of each (pixel, group, tap) sample is ONE hardware-filtered texture fetch (8 fractional weight bits) instead of four
 * loads and ~30 blend instructions: the op is bound by the L1TEX data stage, not by HBM or issue (DESIGN.md).
 *   x_q4t  [xB, 16, H+3, Wpt, 4] fp16 from cdfo_pack_q4t (Wpt = cdfo_q4t_pitch(W); 512-byte aligned base)
 *   fields [B, 9 taps, dg/gp, H, W, gp] x fp16x4 (dy, dx, mask, 0), gp = 2 when dg = 16 else 1: learned residual and mask as
 *          cdfo_mv_offset_head_sm100_fwd writes them (a warp's 32 pixels x gp groups are contiguous; 16-byte aligned)
 *   mv     [B, 2, H, W] fp32 (x, y) or NULL: decoded MV prior, added as offset + flow.flip(1).repeat(...) (arch:3347)
 *   wpk    73728 bytes from cdfo_dcn_tex_sm100_pack_weight (fp16); bias [64] fp32 or NULL
 *   y / out_mode / num_ctas / x_batch: as cdfo_dcn_sm100_fwd (x_batch * 16 * (H + 3) <= 65000 texture rows); fields_bstride in 8-byte elements (<= 0: dense).
 * Texture descriptors over x_q4t are created on first use and cached by (device, pointer, shape); they own no memory. */
int cdfo_dcn_tex_sm100_fwd(const void *x_q4t, const void *fields, const float *mv, const void *wpk, const float *bias,
                           void *y, int B, int H, int W, int dg, int out_mode, int num_ctas, int x_batch,
                           long long fields_bstride, void *stream);
/* How cdfo_dcn_tex_sm100_fwd reads dense dg = 16 fields: 1 (default) = tiled TMA boxes into a shared-memory ring, 0 = per-thread
 * LDG.128 (the path strided fields and dg < 16 always take).  Same results; a measurement switch (tools/bench_dcn.py). */
int cdfo_dcn_tex_sm100_set_fields_path(int use_tma);
/* Same kernel writing straight into the stacked input of tsa_fusion (arch/SIDECVSR_our.py:4463-4466): the batch is
 * group-major (sample s = group * n_seq + sequence; the model's groups are the six neighbour frames), and sample s lands in
 * the 8-channel chunks [group_chunk[group], +8) of y_stack [n_seq, stack_chunks, H, W, 8] bf16 (frame slot * 8). */
int cdfo_dcn_tex_sm100_stacked_fwd(const void *x_q4t, const void *fields, const float *mv, const void *wpk, const float *bias,
                                   void *y_stack, int n_seq, int n_groups, int stack_chunks, const int *group_chunk, int H,
                                   int W, int dg, int x_batch, void *stream);
int cdfo_dcn_tex_sm100_pack_weight(const float *w, void *wpk, void *stream);
/* ---- A5 + A6 fused: conv_offset[-1] on both hidden maps, tanh / sum / sigmoid, + MV prior, DCN -- ONE kernel
 * (csrc/mv_dcn_fused_sm100.cu; arch/SIDECVSR_our.py:3339-3352).  The offset / mask fields never reach HBM.  dg = 16 only.
 *   z_c8      [2 B, 8, H, W, 8] bf16: hidden maps lrelu(conv_offset[0](.)) of the two MDTA outputs, sample b and b + B
 *   head_wpk  cdfo_conv_sm100_pack_weight(432, 64, 3) of conv_offset[-1].weight with its output channels permuted to
 *             n' = T*144 + qs*36 + tl*12 + gi*3 + c  <-  tap = 3 T + tl, group g = 4 qs + gi, c = (dy, dx, m), i.e. reference
 *             channels (2 k, 2 k + 1, 288 + k) with k = g * 9 + tap;  head_bias [432] fp32 permuted the same way
 *   magnitude max_residue_magnitude (10);  x_q4t / mv / dcn_wpk / dcn_bias / y / out_mode / x_batch / num_ctas: as
 *             cdfo_dcn_tex_sm100_fwd
 *   fields_out NULL, or [B, 9, 8, H, W, 2] x fp16x4: debug tap of the fields the kernel computed (same layout and, by
 *             construction, the same bits as cdfo_mv_offset_head_dual_sm100_fwd writes) */
int cdfo_mv_head_dcn_fused_sm100_fwd(const void *z_c8, const void *head_wpk, const float *head_bias, float magnitude,
                                     const void *x_q4t, const float *mv, const void *dcn_wpk, const float *dcn_bias, void *y,
                                     void *fields_out, int B, int H, int W, int out_mode, int x_batch, int num_ctas, void *stream);
/* Same, writing into the stacked input of tsa_fusion like cdfo_dcn_tex_sm100_stacked_fwd. */
int cdfo_mv_head_dcn_fused_sm100_stacked_fwd(const void *z_c8, const void *head_wpk, const float *head_bias, float magnitude,
                                             const void *x_q4t, const float *mv, const void *dcn_wpk, const float *dcn_bias,
                                             void *y_stack, int n_seq, int n_groups, int stack_chunks, const int *group_chunk,
                                             int H, int W, int x_batch, void *stream);
/* NCHW fp32 -> [B, C/4, H+3, Wpt, 4] fp16 (saturated to +-65504), zero border 1 before / 2 after, zero pitch padding. */
int cdfo_pack_q4t(const float *x_nchw, void *x_q4t, int B, int C, int H, int W, void *stream);
int cdfo_q4t_pitch(int W);
size_t cdfo_q4t_bytes(int B, int C, int H, int W);
/* ---- 3x3 / stride 1 / padding 1 convolution, tcgen05 implicit GEMM with a TMA-staged halo (A9, heads of A5, A4) ----
 * Replaces nn.Conv2d(Cin, Cout, 3, 1, 1) on the path: conv_offset.{0,2} (arch/SIDECVSR_our.py:3271-3275),
 * ResidualBlock_noBN.conv{1,2} (:254-271), conv_expand_fea_r (:4382).  Cin % 64 == 0, Cout % 16 == 0.
 *   x_c8 [B, Cin/8, H, W, 8] bf16; wpk from cdfo_conv3x3_sm100_pack_weight (cdfo_conv3x3_sm100_weight_bytes bytes);
 *   bias [Cout] fp32 or NULL; act 0 none / 1 ReLU / 2 LeakyReLU(0.1); resid_c8 (same shape as a c8 output) or NULL is
 *   added after the activation; y: out_mode 0 = [B, Cout, H, W] fp32, 1 = [B, Cout/8, H, W, 8] bf16,
 *   2 = [B, Cout/32, 2H, 2W, 8] bf16 = PixelShuffle(2) of the result when the caller packed the weights / bias with output
 *   channels ordered n' = (2i+j)*(Cout/4) + c (PixelShuffle: channel 4c+2i+j -> (c, 2h+i, 2w+j)): upconv + PixelShuffle +
 *   LeakyReLU of the tail (arch/SIDECVSR_our.py:4473-4476) in one launch (cdfo_conv_sm100_fwd with ksize = 1). */
int cdfo_conv3x3_sm100_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, void *y,
                           int B, int Cin, int Cout, int H, int W, int act, int out_mode, void *stream);
/* ---- offset / mask head of MVDualAttAlignment (arch/SIDECVSR_our.py:3274, :3339-3350) fused into the conv epilogue ----
 * The caller packs conv_offset[-1] with its output channels permuted into triples (dy, dx, m) in the order k' = tap*dg + g
 * (reference channels 2k, 2k+1, dg*18 + k with k = g*9 + tap).  out = "fields" [B, 9 taps, dg/gp, H, W, gp] x fp16x4 (dy, dx, m, 0):
 *   first == NULL : (magnitude*tanh(dy), magnitude*tanh(dx), m)                                  (evaluation on out_1)
 *   first != NULL : (first.dy + magnitude*tanh(dy), first.dx + magnitude*tanh(dx), sigmoid(first.m + m))
 *                   (evaluation on out_2; first = the previous call's output) = offset_1 + offset_2 and the mask;
 *   the MV prior (+ flow.flip(1).repeat) is added by cdfo_dcn_sm100_fwd (off_dtype = CDFO_FIELDS_F16X4).
 *   z_c8 [B, Cin/8, H, W, 8] bf16. */
int cdfo_mv_offset_head_sm100_fwd(const void *z_c8, const void *wpk, const float *bias, const void *first, void *out,
                                  int B, int Cin, int dg, int H, int W, float magnitude, void *stream);
/* Both evaluations in ONE launch: z_c8 [2 B,Cin/8,H,W,8] holds the two hidden maps (sample b and b + B); every CTA computes the same
 * pixel tile of both back to back and keeps the first evaluation in registers (rounded to fp16 exactly as the two-launch path
 * stores it: bit-identical fields), so the intermediate fields (1152 B per pixel written, then read) never reach HBM. */
int cdfo_mv_offset_head_dual_sm100_fwd(const void *z_c8, const void *wpk, const float *bias, void *out, int B, int Cin, int dg, int H,
                                       int W, float magnitude, void *stream);
/* conv_last (Cin -> 1, 3x3; weight packed with Cout padded to 16) + bias + bilinear x4 skip (align_corners=False) of the
 * 1-channel LR image lr [B, H/4, W/4] fp32 (arch/SIDECVSR_our.py:4477-4480); x_c8 [B, Cin/8, H, W, 8] bf16; y [B, 1, H, W] fp32. */
int cdfo_conv_last_skip_sm100_fwd(const void *x_c8, const void *wpk, const float *bias, const float *lr, float *y, int B,
                                  int Cin, int H, int W, void *stream);
int cdfo_conv3x3_sm100_pack_weight(const float *w, void *wpk, int Cout, int Cin, void *stream);
/* The same kernel for kernel size 1 or 3 (stride 1, "same" padding): 1x1 convolutions of the path -- tsa_fusion (448 -> 64,
 * arch/SIDECVSR_our.py:4466), upconv1 / upconv2 (:4473-4475), the trunk's down / up convs (:388-399).  For ksize = 1 the A operand
 * is the pixel tile itself (no halo) and the pipeline runs four 16 KB stages.  weight [Cout, Cin, ksize, ksize] fp32. */
int cdfo_conv_sm100_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, void *y, int B, int Cin,
                        int Cout, int H, int W, int ksize, int act, int out_mode, void *stream);
int cdfo_conv_sm100_pack_weight(const float *w, void *wpk, int Cout, int Cin, int ksize, void *stream);
size_t cdfo_conv_sm100_weight_bytes(int Cout, int Cin, int ksize);
size_t cdfo_conv3x3_sm100_weight_bytes(int Cout, int Cin);
int cdfo_conv3x3_sm100_ntile(int Cout, int Cin);
/* ---- A4 / A5: warp + fusion_out + dual MDTA + project_out (csrc/mdta.cu) ----
 * arch/SIDECVSR_our.py:3303-3337 (mode 0: MVDualAttAlignment, heads = 8, no ReLU after fusion_out) and :3455-3492
 * (mode 1: DualAttAlignment, heads = 4, ReLU after fusion_out, second fusion_out folded in).  All NCHW fp32:
 *   x [x_batch,64,H,W] query (sample b uses x[b % x_batch]); extra, pred [B,64,H,W]; flow [B,2,H,W] (x, y)
 *   fusion_w [64,128] (no bias); conv_du: du_w1 [4,64], du_b1 [4], du_w2 [64,4], du_b2 [64]; temperature [heads]; proj_w [64,64]
 *   mode 0: out = c8 bf16 [2B, 8, H, W, 8]: samples [0,B) = project_out(attn @ (warped*g)), [B,2B) = project_out(attn @ (pred*g))
 *   mode 1: out = NCHW fp32 [B,64,H,W] = ReLU(fusion_out(cat[o1 + o2, x])); ca_sums [B, cdfo_mdta_parts(B), 64] = per-part
 *           channel sums of out (feed cdfo_channel_gate_fwd: CALayer pooling, arch:2032-2043)
 *   workspace: cdfo_mdta_workspace_bytes(B, H, W, heads) bytes (holds the warped features, fp32). */
int cdfo_mdta_fwd(const float *x, int x_batch, const float *extra, const float *pred, const float *flow,
                  const float *fusion_w, const float *du_w1, const float *du_b1, const float *du_w2, const float *du_b2,
                  const float *temperature, const float *proj_w, int heads, int mode, void *out, float *ca_sums,
                  void *workspace, int B, int H, int W, void *stream);
/* Mode 0 with x, extra, pred as c8 bf16 [.,8,H,W,8] (what their producers write: the tcgen05 convolution's epilogue, the prior
 * convolution, the centre feature packed for the stack): the bilinear gather loads 16 bytes per corner and 8 channels, the warped
 * features live in the workspace as bf16, the arithmetic stays fp32 / TF32.  Same workspace size. */
int cdfo_mdta_c8_fwd(const void *x_c8, int x_batch, const void *extra_c8, const void *pred_c8, const float *flow, const float *fusion_w,
                     const float *du_w1, const float *du_b1, const float *du_w2, const float *du_b2, const float *temperature,
                     const float *proj_w, int heads, void *out_c8, void *workspace, int B, int H, int W, void *stream);
size_t cdfo_mdta_workspace_bytes(int B, int H, int W, int heads);
int cdfo_mdta_parts(int B);
/* gate [B,C] = sigmoid(W2 relu(W1 mean + b1) + b2), mean = (sum over `parts` of partial_sums [B,parts,C]) / HW; w1 [Cmid,C], w2 [C,Cmid]. */
int cdfo_channel_gate_fwd(const float *partial_sums, int parts, const float *w1, const float *b1, const float *w2,
                          const float *b2, float *gate, int B, int C, int Cmid, int HW, void *stream);
/* NCHW fp32 * scale[b][c] -> c8 bf16;  c8 bf16 + add[b % add_batch] (NCHW fp32) -> NCHW fp32. */
int cdfo_pack_c8_scaled(const float *x_nchw, const float *scale, void *x_c8, int B, int C, int H, int W, void *stream);
int cdfo_unpack_c8_add(const void *x_c8, const float *add_nchw, int add_batch, float *y_nchw, int B, int C, int H, int W,
                       void *stream);
/* ---- bilinear x0.5 / x2 (align_corners=False, arch/SIDECVSR_our.py:324-333) on c8 bf16, and the three-scale sum of the
 * trunk's cross-scale block (arch:401-406).  mode 0: y [B,C/8,Ho,Wo,8] = x0.5(a [.,2Ho,2Wo,.]); mode 1: y = x2(a [.,Ho/2,Wo/2,.]);
 * mode 2: y = base + x0.5(a) + x2(b). */
int cdfo_resample_c8(const void *a, const void *b, const void *base, void *y, int B, int C, int Ho, int Wo, int mode, void *stream);
/* ---- A8: LLongRangAttention.forward (arch/SIDECVSR_our.py:2179-2249) after its 1x1 input_conv and the pooled mask logits ----
 *   qv     [B,128,H,W] fp32 = input_conv(x) (q = first 64 channels, v = last 64)          arch:2206,2211
 *   u      [B,64,H,W]  fp32 uniform noise of gumbel_softmax (torch.rand_like, arch:2169)
 *   vmax   [B,64]      fp32 = conv_du_re2(avg_pool(conv_du_re(res)))                        arch:2183-2185
 *   x, x2  [B,64,H,W]  fp32 residual input = x + x2 (x2 may be NULL; the model passes the feature and the residual prior
 *          separately, arch:4449);  out [B,64,H,W] fp32 = fuse(cat[long, loc]) + x + x2  arch:2246-2249
 *   tables [9 + 9 + 64 + 4096] fp32: directW1_conv taps, directH1_conv taps, K1, R (see csrc/lra.cu); beta / bh their biases
 *   fuse_w [64,128] fp32, fuse_b [64];  workspace: cdfo_lra_workspace_bytes(B, H, W) bytes;  H, W multiples of 8.
 * No score tensor is materialised (the reference writes ~3.1 kB of fp32 scores per pixel and call). */
int cdfo_lra_fwd(const float *qv, const float *u, const float *vmax, const float *x, const float *x2, const float *tables,
                 float beta, float bh, const float *fuse_w, const float *fuse_b, float *out, void *workspace, int B, int H, int W,
                 void *stream);
/* Same, with the result leaving as bf16 in channels [channel0, channel0 + 64) of a c8 tensor [B,out_channels/8,H,W,8] -- the second
 * half of the model's cat([fea, x_n]) (arch:4454), the input of conv_expand_fea_r; no fp32 copy of x_n exists. */
/* Column pass operands: 0 (default) = bf16 mma.sync m16n8k16, 1 = TF32 m16n8k8 (the first-generation kernel; A/B switch). */
int cdfo_lra_set_col_precision(int tf32);
/* Column pass: 1 (default) = the tcgen05 kernel (csrc/lra_col_sm100.cu: score tile in tensor memory, bf16 operands; H <= 448), 0 = the
 * warp-level mma.sync kernels of round 1.  A measurement / test switch. */
int cdfo_lra_set_col_tcgen05(int on);
/* 8x8 window pass: 1 (default) = tensor cores (bf16 hi/lo split scores, mma.sync), 0 = round 1's fp32 SIMT kernel. */
int cdfo_lra_set_win_tensor_core(int on);
/* Row pass: 1 (default) = the raw v row arrives by tiled TMA (mbarrier ring; needs W % 4 == 0), 0 = 4-byte cp.async copies. */
int cdfo_lra_set_row_tma(int on);
int cdfo_lra_c8_fwd(const float *qv, const float *u, const float *vmax, const float *x, const float *x2, const float *tables,
                    float beta, float bh, const float *fuse_w, const float *fuse_b, void *out_c8, int out_channels, int channel0,
                    void *workspace, int B, int H, int W, void *stream);
/* ---- 1x1 convolutions of A8 on the tensor cores (csrc/pointwise.cu), NCHW fp32 in / out ----
 *   y[b,co,p] = act(bias[co] + sum_k w[co,k] x[b,k,p]) + resid1[b,co,p] + resid2[b,co,p]        (act 0 none / 1 ReLU)
 *   mode 0: x = in1 + in2 (in2 may be NULL), [B,K,H,W]; supported K -> Co: 64 -> 64 (conv_du_re.0, arch:2183), 64 -> 128 (input_conv
 *           on fea + residual prior, arch:2206/:4449);  mode 1: x = cat(in1, in2), both pixel-major [B,H*W,64], 128 -> 64 (fuse, arch:2246). */
int cdfo_pointwise_conv_fwd(const float *in1, const float *in2, const float *w, const float *bias, const float *resid1,
                            const float *resid2, float *out, int B, int K, int Co, int H, int W, int act, int mode, void *stream);
/* Same, the Co output channels leaving as bf16 in channels [channel0, channel0 + Co) of a c8 tensor [B,out_channels/8,H,W,8]
 * (H * W a multiple of 4). */
int cdfo_pointwise_conv_c8_fwd(const float *in1, const float *in2, const float *w, const float *bias, const float *resid1,
                               const float *resid2, void *out_c8, int B, int K, int Co, int H, int W, int act, int mode,
                               int out_channels, int channel0, void *stream);
size_t cdfo_lra_workspace_bytes(int B, int H, int W);
/* ---- pieces of the feature extraction (SURVEY 8f rank 2), NCHW, dtype CDFO_F32 or CDFO_BF16 storage, fp32 arithmetic ----
 * LayerNorm over the 64 channels of each pixel, WithBias (arch/SIDECVSR_our.py:1169-1198): y = (x - mu) rsqrt(var + eps) gamma + beta. */
int cdfo_layernorm_c_fwd(const void *x, const float *gamma, const float *beta, void *y, int B, int C, int H, int W, float eps,
                         int dtype, void *stream);
/* depthwise 3x3, stride 1, padding 1, no bias (qkv_dwconv, arch:1545-1576): w [C,1,3,3] fp32. */
int cdfo_dwconv3x3_fwd(const void *x, const float *w, void *y, int B, int C, int H, int W, int dtype, void *stream);
/* Per-head Gram matrix and squared norms of the MDTA self-attention (Attention.forward, arch:1545-1576; 8 heads x 8 channels):
 * qk [B,Ctot,H,W] (dtype fp32 / bf16) with q = channels [0,64), k = [64,128);  partial [B,parts,640] fp32 = per pixel range the 512
 * entries G[hd][i][j] = sum_p q[8hd+i] k[8hd+j], then sum_p q[c]^2 (64) and sum_p k[c]^2 (64): the caller adds the parts in order. */
int cdfo_mdta_gram_fwd(const void *qk, float *partial, int B, int Ctot, int H, int W, int parts, int dtype, void *stream);
/* ---- 3x3 convolutions on a CTA PAIR (csrc/conv3x3_pair_sm100.cu): tcgen05.mma cta_group::2, M = 256 pixels over the two SMs of a
 * TPC, each CTA holding the weights of HALF the output channels resident in shared memory.  Supported: Cout = 64 with Cin in
 * {64, 128, 192, 256} (the trunk's 256 -> 64, conv_expand_fea_r, the 64 -> 64 layers) and 64 -> 256 (the trunk's body.0,
 * arch/SIDECVSR_our.py:378-406).  x_c8 [B,Cin/8,H,W,8] bf16 -> y_c8 [B,Cout/8,H,W,8] bf16 = act(conv + bias) + resid_c8
 * (act 0 none / 1 ReLU / 2 LeakyReLU 0.1; bias, resid_c8 may be NULL).  Results are bit-identical to cdfo_conv_sm100_fwd. */
int cdfo_conv3x3_pair_sm100_supported(int Cout, int Cin);
size_t cdfo_conv3x3_pair_sm100_weight_bytes(int Cout, int Cin);
int cdfo_conv3x3_pair_sm100_pack_weight(const float *w, void *wpk, int Cout, int Cin, void *stream);
int cdfo_conv3x3_pair_sm100_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, void *y_c8, int B, int Cin,
                                int Cout, int H, int W, int act, void *stream);
/* Same, with y_planes = 1 storing the output as its four parity planes [B,Cout/8,2 (row parity),2 (column parity),H/2,W/2,8]
 * (H, W even; pixel (h, w) -> plane (h & 1, w & 1) at (h / 2, w / 2)): the input layout of cdfo_conv4x4s2_pair_sm100_planes_fwd;
 * y_planes = 2: y is NCHW fp32 [B,Cout,H,W]. */
int cdfo_conv3x3_pair_sm100_planes_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, void *y, int B,
                                       int Cin, int Cout, int H, int W, int act, int y_planes, void *stream);
/* Same, with bias_edge [9][Cout] fp32 (or NULL): the bias of the border pixels by class (row: top 0 / middle 1 / bottom 2) * 3 + (column: left
 * 0 / middle 1 / right 2); `bias` stays the interior one (class 4).  For a 1x1 convolution composed INTO this 3x3 one (Block_'s down / up 1x1
 * followed by body.0, arch/SIDECVSR_our.py:388-406): its bias passes only under the taps that lie inside the frame. */
int cdfo_conv3x3_pair_sm100_edge_fwd(const void *x_c8, const void *wpk, const float *bias, const float *bias_edge, const void *resid_c8,
                                     void *y, int B, int Cin, int Cout, int H, int W, int act, int y_planes, void *stream);
/* The 64 -> 256 convolution applied to the bilinear x2 of x8_1x [B,8,H2/2,W2/2,8] bf16 (F.interpolate, align_corners=False) without
 * materialising it: y = cdfo_conv3x3_pair_sm100_edge_fwd(cdfo_resample_c8(x8_1x, mode 1), ...) bit for bit, at the 2x size H2 x W2
 * (both even).  Cin = 64, Cout = 256, no residual, y_planes 0 (c8) or 1 (parity planes); bias_edge may be NULL. */
int cdfo_conv3x3_pair_sm100_up2_fwd(const void *x8_1x, const void *wpk, const float *bias, const float *bias_edge, void *y, int B, int Cin,
                                    int Cout, int H2, int W2, int act, int y_planes, void *stream);
/* ---- "3x3 convolution at 2H x 2W followed by bilinear x0.5" as ONE 4x4 / stride-2 convolution on a CTA pair
 * (csrc/conv4x4s2_pair_sm100.cu): the down(body(up(x))) branch of Block_.forward, arch/SIDECVSR_our.py:401-406 with Interpolate(0.5)
 * :324-333.  w3 [64,Cin,3,3] fp32 is the 3x3 weight (pack_weight folds the 2x2 mean into a 4x4 kernel);
 * x_c8 [B,Cin/8,H_in,W_in,8] bf16 (H_in, W_in even) -> y_c8 [B,8,H_in/2,W_in/2,8] bf16 = conv + bias + resid_c8. */
int cdfo_conv4x4s2_pair_sm100_supported(int Cout, int Cin);
size_t cdfo_conv4x4s2_pair_sm100_weight_bytes(int Cin);
int cdfo_conv4x4s2_pair_sm100_pack_weight(const float *w3, void *wpk, int Cin, void *stream);
int cdfo_conv4x4s2_pair_sm100_fwd(const void *x_c8, const void *wpk, const float *bias, const void *resid_c8, void *y_c8, int B, int Cin,
                                  int H_in, int W_in, void *stream);
/* Same, with x_planes = 1 reading x as parity planes [B,Cin/8,2,2,H_in/2,W_in/2,8]: every stride-2 phase window is then a dense
 * TMA box (the plain c8 input is loaded with elementStrides = 2, one L2 request per 16-byte pixel chunk). */
int cdfo_conv4x4s2_pair_sm100_planes_fwd(const void *x, const void *wpk, const float *bias, const void *resid_c8, void *y_c8, int B,
                                         int Cin, int H_in, int W_in, int x_planes, void *stream);
/* Same, closing a whole cross-scale block (Block_.forward, arch/SIDECVSR_our.py:401-406) in the epilogue:
 *   y = conv + bias + resid_c8 + bilinear_x2(up_c8)        up_c8 [B,8,H_in/4,W_in/4,8] bf16 or NULL: the up(body(down(x))) branch
 *   half_c8 = bilinear_x0.5(y) from the fp32 values        [B,8,H_in/4,W_in/4,8] bf16 or NULL: the next block's down(x) input
 * (no separate resampling passes over HBM; H_in, W_in multiples of 4 when either is given). */
int cdfo_conv4x4s2_pair_sm100_block_fwd(const void *x, const void *wpk, const float *bias, const void *resid_c8, const void *up_c8,
                                        void *y_c8, void *half_c8, int B, int Cin, int H_in, int W_in, int x_planes, void *stream);
/* ---- frame I/O of the evaluation loop (SURVEY 8f rank 3) ----
 * Integer planes [n_planes, H_in, W] (src_kind 0 uint8, 1 int8, 2 int16, 3 int32) -> fp32 k / 255 [n_planes, H_out, W], rows
 * H_in..H_out-1 zero: generate_input / generate_PM_input / generate_RM_input (test_LD_37.py:19-29,33-46,64-74; 270 -> 272 rows). */
int cdfo_planes_to_unit_f32(const void *src, int src_kind, float *dst, int n_planes, int H_in, int W, int H_out, void *stream);
/* SR fp32 [n_planes, H_in, W] -> uint8 [n_planes, H_out, W], H_out <= H_in (drops the padded rows): slice, clamp(0, 1) * 255.0,
 * astype(uint8) = truncation, what cv2.imwrite receives at test_LD_37.py:172-180. */
int cdfo_sr_to_u8(const float *sr, uint8_t *out, int n_planes, int H_in, int W, int H_out, void *stream);
/* ---- on-GPU PSNR / SSIM (SURVEY 8f rank 4): metric/psnr_ssim.py:278-317 calculate_psnr, :320-399 _ssim / calculate_ssim as
 * cal_psnr_ssim (:446-484) calls them -- single-channel uint8 frames, crop_border pixels dropped on every edge, the float32
 * / 255 * 255 round trip of to_y_channel, 11x11 Gaussian (sigma 1.5) in fp64 on the valid region.
 *   res, gt   [B, H, W] uint8;  frame_out [B, 2] fp64 = (psnr dB (inf when identical), ssim) or NULL
 *   accum     [B, 3] fp64 or NULL: += (psnr, ssim, 1) per image -- the per-sequence sums cal_psnr_ssim averages over frames
 *   workspace cdfo_psnr_ssim_workspace_bytes(B, H, W, border) bytes.  Summation order is fixed (reproducible). */
size_t cdfo_psnr_ssim_workspace_bytes(int B, int H, int W, int border);
int cdfo_psnr_ssim_u8(const uint8_t *res, const uint8_t *gt, int B, int H, int W, int border, double *frame_out, double *accum,
                      void *workspace, void *stream);
/* tcgen05 plumbing self-test: D[128,64] fp32 = A[128,64] * B[64,64]^T (row-major bf16 inputs). */
int cdfo_umma_selftest(const void *A, const void *B, float *D, int swap_lbo_sbo, void *stream);

/* ---- A8, mask logits after conv_du_re.0 (csrc/lra_mask_logits.cu; arch/SIDECVSR_our.py:2183-2186) ----
 * v_max [B, 64] = ReLU(conv_du_re2(mean_hw ReLU(conv_du_re.2(v)))): v [B, 64, H, W] fp32 = ReLU(conv_du_re.0(res)); w2 [64,64,3,3] / b2 the
 * stride-2 padding-2 convolution, w3 [64,64] / b3 the 1x1 on the pooled vector.  Tensor cores (TF32 mma.sync), the strided activation is
 * never written; workspace: cdfo_lra_mask_logits_workspace_bytes(B, H, W) bytes of tile sums (fixed-order reduction). */
size_t cdfo_lra_mask_logits_workspace_bytes(int B, int H, int W);
int cdfo_lra_mask_logits_fwd(const float *v, const float *w2, const float *b2, const float *w3, const float *b3, float *vmax,
                             void *workspace, int B, int H, int W, void *stream);
/* Stride-2 convolution of the mask logits: 1 (default) = input patches by tiled TMA (mbarrier ring; needs W % 4 == 0),
 * 0 = the 4-byte cp.async kernel.  A measurement / test switch. */
int cdfo_lra_set_logit_tma(int on);

/* ---- feature extraction on c8 bf16 (csrc/features_c8.cu; SURVEY.md 8f rank 2; arch/SIDECVSR_our.py:1441-1475, :1643-1653) ----
 * "c8" = [B, C/8, H, W, 8] bf16.  fp32 arithmetic, fixed reduction orders. */
/* Conv2d(1, Co, 3, 1, 1) on x [B,1,H,W] fp32 (conv_first / conv_second, arch:4376-4377) -> y c8; lrelu != 0 applies LeakyReLU(0.1). */
int cdfo_prior_conv_c8_fwd(const float *x, const float *w, const float *bias, void *y_c8, int B, int Co, int H, int W, int lrelu, void *stream);
/* WithBias LayerNorm over the 64 channels of each pixel (arch:1169-1198). */
int cdfo_layernorm_c8_fwd(const void *x_c8, const float *gamma, const float *beta, void *y_c8, int B, int H, int W, float eps, void *stream);
/* Depthwise 3x3 / stride 1 / padding 1, no bias (qkv_dwconv, arch:1558): w [C, 9] fp32. */
int cdfo_dwconv3x3_c8_fwd(const void *x_c8, const float *w, void *y_c8, int B, int C, int H, int W, void *stream);
/* Per-head Gram q k^T over H*W + squared row norms of q (channels 0..63) and k (64..127) of qkv_c8 [B, C/8 >= 16, H, W, 8], 8 heads x 8
 * channels: partial [B, parts, 640] fp32 = (G [8][8][8] | |q|^2 [64] | |k|^2 [64]) per pixel range. */
int cdfo_mdta_gram_c8_fwd(const void *qkv_c8, float *partial, int B, int C, int H, int W, int parts, void *stream);
/* M [B, 64, 64] = project_out . blockdiag(softmax(G / (|q| |k|) * temperature)) from the partial sums (arch:1567-1576). */
int cdfo_mdta_fold_fwd(const float *partial, const float *temperature, const float *project_out, float *M, int B, int parts, void *stream);
/* out1 = x1 + M v (v = channels [v_channel0, +64) of qkv_c8); out2 (optional) = out1 + x2. */
int cdfo_mdta_apply_c8_fwd(const void *qkv_c8, int C, int v_channel0, const float *M, const void *x1_c8, const void *x2_c8, void *out1_c8,
                           void *out2_c8, int B, int H, int W, void *stream);
/* 16 -> 16 channels, 3x3, stride 2, padding 2, + LeakyReLU(0.1): convolution (transposed = 0, w [co][ci][3][3], Ho = (Hi + 1) / 2 + 1) or
 * transposed convolution (transposed = 1, w [ci][co][3][3], Ho = 2 Hi - 3 or 2 Hi - 2 with output_padding 1) of the side branch
 * (arch:1815-1832).  y_c8 has y_channels >= 16 channels; channels 0..15 are written. */
int cdfo_conv16_c8_fwd(const void *x_c8, const float *w, const float *bias, void *y_c8, int B, int Hi, int Wi, int Ho, int Wo, int y_channels,
                       int transposed, void *stream);
/* SpatialAttention (arch:1883-1899) on a 16-channel c8 map: y = x * sigmoid(conv7x7([max_c x, mean_c x]) + bias); w [1][2][7][7];
 * pooled_ws: B * H * W * 8 bytes of scratch. */
int cdfo_spatial_gate_c8_fwd(const void *x_c8, const float *w, const float *bias, void *pooled_ws, void *y_c8, int B, int H, int W, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CDFO_B200_H_ */
