"""Process-wide switches of the host side."""
import os

# Route deformable convolutions of the model's hot shape (64->64, 3x3, s=p=d=1, groups=1) to the tcgen05
# implicit-GEMM kernel (bf16 operands, fp32 accumulate).  False: every call takes the fp32 catch-all kernel.
tensor_core = True

# Gather of the fused alignment path (MVDualAttAlignment: head fields -> DCN):
#   "tex"   bilinear footprint fetched by the texture units (cdfo_dcn_tex_sm100_fwd; 8-bit filter weights, fp16 operands)
#   "exact" fp32 coordinate / weight arithmetic of the reference with LDG gathers (cdfo_dcn_sm100_fwd; bf16 operands)
dcn_gather = "tex"

# 3x3 convolutions with >= 128 input and 64 output channels (the trunk's 256 -> 64): True = the two-SM kernel (CTA pair,
# tcgen05.mma cta_group::2, weights resident, cdfo_conv3x3_pair_sm100_fwd); False = the single-SM kernel that streams the weights.
conv_pair = os.environ.get("CDFO_CONV_PAIR", "1") != "0"

# Block_'s down(body(up(x))) branch: True = its last 3x3 convolution and the bilinear x0.5 that follows run as one 4x4 / stride-2
# convolution at the output resolution (cdfo_conv4x4s2_pair_sm100_fwd, 2.25x fewer FLOPs); False = conv at 2x + resample kernel.
conv_fold_half = os.environ.get("CDFO_CONV_FOLD_HALF", "1") != "0"

# With conv_fold_half: True = the 2x-resolution intermediate of that branch is written by the 64 -> 256 convolution as its four parity
# planes ([B, C/8, 2, 2, H, W, 8]), so every stride-2 phase window of the folded convolution is a dense TMA box; False = plain c8,
# loaded with elementStrides = 2 (every 16-byte pixel chunk drags a 32-byte L2 sector: 1.85 GB instead of 1.16 GB of L2 -> SM traffic per
# launch at 2 x 544x960).  Measured (tools/bench_conv.py) once the MMA issuer stopped being the bottleneck: 193.6 -> 153.8 us for the
# folded convolution against +16 us for the producer's scattered stores.
conv_parity_planes = os.environ.get("CDFO_CONV_PARITY_PLANES", "1") != "0"
# With conv_fold_half: True = the folded convolution's epilogue closes the block (adds the bilinear x2 of the half-resolution branch and writes
# the x0.5 of the sum for the next block): no resampling pass over HBM between the blocks of a group.  False = round 1's resample kernels.
trunk_fused_resample = os.environ.get("CDFO_TRUNK_FUSED_RESAMPLE", "1") != "0"

# Offset / mask head of MVDualAttAlignment: True = both evaluations of conv_offset[-1] in one launch (the first one stays in the
# epilogue's registers, cdfo_mv_offset_head_dual_sm100_fwd); False = two launches with the intermediate fields in HBM.
head_dual = os.environ.get("CDFO_HEAD_DUAL", "1") != "0"

# MVDualAttAlignment (dg = 16, texture gather): True = conv_offset[-1] on both hidden maps + tanh / sigmoid + MV prior + DCN as ONE kernel
# (cdfo_mv_head_dcn_fused_sm100_fwd: the offset / mask fields never reach HBM); False = dual head launch -> fields in HBM -> DCN kernel.
fused_head_dcn = os.environ.get("CDFO_FUSED_HEAD_DCN", "1") != "0"

# Feature extraction (conv_first / conv_second + PAItransformerSA_2) when model.lowp is bf16: True = this repo's kernels on c8 bf16
# (cdfo_b200/features.py: tcgen05 convolutions + csrc/features_c8.cu, no cuDNN / cuBLAS / ATen launch, bit-identical reruns);
# False = round 1's path (cuDNN bf16 convolutions under autocast + own LayerNorm / depthwise / Gram kernels).  model.lowp = None
# always takes the fp32 cuDNN path (a debugging reference, not the benchmarked configuration).
features_c8 = os.environ.get("CDFO_FEATURES_C8", "1") != "0"
# True: on the fused-alignment path the MDTA kernels of MVDualAttAlignment read c8 bf16 inputs (conv_expand_fea_r's output, the ufs prior
# features, the packed centre feature) and keep the warped features in bf16 (cdfo_mdta_c8_fwd); False: fp32 NCHW copies as in round 1.
mdta_c8 = os.environ.get("CDFO_MDTA_C8", "1") != "0"
# True: the down / up 1x1 convolutions of a cross-scale block are composed into body.0's 3x3 weights (they commute with the bilinear
# resampling; the 1x1 bias becomes a border-class bias table of the 3x3 kernel's epilogue): 42 fewer launches per trunk.
trunk_compose_1x1 = os.environ.get("CDFO_TRUNK_COMPOSE_1X1", "1") != "0"
# With trunk_compose_1x1 and conv_fold_half: True = body.0 of the down(body(up(x))) branch builds its A operand from the 1x image (bilinear x2 in
# the producer, cdfo_conv3x3_pair_sm100_up2_fwd; bit-identical): the 2x input tensor is never written.  False = resample kernel + convolution.
trunk_fused_upsample = os.environ.get("CDFO_TRUNK_FUSED_UPSAMPLE", "1") != "0"
# True: the mask logits of LLongRangAttention start from the ONE-channel residual map (conv_expand_rms composed with conv_du_re.0 + ReLU as one
# direct 1 -> 64 convolution) instead of reading the 64-channel prior features through a 1x1 convolution kernel.
lra_logits_from_prior = os.environ.get("CDFO_LRA_LOGITS_FROM_PRIOR", "1") != "0"
