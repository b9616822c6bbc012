"""Process-wide switches of the host side."""
import os

# Route deformable convolutions of the model's hot shape (64->64, 3x3, s=p=d=1, groups=1) to the tcgen05
# implicit-GEMM kernel (bf16 operands, fp32 accumulate).  False: every call takes the fp32 catch-all kernel.
tensor_core = True

# Gather of the fused alignment path (MVDualAttAlignment: head fields -> DCN):
#   "tex"   bilinear footprint fetched by the texture units (cdfo_dcn_tex_sm100_fwd; 8-bit filter weights, fp16 operands)
#   "exact" fp32 coordinate / weight arithmetic of the reference with LDG gathers (cdfo_dcn_sm100_fwd; bf16 operands)
dcn_gather = "tex"

# Plain 3x3 convolutions that both kernels can serve (>= 128 input and 64 output channels, e.g. the trunk's 256 -> 64): True = the two-SM
# kernel (CTA pair, tcgen05.mma cta_group::2, weights resident, cdfo_conv3x3_pair_sm100_fwd); False = the single-SM kernel that streams the
# weights.  Calls that only the CTA-pair kernel serves (parity-plane output, border-class bias, conv.conv3x3_up2, conv.conv3x3_then_half)
# take it either way.
conv_pair = os.environ.get("CDFO_CONV_PAIR", "1") != "0"

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
# True: the mask logits of LLongRangAttention start from the ONE-channel residual map (conv_expand_rms composed with conv_du_re.0 + ReLU as one
# direct 1 -> 64 convolution) instead of reading the 64-channel prior features through a 1x1 convolution kernel.
lra_logits_from_prior = os.environ.get("CDFO_LRA_LOGITS_FROM_PRIOR", "1") != "0"
