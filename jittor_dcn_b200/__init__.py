"""jittor_dcn_b200 — B200-native engine behind the reference's DeformConv2d / TorchDeformConv2d.

Only what the hot path needs: the C-ABI library (csrc/ -> libdcn_b200.so), its ctypes
binding and the two module classes that mirror the reference's operator interface.
"""
from ._lib import (DCN_V3_FLAG_SOFTMAX_MASK, DCN_V4_FLAG_REMOVE_CENTER, DcnError, DcnMsdaShape, DcnShape, DcnV3Shape,
                   FLAG_ACCUM_GRAD_X, FLAG_FORCE_SIMT, FLAG_NO_GRAD_X, FLAG_RELU_OUT,
                   OPERAND_BF16, OPERAND_FP16, OPERAND_FP32, VARIANT_DCNV1, VARIANT_JITTOR, VARIANT_TORCH, load, make_shape)
from .deform_conv import DeformConv2d
from .functional import (batch_norm_relu, clear_workspaces, dcn_backward, dcn_backward_modulated, dcn_corners,
                         dcn_forward, dcn_forward_modulated, dcn_layer_backward, dcn_layer_forward,
                         dcn_layer_backward_modulated, dcn_layer_forward_modulated, dcn_offset_conv_forward,
                         dcn_offset_conv_forward_modulated, deform_conv2d, deform_conv2d_modulated, deform_conv2d_v1,
                         deform_layer, layer_supported, modulated_deform_layer, modulated_layer_supported,
                         MSDeformAttnFunction, dcn_msda_backward, dcn_msda_forward, ms_deform_attn,
                         DCNv3Function, dcn_v3_backward, dcn_v3_forward, dcnv3_core,
                         DCNv4Function, dcn_v4_backward, dcn_v4_forward, dcnv4_core, dcnv4_row_floats)
from .dcnv3 import DCNv3
from .dcnv4 import DCNv4
from .msda import MSDeformAttn
from .chain import ChainedDeformStages
from .roi_pool import DeformPSRoIPool, DeformRoIPool
from .torch_module import (BatchNormReLU2d, ModulatedDeformConv2dPack, StemConv2d, TorchDeformConv2d,
                           TorchDeformConv2dJittorSemantics, TorchvisionDeformConv2d, fuse_eval_bn_relu)

__all__ = [
    "DeformConv2d", "TorchDeformConv2d", "BatchNormReLU2d", "batch_norm_relu", "TorchDeformConv2dJittorSemantics", "deform_conv2d",
    "dcn_forward", "dcn_backward", "dcn_corners", "deform_conv2d_v1", "VARIANT_DCNV1", "load", "make_shape", "DcnShape", "DcnError",
    "VARIANT_JITTOR", "VARIANT_TORCH", "OPERAND_FP32", "OPERAND_BF16", "OPERAND_FP16", "FLAG_ACCUM_GRAD_X",
    "FLAG_FORCE_SIMT", "FLAG_NO_GRAD_X", "FLAG_RELU_OUT", "clear_workspaces", "dcn_offset_conv_forward", "dcn_layer_forward", "dcn_layer_backward", "deform_layer",
    "layer_supported", "fuse_eval_bn_relu", "DeformRoIPool", "DeformPSRoIPool", "ChainedDeformStages", "StemConv2d",
    "dcn_forward_modulated", "dcn_backward_modulated", "deform_conv2d_modulated", "TorchvisionDeformConv2d",
    "dcn_offset_conv_forward_modulated", "dcn_layer_forward_modulated", "dcn_layer_backward_modulated",
    "modulated_deform_layer", "modulated_layer_supported", "ModulatedDeformConv2dPack",
    "DcnMsdaShape", "dcn_msda_forward", "dcn_msda_backward", "MSDeformAttnFunction", "ms_deform_attn", "MSDeformAttn",
    "DcnV3Shape", "DCN_V3_FLAG_SOFTMAX_MASK", "dcn_v3_forward", "dcn_v3_backward", "DCNv3Function", "dcnv3_core",
    "DCNv3",
    "DCN_V4_FLAG_REMOVE_CENTER", "dcn_v4_forward", "dcn_v4_backward", "DCNv4Function", "dcnv4_core", "dcnv4_row_floats",
    "DCNv4",
]
