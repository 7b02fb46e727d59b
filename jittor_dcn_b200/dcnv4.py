"""The DCNv4 module on the engine's kernels.

``DCNv4`` restates ``DCNv4_op/DCNv4/modules/dcnv4.py`` of the DCNv4 repository (FlashInternImage): the constructor,
attributes, submodules and initialisation, and ``forward`` on ``[N, L, C]`` tokens.  Those names and defaults are
restated from the repository as remembered; its sources were not available when this was written, so the state-dict
keys have not been checked against an upstream checkpoint.  The core runs on csrc/dcn_dcnv3.cu through
``DCNv4Function``.
"""
import torch
import torch.nn.functional as F
from torch import nn
from torch.nn.init import constant_, xavier_uniform_

from .functional import DCNv4Function, dcnv4_row_floats

_GROUP_CHANNELS = (16, 32, 64, 128, 256)


class CenterFeatureScaleModule(nn.Module):
    def forward(self, query, center_feature_scale_proj_weight, center_feature_scale_proj_bias):
        return F.linear(query, weight=center_feature_scale_proj_weight, bias=center_feature_scale_proj_bias).sigmoid()


class DCNv4(nn.Module):
    def __init__(self, channels=64, kernel_size=3, stride=1, pad=1, dilation=1, group=4, offset_scale=1.0,
                 dw_kernel_size=None, center_feature_scale=False, remove_center=False, output_bias=True,
                 without_pointwise=False):
        """
        DCNv4 Module
        :param channels           number of input (and output) channels, group * group_channels
        :param kernel_size        sampling grid of kernel_size x kernel_size points per group
        :param offset_scale       scales the dilation grid and the offsets
        :param dw_kernel_size     if set, a depthwise conv of this kernel feeds offset_mask (offset_mask_dw)
        :param remove_center      drop the kernel's centre point (odd kernel_size only)
        :param output_bias        bias of output_proj
        :param without_pointwise  no value_proj / output_proj: the core runs on the input itself
        """
        super().__init__()
        if channels % group != 0:
            raise ValueError(f'channels must be divisible by group, but got {channels} and {group}')
        _d_per_group = channels // group
        if _d_per_group not in _GROUP_CHANNELS:
            raise ValueError(f'DCNv4: channels // group = {_d_per_group} channels per group is not supported '
                             f'(one of {_GROUP_CHANNELS})')
        if remove_center and kernel_size % 2 == 0:
            raise ValueError(f'DCNv4: remove_center needs an odd kernel_size, got {kernel_size}')

        self.offset_scale = offset_scale
        self.channels = channels
        self.kernel_size = kernel_size
        self.stride = stride
        self.dilation = dilation
        self.pad = pad
        self.group = group
        self.group_channels = channels // group
        self.dw_kernel_size = dw_kernel_size
        self.center_feature_scale = center_feature_scale
        self.remove_center = int(remove_center)
        self.without_pointwise = without_pointwise

        self.K = group * (kernel_size * kernel_size - self.remove_center)
        if dw_kernel_size is not None:
            self.offset_mask_dw = nn.Conv2d(channels, channels, dw_kernel_size, stride=1,
                                            padding=(dw_kernel_size - 1) // 2, groups=channels)
        self.offset_mask = nn.Linear(channels, dcnv4_row_floats(kernel_size, kernel_size, group, remove_center))
        if not without_pointwise:
            self.value_proj = nn.Linear(channels, channels)
            self.output_proj = nn.Linear(channels, channels, bias=output_bias)
        self._reset_parameters()

        if center_feature_scale:
            self.center_feature_scale_proj_weight = nn.Parameter(torch.zeros((group, channels), dtype=torch.float))
            self.center_feature_scale_proj_bias = nn.Parameter(
                torch.tensor(0.0, dtype=torch.float).view((1,)).repeat(group, ))
            self.center_feature_scale_module = CenterFeatureScaleModule()

    def _reset_parameters(self):
        constant_(self.offset_mask.weight.data, 0.)
        constant_(self.offset_mask.bias.data, 0.)
        if not self.without_pointwise:
            xavier_uniform_(self.value_proj.weight.data)
            constant_(self.value_proj.bias.data, 0.)
            xavier_uniform_(self.output_proj.weight.data)
            if self.output_proj.bias is not None:
                constant_(self.output_proj.bias.data, 0.)

    def forward(self, input, shape=None):
        """
        :param input   (N, L, C) tokens of an H x W image, row-major
        :param shape   (H, W); default: a square image, H = W = sqrt(L)
        :return output (N, L, C)
        """
        N, L, C = input.shape
        if shape is not None:
            H, W = shape
        else:
            H, W = int(L ** 0.5), int(L ** 0.5)

        x = input
        if not self.without_pointwise:
            x = self.value_proj(x)
        x = x.reshape(N, H, W, -1)
        if self.dw_kernel_size is not None:
            offset_mask_input = self.offset_mask_dw(input.view(N, H, W, C).permute(0, 3, 1, 2))
            offset_mask_input = offset_mask_input.permute(0, 2, 3, 1).view(N, L, C)
        else:
            offset_mask_input = input
        offset_mask = self.offset_mask(offset_mask_input).reshape(N, H, W, -1)

        x_proj = x
        dtype = x.dtype
        # bfloat16 or float16 x and offset_mask of one dtype (autocast, module.half()) go to the core as they are; any
        # other mix (e.g. without_pointwise under autocast) runs on float32 copies, and the output comes back in x's dtype
        half = x.dtype in (torch.bfloat16, torch.float16) and offset_mask.dtype == x.dtype
        with torch.autocast(device_type=input.device.type, enabled=False):
            x = DCNv4Function.apply(
                *((x, offset_mask) if half else (x.float(), offset_mask.float())),
                self.kernel_size, self.kernel_size,
                self.stride, self.stride,
                self.pad, self.pad,
                self.dilation, self.dilation,
                self.group, self.group_channels,
                self.offset_scale,
                256,
                self.remove_center).type(dtype)

        if self.center_feature_scale:
            center_feature_scale = self.center_feature_scale_module(
                x, self.center_feature_scale_proj_weight, self.center_feature_scale_proj_bias)
            # N, H, W, groups -> N, H, W, groups, 1 -> N, H, W, groups, _d_per_group -> N, H, W, channels
            center_feature_scale = center_feature_scale[..., None].repeat(
                1, 1, 1, 1, self.channels // self.group).flatten(-2)
            x = x * (1 - center_feature_scale) + x_proj * center_feature_scale

        x = x.view(N, L, -1)
        if not self.without_pointwise:
            x = self.output_proj(x)
        return x
