"""DCNv4 defined through the DCNv3 references (oracle/dcnv3_reference.py).  TEST INFRA: the product never imports it.

DCNv4's core is DCNv3's with the mask used as given (no softmax), offsets and mask packed into one tensor
offset_mask [N, Ho, Wo, Cm], Cm = ceil(3*G*K / 8)*8 (group g owns floats [g*3K, g*3K + 3K) of each pixel: 2K interleaved
(dx, dy), then K mask values; the rest is padding), and remove_center, which drops the centre point of an odd kernel
(K = kh*kw - 1).  ``unpack`` turns offset_mask into DCNv3's offset / mask, with the centre point reinserted at offset 0
and mask 0, so that every DCNv3 reference evaluates DCNv4; autograd through ``unpack`` packs the gradients back (0 in
the padding, the centre point's gradients dropped).  ``DCNv4Ref`` restates the module of the DCNv4 repository on the
composition.
"""
import torch
import torch.nn.functional as F
from torch import nn
from torch.nn.init import constant_, xavier_uniform_

from . import dcnv3_reference


def points(kernel_h, kernel_w, remove_center):
    """K, and the index c of the centre point in DCNv3's x-major order (None without remove_center)."""
    if not remove_center:
        return kernel_h * kernel_w, None
    return kernel_h * kernel_w - 1, (kernel_w // 2) * kernel_h + kernel_h // 2


def row_floats(kernel_h, kernel_w, group, remove_center):
    K, _ = points(kernel_h, kernel_w, remove_center)
    return (3 * group * K + 7) // 8 * 8


def unpack(offset_mask, kernel_h, kernel_w, group, remove_center):
    """offset_mask [N, Ho, Wo, Cm] -> DCNv3's offset [N, Ho, Wo, G*P*2], mask [N, Ho, Wo, G*P] with P = kh*kw (the
    removed centre point, if any, at offset 0 and mask 0).  Differentiable; the padding columns are never read."""
    N, Ho, Wo, _ = offset_mask.shape
    K, c = points(kernel_h, kernel_w, remove_center)
    om = offset_mask[..., :3 * group * K].reshape(N, Ho, Wo, group, 3 * K)
    off = om[..., :2 * K].reshape(N, Ho, Wo, group, K, 2)
    m = om[..., 2 * K:]
    if c is not None:
        off = torch.cat([off[..., :c, :], off.new_zeros(N, Ho, Wo, group, 1, 2), off[..., c:, :]], 4)
        m = torch.cat([m[..., :c], m.new_zeros(N, Ho, Wo, group, 1), m[..., c:]], 4)
    return off.reshape(N, Ho, Wo, -1), m.reshape(N, Ho, Wo, -1)


def dcnv4_core_pytorch(input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                       dilation_w, group, group_channels, offset_scale, remove_center=False):
    """DCNv4 on InternImage's grid_sample composition (dcnv3_core_pytorch)."""
    off, m = unpack(offset_mask, kernel_h, kernel_w, group, remove_center)
    return dcnv3_reference.dcnv3_core_pytorch(input, off, m, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                                              dilation_h, dilation_w, group, group_channels, offset_scale)


def reference(input, offset_mask, geo, grad_out=None, remove_center=False):
    """float64 CPU evaluation on dcnv3_reference.dcnv3_core_pixels (exact pixel coordinates: the gradient reference)
    -> out, or (out, grad_input, grad_offset_mask).  geo = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
    dilation_h, dilation_w, group, group_channels, offset_scale)."""
    x, om = (torch.as_tensor(t).detach().cpu().double().requires_grad_(grad_out is not None)
             for t in (input, offset_mask))
    off, m = unpack(om, geo[0], geo[1], geo[8], remove_center)
    out = dcnv3_reference.dcnv3_core_pixels(x, off, m, *geo)
    if grad_out is None:
        return out.detach()
    g = torch.as_tensor(grad_out).detach().cpu().double()
    gx, gom = torch.autograd.grad(out, [x, om], g)
    return out.detach(), gx, gom


class CenterFeatureScaleModule(nn.Module):
    def forward(self, query, center_feature_scale_proj_weight, center_feature_scale_proj_bias):
        return F.linear(query, weight=center_feature_scale_proj_weight, bias=center_feature_scale_proj_bias).sigmoid()


class DCNv4Ref(nn.Module):
    """The DCNv4 repository's DCNv4 module (restated from memory, as the engine's module is) with dcnv4_core_pytorch as
    its core.  core_fp32: under autocast the core runs on float32 operands and its output is cast back, as the
    engine's module does."""

    def __init__(self, channels=64, kernel_size=3, stride=1, pad=1, dilation=1, group=4, offset_scale=1.0,
                 dw_kernel_size=None, center_feature_scale=False, remove_center=False, output_bias=True,
                 without_pointwise=False, core_fp32=False):
        super().__init__()
        self.core_fp32 = core_fp32
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
        if dw_kernel_size is not None:
            self.offset_mask_dw = nn.Conv2d(channels, channels, dw_kernel_size, stride=1,
                                            padding=(dw_kernel_size - 1) // 2, groups=channels)
        self.offset_mask = nn.Linear(channels, row_floats(kernel_size, kernel_size, group, remove_center))
        if not without_pointwise:
            self.value_proj = nn.Linear(channels, channels)
            self.output_proj = nn.Linear(channels, channels, bias=output_bias)
        constant_(self.offset_mask.weight.data, 0.)
        constant_(self.offset_mask.bias.data, 0.)
        if not without_pointwise:
            xavier_uniform_(self.value_proj.weight.data)
            constant_(self.value_proj.bias.data, 0.)
            xavier_uniform_(self.output_proj.weight.data)
            if self.output_proj.bias is not None:
                constant_(self.output_proj.bias.data, 0.)
        if center_feature_scale:
            self.center_feature_scale_proj_weight = nn.Parameter(torch.zeros((group, channels), dtype=torch.float))
            self.center_feature_scale_proj_bias = nn.Parameter(
                torch.tensor(0.0, dtype=torch.float).view((1,)).repeat(group, ))
            self.center_feature_scale_module = CenterFeatureScaleModule()

    def forward(self, input, shape=None):
        N, L, C = input.shape
        H, W = shape if shape is not None else (int(L ** 0.5), int(L ** 0.5))
        x = input if self.without_pointwise else self.value_proj(input)
        x = x.reshape(N, H, W, -1)
        if self.dw_kernel_size is not None:
            omi = self.offset_mask_dw(input.view(N, H, W, C).permute(0, 3, 1, 2)).permute(0, 2, 3, 1).reshape(N, L, C)
        else:
            omi = input
        offset_mask = self.offset_mask(omi).reshape(N, H, W, -1)
        x_proj = x
        dtype = x.dtype
        geo = (self.kernel_size, self.kernel_size, self.stride, self.stride, self.pad, self.pad, self.dilation,
               self.dilation, self.group, self.group_channels, self.offset_scale)
        if self.core_fp32 and dtype in (torch.float16, torch.bfloat16):
            with torch.autocast(device_type=input.device.type, enabled=False):
                x = dcnv4_core_pytorch(x.float(), offset_mask.float(), *geo, self.remove_center).type(dtype)
        else:
            x = dcnv4_core_pytorch(x, offset_mask.type(dtype), *geo, self.remove_center)
        if self.center_feature_scale:
            center_feature_scale = self.center_feature_scale_module(
                x, self.center_feature_scale_proj_weight, self.center_feature_scale_proj_bias)
            center_feature_scale = center_feature_scale[..., None].repeat(
                1, 1, 1, 1, self.channels // self.group).flatten(-2)
            x = x * (1 - center_feature_scale) + x_proj * center_feature_scale
        x = x.reshape(N, L, -1)
        return x if self.without_pointwise else self.output_proj(x)
