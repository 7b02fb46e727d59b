"""DCNv3 as InternImage writes it in PyTorch.  TEST INFRA: the product never imports it.

``dcnv3_core_pytorch`` restates the grid_sample composition of InternImage's ``ops_dcnv3/functions/dcnv3_func.py``;
``dcnv3_core_pixels`` is the same operator on exact pixel coordinates, whose float64 autograd is the reference for
the output and the gradients of input, offset and mask (see its docstring for why).  One deliberate
difference: the original pads with ``F.pad(input, [0, 0, pad_h, pad_h, pad_w, pad_w])``, which pads the width by
pad_h and the height by pad_w (the same thing in every InternImage model, where pad_h == pad_w).  The CUDA extension
pads the height by pad_h, and so does this restatement, so rectangular paddings are pinned to the CUDA semantics.
``points_loop`` evaluates the same operator sample by sample from the coordinate formula, and ``DCNv3Ref`` restates the
module of ``ops_dcnv3/modules/dcnv3.py`` on the composition, with the softmax of the mask outside the core.
"""
import math

import torch
import torch.nn.functional as F
from torch import nn
from torch.nn.init import constant_, xavier_uniform_


def _get_reference_points(spatial_shapes, device, kernel_h, kernel_w, dilation_h, dilation_w, stride_h, stride_w,
                          dtype):
    _, H_, W_, _ = spatial_shapes
    H_out = (H_ - (dilation_h * (kernel_h - 1) + 1)) // stride_h + 1
    W_out = (W_ - (dilation_w * (kernel_w - 1) + 1)) // stride_w + 1
    ref_y, ref_x = torch.meshgrid(
        torch.linspace((dilation_h * (kernel_h - 1)) // 2 + 0.5,
                       (dilation_h * (kernel_h - 1)) // 2 + 0.5 + (H_out - 1) * stride_h,
                       H_out, dtype=dtype, device=device),
        torch.linspace((dilation_w * (kernel_w - 1)) // 2 + 0.5,
                       (dilation_w * (kernel_w - 1)) // 2 + 0.5 + (W_out - 1) * stride_w,
                       W_out, dtype=dtype, device=device), indexing="ij")
    ref_y = ref_y.reshape(-1)[None] / H_
    ref_x = ref_x.reshape(-1)[None] / W_
    return torch.stack((ref_x, ref_y), -1).reshape(1, H_out, W_out, 1, 2)


def _generate_dilation_grids(spatial_shapes, kernel_h, kernel_w, dilation_h, dilation_w, group, device, dtype):
    _, H_, W_, _ = spatial_shapes
    x, y = torch.meshgrid(
        torch.linspace(-((dilation_w * (kernel_w - 1)) // 2),
                       -((dilation_w * (kernel_w - 1)) // 2) + (kernel_w - 1) * dilation_w,
                       kernel_w, dtype=dtype, device=device),
        torch.linspace(-((dilation_h * (kernel_h - 1)) // 2),
                       -((dilation_h * (kernel_h - 1)) // 2) + (kernel_h - 1) * dilation_h,
                       kernel_h, dtype=dtype, device=device), indexing="ij")
    grid = torch.stack([x / W_, y / H_], -1).reshape(-1, 1, 2).repeat(1, group, 1).permute(1, 0, 2)
    return grid.reshape(1, 1, 1, group * kernel_h * kernel_w, 2)


def dcnv3_core_pytorch(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                       dilation_w, group, group_channels, offset_scale):
    input = F.pad(input, [0, 0, pad_w, pad_w, pad_h, pad_h])   # (C), W, H: see the module docstring
    N_, H_in, W_in, _ = input.shape
    _, H_out, W_out, _ = offset.shape
    ref = _get_reference_points(input.shape, input.device, kernel_h, kernel_w, dilation_h, dilation_w, stride_h,
                                stride_w, input.dtype)
    grid = _generate_dilation_grids(input.shape, kernel_h, kernel_w, dilation_h, dilation_w, group, input.device,
                                    input.dtype)
    spatial_norm = torch.tensor([W_in, H_in], dtype=input.dtype).reshape(1, 1, 1, 2).repeat(
        1, 1, 1, group * kernel_h * kernel_w).to(input.device)
    sampling_locations = (ref + grid * offset_scale).repeat(N_, 1, 1, 1, 1).flatten(3, 4) + \
        offset * offset_scale / spatial_norm
    P_ = kernel_h * kernel_w
    sampling_grids = 2 * sampling_locations - 1
    input_ = input.view(N_, H_in * W_in, group * group_channels).transpose(1, 2).reshape(
        N_ * group, group_channels, H_in, W_in)
    sampling_grid_ = sampling_grids.view(N_, H_out * W_out, group, P_, 2).transpose(1, 2).flatten(0, 1)
    sampling_input_ = F.grid_sample(input_, sampling_grid_, mode='bilinear', padding_mode='zeros',
                                    align_corners=False)
    mask = mask.view(N_, H_out * W_out, group, P_).transpose(1, 2).reshape(N_ * group, 1, H_out * W_out, P_)
    output = (sampling_input_ * mask).sum(-1).view(N_, group * group_channels, H_out * W_out)
    return output.transpose(1, 2).reshape(N_, H_out, W_out, -1).contiguous()


def out_extent(H, W, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w):
    return ((H + 2 * pad_h - (dilation_h * (kernel_h - 1) + 1)) // stride_h + 1,
            (W + 2 * pad_w - (dilation_w * (kernel_w - 1) + 1)) // stride_w + 1)


def sample_coordinates(Ho, Wo, offset, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                       group, offset_scale):
    """Unpadded pixel coordinates (x, y) [N, Ho, Wo, G, P] of every sample, from the formula of the C header."""
    N = offset.shape[0]
    P = kernel_h * kernel_w
    off = offset.reshape(N, Ho, Wo, group, P, 2)
    hw, hh = (dilation_w * (kernel_w - 1)) // 2, (dilation_h * (kernel_h - 1)) // 2
    p = torch.arange(P)
    i, j = p // kernel_h, p % kernel_h                                 # x-major: p = i*kernel_h + j
    wo = torch.arange(Wo).view(1, 1, Wo, 1, 1)
    ho = torch.arange(Ho).view(1, Ho, 1, 1, 1)
    x = wo * stride_w - pad_w + hw + (i * dilation_w - hw + off[..., 0]) * offset_scale
    y = ho * stride_h - pad_h + hh + (j * dilation_h - hh + off[..., 1]) * offset_scale
    return x, y


def points_loop(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                group, group_channels, offset_scale):
    """The operator one sample at a time (bilinear with zero corners outside the image), in float64."""
    input, offset, mask = (torch.as_tensor(t).double() for t in (input, offset, mask))
    N, H, W, C = input.shape
    Ho, Wo = out_extent(H, W, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w)
    P = kernel_h * kernel_w
    xs, ys = sample_coordinates(Ho, Wo, offset, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                                dilation_w, group, offset_scale)
    m = mask.reshape(N, Ho, Wo, group, P)
    out = torch.zeros(N, Ho, Wo, group, group_channels, dtype=torch.float64)
    img = input.reshape(N, H, W, group, group_channels)
    for n in range(N):
        for ho in range(Ho):
            for wo in range(Wo):
                for g in range(group):
                    for p in range(P):
                        x, y = float(xs[n, ho, wo, g, p]), float(ys[n, ho, wo, g, p])
                        x0, y0 = math.floor(x), math.floor(y)
                        fx, fy = x - x0, y - y0
                        val = torch.zeros(group_channels, dtype=torch.float64)
                        for dy, dx, w in ((0, 0, (1 - fy) * (1 - fx)), (0, 1, (1 - fy) * fx), (1, 0, fy * (1 - fx)),
                                          (1, 1, fy * fx)):
                            if 0 <= y0 + dy < H and 0 <= x0 + dx < W:
                                val += w * img[n, y0 + dy, x0 + dx, g]
                        out[n, ho, wo, g] += m[n, ho, wo, g, p] * val
    return out.reshape(N, Ho, Wo, C)


def dcnv3_core_pixels(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                      dilation_w, group, group_channels, offset_scale):
    """The same operator written on pixel coordinates (the formula of the C header), vectorised and differentiable.
    The gradient reference: dcnv3_core_pytorch reaches the pixel coordinate through a normalisation and back, whose
    float64 rounding can move a coordinate that is exactly an integer (offsets on a 2^-10 grid make many) to the other
    side of it, where the offset gradient is the other one-sided derivative.  Here the coordinate is exact, as in the
    kernels, so both take the same cell."""
    N, H, W, C = input.shape
    Ho, Wo = out_extent(H, W, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w)
    P = kernel_h * kernel_w
    x, y = sample_coordinates(Ho, Wo, offset, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                              dilation_w, group, offset_scale)
    x0, y0 = torch.floor(x).detach(), torch.floor(y).detach()
    fx, fy = x - x0, y - y0
    img = input.reshape(N, H * W, group, group_channels)
    nidx = torch.arange(N).view(N, 1, 1, 1, 1)
    gidx = torch.arange(group).view(1, 1, 1, group, 1)
    out = 0
    for dy, dx, w in ((0, 0, (1 - fy) * (1 - fx)), (0, 1, (1 - fy) * fx), (1, 0, fy * (1 - fx)), (1, 1, fy * fx)):
        yy, xx = y0 + dy, x0 + dx
        valid = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
        idx = (yy.clamp(0, H - 1) * W + xx.clamp(0, W - 1)).long()
        out = out + (w * valid)[..., None] * img[nidx, idx, gidx]
    m = mask.reshape(N, Ho, Wo, group, P)
    return (out * m[..., None]).sum(4).reshape(N, Ho, Wo, C)


def reference(input, offset, mask, geo, grad_out=None, softmax_mask=False):
    """float64 CPU evaluation (dcnv3_core_pixels, which tests/test_dcnv3.py checks against the grid_sample composition,
    the per-point loop and the MSDA reference) -> out, or (out, grad_input, grad_offset, grad_mask).  geo =
    (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels, offset_scale).
    softmax_mask: `mask` holds logits, softmax over each group's points first (grad_mask is the logits' gradient)."""
    x, off, m = (torch.as_tensor(t).detach().cpu().double().requires_grad_(grad_out is not None)
                 for t in (input, offset, mask))
    group, P = geo[8], geo[0] * geo[1]
    mm = F.softmax(m.reshape(m.shape[:3] + (group, P)), -1).reshape(m.shape) if softmax_mask else m
    out = dcnv3_core_pixels(x, off, mm, *geo)
    if grad_out is None:
        return out.detach()
    g = torch.as_tensor(grad_out).detach().cpu().double()
    gx, goff, gm = torch.autograd.grad(out, [x, off, m], g)
    return out.detach(), gx, goff, gm


class _Permute(nn.Module):
    def __init__(self, *dims):
        super().__init__()
        self.dims = dims

    def forward(self, x):
        return x.permute(*self.dims)


class DCNv3Ref(nn.Module):
    """InternImage's DCNv3 module (LayerNorm + GELU in dw_conv, as its defaults) with dcnv3_core_pytorch as its core
    and the softmax of the mask outside it.  core_fp32: under autocast the core runs on float32 operands and its output
    is cast back, as the engine's module does (the composition itself would build its sampling grid in bf16)."""

    def __init__(self, channels=64, kernel_size=3, dw_kernel_size=None, stride=1, pad=1, dilation=1, group=4,
                 offset_scale=1.0, center_feature_scale=False, core_fp32=False):
        super().__init__()
        self.core_fp32 = core_fp32
        dw_kernel_size = dw_kernel_size if dw_kernel_size is not None else kernel_size
        self.offset_scale = offset_scale
        self.channels = channels
        self.kernel_size = kernel_size
        self.stride = stride
        self.dilation = dilation
        self.pad = pad
        self.group = group
        self.group_channels = channels // group
        self.center_feature_scale = center_feature_scale
        self.dw_conv = nn.Sequential(
            nn.Conv2d(channels, channels, kernel_size=dw_kernel_size, stride=1, padding=(dw_kernel_size - 1) // 2,
                      groups=channels),
            nn.Sequential(_Permute(0, 2, 3, 1), nn.LayerNorm(channels, eps=1e-6)),
            nn.GELU())
        self.offset = nn.Linear(channels, group * kernel_size * kernel_size * 2)
        self.mask = nn.Linear(channels, group * kernel_size * kernel_size)
        self.input_proj = nn.Linear(channels, channels)
        self.output_proj = nn.Linear(channels, channels)
        constant_(self.offset.weight.data, 0.)
        constant_(self.offset.bias.data, 0.)
        constant_(self.mask.weight.data, 0.)
        constant_(self.mask.bias.data, 0.)
        xavier_uniform_(self.input_proj.weight.data)
        constant_(self.input_proj.bias.data, 0.)
        xavier_uniform_(self.output_proj.weight.data)
        constant_(self.output_proj.bias.data, 0.)
        if center_feature_scale:
            self.center_feature_scale_proj_weight = nn.Parameter(torch.zeros((group, channels), dtype=torch.float))
            self.center_feature_scale_proj_bias = nn.Parameter(
                torch.tensor(0.0, dtype=torch.float).view((1,)).repeat(group, ))

    def forward(self, input):
        N, H, W, _ = input.shape
        x = self.input_proj(input)
        x_proj = x
        dtype = x.dtype
        x1 = input.permute(0, 3, 1, 2)
        x1 = self.dw_conv(x1)
        offset = self.offset(x1)
        mask = self.mask(x1).reshape(N, H, W, self.group, -1)
        mask = F.softmax(mask, -1).reshape(N, H, W, -1).type(dtype)
        geo = (self.kernel_size, self.kernel_size, self.stride, self.stride, self.pad, self.pad, self.dilation,
               self.dilation, self.group, self.group_channels, self.offset_scale)
        if self.core_fp32 and dtype in (torch.float16, torch.bfloat16):
            with torch.autocast(device_type=input.device.type, enabled=False):
                x = dcnv3_core_pytorch(x.float(), offset.float(), mask.float(), *geo).type(dtype)
        else:
            x = dcnv3_core_pytorch(x, offset, mask, *geo)
        if self.center_feature_scale:
            center_feature_scale = F.linear(x1, self.center_feature_scale_proj_weight,
                                            self.center_feature_scale_proj_bias).sigmoid()
            center_feature_scale = center_feature_scale[..., None].repeat(
                1, 1, 1, 1, self.channels // self.group).flatten(-2)
            x = x * (1 - center_feature_scale) + x_proj * center_feature_scale
        return self.output_proj(x)
