"""`TorchDeformConv2d` — drop-in for the class of the same name in the reference's train.py:70-140.

Same constructor, attributes, parameter names/shapes (state_dict compatible:
``weight``, ``bias``, ``offset_conv.weight``, ``offset_conv.bias``) and initialisation
(train.py:87-93).  ``forward`` keeps the companion offset convolution as a framework conv
(train.py:98) and hands everything after it (train.py:102-140 and its autograd) to the
B200 engine.
"""
import math

import torch
import torch.nn as nn

from . import _lib
from .functional import (batch_norm_relu, batch_norm_relu_staged, deform_conv2d, deform_conv2d_v1, deform_layer,
                         deform_layer_framed, layer_supported, modulated_deform_layer, modulated_layer_supported,
                         stem_conv, stem_conv_supported)


class TorchDeformConv2d(nn.Module):
    variant = _lib.VARIANT_TORCH

    def __init__(self, in_channels, out_channels, kernel_size=3, stride=1, padding=1, bias=True):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = kernel_size if isinstance(kernel_size, tuple) else (kernel_size, kernel_size)
        self.stride = stride if isinstance(stride, tuple) else (stride, stride)
        self.padding = padding if isinstance(padding, tuple) else (padding, padding)
        self.N = self.kernel_size[0] * self.kernel_size[1]
        self.operand = _lib.OPERAND_FP32
        self.engine_flags = 0
        # True: a private scratch buffer of backward-phase size lives from forward to backward so
        # that the backward pass reuses the staged channels-last copy of x (no second transpose);
        # costs device memory between the two passes, saves one full pass over x
        self.keep_staged_input = False
        # True (default): when the shape allows it, the companion offset convolution runs on the engine as well
        # (a plain mode of the tcgen05 kernels, SURVEY 8f.1) and the whole layer is ONE autograd node; otherwise —
        # or for CPU inputs, bf16 operands, unsupported channel counts — offset_conv stays a framework convolution
        self.engine_offset_conv = True

        # companion offset conv: C -> 2N, same k/s/p (train.py:80-85)
        self.offset_conv = nn.Conv2d(in_channels, 2 * self.N, kernel_size=self.kernel_size,
                                     stride=self.stride, padding=self.padding)
        # He-style normal init of the main weight, zero bias (train.py:87-90)
        std = math.sqrt(2.0 / (in_channels * self.kernel_size[0] * self.kernel_size[1]))
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels, *self.kernel_size))
        nn.init.normal_(self.weight, mean=0.0, std=std)
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None
        # offsets start at zero (train.py:92-93)
        nn.init.zeros_(self.offset_conv.weight)
        nn.init.zeros_(self.offset_conv.bias)

    def _whole_layer_on_engine(self, x):
        return (self.engine_offset_conv and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4
                and self.operand == _lib.OPERAND_FP32 and self.weight.is_cuda
                and layer_supported(x.shape, self.out_channels, self.kernel_size, self.stride, self.padding,
                                    self.variant, self.operand, self.engine_flags))

    def forward(self, x):
        if self._whole_layer_on_engine(x):
            return deform_layer(x, self.offset_conv.weight, self.offset_conv.bias, self.weight, self.bias,
                                self.kernel_size, self.stride, self.padding, self.variant, self.engine_flags,
                                keep_staged=self.keep_staged_input and torch.is_grad_enabled())
        offset = self.offset_conv(x)
        return deform_conv2d(x, offset, self.weight, self.bias, self.kernel_size, self.stride,
                             self.padding, self.variant, self.operand, self.engine_flags,
                             keep_staged=self.keep_staged_input and torch.is_grad_enabled())

    def consumer_cfg(self):
        """What a staged post-op needs to know about this layer to write its staged input (SURVEY 8f.2)."""
        return (self.out_channels, self.kernel_size, self.stride, self.padding, self.variant, self.engine_flags)

    def forward_staged(self, xt, in_hw):
        """forward on an input that a staged post-op (BatchNormReLU2d.forward_staged) already wrote as this layer's
        channels-last staging copy; in_hw = (H, W) of the logical input."""
        return deform_layer_framed(xt, (self.in_channels, int(in_hw[0]), int(in_hw[1])), self.offset_conv.weight,
                                   self.offset_conv.bias, self.weight, self.bias, self.kernel_size, self.stride,
                                   self.padding, self.variant, self.engine_flags)

    def extra_repr(self):
        return (f"{self.in_channels}, {self.out_channels}, kernel_size={self.kernel_size}, "
                f"stride={self.stride}, padding={self.padding}, bias={self.bias is not None}")


class TorchDeformConv2dJittorSemantics(TorchDeformConv2d):
    """PyTorch-hosted module with the Jittor operator's semantics (deform_conv.py:56-81):
    normalisation by the OUTPUT extent and (n, c)-ordered columns."""
    variant = _lib.VARIANT_JITTOR


def fuse_eval_bn_relu(layer, bn):
    """`relu(bn(layer(x)))` of the reference's detector (train.py:167-170, 329-332) for INFERENCE as one engine call:
    returns a copy of `layer` whose weight / bias carry the eval-mode BatchNorm (running statistics) and whose forward
    epilogue applies the ReLU (DCN_FLAG_RELU_OUT, SURVEY 8f.2) — no separate post-op pass over the output.
    The offset branch is untouched (BatchNorm acts on the layer's output only)."""
    if bn.training:
        raise ValueError("fuse_eval_bn_relu folds RUNNING statistics: call bn.eval() first")
    import copy
    fused = copy.deepcopy(layer)
    with torch.no_grad():
        inv = torch.rsqrt(bn.running_var + bn.eps)
        scale = inv * (bn.weight if bn.weight is not None else 1.0)
        shift = (bn.bias if bn.bias is not None else 0.0) - bn.running_mean * scale
        fused.weight.mul_(scale.view(-1, 1, 1, 1))
        old_bias = fused.bias if fused.bias is not None else torch.zeros_like(scale)
        fused.bias = nn.Parameter(old_bias * scale + shift)
    fused.engine_flags = layer.engine_flags | _lib.FLAG_RELU_OUT
    return fused


class BatchNormReLU2d(nn.BatchNorm2d):
    """`relu(bn(x))` of the reference's detector (train.py:167-170, 329-332) as one module: the parameters,
    buffers and state-dict keys of ``nn.BatchNorm2d`` (``weight``, ``bias``, ``running_mean``, ``running_var``,
    ``num_batches_tracked``), evaluated by the engine's batch-norm kernels with the ReLU fused (SURVEY 8f.2).
    The framework's kernels run one CTA per channel and take most of the detector step on B200."""

    def forward(self, x):
        if x.dim() != 4 or x.dtype != torch.float32:
            raise ValueError("BatchNormReLU2d expects a float32 NCHW tensor")
        use_batch_stats = self.training or not self.track_running_stats
        if use_batch_stats and x.numel() // x.shape[1] == 1:
            # same refusal as nn.BatchNorm2d (torch.nn.functional._verify_batch_size)
            raise ValueError(f"Expected more than 1 value per channel when training, got input size {x.size()}")
        momentum = 0.0 if self.momentum is None else self.momentum
        if self.training and self.track_running_stats and self.num_batches_tracked is not None:
            self.num_batches_tracked.add_(1)
            if self.momentum is None:
                momentum = 1.0 / float(self.num_batches_tracked)
        return self._apply_op(x, use_batch_stats, momentum, None)

    def forward_staged(self, x, consumer):
        """relu(bn(x)) written directly as the staged channels-last input of `consumer` (a TorchDeformConv2d): returns
        the tensor to hand to consumer.forward_staged (SURVEY 8f.2; csrc/dcn_bn.cu: bn_stage_kernel)."""
        if x.dim() != 4 or x.dtype != torch.float32 or not x.is_cuda:
            raise ValueError("BatchNormReLU2d.forward_staged expects a float32 NCHW CUDA tensor")
        use_batch_stats = self.training or not self.track_running_stats
        momentum = 0.0 if self.momentum is None else self.momentum
        if self.training and self.track_running_stats and self.num_batches_tracked is not None:
            self.num_batches_tracked.add_(1)
            if self.momentum is None:
                momentum = 1.0 / float(self.num_batches_tracked)
        return self._apply_op(x, use_batch_stats, momentum, consumer.consumer_cfg())

    def _apply_op(self, x, use_batch_stats, momentum, consumer_cfg):
        rm = self.running_mean if self.track_running_stats else None
        rv = self.running_var if self.track_running_stats else None
        if consumer_cfg is not None:
            return batch_norm_relu_staged(x, self.weight, self.bias, rm, rv, use_batch_stats, momentum, self.eps,
                                          consumer_cfg)
        return batch_norm_relu(x, self.weight, self.bias, rm, rv, use_batch_stats, momentum, self.eps)


class StemConv2d(nn.Conv2d):
    """``nn.Conv2d`` (same parameters, initialisation and state-dict keys) whose 3 x 3 / stride 1 / padding 1 case on
    the network input — the detector's ``conv1 = Conv2d(1, 16, 3, 1, 1)``, train.py:145 / :307 — runs on the engine's
    two streaming kernels (csrc/dcn_stem.cu); every other configuration, a CPU tensor or an input that wants a
    gradient takes the framework's convolution unchanged."""

    def forward(self, x):
        if (self.stride == (1, 1) and self.padding == (1, 1) and self.dilation == (1, 1) and self.groups == 1
                and self.padding_mode == "zeros" and stem_conv_supported(x, self.weight)):
            return stem_conv(x, self.weight, self.bias)
        return super().forward(x)


class TorchvisionDeformConv2d(nn.Module):
    """Drop-in for ``torchvision.ops.DeformConv2d``: the same constructor, attributes, parameters (``weight``,
    ``bias``: state dicts load unchanged), initialisation (``reset_parameters``) and ``forward(input, offset,
    mask=None)``.  ``mask=None`` is deformable convolution v1, a mask [B, kh*kw, H_out, W_out] makes it the
    modulated form (DCNv2); both run on the engine (``deform_conv2d_v1``).  One offset group; ``dilation`` and
    ``groups`` other than 1 are refused at construction."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True):
        super().__init__()
        if in_channels % groups != 0:
            raise ValueError("in_channels must be divisible by groups")
        if out_channels % groups != 0:
            raise ValueError("out_channels must be divisible by groups")
        if groups != 1:
            raise ValueError(f"TorchvisionDeformConv2d: groups={groups} is not supported (only 1)")
        if _lib._pair(dilation) != (1, 1):
            raise ValueError(f"TorchvisionDeformConv2d: dilation={dilation} is not supported (only 1)")
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _lib._pair(kernel_size)
        self.stride = _lib._pair(stride)
        self.padding = _lib._pair(padding)
        self.dilation = _lib._pair(dilation)
        self.groups = groups
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels // groups, self.kernel_size[0],
                                               self.kernel_size[1]))
        if bias:
            self.bias = nn.Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        # the same draws, in the same order, as torchvision.ops.DeformConv2d.reset_parameters
        nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        if self.bias is not None:
            fan_in, _ = nn.init._calculate_fan_in_and_fan_out(self.weight)
            bound = 1 / math.sqrt(fan_in)
            nn.init.uniform_(self.bias, -bound, bound)

    def forward(self, input, offset, mask=None):
        return deform_conv2d_v1(input, offset, self.weight, self.bias, stride=self.stride, padding=self.padding,
                                dilation=self.dilation, mask=mask)

    def extra_repr(self):
        s = f"{self.in_channels}, {self.out_channels}, kernel_size={self.kernel_size}, stride={self.stride}"
        s += f", padding={self.padding}" if self.padding != (0, 0) else ""
        s += f", dilation={self.dilation}" if self.dilation != (1, 1) else ""
        s += f", groups={self.groups}" if self.groups != 1 else ""
        s += ", bias=False" if self.bias is None else ""
        return s


class ModulatedDeformConv2dPack(nn.Module):
    """Drop-in for mmcv's ``ModulatedDeformConv2dPack`` (the ``DCNv2`` layer of mmdet's ResNet backbones): the same
    constructor, parameters (``weight``, ``bias``, ``conv_offset.weight``, ``conv_offset.bias``: mmcv checkpoints load
    unchanged) and initialisation (mmcv's ``init_weights``).  ``conv_offset`` has 3N = 3 * kh * kw outputs; channels
    [0, 2N) are the offsets and channels [2N, 3N) one mask logit per tap, mask = sigmoid(logit).

    ``forward`` runs the whole layer (that conv, the sigmoid and the modulated span) as ONE autograd node on the
    engine when the input is a float32 CUDA tensor and ``modulated_layer_supported`` covers the shape; otherwise, or
    with ``engine_offset_conv = False``, it computes mmcv's composition: ``conv_offset`` as a framework convolution,
    chunk / cat / sigmoid, and ``deform_conv2d_v1(..., mask=)`` as the span.  One offset group; ``dilation``,
    ``groups`` and ``deform_groups`` other than 1 are refused at construction."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 deform_groups=1, bias=True):
        super().__init__()
        if _lib._pair(dilation) != (1, 1):
            raise ValueError(f"ModulatedDeformConv2dPack: dilation={dilation} is not supported (only 1)")
        if groups != 1:
            raise ValueError(f"ModulatedDeformConv2dPack: groups={groups} is not supported (only 1)")
        if deform_groups != 1:
            raise ValueError(f"ModulatedDeformConv2dPack: deform_groups={deform_groups} is not supported (only 1)")
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _lib._pair(kernel_size)
        self.stride = _lib._pair(stride)
        self.padding = _lib._pair(padding)
        self.dilation = _lib._pair(dilation)
        self.groups = groups
        self.deform_groups = deform_groups
        self.engine_flags = 0
        # True (default): the whole layer is one autograd node on the engine when the shape allows it; False: the
        # framework convolution + chunk / cat / sigmoid + the engine's modulated span, as mmcv composes it
        self.engine_offset_conv = True
        # True: a private scratch buffer lives from forward to backward so that the backward pass reuses the staged
        # channels-last copy of x (one pass over x saved, device memory held in between)
        self.keep_staged_input = False
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels // groups, *self.kernel_size))
        if bias:
            self.bias = nn.Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        # the same draws, in the same order, as mmcv: init_weights() in the base constructor, the framework's default
        # initialisation of conv_offset, then init_weights() again (which also zeroes conv_offset)
        self._init_main()
        self.conv_offset = nn.Conv2d(in_channels, deform_groups * 3 * self.kernel_size[0] * self.kernel_size[1],
                                     kernel_size=self.kernel_size, stride=self.stride, padding=self.padding,
                                     dilation=self.dilation, bias=True)
        self.init_weights()

    def _init_main(self):
        n = self.in_channels * self.kernel_size[0] * self.kernel_size[1]
        stdv = 1.0 / math.sqrt(n)
        with torch.no_grad():
            self.weight.uniform_(-stdv, stdv)
            if self.bias is not None:
                self.bias.zero_()

    def init_weights(self):
        self._init_main()
        with torch.no_grad():
            self.conv_offset.weight.zero_()
            self.conv_offset.bias.zero_()

    def _whole_layer_on_engine(self, x):
        return (self.engine_offset_conv and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4
                and self.weight.is_cuda and self.weight.dtype == torch.float32
                and self.conv_offset.weight.dtype == torch.float32
                and modulated_layer_supported(x.shape, self.out_channels, self.kernel_size, self.stride, self.padding,
                                              self.engine_flags))

    def forward(self, x):
        if self._whole_layer_on_engine(x):
            return modulated_deform_layer(x, self.conv_offset.weight, self.conv_offset.bias, self.weight, self.bias,
                                          self.kernel_size, self.stride, self.padding, self.engine_flags,
                                          keep_staged=self.keep_staged_input and torch.is_grad_enabled())
        out = self.conv_offset(x)
        o1, o2, mask = torch.chunk(out, 3, dim=1)
        offset = torch.cat((o1, o2), dim=1)
        mask = torch.sigmoid(mask)
        return deform_conv2d_v1(x, offset, self.weight, self.bias, stride=self.stride, padding=self.padding,
                                dilation=self.dilation, mask=mask)

    def extra_repr(self):
        s = f"{self.in_channels}, {self.out_channels}, kernel_size={self.kernel_size}, stride={self.stride}"
        s += f", padding={self.padding}" if self.padding != (0, 0) else ""
        s += ", bias=False" if self.bias is None else ""
        return s
