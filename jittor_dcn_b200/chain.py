"""Chained inference (SURVEY.md 8f.2): consecutive `relu(bn(dcn(x)))` stages (train.py:167-170, 329-332) with
channels-last activations BETWEEN the engine layers.

Every stage is one `dcn_layer_forward_chained` call: offset conv + DCN forward on the engine, eval-mode BatchNorm
folded into weight / bias, ReLU in the epilogue (DCN_FLAG_RELU_OUT), and the epilogue writes straight into the framed
channels-last staging copy of the NEXT stage, which therefore runs with DCN_FLAG_XT_STAGED.  Only the first stage
stages its NCHW input and only the last one writes NCHW: one layout pass per network instead of one per layer.
Inference only (training-mode BatchNorm needs the statistics of the complete output before anything is normalised).
"""
import ctypes

import torch
import torch.nn as nn

from . import _lib
from .functional import _dev_ready, _run
from .torch_module import fuse_eval_bn_relu


class ChainedDeformStages(nn.Module):
    def __init__(self, stages):
        """stages: [(TorchDeformConv2d, nn.BatchNorm2d in eval mode), ...] in execution order."""
        super().__init__()
        self.layers = nn.ModuleList([fuse_eval_bn_relu(layer, bn) for layer, bn in stages])
        self._plan = None

    def _build(self, x):
        lib = _lib.load()
        B, C, H, W = (int(v) for v in x.shape)
        plan = []
        for layer in self.layers:
            flags = layer.engine_flags | _lib.FLAG_RELU_OUT
            shp = _lib.make_shape(B, C, layer.out_channels, H, W, layer.kernel_size, layer.stride, layer.padding,
                                  layer.variant, _lib.OPERAND_FP32, flags)
            if _lib.path_name(shp, _lib.PHASE_LAYER_FORWARD) != "umma":
                raise _lib.DcnError(f"chained inference needs every stage on the tensor path; {tuple(x.shape)} -> "
                                    f"{layer} is not")
            Ho, Wo = _lib.output_hw(shp)
            need = int(lib.dcn_workspace_bytes(ctypes.byref(shp), _lib.PHASE_LAYER_FORWARD))
            ws = torch.empty(need, dtype=torch.uint8, device=x.device)
            off = torch.empty((B, 2 * layer.N, Ho, Wo), dtype=torch.float32, device=x.device)
            plan.append(dict(shape=shp, ws=ws, off=off, out_hw=(Ho, Wo)))
            C, H, W = layer.out_channels, Ho, Wo
        for st in plan[1:]:     # the frame of every chained input is zeroed once; the epilogues write interior pixels only
            _run("dcn_staged_input_clear", x.device, st["shape"], (st["ws"],))
        self._plan = (tuple(x.shape), x.device, plan)
        return plan

    @torch.no_grad()
    def forward(self, x):
        if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 4:
            raise ValueError("ChainedDeformStages expects a float32 NCHW CUDA tensor")
        x = _dev_ready(x)
        plan = self._plan[2] if self._plan and self._plan[0] == tuple(x.shape) and self._plan[1] == x.device \
            else self._build(x)
        last = len(plan) - 1
        out = None
        for i, (layer, st) in enumerate(zip(self.layers, plan)):
            shp = st["shape"]
            shp.flags = layer.engine_flags | _lib.FLAG_RELU_OUT | (_lib.FLAG_XT_STAGED if i > 0 else 0)
            src = x if i == 0 else st["ws"]           # chained stages never read `x`: their input is staged
            ow, ob = layer.offset_conv.weight, layer.offset_conv.bias
            if i < last:
                _run("dcn_layer_forward_chained", x.device, shp,
                     (plan[i + 1]["shape"], src, ow, ob, layer.weight, layer.bias, st["off"], plan[i + 1]["ws"]),
                     ws=st["ws"])
            else:
                Ho, Wo = st["out_hw"]
                out = torch.empty((shp.B, shp.O, Ho, Wo), dtype=torch.float32, device=x.device)
                _run("dcn_layer_forward", x.device, shp, (src, ow, ob, layer.weight, layer.bias, st["off"], out),
                     ws=st["ws"])
        return out
