"""`DeformRoIPool` / `DeformPSRoIPool` — the reference's two RoI modules (deform_conv.py:83-157, 160-241; SURVEY.md 8f.4)
on the engine, PyTorch-hosted (the reference classes are Jittor modules; `execute` is aliased to `forward`).

Only `output_size == 1` is accepted: both reference modules sum the per-bin values over the bin axis and then reshape
`[num_rois, C]` to `[num_rois, C, pooled_h, pooled_w]` (deform_conv.py:137-157, 236-241), which raises for any other
size — there is no behaviour to reproduce.  Constructor arguments, their defaults and the dead ones (`sampling_ratio`,
`group_size`) are the reference's.
"""
import torch
import torch.nn as nn

from . import _lib
from .functional import _dev_ready, _run


class _RoIPoolFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, features, rois, offsets, kind, spatial_scale, trans_std, no_trans):
        if not features.is_cuda:
            raise _lib.DcnError("jittor_dcn_b200 RoI pooling needs CUDA tensors: there is no CPU path")
        f, r = _dev_ready(features), _dev_ready(rois.to(features.device))
        o = None if offsets is None else _dev_ready(offsets.to(features.device).reshape(rois.shape[0], -1)[:, :2])
        B, C, H, W = f.shape
        R = r.shape[0]
        out = torch.empty((R, C), dtype=torch.float32, device=f.device)
        _run("dcn_roi_pool_forward", f.device, None,
             (kind, B, C, H, W, R, f, r, o, float(spatial_scale), float(trans_std), int(no_trans), out))
        ctx.save_for_backward(f, r, o if o is not None else torch.empty(0, device=f.device))
        ctx.cfg = (kind, spatial_scale, trans_std, no_trans, offsets is not None, None if offsets is None else offsets.shape)
        return out.view(R, C, 1, 1)

    @staticmethod
    def backward(ctx, grad_out):
        f, r, o = ctx.saved_tensors
        kind, spatial_scale, trans_std, no_trans, has_off, off_shape = ctx.cfg
        B, C, H, W = f.shape
        R = r.shape[0]
        g = _dev_ready(grad_out.reshape(R, C))
        gf = torch.empty_like(f) if ctx.needs_input_grad[0] else None
        go = torch.empty((R, 2), dtype=torch.float32, device=f.device) if (has_off and ctx.needs_input_grad[2]) else None
        _run("dcn_roi_pool_backward", f.device, None,
             (kind, B, C, H, W, R, f, r, o if has_off else None, float(spatial_scale), float(trans_std), int(no_trans),
              g, gf, go))
        if go is not None:
            full = torch.zeros(off_shape, dtype=torch.float32, device=f.device).reshape(R, -1)
            full[:, :2] = go
            go = full.reshape(off_shape)
        return gf, None, go, None, None, None, None


def _one_by_one(output_size, who):
    size = output_size if isinstance(output_size, tuple) else (output_size, output_size)
    if tuple(int(v) for v in size) != (1, 1):
        raise ValueError(
            f"{who}: only output_size 1 is defined — the reference sums over the bin axis and then reshapes "
            "[num_rois, C] to [num_rois, C, pooled_h, pooled_w] (deform_conv.py:137-157 / 236-241), which fails for any "
            "other size")
    return (1, 1)


class DeformRoIPool(nn.Module):
    """deform_conv.py:83-157.  features [B,C,H,W], rois [R,5] = (batch index, x1, y1, x2, y2), offsets [R,1,2]
    (fractions of the roi extent) -> [R,C,1,1]."""

    def __init__(self, output_size, spatial_scale=1.0, sampling_ratio=1):
        super().__init__()
        self.output_size = _one_by_one(output_size, "DeformRoIPool")
        self.spatial_scale = spatial_scale
        self.sampling_ratio = sampling_ratio      # dead in the reference as well

    def forward(self, features, rois, offsets):
        return _RoIPoolFunction.apply(features, rois, offsets, _lib.ROI_POOL, self.spatial_scale, 1.0, False)

    execute = forward


class DeformPSRoIPool(nn.Module):
    """deform_conv.py:160-241.  offsets [R,2] (x, y of part 0), scaled by the roi extent and `trans_std`; ignored with
    `no_trans`.  With one bin every output channel reads the input channel of the same index (:224-226)."""

    def __init__(self, output_size, spatial_scale=1.0, sampling_ratio=1, no_trans=False, group_size=1, part_size=None,
                 trans_std=0.1):
        super().__init__()
        self.output_size = _one_by_one(output_size, "DeformPSRoIPool")
        self.spatial_scale = spatial_scale
        self.sampling_ratio = sampling_ratio
        self.no_trans = no_trans
        self.group_size = group_size
        self.part_size = _one_by_one(part_size, "DeformPSRoIPool(part_size)") if part_size else self.output_size
        self.trans_std = trans_std

    def forward(self, features, rois, offsets=None):
        if offsets is None and not self.no_trans:
            raise ValueError("DeformPSRoIPool: offsets are required unless no_trans=True")
        return _RoIPoolFunction.apply(features, rois, None if self.no_trans else offsets, _lib.PSROI_POOL,
                                      self.spatial_scale, self.trans_std, self.no_trans)

    execute = forward
