"""Tensor-level entry points: torch tensors in, raw device pointers across the C ABI.

PyTorch is used for device memory, streams and autograd plumbing only; all arithmetic of
the operator happens in libdcn_b200.so.
"""
import ctypes

import torch

from . import _lib
from ._lib import (FLAG_ACCUM_GRAD_X, FLAG_FORCE_SIMT, FLAG_NO_GRAD_X, FLAG_RELU_OUT, FLAG_XT_STAGED, OPERAND_BF16, OPERAND_FP32,
                   PHASE_BACKWARD, PHASE_FORWARD, PHASE_LAYER_BACKWARD, PHASE_LAYER_BACKWARD_MODULATED,
                   PHASE_LAYER_FORWARD, PHASE_LAYER_FORWARD_MODULATED, VARIANT_DCNV1, VARIANT_JITTOR, VARIANT_TORCH)

_workspaces = {}
_captured = []   # scratch buffers whose addresses are baked into CUDA graphs: alive until clear_workspaces()


def _workspace(device, stream_id, nbytes):
    """Caller-owned scratch, one growing buffer per (device, stream).

    While the stream is being captured into a CUDA graph the call gets a PRIVATE buffer that is never freed or
    handed out again (a replay reads and writes the captured address; the shared cache may be re-allocated by a
    later, larger eager call).  clear_workspaces() drops everything — only once such graphs are gone."""
    if torch.cuda.is_current_stream_capturing():
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _captured.append(ws)
        return ws
    key = (device.index, stream_id)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def clear_workspaces():
    """Release the cached scratch buffers (all devices / streams) and the ones captured CUDA graphs point at.
    Call only when no such graph will be replayed again."""
    _workspaces.clear()
    del _captured[:]


def _dev_ready(t, dtype=torch.float32):
    """Dense, 16-byte aligned tensor of the wanted dtype on its current CUDA device."""
    if t is None:
        return None
    if t.dtype != dtype:
        t = t.to(dtype)
    t = t.contiguous()
    if t.data_ptr() % 16:
        t = t.clone(memory_format=torch.contiguous_format)
    return t


def _compute_device(x):
    if x.is_cuda:
        return x.device
    if not torch.cuda.is_available():
        raise _lib.DcnError("jittor_dcn_b200 needs a CUDA device (B200, sm_100a): there is no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def _to_device(t, dev):
    """Host tensors are staged through pinned memory (the reference feeds CPU tensors,
    train.py:239); CUDA tensors are used in place."""
    if t is None or t.device == dev:
        return t
    if t.device.type == "cpu":
        t = t.detach().contiguous()
        try:
            t = t.pin_memory()
        except RuntimeError:
            pass
        return t.to(dev, non_blocking=True)
    return t.to(dev)


def _shape_of(x, weight, kernel_size, stride, padding, variant, operand, flags):
    B, C, H, W = x.shape
    O = weight.shape[0]
    return _lib.make_shape(B, C, O, H, W, kernel_size, stride, padding, variant, operand, flags)


def staged_workspace(x, weight, kernel_size=3, stride=1, padding=1, variant=VARIANT_TORCH,
                     operand=OPERAND_FP32, flags=0):
    """A private scratch buffer big enough for BOTH phases of one layer call, or None when either
    phase would not run on the tensor path.  Passing it to dcn_forward and then to dcn_backward
    (xt_staged=True) lets the backward pass reuse the staged copy of x (DCN_FLAG_XT_STAGED)."""
    lib = _lib.load()
    shp = _shape_of(x, weight, kernel_size, stride, padding, variant, operand, flags)
    names = [_lib.path_name(shp, ph) for ph in (PHASE_FORWARD, PHASE_BACKWARD)]
    if names not in (["umma", "umma"], ["gemm", "gemm"]):      # both keep the forward's staging at the workspace head
        return None
    need = max(lib.dcn_workspace_bytes(ctypes.byref(shp), PHASE_FORWARD),
               lib.dcn_workspace_bytes(ctypes.byref(shp), PHASE_BACKWARD))
    return torch.empty(need, dtype=torch.uint8, device=x.device)


def _run(entry, dev, shp, args, phase=None, ws=None):
    """lib.<entry>(shp, *args[, workspace, workspace_bytes], stream) under the device guard of `dev` on its current
    stream, then its status checked.  shp: the shape structure the entry point takes first, None for one that takes
    none.  Tensors pass as their device pointers, ctypes structures by reference, None as NULL and everything else as
    it is.  The call takes a workspace when `ws` or `phase` is given: `ws`, or else the cached scratch buffer that
    `phase` needs for `shp`."""
    lib = _lib.load()
    args = [ctypes.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else
            ctypes.byref(a) if isinstance(a, ctypes.Structure) else a for a in (args if shp is None else (shp, *args))]
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        if ws is None and phase is not None:
            ws = _workspace(dev, stream.cuda_stream, lib.dcn_workspace_bytes(args[0], phase))
        if ws is not None:
            args += [ctypes.c_void_p(ws.data_ptr()), ws.numel()]
        rc = getattr(lib, entry)(*args, ctypes.c_void_p(stream.cuda_stream))
    _lib.check(rc, entry)


def dcn_forward(x, offset, weight, bias, kernel_size=3, stride=1, padding=1, variant=VARIANT_TORCH,
                operand=OPERAND_FP32, flags=0, ws=None):
    """out[B,O,Ho,Wo] = engine forward on CUDA tensors (no autograd)."""
    return _span_forward(x, offset, None, weight, bias, kernel_size, stride, padding, variant, operand, flags, ws)


def dcn_backward(x, offset, weight, grad_out, has_bias, kernel_size=3, stride=1, padding=1,
                 variant=VARIANT_TORCH, operand=OPERAND_FP32, flags=0, need_grad_x=True, ws=None,
                 xt_staged=False, grad_x=None):
    """-> grad_x (or None), grad_offset, grad_weight, grad_bias (or None); all float32.
    ws / xt_staged: the buffer from staged_workspace() that the matching dcn_forward used.
    grad_x: an existing float32 gradient of x's shape to ACCUMULATE into (DCN_FLAG_ACCUM_GRAD_X; e.g. the
    term the companion offset conv contributes); without it the flag is refused — the library would add into
    whatever the freshly allocated output buffer happens to hold."""
    gx, goff, _, gw, gb = _span_backward(x, offset, None, weight, grad_out, has_bias, kernel_size, stride, padding,
                                         variant, operand, flags, need_grad_x, ws, xt_staged, grad_x)
    return gx, goff, gw, gb


# ---- modulated deformable convolution (DCNv2): DCNv1 sampling, every sample scaled by mask[b, n, p] ----------------
def dcn_forward_modulated(x, offset, mask, weight, bias, kernel_size=3, stride=1, padding=1, operand=OPERAND_FP32,
                          flags=0, ws=None):
    """out[B,O,Ho,Wo] = modulated DCNv1 forward on CUDA tensors (no autograd); mask [B, kh*kw, Ho, Wo] float32
    (torchvision's tap order, any values).  Arguments otherwise as dcn_forward with variant = VARIANT_DCNV1."""
    return _span_forward(x, offset, mask, weight, bias, kernel_size, stride, padding, VARIANT_DCNV1, operand, flags, ws)


def dcn_backward_modulated(x, offset, mask, weight, grad_out, has_bias, kernel_size=3, stride=1, padding=1,
                           operand=OPERAND_FP32, flags=0, need_grad_x=True, ws=None, xt_staged=False, grad_x=None):
    """-> grad_x (or None), grad_offset, grad_mask, grad_weight, grad_bias (or None); all float32.
    Arguments as dcn_backward with variant = VARIANT_DCNV1, plus the forward's mask."""
    return _span_backward(x, offset, mask, weight, grad_out, has_bias, kernel_size, stride, padding, VARIANT_DCNV1,
                          operand, flags, need_grad_x, ws, xt_staged, grad_x)


def _check_mask(mask, shp, Ho, Wo):
    N = shp.kh * shp.kw
    if tuple(mask.shape) != (shp.B, N, Ho, Wo):
        raise ValueError(f"mask shape {tuple(mask.shape)} != {(shp.B, N, Ho, Wo)} ([B, kh*kw, H_out, W_out])")


# the span calls: mask None = unmodulated (dcn_forward / dcn_backward), else DCN_VARIANT_DCNV1 modulated
def _span_forward(x, offset, mask, weight, bias, kernel_size, stride, padding, variant, operand, flags, ws):
    shp = _shape_of(x, weight, kernel_size, stride, padding, variant, operand, flags)
    Ho, Wo = _lib.output_hw(shp)
    N = shp.kh * shp.kw
    if tuple(offset.shape) != (shp.B, 2 * N, Ho, Wo):
        raise ValueError(f"offset shape {tuple(offset.shape)} != {(shp.B, 2 * N, Ho, Wo)}")
    if tuple(weight.shape) != (shp.O, shp.C, shp.kh, shp.kw):
        raise ValueError(f"weight shape {tuple(weight.shape)} != {(shp.O, shp.C, shp.kh, shp.kw)}")
    if mask is not None:
        _check_mask(mask, shp, Ho, Wo)
    act = torch.bfloat16 if operand == OPERAND_BF16 else torch.float32
    x, weight = _dev_ready(x, act), _dev_ready(weight, act)
    offset, mask, bias = _dev_ready(offset), _dev_ready(mask), _dev_ready(bias)
    out = torch.empty((shp.B, shp.O, Ho, Wo), dtype=torch.float32, device=x.device)
    if mask is None:
        _run("dcn_forward", x.device, shp, (x, offset, weight, bias, out), phase=PHASE_FORWARD, ws=ws)
    else:
        _run("dcn_forward_modulated", x.device, shp, (x, offset, mask, weight, bias, out), phase=PHASE_FORWARD, ws=ws)
    return out


def _span_backward(x, offset, mask, weight, grad_out, has_bias, kernel_size, stride, padding, variant, operand, flags,
                   need_grad_x, ws, xt_staged, grad_x):
    """-> grad_x, grad_offset, grad_mask (None without a mask), grad_weight, grad_bias."""
    if grad_x is not None:
        if not need_grad_x:
            raise ValueError("grad_x given but need_grad_x is False")
        if grad_x.dtype != torch.float32 or tuple(grad_x.shape) != tuple(x.shape) or not grad_x.is_contiguous() \
                or grad_x.data_ptr() % 16:
            raise ValueError("grad_x must be a dense, 16-byte aligned float32 tensor of x's shape")
        flags |= FLAG_ACCUM_GRAD_X
    elif flags & FLAG_ACCUM_GRAD_X:
        raise ValueError("FLAG_ACCUM_GRAD_X needs the tensor to accumulate into: pass grad_x=")
    if not need_grad_x:
        flags |= FLAG_NO_GRAD_X
    if xt_staged and ws is not None:
        flags |= FLAG_XT_STAGED
    shp = _shape_of(x, weight, kernel_size, stride, padding, variant, operand, flags)
    Ho, Wo = _lib.output_hw(shp)
    N = shp.kh * shp.kw
    if mask is not None:
        _check_mask(mask, shp, Ho, Wo)
    act = torch.bfloat16 if operand == OPERAND_BF16 else torch.float32
    x, weight, grad_out = _dev_ready(x, act), _dev_ready(weight, act), _dev_ready(grad_out, act)
    offset, mask = _dev_ready(offset), _dev_ready(mask)
    dev = x.device
    gx = grad_x if grad_x is not None else (torch.empty(x.shape, dtype=torch.float32, device=dev) if need_grad_x else None)
    goff = torch.empty((shp.B, 2 * N, Ho, Wo), dtype=torch.float32, device=dev)
    gw = torch.empty(weight.shape, dtype=torch.float32, device=dev)
    gb = torch.empty((shp.O,), dtype=torch.float32, device=dev) if has_bias else None
    if mask is None:
        gmask = None
        _run("dcn_backward", dev, shp, (x, offset, weight, grad_out, gx, goff, gw, gb), phase=PHASE_BACKWARD, ws=ws)
    else:
        gmask = torch.empty((shp.B, N, Ho, Wo), dtype=torch.float32, device=dev)
        _run("dcn_backward_modulated", dev, shp, (x, offset, mask, weight, grad_out, gx, goff, gmask, gw, gb),
             phase=PHASE_BACKWARD, ws=ws)
    return gx, goff, gmask, gw, gb


# ---- whole layer: companion offset conv + DCN span on the engine (SURVEY 8f.1) -----------------------------------
# The modulated layer (mmcv's ModulatedDeformConv2dPack) shares every body below: its conv has 3N outputs (offsets,
# then one mask logit per tap, the mask being their sigmoid), DCNv1 sampling, and phases of its own.
_PHASES = {False: (PHASE_LAYER_FORWARD, PHASE_LAYER_BACKWARD),
           True: (PHASE_LAYER_FORWARD_MODULATED, PHASE_LAYER_BACKWARD_MODULATED)}


def layer_supported(x_shape, out_channels, kernel_size=3, stride=1, padding=1, variant=VARIANT_TORCH,
                    operand=OPERAND_FP32, flags=0):
    """True when dcn_layer_forward / dcn_layer_backward cover the shape (both phases on the tensor path)."""
    return _layer_supported(x_shape, out_channels, kernel_size, stride, padding, variant, operand, flags, False)


def layer_workspace(x, weight, kernel_size=3, stride=1, padding=1, variant=VARIANT_TORCH, flags=0):
    """One scratch buffer big enough for dcn_layer_forward AND dcn_layer_backward of this layer: handing the same
    buffer to both lets the backward pass reuse the staged copy of x (DCN_FLAG_XT_STAGED)."""
    return _layer_workspace(x, weight, kernel_size, stride, padding, variant, flags, False)


def dcn_offset_conv_forward(x, offset_weight, offset_bias, out_channels, kernel_size=3, stride=1, padding=1,
                            variant=VARIANT_TORCH, flags=0, ws=None, xt_staged=False):
    """offset[B,2N,Ho,Wo] = the companion offset convolution on the engine (a plain mode of the tcgen05 forward
    kernel).  `variant` / out_channels describe the DCN layer the offsets are for: the staged copy of x is laid out
    for it, so a following dcn_forward(..., ws=ws, xt_staged=True) reuses it."""
    return _offset_conv_forward(x, offset_weight, offset_bias, out_channels, kernel_size, stride, padding, variant,
                                flags, ws, xt_staged, False)[0]


def dcn_layer_forward(x, offset_weight, offset_bias, weight, bias, kernel_size=3, stride=1, padding=1,
                      variant=VARIANT_TORCH, flags=0, ws=None):
    """-> (offset, out): offset conv + DCN forward, x staged once (no autograd)."""
    offset, _, out = _layer_forward(x, offset_weight, offset_bias, weight, bias, kernel_size, stride, padding, variant,
                                    flags, ws, False)
    return offset, out


def dcn_layer_backward(x, offset, offset_weight, weight, grad_out, has_offset_bias=True, has_bias=True, kernel_size=3,
                       stride=1, padding=1, variant=VARIANT_TORCH, flags=0, need_grad_x=True, ws=None, xt_staged=False):
    """-> grad_x (or None), grad_offset_weight, grad_offset_bias (or None), grad_weight, grad_bias (or None).
    grad_offset stays inside the workspace; the offset conv's data gradient is accumulated on chip-side buffers."""
    return _layer_backward(x, offset, None, offset_weight, weight, grad_out, has_offset_bias, has_bias, kernel_size,
                           stride, padding, variant, flags, need_grad_x, ws, xt_staged)


def deform_layer(x, offset_weight, offset_bias, weight, bias=None, kernel_size=3, stride=1, padding=1,
                 variant=VARIANT_TORCH, flags=0, keep_staged=False):
    """Differentiable whole layer on the engine (CUDA float32 tensors; check layer_supported() first)."""
    cfg = (_lib._pair(kernel_size), _lib._pair(stride), _lib._pair(padding), variant, flags, bool(keep_staged), False)
    return DeformLayerFunction.apply(x, offset_weight, offset_bias, weight, bias, cfg)


# ---- whole modulated layer: mmcv's ModulatedDeformConv2dPack (3N-channel offset-and-mask conv + DCNv2 span) --------
def modulated_layer_supported(x_shape, out_channels, kernel_size, stride, padding, flags=0):
    """True when dcn_layer_forward_modulated / dcn_layer_backward_modulated cover the shape (fp32, tensor path)."""
    return _layer_supported(x_shape, out_channels, kernel_size, stride, padding, VARIANT_DCNV1, OPERAND_FP32, flags,
                            True)


def modulated_layer_workspace(x, weight, kernel_size, stride, padding, flags=0):
    """One scratch buffer for both modulated layer calls: the backward pass reuses the staged copy of x."""
    return _layer_workspace(x, weight, kernel_size, stride, padding, VARIANT_DCNV1, flags, True)


def dcn_offset_conv_forward_modulated(x, offset_weight, offset_bias, out_channels, kernel_size=3, stride=1, padding=1,
                                      flags=0, ws=None, xt_staged=False):
    """-> (offset [B,2N,Ho,Wo], mask [B,N,Ho,Wo]): the modulated layer's 3N-channel conv on the engine, channels
    [0, 2N) as offsets and sigmoid(channels [2N, 3N)) as the mask (no autograd)."""
    return _offset_conv_forward(x, offset_weight, offset_bias, out_channels, kernel_size, stride, padding,
                                VARIANT_DCNV1, flags, ws, xt_staged, True)


def dcn_layer_forward_modulated(x, offset_weight, offset_bias, weight, bias, kernel_size=3, stride=1, padding=1,
                                flags=0, ws=None):
    """-> (offset, mask, out): offset-and-mask conv + modulated DCN forward, x staged once (no autograd)."""
    return _layer_forward(x, offset_weight, offset_bias, weight, bias, kernel_size, stride, padding, VARIANT_DCNV1,
                          flags, ws, True)


def dcn_layer_backward_modulated(x, offset, mask, offset_weight, weight, grad_out, has_offset_bias=True, has_bias=True,
                                 kernel_size=3, stride=1, padding=1, flags=0, need_grad_x=True, ws=None,
                                 xt_staged=False):
    """-> grad_x (or None), grad_offset_weight, grad_offset_bias (or None), grad_weight, grad_bias (or None).
    offset / mask: what dcn_layer_forward_modulated returned.  The gradients of offset and mask stay in the workspace."""
    return _layer_backward(x, offset, mask, offset_weight, weight, grad_out, has_offset_bias, has_bias, kernel_size,
                           stride, padding, VARIANT_DCNV1, flags, need_grad_x, ws, xt_staged)


def modulated_deform_layer(x, offset_weight, offset_bias, weight, bias=None, kernel_size=3, stride=1, padding=1,
                           flags=0, keep_staged=False):
    """Differentiable whole modulated layer on the engine (CUDA float32 tensors; check modulated_layer_supported()
    first).  offset_weight [3N, C, kh, kw]: offsets, then one mask logit per tap (mmcv's conv_offset)."""
    cfg = (_lib._pair(kernel_size), _lib._pair(stride), _lib._pair(padding), VARIANT_DCNV1, flags & ~FLAG_RELU_OUT,
           bool(keep_staged), True)
    return DeformLayerFunction.apply(x, offset_weight, offset_bias, weight, bias, cfg)


# the layer bodies: modulated False = dcn_layer_* (2N-channel offset conv), True = dcn_layer_*_modulated
def _layer_supported(x_shape, out_channels, kernel_size, stride, padding, variant, operand, flags, modulated):
    B, C, H, W = (int(v) for v in x_shape)
    shp = _lib.make_shape(B, C, int(out_channels), H, W, kernel_size, stride, padding, variant, operand, flags)
    return all(_lib.path_name(shp, ph) == "umma" for ph in _PHASES[modulated])


def _layer_workspace(x, weight, kernel_size, stride, padding, variant, flags, modulated):
    shp = _shape_of(x, weight, kernel_size, stride, padding, variant, OPERAND_FP32, flags)
    return torch.empty(_layer_bytes(shp, modulated), dtype=torch.uint8, device=x.device)


def _layer_bytes(shp, modulated=False):
    """Bytes of one workspace for both calls of the layer; 0 when it does not run on the tensor path."""
    lib = _lib.load()
    return max(lib.dcn_workspace_bytes(ctypes.byref(shp), ph) for ph in _PHASES[modulated])


def _check_offset_weight(offset_weight, shp, modulated):
    n = 3 if modulated else 2
    want = (n * shp.kh * shp.kw, shp.C, shp.kh, shp.kw)
    if tuple(offset_weight.shape) != want:
        raise ValueError(f"offset_weight shape {tuple(offset_weight.shape)} != {want}" +
                         (" (3N outputs: offsets, then one mask logit per tap)" if modulated else ""))


def _offset_conv_forward(x, offset_weight, offset_bias, out_channels, kernel_size, stride, padding, variant, flags, ws,
                         xt_staged, modulated):
    """-> (offset, mask or None)"""
    B, C, H, W = x.shape
    if xt_staged and ws is not None:
        flags |= FLAG_XT_STAGED
    shp = _lib.make_shape(B, C, int(out_channels), H, W, kernel_size, stride, padding, variant, OPERAND_FP32, flags)
    Ho, Wo = _lib.output_hw(shp)
    N = shp.kh * shp.kw
    _check_offset_weight(offset_weight, shp, modulated)
    x, offset_weight, offset_bias = _dev_ready(x), _dev_ready(offset_weight), _dev_ready(offset_bias)
    offset = torch.empty((B, 2 * N, Ho, Wo), dtype=torch.float32, device=x.device)
    if not modulated:
        _run("dcn_offset_conv_forward", x.device, shp, (x, offset_weight, offset_bias, offset),
             phase=PHASE_LAYER_FORWARD, ws=ws)
        return offset, None
    mask = torch.empty((B, N, Ho, Wo), dtype=torch.float32, device=x.device)
    _run("dcn_offset_conv_forward_modulated", x.device, shp, (x, offset_weight, offset_bias, offset, mask),
         phase=PHASE_LAYER_FORWARD_MODULATED, ws=ws)
    return offset, mask


def _layer_forward(x, offset_weight, offset_bias, weight, bias, kernel_size, stride, padding, variant, flags, ws,
                   modulated):
    """-> (offset, mask or None, out)"""
    shp = _shape_of(x, weight, kernel_size, stride, padding, variant, OPERAND_FP32, flags)
    return _layer_forward_shaped(shp, _dev_ready(x), offset_weight, offset_bias, weight, bias, ws, modulated)


def _layer_forward_shaped(shp, x, offset_weight, offset_bias, weight, bias, ws, modulated):
    """_layer_forward once the shape is built; x is the dense input, or the workspace whose head holds it staged."""
    Ho, Wo = _lib.output_hw(shp)
    N = shp.kh * shp.kw
    _check_offset_weight(offset_weight, shp, modulated)
    weight, bias = _dev_ready(weight), _dev_ready(bias)
    offset_weight, offset_bias = _dev_ready(offset_weight), _dev_ready(offset_bias)
    offset = torch.empty((shp.B, 2 * N, Ho, Wo), dtype=torch.float32, device=x.device)
    out = torch.empty((shp.B, shp.O, Ho, Wo), dtype=torch.float32, device=x.device)
    if not modulated:
        _run("dcn_layer_forward", x.device, shp, (x, offset_weight, offset_bias, weight, bias, offset, out),
             phase=PHASE_LAYER_FORWARD, ws=ws)
        return offset, None, out
    mask = torch.empty((shp.B, N, Ho, Wo), dtype=torch.float32, device=x.device)
    _run("dcn_layer_forward_modulated", x.device, shp, (x, offset_weight, offset_bias, weight, bias, offset, mask, out),
         phase=PHASE_LAYER_FORWARD_MODULATED, ws=ws)
    return offset, mask, out


def _layer_backward(x, offset, mask, offset_weight, weight, grad_out, has_offset_bias, has_bias, kernel_size, stride,
                    padding, variant, flags, need_grad_x, ws, xt_staged):
    """mask None: dcn_layer_backward, else dcn_layer_backward_modulated"""
    if not need_grad_x:
        flags |= FLAG_NO_GRAD_X
    if xt_staged and ws is not None:
        flags |= FLAG_XT_STAGED
    shp = _shape_of(x, weight, kernel_size, stride, padding, variant, OPERAND_FP32, flags)
    x = _dev_ready(x)
    gx = torch.empty(x.shape, dtype=torch.float32, device=x.device) if need_grad_x else None
    return _layer_backward_shaped(shp, x, gx, offset, mask, offset_weight, weight, grad_out, has_offset_bias, has_bias,
                                  ws)


def _layer_backward_shaped(shp, x, gx, offset, mask, offset_weight, weight, grad_out, has_offset_bias, has_bias, ws):
    """_layer_backward once the shape is built; x as in _layer_forward_shaped, gx its gradient buffer or None."""
    _check_offset_weight(offset_weight, shp, mask is not None)
    weight, grad_out = _dev_ready(weight), _dev_ready(grad_out)
    offset, mask, offset_weight = _dev_ready(offset), _dev_ready(mask), _dev_ready(offset_weight)
    dev = x.device
    gwoff = torch.empty(offset_weight.shape, dtype=torch.float32, device=dev)
    gboff = torch.empty((offset_weight.shape[0],), dtype=torch.float32, device=dev) if has_offset_bias else None
    gw = torch.empty(weight.shape, dtype=torch.float32, device=dev)
    gb = torch.empty((shp.O,), dtype=torch.float32, device=dev) if has_bias else None
    if mask is None:
        _run("dcn_layer_backward", dev, shp, (x, offset, offset_weight, weight, grad_out, gx, gwoff, gboff, gw, gb),
             phase=PHASE_LAYER_BACKWARD, ws=ws)
    else:
        _run("dcn_layer_backward_modulated", dev, shp,
             (x, offset, mask, offset_weight, weight, grad_out, gx, gwoff, gboff, gw, gb),
             phase=PHASE_LAYER_BACKWARD_MODULATED, ws=ws)
    return gx, gwoff, gboff, gw, gb


class DeformLayerFunction(torch.autograd.Function):
    """The whole reference module forward (offset conv + sampling + GEMM, deform_conv.py:56-81 / train.py:95-140)
    and its autograd as ONE node on the engine: x is staged once per step, grad_offset never reaches HBM as a
    framework tensor, and the two data-gradient terms are summed before the single transposition back to NCHW.
    cfg[-1] (modulated): mmcv's ModulatedDeformConv2dPack.forward (conv_offset, chunk / cat, sigmoid,
    modulated_deform_conv2d) instead, where neither the [B, 3N, Ho, Wo] conv output nor the gradients of offset and
    mask reach HBM as framework tensors."""

    @staticmethod
    def forward(ctx, x, offset_weight, offset_bias, weight, bias, cfg):
        kernel_size, stride, padding, variant, flags, keep_staged, modulated = cfg
        ctx.ws = _layer_workspace(x, weight, kernel_size, stride, padding, variant, flags, modulated) \
            if keep_staged else None
        offset, mask, out = _layer_forward(x, offset_weight, offset_bias, weight, bias, kernel_size, stride, padding,
                                           variant, flags, ctx.ws, modulated)
        # DCN_FLAG_RELU_OUT: the epilogue applied the ReLU; the backward entry points want the gradient of the
        # pre-activation sum, i.e. grad_out masked with out > 0
        ctx.relu = bool(flags & FLAG_RELU_OUT)
        ctx.save_for_backward(x, offset, mask, offset_weight, weight, *((out,) if ctx.relu else ()))
        ctx.cfg = cfg
        ctx.has = (offset_bias is not None, bias is not None)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, offset, mask, offset_weight, weight = ctx.saved_tensors[:5]
        if ctx.relu:
            grad_out = grad_out * (ctx.saved_tensors[5] > 0)
        kernel_size, stride, padding, variant, flags = ctx.cfg[:5]
        gx, gwoff, gboff, gw, gb = _layer_backward(
            x, offset, mask, offset_weight, weight, grad_out, ctx.has[0], ctx.has[1], kernel_size, stride, padding,
            variant, flags & ~FLAG_ACCUM_GRAD_X, ctx.needs_input_grad[0], ctx.ws, ctx.ws is not None)
        ctx.ws = None
        return gx, gwoff, gboff, gw, gb, None


def dcn_corners(offset, in_hw, kernel_size=3, stride=1, padding=1, variant=VARIANT_TORCH):
    """Sampling geometry only: y0, x0 [B,N,Ho,Wo] int32 and w4 [B,N,Ho,Wo,4] float32."""
    B = offset.shape[0]
    shp = _lib.make_shape(B, 1, 1, in_hw[0], in_hw[1], kernel_size, stride, padding, variant)
    Ho, Wo = _lib.output_hw(shp)
    N = shp.kh * shp.kw
    offset = _dev_ready(offset)
    dev = offset.device
    y0 = torch.empty((B, N, Ho, Wo), dtype=torch.int32, device=dev)
    x0 = torch.empty_like(y0)
    w4 = torch.empty((B, N, Ho, Wo, 4), dtype=torch.float32, device=dev)
    _run("dcn_debug_corners", dev, shp, (offset, y0, x0, w4))
    return y0, x0, w4


class DeformConvFunction(torch.autograd.Function):
    """autograd node standing where the reference has grid_sample + matmul + their autograd
    (train.py:102-140 forward, train.py:249 backward).  With a mask (the last input): the modulated DCNv1 operator
    (DCNv2), differentiable in the mask as well.  Host tensors are answered on their device."""

    @staticmethod
    def forward(ctx, x, offset, weight, bias, cfg, mask=None):
        kernel_size, stride, padding, variant, operand, flags, keep_staged = cfg
        home = x.device
        dev = _compute_device(x)
        xd, od, md, wd = (_to_device(t, dev) for t in (x, offset, mask, weight))
        bd = _to_device(bias, dev)
        act = torch.bfloat16 if operand == OPERAND_BF16 else torch.float32
        ctx.ws = None
        if keep_staged and xd.dtype == act and xd.is_contiguous():
            # private scratch that lives until backward: its head keeps the staged copy of x
            ctx.ws = staged_workspace(xd, wd, kernel_size, stride, padding, variant, operand, flags)
        out = _span_forward(xd, od, md, wd, bd, kernel_size, stride, padding, variant, operand, flags, ctx.ws)
        ctx.relu = bool(flags & FLAG_RELU_OUT)    # see DeformLayerFunction
        ctx.save_for_backward(xd, od, md, wd, *((out,) if ctx.relu else ()))
        ctx.cfg, ctx.home, ctx.has_bias = cfg, home, bias is not None
        ctx.dtypes = (x.dtype, offset.dtype, weight.dtype, None if mask is None else mask.dtype)
        return out if home == dev else out.to(home)

    @staticmethod
    def backward(ctx, grad_out):
        xd, od, md, wd = ctx.saved_tensors[:4]
        kernel_size, stride, padding, variant, operand, flags = ctx.cfg[:6]
        flags &= ~FLAG_ACCUM_GRAD_X     # autograd sums gradient terms itself; the output buffer here is fresh
        dev = xd.device
        grad_out = _to_device(grad_out, dev)
        if ctx.relu:
            grad_out = grad_out * (ctx.saved_tensors[4] > 0)
        gx, goff, gmask, gw, gb = _span_backward(xd, od, md, wd, grad_out, ctx.has_bias, kernel_size, stride, padding,
                                                 variant, operand, flags, ctx.needs_input_grad[0], ctx.ws,
                                                 ctx.ws is not None, None)
        ctx.ws = None
        home = ctx.home

        def back(t, dtype):
            if t is None:
                return None
            t = t.to(dtype) if t.dtype != dtype else t
            return t if home == dev else t.to(home)

        return (back(gx, ctx.dtypes[0]), back(goff, ctx.dtypes[1]), back(gw, ctx.dtypes[2]),
                back(gb, torch.float32), None, back(gmask, ctx.dtypes[3]))


def deform_conv2d(x, offset, weight, bias=None, kernel_size=3, stride=1, padding=1,
                  variant=VARIANT_TORCH, operand=OPERAND_FP32, flags=0, keep_staged=False):
    """Differentiable DeformConv2d core: everything after the offset conv.
    keep_staged: hold a private scratch buffer (backward-phase size) from forward to backward so
    that the backward pass reuses the staged copy of x instead of transposing it again."""
    cfg = (_lib._pair(kernel_size), _lib._pair(stride), _lib._pair(padding), variant, operand, flags,
           bool(keep_staged))
    return DeformConvFunction.apply(x, offset, weight, bias, cfg)


def deform_conv2d_modulated(x, offset, mask, weight, bias=None, kernel_size=3, stride=1, padding=1,
                            operand=OPERAND_FP32, flags=0):
    """Differentiable modulated DCNv1 (DCNv2) core: mask [B, kh*kw, Ho, Wo] scales every sample."""
    cfg = (_lib._pair(kernel_size), _lib._pair(stride), _lib._pair(padding), VARIANT_DCNV1, operand,
           flags & ~FLAG_RELU_OUT, False)
    return DeformConvFunction.apply(x, offset, weight, bias, cfg, mask)


def _out_hw(H, W, kernel_size, stride, padding):
    (kh, kw), (sh, sw), (ph, pw) = kernel_size, stride, padding
    return (H + 2 * ph - kh) // sh + 1, (W + 2 * pw - kw) // sw + 1


def deform_conv2d_v1(input, offset, weight, bias=None, stride=1, padding=0, dilation=1, mask=None):
    """Standard deformable convolution with the call signature (and semantics) of
    ``torchvision.ops.deform_conv2d(input, offset, weight, bias, stride, padding, dilation, mask)`` for one offset
    group and dilation 1 — the same kernels as the reference's operators with the textbook coordinate generator
    (SURVEY.md 8f.3).  mask=None: DCNv1, differentiable in input, offset, weight and bias.  mask [B, kh*kw, Ho, Wo]:
    modulated (DCNv2), every sample scaled by its mask value (no range or sigmoid applied), differentiable in the mask
    as well."""
    if _lib._pair(dilation) != (1, 1):
        raise ValueError(f"deform_conv2d_v1: dilation {dilation} is not supported (only 1)")
    kernel_size = (int(weight.shape[2]), int(weight.shape[3]))
    B, _, H, W = (int(v) for v in input.shape)
    Ho, Wo = _out_hw(H, W, kernel_size, _lib._pair(stride), _lib._pair(padding))
    N = kernel_size[0] * kernel_size[1]
    if tuple(offset.shape) != (B, 2 * N, Ho, Wo):
        raise ValueError(f"deform_conv2d_v1: offset shape {tuple(offset.shape)} != {(B, 2 * N, Ho, Wo)} "
                         "(one offset group: [B, 2*kh*kw, H_out, W_out])")
    if mask is None:
        return deform_conv2d(input, offset, weight, bias, kernel_size, stride, padding, variant=VARIANT_DCNV1)
    if tuple(mask.shape) != (B, N, Ho, Wo):
        raise ValueError(f"deform_conv2d_v1: mask shape {tuple(mask.shape)} != {(B, N, Ho, Wo)} "
                         "([B, kh*kw, H_out, W_out])")
    return deform_conv2d_modulated(input, offset, mask, weight, bias, kernel_size, stride, padding)


# ---- post-op: BatchNorm2d + ReLU (SURVEY 8f.2; train.py:167-170) -------------------------------------
class BatchNormReLUFunction(torch.autograd.Function):
    """relu(batch_norm(x)) on the engine's own kernels (csrc/dcn_bn.cu).  running_mean / running_var are
    updated in place in training mode, exactly as nn.BatchNorm2d does."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, training, momentum, eps):
        home = x.device
        dev = _compute_device(x)
        xd = _dev_ready(_to_device(x, dev))
        B, C = xd.shape[0], xd.shape[1]
        HW = xd.numel() // (B * C)
        wd, bd = _dev_ready(_to_device(weight, dev)), _dev_ready(_to_device(bias, dev))
        rm, rv = _to_device(running_mean, dev), _to_device(running_var, dev)
        y = torch.empty_like(xd)
        saved = torch.empty(4 * C, dtype=torch.float32, device=dev)
        _run("dcn_bn_relu_forward", dev, None,
             (B, C, HW, 1 if training else 0, xd, wd, bd, rm, rv, float(momentum), float(eps), y, saved),
             ws=_bn_workspace(dev, C))
        if training and running_mean is not None and rm is not running_mean:
            running_mean.copy_(rm)       # host-resident module: write the updated statistics back
            running_var.copy_(rv)
        ctx.save_for_backward(xd, saved)
        ctx.training, ctx.home = bool(training), home
        ctx.has_affine = (weight is not None, bias is not None)
        return y if home == dev else y.to(home)

    @staticmethod
    def backward(ctx, grad_y):
        xd, saved = ctx.saved_tensors
        dev = xd.device
        B, C = xd.shape[0], xd.shape[1]
        HW = xd.numel() // (B * C)
        gy = _dev_ready(_to_device(grad_y, dev))
        gx, gg, gb = _bn_grads(ctx, xd)
        _run("dcn_bn_relu_backward", dev, None, (B, C, HW, 1 if ctx.training else 0, xd, gy, saved, gx, gg, gb),
             ws=_bn_workspace(dev, C))
        home = ctx.home

        def back(t):
            return t if t is None or home == dev else t.to(home)

        return back(gx), back(gg), back(gb), None, None, None, None, None


def _bn_workspace(dev, C):
    """The scratch buffer the BatchNorm kernels take for C channels."""
    return torch.empty(_lib.load().dcn_bn_workspace_bytes(C), dtype=torch.uint8, device=dev)


def _bn_grads(ctx, x):
    """The BatchNorm backward's outputs for input x: grad_x if autograd wants it, grad_gamma / grad_beta for the affine
    parameters the node was given (None otherwise)."""
    C = x.shape[1]
    gx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
    gg, gb = (torch.empty(C, dtype=torch.float32, device=x.device) if has else None for has in ctx.has_affine)
    return gx, gg, gb


def batch_norm_relu(x, weight, bias, running_mean, running_var, training, momentum=0.1, eps=1e-5):
    """relu(F.batch_norm(x, running_mean, running_var, weight, bias, training, momentum, eps)) for NCHW float32."""
    return BatchNormReLUFunction.apply(x, weight, bias, running_mean, running_var, training, momentum, eps)


# ---- training: channels-last hand-over between a layer's post-op and the next layer (SURVEY 8f.2) ----------------
# The post-op writes the NEXT layer's staged input (framed channels-last copy at the head of that layer's workspace);
# the tensor that travels between the two autograd nodes is a float32 view of that workspace head, and its gradient
# is the consumer's channels-last grad_x accumulator (DCN_FLAG_GRAD_X_FRAMED) — nothing crosses the boundary in NCHW.
def stem_conv_supported(x, weight):
    """dcn_stem_conv_* takes this convolution (csrc/dcn_stem.cu: 3 x 3, stride 1, padding 1, Cin <= 4, O in {16, 32},
    W % 4 == 0, float32 CUDA tensors, no input gradient wanted)."""
    return (x.is_cuda and x.dim() == 4 and x.dtype == torch.float32 and weight.dtype == torch.float32
            and tuple(weight.shape[2:]) == (3, 3) and weight.shape[1] == x.shape[1] <= 4
            and weight.shape[0] in (16, 32) and x.shape[3] % 4 == 0 and not x.requires_grad)


class StemConvFunction(torch.autograd.Function):
    """conv2d(x, weight, bias, stride 1, padding 1) of the detector's first layer (train.py:145,166) on the engine's two
    streaming kernels.  x is the network input: no gradient flows to it."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        xd, wd = _dev_ready(x), _dev_ready(weight)
        bd = _dev_ready(bias) if bias is not None else None
        B, Cin, H, W = xd.shape
        O = wd.shape[0]
        out = torch.empty(B, O, H, W, dtype=torch.float32, device=xd.device)
        _run("dcn_stem_conv_forward", xd.device, None, (B, Cin, O, H, W, xd, wd, bd, out))
        ctx.save_for_backward(xd)
        ctx.O, ctx.has_bias = O, bias is not None
        return out

    @staticmethod
    def backward(ctx, grad_out):
        xd, = ctx.saved_tensors
        B, Cin, H, W = xd.shape
        go = _dev_ready(grad_out)
        gw = torch.empty(ctx.O, Cin, 3, 3, dtype=torch.float32, device=xd.device)
        gb = torch.empty(ctx.O, dtype=torch.float32, device=xd.device)
        _run("dcn_stem_conv_backward", xd.device, None, (B, Cin, ctx.O, H, W, xd, go, gw, gb))
        return None, gw, gb if ctx.has_bias else None


def stem_conv(x, weight, bias=None):
    """The detector's conv1 on the engine; the caller checks stem_conv_supported first."""
    return StemConvFunction.apply(x, weight, bias)


def _framed_view(ws, B, H, W, C):
    n = B * (H + 3) * (W + 2) * C
    return ws[:4 * n].view(torch.float32).view(B, H + 3, W + 2, C)


def _storage_tensor(t):
    """uint8 tensor over the WHOLE storage `t` lives in (the workspace a staged tensor is the head of)."""
    return torch.empty(0, dtype=torch.uint8, device=t.device).set_(t.untyped_storage())


def _consumer_shape(x_shape, consumer):
    out_channels, kernel_size, stride, padding, variant, flags = consumer
    B, C, H, W = (int(v) for v in x_shape)
    return _lib.make_shape(B, C, int(out_channels), H, W, kernel_size, stride, padding, variant, OPERAND_FP32, flags)


class BatchNormReLUStagedFunction(torch.autograd.Function):
    """relu(batch_norm(x)) whose result is written as the staged input of `consumer` (a DCN layer).  Returns the float32
    view [B, H + 3, W + 2, C] of the consumer's workspace head."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, training, momentum, eps, consumer):
        x = _dev_ready(x)
        B, C, H, W = x.shape
        shp = _consumer_shape(x.shape, consumer)
        need = _layer_bytes(shp)
        if need == 0:
            raise _lib.DcnError("staged post-op: the consumer layer does not run on the tensor path")
        dev = x.device
        consumer_ws = torch.empty(need, dtype=torch.uint8, device=dev)
        saved = torch.empty(4 * C, dtype=torch.float32, device=dev)
        _run("dcn_bn_relu_forward_staged", dev, shp,
             (1 if training else 0, x, weight, bias, running_mean, running_var, float(momentum), float(eps),
              consumer_ws, saved), ws=_bn_workspace(dev, C))
        ctx.save_for_backward(x, saved)
        ctx.consumer, ctx.training = consumer, bool(training)
        ctx.has_affine = (weight is not None, bias is not None)
        return _framed_view(consumer_ws, B, H, W, C)

    @staticmethod
    def backward(ctx, grad_staged):
        x, saved = ctx.saved_tensors
        shp = _consumer_shape(x.shape, ctx.consumer)
        g = _dev_ready(grad_staged)
        gx, gg, gb = _bn_grads(ctx, x)
        _run("dcn_bn_relu_backward_staged", x.device, shp, (1 if ctx.training else 0, x, g, saved, gx, gg, gb),
             ws=_bn_workspace(x.device, x.shape[1]))
        return gx, gg, gb, None, None, None, None, None, None


def batch_norm_relu_staged(x, weight, bias, running_mean, running_var, training, momentum, eps, consumer):
    """consumer = (out_channels, kernel_size, stride, padding, variant, flags) of the DCN layer that reads the result."""
    return BatchNormReLUStagedFunction.apply(x, weight, bias, running_mean, running_var, training, momentum, eps, consumer)


class DeformLayerFramedFunction(torch.autograd.Function):
    """The whole layer (offset conv + DCN span) on an input that is ALREADY staged: `xt` is the view a staged post-op
    returned (head of this layer's workspace).  Its gradient is returned in the same framed channels-last layout."""

    @staticmethod
    def forward(ctx, xt, offset_weight, offset_bias, weight, bias, cfg):
        (C, H, W), kernel_size, stride, padding, variant, flags = cfg
        B = int(xt.shape[0])
        if tuple(xt.shape) != (B, H + 3, W + 2, C) or xt.dtype != torch.float32 or not xt.is_contiguous():
            raise ValueError(f"staged input of shape {tuple(xt.shape)} does not match the layer input {(B, C, H, W)}")
        ws = _storage_tensor(xt)
        shp = _lib.make_shape(B, C, int(weight.shape[0]), H, W, kernel_size, stride, padding, variant, OPERAND_FP32,
                              flags | FLAG_XT_STAGED)
        need = _layer_bytes(shp)
        if need == 0 or ws.numel() < need or xt.data_ptr() != ws.data_ptr():
            raise _lib.DcnError("staged input is not the head of a workspace of this layer")
        offset, _, out = _layer_forward_shaped(shp, ws, offset_weight, offset_bias, weight, bias, ws, False)
        ctx.relu = bool(flags & FLAG_RELU_OUT)
        ctx.save_for_backward(xt, offset, offset_weight, weight, *((out,) if ctx.relu else ()))
        ctx.cfg = cfg
        ctx.has = (offset_bias is not None, bias is not None)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        xt, offset, offset_weight, weight = ctx.saved_tensors[:4]
        if ctx.relu:
            grad_out = grad_out * (ctx.saved_tensors[4] > 0)
        (C, H, W), kernel_size, stride, padding, variant, flags = ctx.cfg
        ws = _storage_tensor(xt)
        need_gx = ctx.needs_input_grad[0]
        fl = (flags & ~FLAG_ACCUM_GRAD_X) | FLAG_XT_STAGED | _lib.FLAG_GRAD_X_FRAMED | (0 if need_gx else FLAG_NO_GRAD_X)
        shp = _lib.make_shape(int(xt.shape[0]), C, int(weight.shape[0]), H, W, kernel_size, stride, padding, variant,
                              OPERAND_FP32, fl)
        gxt = torch.empty_like(xt) if need_gx else None
        grads = _layer_backward_shaped(shp, ws, gxt, offset, None, offset_weight, weight, grad_out, *ctx.has, ws)
        return grads + (None,)


def deform_layer_framed(xt, in_chw, offset_weight, offset_bias, weight, bias=None, kernel_size=3, stride=1, padding=1,
                        variant=VARIANT_TORCH, flags=0):
    """Whole layer on a staged input (see batch_norm_relu_staged); in_chw = (C, H, W) of the layer's logical input."""
    cfg = (tuple(int(v) for v in in_chw), _lib._pair(kernel_size), _lib._pair(stride), _lib._pair(padding), variant, flags)
    return DeformLayerFramedFunction.apply(xt, offset_weight, offset_bias, weight, bias, cfg)


# ---- multi-scale deformable attention (Deformable DETR's MSDeformAttn core; csrc/dcn_msda.cu) --------------------
def _msda_inputs(value, spatial_shapes, level_start_index, sampling_locations, attention_weights):
    """Checks shapes, dtypes and devices from tensor metadata only (no host synchronisation, so the call can be
    captured in a CUDA graph) -> (DcnMsdaShape, dense 16-byte aligned device tensors)."""
    floats = (("value", value), ("sampling_locations", sampling_locations), ("attention_weights", attention_weights))
    for name, t in floats:
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32:
            raise ValueError(f"ms_deform_attn: {name} must be a float32 tensor, got "
                             f"{getattr(t, 'dtype', type(t).__name__)} (the kernels are float32 only)")
    for name, t in floats:
        if not t.is_cuda:
            raise ValueError(f"ms_deform_attn: {name} must be a CUDA tensor: there is no CPU path")
    dev = value.device
    for name, t in (("sampling_locations", sampling_locations), ("attention_weights", attention_weights)):
        if t.device != dev:
            raise ValueError(f"ms_deform_attn: {name} is on {t.device}, value on {dev}")
    for name, t in (("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index)):
        if not isinstance(t, torch.Tensor) or t.is_floating_point() or t.is_complex() or t.dtype == torch.bool:
            raise ValueError(f"ms_deform_attn: {name} must be an integer tensor, got "
                             f"{getattr(t, 'dtype', type(t).__name__)}")
    if value.dim() != 4:
        raise ValueError(f"ms_deform_attn: value must be [B, S, M, D], got shape {tuple(value.shape)}")
    B, S, M, D = (int(v) for v in value.shape)
    if spatial_shapes.dim() != 2 or spatial_shapes.shape[1] != 2:
        raise ValueError(f"ms_deform_attn: spatial_shapes must be [L, 2], got shape {tuple(spatial_shapes.shape)}")
    L = int(spatial_shapes.shape[0])
    if tuple(level_start_index.shape) != (L,):
        raise ValueError(f"ms_deform_attn: level_start_index shape {tuple(level_start_index.shape)} != {(L,)}")
    if sampling_locations.dim() != 6:
        raise ValueError("ms_deform_attn: sampling_locations must be [B, Q, M, L, P, 2], got shape "
                         f"{tuple(sampling_locations.shape)}")
    Q, P = int(sampling_locations.shape[1]), int(sampling_locations.shape[4])
    if tuple(sampling_locations.shape) != (B, Q, M, L, P, 2):
        raise ValueError(f"ms_deform_attn: sampling_locations shape {tuple(sampling_locations.shape)} != "
                         f"{(B, Q, M, L, P, 2)} (value [B, S, M, D] = {(B, S, M, D)}, spatial_shapes [L, 2])")
    if tuple(attention_weights.shape) != (B, Q, M, L, P):
        raise ValueError(f"ms_deform_attn: attention_weights shape {tuple(attention_weights.shape)} != "
                         f"{(B, Q, M, L, P)}")
    if max(B, S, Q, M, D, L, P) > 0x7fffffff:
        raise ValueError(f"ms_deform_attn: an extent of {(B, S, Q, M, D, L, P)} exceeds 2^31 - 1")
    shp = _lib.DcnMsdaShape(B, S, Q, M, D, L, P, 0)
    idx = tuple(_dev_ready(_to_device(t, dev), torch.int64) for t in (spatial_shapes, level_start_index))
    return (shp, _dev_ready(value)) + idx + (_dev_ready(sampling_locations), _dev_ready(attention_weights))


def dcn_msda_forward(value, spatial_shapes, level_start_index, sampling_locations, attention_weights):
    """out [B, Q, M*D] of multi-scale deformable attention on CUDA tensors (no autograd)."""
    shp, v, ss, ls, loc, aw = _msda_inputs(value, spatial_shapes, level_start_index, sampling_locations,
                                           attention_weights)
    out = torch.empty((shp.B, shp.Q, shp.M * shp.D), dtype=torch.float32, device=v.device)
    _run("dcn_msda_forward", v.device, shp, (v, ss, ls, loc, aw, out))
    return out


def dcn_msda_backward(value, spatial_shapes, level_start_index, sampling_locations, attention_weights, grad_out,
                      need=(True, True, True)):
    """(grad_value, grad_sampling_locations, grad_attention_weights); need[i] False -> None, not computed."""
    shp, v, ss, ls, loc, aw = _msda_inputs(value, spatial_shapes, level_start_index, sampling_locations,
                                           attention_weights)
    if tuple(grad_out.shape) != (shp.B, shp.Q, shp.M * shp.D):
        raise ValueError(f"ms_deform_attn: grad_out shape {tuple(grad_out.shape)} != {(shp.B, shp.Q, shp.M * shp.D)}")
    go = _dev_ready(_to_device(grad_out, v.device))
    gv, gl, ga = (torch.empty_like(t) if n else None for t, n in zip((v, loc, aw), need))
    if gv is None and gl is None and ga is None:
        return None, None, None
    _run("dcn_msda_backward", v.device, shp, (v, ss, ls, loc, aw, go, gv, gl, ga))
    return gv, gl, ga


class MSDeformAttnFunction(torch.autograd.Function):
    """Multi-scale deformable attention core as one autograd node, with the positional interface of Deformable DETR's
    ``MSDeformAttnFunction`` and mmcv's ``MultiScaleDeformableAttnFunction``:

        MSDeformAttnFunction.apply(value, value_spatial_shapes, value_level_start_index,
                                   sampling_locations, attention_weights, im2col_step) -> [B, Q, M*D]

    value [B, S, M, D] f32, spatial_shapes [L, 2] and level_start_index [L] integer tensors (kept on the device: the
    node never synchronises with the host and can be captured in a CUDA graph), sampling_locations [B, Q, M, L, P, 2]
    and attention_weights [B, Q, M, L, P] f32, all on one CUDA device.  ``im2col_step`` is accepted and ignored: it
    exists only so that calls written for those implementations run unchanged.  Differentiable in value,
    sampling_locations and attention_weights; only the gradients autograd asks for are computed."""

    @staticmethod
    def forward(ctx, value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights,
                im2col_step=64):
        out = dcn_msda_forward(value, value_spatial_shapes, value_level_start_index, sampling_locations,
                               attention_weights)
        ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index, sampling_locations,
                              attention_weights)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        need = (ctx.needs_input_grad[0], ctx.needs_input_grad[3], ctx.needs_input_grad[4])
        gv, gl, ga = dcn_msda_backward(*ctx.saved_tensors, grad_output, need=need)
        return gv, None, None, gl, ga, None


def ms_deform_attn(value, spatial_shapes, level_start_index, sampling_locations, attention_weights):
    """Differentiable multi-scale deformable attention core (see MSDeformAttnFunction):
    out[b, q, m*D + d] = sum_{l,p} a[b,q,m,l,p] * bilinear(value_l[b, :, :, m, d], x*W_l - 0.5, y*H_l - 0.5)."""
    return MSDeformAttnFunction.apply(value, spatial_shapes, level_start_index, sampling_locations, attention_weights,
                                      64)


# ---- DCNv3 (InternImage's ops_dcnv3 core; csrc/dcn_dcnv3.cu) ------------------------------------------------------
def _grid_inputs(what, floats, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
                 group_channels):
    """The checks DCNv3 and DCNv4 share, on tensor metadata only: dtypes and devices of `floats` ((name, tensor), input
    first), the geometry and the input's shape -> (N, H, W, C, Ho, Wo)."""
    for name, t in floats:
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32:
            raise ValueError(f"{what}: {name} must be a float32 tensor, got "
                             f"{getattr(t, 'dtype', type(t).__name__)} (the kernels are float32 only)")
    for name, t in floats:
        if not t.is_cuda:
            raise ValueError(f"{what}: {name} must be a CUDA tensor: there is no CPU path")
    input = floats[0][1]
    dev = input.device
    for name, t in floats[1:]:
        if t.device != dev:
            raise ValueError(f"{what}: {name} is on {t.device}, input on {dev}")
    geo = dict(kernel_h=kernel_h, kernel_w=kernel_w, stride_h=stride_h, stride_w=stride_w, pad_h=pad_h, pad_w=pad_w,
               dilation_h=dilation_h, dilation_w=dilation_w, group=group, group_channels=group_channels)
    for name, v in geo.items():
        if isinstance(v, bool) or not isinstance(v, int):
            raise ValueError(f"{what}: {name} must be an int, got {v!r}")
        if v < (0 if name.startswith("pad") else 1):
            raise ValueError(f"{what}: {name} = {v} is out of range (paddings >= 0, everything else >= 1)")
    if input.dim() != 4:
        raise ValueError(f"{what}: input must be [N, H, W, group*group_channels], got shape {tuple(input.shape)}")
    N, H, W, C = (int(v) for v in input.shape)
    if C != group * group_channels:
        raise ValueError(f"{what}: input has {C} channels, group*group_channels = {group}*{group_channels} = "
                         f"{group * group_channels}")
    Ho = (H + 2 * pad_h - (dilation_h * (kernel_h - 1) + 1)) // stride_h + 1
    Wo = (W + 2 * pad_w - (dilation_w * (kernel_w - 1) + 1)) // stride_w + 1
    if Ho < 1 or Wo < 1:
        raise ValueError(f"{what}: empty output {Ho} x {Wo}: the dilated kernel does not fit the padded {H} x {W} "
                         "input")
    return N, H, W, C, Ho, Wo


def _dcnv3_inputs(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                  group, group_channels, softmax_mask):
    """Checks shapes, dtypes and devices from tensor metadata only (no host synchronisation, so the call can be
    captured in a CUDA graph) -> (DcnV3Shape, dense 16-byte aligned input, offset, mask)."""
    N, H, W, C, Ho, Wo = _grid_inputs("dcnv3", (("input", input), ("offset", offset), ("mask", mask)), kernel_h,
                                      kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
                                      group_channels)
    P = kernel_h * kernel_w
    if tuple(offset.shape) != (N, Ho, Wo, group * P * 2):
        raise ValueError(f"dcnv3: offset shape {tuple(offset.shape)} != {(N, Ho, Wo, group * P * 2)} "
                         f"(input {(N, H, W, C)}, {kernel_h}x{kernel_w} kernel, {group} groups)")
    if tuple(mask.shape) != (N, Ho, Wo, group * P):
        raise ValueError(f"dcnv3: mask shape {tuple(mask.shape)} != {(N, Ho, Wo, group * P)}")
    if max(N, H, W, C) > 0x7fffffff:
        raise ValueError(f"dcnv3: an extent of {(N, H, W, C)} exceeds 2^31 - 1")
    shp = _lib.DcnV3Shape(N, H, W, group, group_channels, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                          dilation_h, dilation_w, _lib.DCN_V3_FLAG_SOFTMAX_MASK if softmax_mask else 0)
    return shp, _dev_ready(input), _dev_ready(offset), _dev_ready(mask)


def dcn_v3_forward(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                   group, group_channels, offset_scale, softmax_mask=False):
    """out [N, Ho, Wo, group*group_channels] of the DCNv3 core on CUDA tensors (no autograd).  softmax_mask: `mask`
    holds logits and the core applies InternImage's softmax over the kernel_h*kernel_w points of each group."""
    shp, x, off, m = _dcnv3_inputs(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                                   dilation_h, dilation_w, group, group_channels, softmax_mask)
    out = torch.empty(tuple(off.shape[:3]) + (group * group_channels,), dtype=torch.float32, device=x.device)
    _run("dcn_v3_forward", x.device, shp, (float(offset_scale), x, off, m, out))
    return out


def dcn_v3_backward(input, offset, mask, grad_out, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                    dilation_w, group, group_channels, offset_scale, softmax_mask=False, need=(True, True, True)):
    """(grad_input, grad_offset, grad_mask); need[i] False -> None, not computed.  With softmax_mask, grad_mask is
    the gradient of the logits."""
    shp, x, off, m = _dcnv3_inputs(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                                   dilation_h, dilation_w, group, group_channels, softmax_mask)
    want = tuple(off.shape[:3]) + (group * group_channels,)
    if not isinstance(grad_out, torch.Tensor) or tuple(grad_out.shape) != want:
        raise ValueError(f"dcnv3: grad_out shape {tuple(getattr(grad_out, 'shape', ()))} != {want}")
    go = _dev_ready(_to_device(grad_out, x.device))
    gx, goff, gm = (torch.empty_like(t) if n else None for t, n in zip((x, off, m), need))
    if gx is None and goff is None and gm is None:
        return None, None, None
    _run("dcn_v3_backward", x.device, shp, (float(offset_scale), x, off, m, go, gx, goff, gm))
    return gx, goff, gm


class DCNv3Function(torch.autograd.Function):
    """The DCNv3 core as one autograd node, with the positional interface of InternImage's ``DCNv3Function``:

        DCNv3Function.apply(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                            dilation_h, dilation_w, group, group_channels, offset_scale, im2col_step,
                            remove_center=False) -> [N, Ho, Wo, group*group_channels]

    input [N, H, W, group*group_channels], offset [N, Ho, Wo, group*P*2] ((dx, dy) per point, points x-major:
    p = i*kernel_h + j for kernel column i and row j), mask [N, Ho, Wo, group*P], float32 on one CUDA device.
    ``im2col_step`` is accepted and ignored: it exists only so that calls written for InternImage run unchanged.
    ``remove_center=True`` is refused.  A trailing ``softmax_mask=True`` (not in InternImage's signature) makes `mask`
    logits and applies InternImage's per-group softmax inside the node.  Differentiable in input, offset and mask;
    only the gradients autograd asks for are computed, and the node never synchronises with the host."""

    @staticmethod
    def forward(ctx, input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                dilation_w, group, group_channels, offset_scale, im2col_step=256, remove_center=False,
                softmax_mask=False):
        if remove_center:
            raise ValueError("dcnv3: remove_center=True is not supported")
        ctx.geo = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
                   group_channels, offset_scale, bool(softmax_mask))
        out = dcn_v3_forward(input, offset, mask, *ctx.geo)
        ctx.save_for_backward(input, offset, mask)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        need = tuple(ctx.needs_input_grad[:3])
        gx, goff, gm = dcn_v3_backward(*ctx.saved_tensors, grad_output, *ctx.geo, need=need)
        return (gx, goff, gm) + (None,) * 14


def dcnv3_core(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
               group, group_channels, offset_scale, softmax_mask=False):
    """Differentiable DCNv3 core (see DCNv3Function):
    out[n, ho, wo, g*Gc + c] = sum_p m[n, ho, wo, g*P + p] * bilinear(input[n, :, :, g*Gc + c], y_p, x_p),
    m = softmax over each group's P entries of `mask` if softmax_mask, else `mask` itself."""
    return DCNv3Function.apply(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                               dilation_w, group, group_channels, offset_scale, 256, False, softmax_mask)


# ---- DCNv4 (the DCNv4 repository's DCNv4Function core; csrc/dcn_dcnv3.cu) ------------------------------------------
def dcnv4_row_floats(kernel_h, kernel_w, group, remove_center=False):
    """Cm, the floats per pixel of DCNv4's offset_mask: ceil(3*group*K / 8)*8 with K = kernel_h*kernel_w - remove_center
    points per group."""
    K = kernel_h * kernel_w - int(bool(remove_center))
    return (3 * group * K + 7) // 8 * 8


def _dcnv4_inputs(input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                  group, group_channels, remove_center):
    """As _dcnv3_inputs, for the packed offset_mask -> (DcnV3Shape, dense 16-byte aligned input, offset_mask)."""
    N, H, W, C, Ho, Wo = _grid_inputs("dcnv4", (("input", input), ("offset_mask", offset_mask)), kernel_h, kernel_w,
                                      stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels)
    rc = bool(remove_center)
    if rc and (kernel_h % 2 == 0 or kernel_w % 2 == 0):
        raise ValueError(f"dcnv4: remove_center needs an odd kernel, got {kernel_h} x {kernel_w}")
    K = kernel_h * kernel_w - rc
    if K == 0:
        raise ValueError("dcnv4: a 1 x 1 kernel with remove_center has no points (K = 0)")
    Cm = dcnv4_row_floats(kernel_h, kernel_w, group, rc)
    if offset_mask.dim() != 4 or tuple(offset_mask.shape[:3]) != (N, Ho, Wo):
        raise ValueError(f"dcnv4: offset_mask shape {tuple(offset_mask.shape)} != {(N, Ho, Wo, Cm)} "
                         f"(input {(N, H, W, C)}, {kernel_h}x{kernel_w} kernel)")
    if int(offset_mask.shape[-1]) != Cm:
        raise ValueError(f"dcnv4: offset_mask has {int(offset_mask.shape[-1])} floats per pixel, expected "
                         f"Cm = ceil(3*group*K / 8)*8 = ceil(3*{group}*{K} / 8)*8 = {Cm} "
                         f"(K = {kernel_h}*{kernel_w}{' - 1, remove_center' if rc else ''})")
    if max(N, H, W, C) > 0x7fffffff:
        raise ValueError(f"dcnv4: an extent of {(N, H, W, C)} exceeds 2^31 - 1")
    shp = _lib.DcnV3Shape(N, H, W, group, group_channels, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                          dilation_h, dilation_w, _lib.DCN_V4_FLAG_REMOVE_CENTER if rc else 0)
    return shp, _dev_ready(input), _dev_ready(offset_mask)


def dcn_v4_forward(input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                   group, group_channels, offset_scale, remove_center=False):
    """out [N, Ho, Wo, group*group_channels] of the DCNv4 core on CUDA tensors (no autograd)."""
    shp, x, om = _dcnv4_inputs(input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                               dilation_w, group, group_channels, remove_center)
    out = torch.empty(tuple(om.shape[:3]) + (group * group_channels,), dtype=torch.float32, device=x.device)
    _run("dcn_v4_forward", x.device, shp, (float(offset_scale), x, om, out))
    return out


def dcn_v4_backward(input, offset_mask, grad_out, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                    dilation_w, group, group_channels, offset_scale, remove_center=False, need=(True, True)):
    """(grad_input, grad_offset_mask); need[i] False -> None, not computed.  grad_offset_mask has offset_mask's packed
    layout, with +0.0 in the padding columns."""
    shp, x, om = _dcnv4_inputs(input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                               dilation_w, group, group_channels, remove_center)
    want = tuple(om.shape[:3]) + (group * group_channels,)
    if not isinstance(grad_out, torch.Tensor) or tuple(grad_out.shape) != want:
        raise ValueError(f"dcnv4: grad_out shape {tuple(getattr(grad_out, 'shape', ()))} != {want}")
    go = _dev_ready(_to_device(grad_out, x.device))
    gx, gom = (torch.empty_like(t) if n else None for t, n in zip((x, om), need))
    if gx is None and gom is None:
        return None, None
    _run("dcn_v4_backward", x.device, shp, (float(offset_scale), x, om, go, gx, gom))
    return gx, gom


class DCNv4Function(torch.autograd.Function):
    """The DCNv4 core as one autograd node, with the positional interface of the DCNv4 repository's ``DCNv4Function``:

        DCNv4Function.apply(input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                            dilation_h, dilation_w, group, group_channels, offset_scale, im2col_step,
                            remove_center) -> [N, Ho, Wo, group*group_channels]

    input [N, H, W, group*group_channels], offset_mask [N, Ho, Wo, Cm] with Cm = ceil(3*group*K / 8)*8 and
    K = kernel_h*kernel_w - remove_center: group g owns floats [g*3K, g*3K + 3K) of each pixel, first K interleaved
    (dx, dy) offsets, then K mask values (used as given: no softmax); the remaining columns are padding and never read.
    Points are DCNv3's, x-major (p = i*kernel_h + j for kernel column i and row j), with the centre point of an odd
    kernel dropped when remove_center is set.  float32 on one CUDA device.  ``im2col_step`` is accepted and ignored.
    Differentiable in input and offset_mask; only the gradients autograd asks for are computed, and the node never
    synchronises with the host."""

    @staticmethod
    def forward(ctx, input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                group, group_channels, offset_scale, im2col_step=256, remove_center=False):
        ctx.geo = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels,
                   offset_scale, bool(remove_center))
        out = dcn_v4_forward(input, offset_mask, *ctx.geo)
        ctx.save_for_backward(input, offset_mask)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        need = tuple(ctx.needs_input_grad[:2])
        gx, gom = dcn_v4_backward(*ctx.saved_tensors, grad_output, *ctx.geo, need=need)
        return (gx, gom) + (None,) * 13


def dcnv4_core(input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
               group, group_channels, offset_scale, remove_center=False):
    """Differentiable DCNv4 core (see DCNv4Function): DCNv3's operator with the packed offset_mask, the mask used as
    given, and optionally the kernel's centre point removed."""
    return DCNv4Function.apply(input, offset_mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                               dilation_w, group, group_channels, offset_scale, 256, remove_center)
