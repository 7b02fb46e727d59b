"""The whole modulated layer (mmcv's ModulatedDeformConv2dPack) on the engine: the offset-and-mask conv, its sigmoid
and the modulated span as one autograd node.

The reference is live: F.conv2d -> chunk / cat -> sigmoid -> torchvision.ops.deform_conv2d(mask=), float64 on the CPU.
Where floor() of a sampling coordinate could flip between the engine's fp32 offsets and the float64 ones, the reference
samples at the engine's offsets (forward value) while its gradient still flows through the float64 conv:
z_off + (offset_engine - z_off).detach().
"""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from tests.util import rel_err

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-4
GRAD_TOL = 1e-3


def _module(C, O, k, s, p, bias=True, seed=0, offset_scale=1.0):
    """A module with random parameters: offsets of a few pixels, mask logits around 0."""
    torch.manual_seed(seed)
    m = dcn.ModulatedDeformConv2dPack(C, O, k, stride=s, padding=p, bias=bias)
    with torch.no_grad():
        kk = m.kernel_size[0] * m.kernel_size[1]
        m.conv_offset.weight.normal_(0.0, offset_scale / np.sqrt(C * kk))
        m.conv_offset.bias.uniform_(-0.5, 0.5)
        if bias:
            m.bias.uniform_(-0.1, 0.1)
    return m.cuda()


def _reference(m, x, gout, off_engine=None, need_gx=True):
    """out and gradients (x, weight, bias, conv_offset.weight, conv_offset.bias) of mmcv's composition in float64."""
    from torchvision.ops import deform_conv2d
    x64 = x.detach().cpu().double().requires_grad_(need_gx)
    w = m.weight.detach().cpu().double().requires_grad_(True)
    b = m.bias.detach().cpu().double().requires_grad_(True) if m.bias is not None else None
    wo = m.conv_offset.weight.detach().cpu().double().requires_grad_(True)
    bo = m.conv_offset.bias.detach().cpu().double().requires_grad_(True)
    z = F.conv2d(x64, wo, bo, m.stride, m.padding)
    o1, o2, ml = torch.chunk(z, 3, dim=1)
    off = torch.cat((o1, o2), dim=1)
    if off_engine is not None:
        off = off + (off_engine.detach().cpu().double() - off).detach()
    out = deform_conv2d(x64, off, w, b, m.stride, m.padding, mask=torch.sigmoid(ml))
    out.backward(gout.detach().cpu().double())
    grads = [x64.grad if need_gx else None, w.grad, b.grad if b is not None else None, wo.grad, bo.grad]
    return out.detach(), grads


def _engine(m, x, gout):
    x = x.detach().clone().requires_grad_(x.requires_grad)
    m.zero_grad(set_to_none=True)
    out = m(x)
    out.backward(gout)
    grads = [x.grad, m.weight.grad, m.bias.grad if m.bias is not None else None, m.conv_offset.weight.grad,
             m.conv_offset.bias.grad]
    return out.detach(), grads


def _engine_offsets(m, x):
    off, mask, _ = dcn.dcn_layer_forward_modulated(x.detach(), m.conv_offset.weight.detach(),
                                                   m.conv_offset.bias.detach(), m.weight.detach(),
                                                   None if m.bias is None else m.bias.detach(), m.kernel_size,
                                                   m.stride, m.padding)
    return off, mask


# ---- the offset-and-mask conv ----------------------------------------------------------------------------------
@pytest.mark.parametrize("shape, kernel", [
    # B, C, O, H, W, k, s, p
    ((2, 64, 64, 16, 16, 3, 1, 1), "conv_offset_mask_fwd_kernel"),        # shifted-view kernels
    ((2, 128, 128, 14, 10, 3, 2, 1), "conv_offset_mask_fwd_kernel"),
    ((2, 64, 32, 9, 11, (1, 3), 1, 1), "conv_offset_mask_fwd_kernel"),    # 3N = 9
    ((2, 16, 16, 20, 20, 3, 1, 1), "conv_small_mask_fwd_kernel"),         # warp-MMA kernels
    ((3, 32, 32, 17, 13, 3, 2, 1), "conv_small_mask_fwd_kernel"),
])
def test_offset_and_mask_conv_matches_conv2d_and_sigmoid(shape, kernel):
    B, C, O, H, W, k, s, p = shape
    kh, kw = _lib._pair(k)
    N = kh * kw
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, C, H, W, generator=g)
    wo = torch.randn(3 * N, C, kh, kw, generator=g) / np.sqrt(C * N)
    bo = torch.randn(3 * N, generator=g)
    _lib.profile_begin()
    off, mask = dcn.dcn_offset_conv_forward_modulated(x.cuda(), wo.cuda(), bo.cuda(), O, k, s, p)
    torch.cuda.synchronize()
    prof = _lib.profile_end()
    assert kernel in prof, prof
    z = F.conv2d(x.double(), wo.double(), bo.double(), s, p)
    assert rel_err(off.cpu(), z[:, :2 * N]) <= 2e-5
    bound = 0.25 * 2e-5 * float(z.abs().max()) + 1e-6
    assert float((mask.cpu().double() - torch.sigmoid(z[:, 2 * N:])).abs().max()) <= bound


# ---- the module against the float64 reference ------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [
    # B, C, O, H, W, s, bias, keep_staged, x.requires_grad
    (2, 64, 64, 16, 16, 1, True, False, True),
    (2, 64, 48, 20, 12, 2, False, True, True),      # non-square, stride 2, no bias
    (2, 16, 32, 24, 24, 2, True, True, True),       # warp-MMA conv kernels
    (2, 32, 32, 13, 19, 1, True, False, False),     # input without requires_grad
    (2, 128, 128, 14, 14, 2, True, False, True),    # stride 2 at 128 channels: plain-mode conv backward
    (1, 512, 512, 7, 7, 1, True, True, True),       # O = 512: output-channel groups
])
def test_module_matches_the_float64_composition(cfg):
    B, C, O, H, W, s, bias, keep, xgrad = cfg
    m = _module(C, O, 3, s, 1, bias=bias, seed=B * C + O)
    m.keep_staged_input = keep
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, C, H, W, generator=g).cuda().requires_grad_(xgrad)
    assert m._whole_layer_on_engine(x)
    Ho, Wo = (H + 2 - 3) // s + 1, (W + 2 - 3) // s + 1
    gout = torch.randn(B, O, Ho, Wo, generator=g).cuda()
    out, grads = _engine(m, x, gout)
    off_e, _ = _engine_offsets(m, x)
    ref_out, ref_grads = _reference(m, x, gout, off_engine=off_e, need_gx=xgrad)
    assert rel_err(out.cpu(), ref_out) <= FWD_TOL
    for name, a, r in zip(("x", "weight", "bias", "conv_offset.weight", "conv_offset.bias"), grads, ref_grads):
        if r is None:
            assert a is None, name
            continue
        assert rel_err(a.cpu(), r) <= GRAD_TOL, name


def test_fresh_module_is_half_a_convolution():
    torch.manual_seed(2)
    m = dcn.ModulatedDeformConv2dPack(64, 64, 3, padding=1).cuda()
    with torch.no_grad():
        m.bias.uniform_(-0.2, 0.2)
    x = torch.randn(2, 64, 16, 16, device="cuda")
    out = m(x)
    ref = 0.5 * F.conv2d(x.double().cpu(), m.weight.detach().double().cpu(), None, 1, 1) + \
        m.bias.detach().double().cpu().view(1, -1, 1, 1)
    assert rel_err(out.detach().cpu(), ref) <= FWD_TOL
    out.square().sum().backward()
    assert float(m.conv_offset.weight.grad.abs().max()) > 0
    assert float(m.conv_offset.bias.grad.abs().max()) > 0


# ---- one node against two nodes --------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [
    # B, C, O, H, W, s: ResNet C3 - C5 (stride 1 and 2) and cfg2 in DCNv1 mode, at reduced batch
    (2, 128, 128, 28, 28, 1), (2, 128, 128, 56, 56, 2),
    (2, 256, 256, 14, 14, 1), (2, 256, 256, 28, 28, 2),
    (2, 512, 512, 7, 7, 1), (2, 512, 512, 14, 14, 2),
    (4, 64, 64, 128, 128, 1),
])
def test_one_node_matches_the_two_node_composition(shape):
    """The composition samples at the engine's offsets (checked against the framework conv to 2e-5 first): offsets
    that differ in the last bits flip floor() for a handful of the 10^6 samples at 128 x 128, and each flip moves one
    grad_offset element, i.e. a 3 x 3 x C patch of grad_x through the conv's backward (see tests/test_gpu_layer.py)."""
    B, C, O, H, W, s = shape
    one = _module(C, O, 3, s, 1, seed=C + s, offset_scale=0.5)
    two = copy.deepcopy(one)
    two.engine_offset_conv = False
    g = torch.Generator().manual_seed(9)
    x = torch.randn(B, C, H, W, generator=g).cuda().requires_grad_(True)
    assert one._whole_layer_on_engine(x) and not two._whole_layer_on_engine(x)
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    gout = torch.randn(B, O, Ho, Wo, generator=g).cuda()
    off_e, _ = _engine_offsets(one, x)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False   # the framework conv in fp32, like the engine's hi/lo split
    try:
        x2 = x.detach().clone().requires_grad_(True)
        o1, o2, ml = torch.chunk(two.conv_offset(x2), 3, dim=1)
        off = torch.cat((o1, o2), dim=1)
        assert rel_err(off_e.cpu(), off.detach().cpu()) <= 2e-5
        off = off + (off_e - off).detach()
        out2 = dcn.deform_conv2d_v1(x2, off, two.weight, two.bias, two.stride, two.padding, mask=torch.sigmoid(ml))
        out2.backward(gout)
        out2 = out2.detach()
        grads2 = [x2.grad, two.weight.grad, two.bias.grad, two.conv_offset.weight.grad, two.conv_offset.bias.grad]
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                            torch.profiler.ProfilerActivity.CUDA]) as prof:
        out1, grads1 = _engine(one, x, gout)
        torch.cuda.synchronize()
    ops = [e.key for e in prof.key_averages()]
    assert not any(k in ("aten::conv2d", "aten::convolution", "aten::_convolution", "aten::cudnn_convolution",
                         "aten::convolution_backward") for k in ops), ops
    assert not any("cudnn" in k.lower() for k in ops), ops
    assert rel_err(out1.cpu(), out2.cpu()) <= FWD_TOL
    for name, a, b in zip(("x", "weight", "bias", "conv_offset.weight", "conv_offset.bias"), grads1, grads2):
        assert rel_err(a.cpu(), b.cpu()) <= GRAD_TOL, name


# ---- shapes outside the layer path -----------------------------------------------------------------------------
@pytest.mark.parametrize("C, flags", [(4, 0), (64, dcn.FLAG_FORCE_SIMT)])
def test_fallback_gives_the_composition(C, flags):
    m = _module(C, 16, 3, 1, 1, seed=4)
    m.engine_flags = flags
    x = torch.randn(2, C, 12, 10, device="cuda").requires_grad_(True)
    assert not m._whole_layer_on_engine(x)
    gout = torch.randn(2, 16, 12, 10, device="cuda")
    out, grads = _engine(m, x, gout)
    ref_out, ref_grads = _reference(m, x, gout)
    assert rel_err(out.cpu(), ref_out) <= FWD_TOL
    for a, r in zip(grads, ref_grads):
        assert rel_err(a.cpu(), r) <= GRAD_TOL


# ---- CUDA graphs -----------------------------------------------------------------------------------------------
def test_module_step_replays_from_a_cuda_graph():
    m = _module(64, 64, 3, 1, 1, seed=8)
    x = torch.randn(2, 64, 16, 16, device="cuda").requires_grad_(True)
    gout = torch.randn(2, 64, 16, 16, device="cuda")
    eager_out, eager_grads = _engine(m, x, gout)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            x.grad = None
            m(x).backward(gout)
    torch.cuda.current_stream().wait_stream(side)
    m.zero_grad(set_to_none=True)
    x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = m(x)
        static_out.backward(gout)
    graph.replay()
    torch.cuda.synchronize()
    replay = [x.grad, m.weight.grad, m.bias.grad, m.conv_offset.weight.grad, m.conv_offset.bias.grad]
    assert rel_err(static_out.detach().cpu(), eager_out.cpu()) <= 1e-6
    for name, a, b in zip(("x", "weight", "bias", "conv_offset.weight", "conv_offset.bias"), replay, eager_grads):
        assert rel_err(a.cpu(), b.cpu()) <= 1e-6, name
