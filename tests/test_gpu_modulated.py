"""Modulated deformable convolution (DCNv2) on the GPU: the dcnv2_* torchvision fixtures on both kernel families, the
backward branches, mask edge cases, bf16 operands, output-channel groups, flags, the Python / module interface,
CUDA-graph capture and the full-size cfg2 shape."""
import numpy as np
import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from jittor_dcn_b200.functional import dcn_backward_modulated, dcn_forward_modulated, staged_workspace
from tests.util import golden, golden_names, rel_err

pytestmark = pytest.mark.gpu

FORCE_SIMT = dcn.FLAG_FORCE_SIMT
BF16 = dcn.OPERAND_BF16


def _cfg(g):
    B, C, O, H, W, kh, kw, sh, sw, ph, pw = (int(v) for v in g["cfg"])
    return B, C, O, H, W, (kh, kw), (sh, sw), (ph, pw)


def _path(B, C, O, H, W, k, s, p, operand=dcn.OPERAND_FP32, flags=0):
    shp = dcn.make_shape(B, C, O, H, W, k, s, p, dcn.VARIANT_DCNV1, operand, flags)
    return [_lib.path_name(shp, ph) for ph in (_lib.PHASE_FORWARD, _lib.PHASE_BACKWARD)]


def _tv_ref(x, off, mask, w, b, gout, s, p):
    """torchvision's CPU operator in float64: out and the five gradients."""
    from torchvision.ops import deform_conv2d
    ts = [torch.as_tensor(np.asarray(a)).double().requires_grad_(True) for a in (x, off, mask, w)]
    tb = torch.as_tensor(np.asarray(b)).double().requires_grad_(True) if b is not None else None
    out = deform_conv2d(ts[0], ts[1], ts[3], tb, stride=s, padding=p, mask=ts[2])
    grads = torch.autograd.grad(out, ts + ([tb] if tb is not None else []), torch.as_tensor(np.asarray(gout)).double())
    gx, goff, gmask, gw = (t.numpy() for t in grads[:4])
    gb = grads[4].numpy() if tb is not None else None
    return out.detach().numpy(), (gx, goff, gmask, gw, gb)


def _run(x, off, mask, w, b, gout, k, s, p, flags=0, operand=dcn.OPERAND_FP32):
    cu = lambda a: torch.as_tensor(np.asarray(a)).cuda() if a is not None else None   # noqa: E731
    tx, toff, tm, tw, tb, tg = (cu(a) for a in (x, off, mask, w, b, gout))
    out = dcn_forward_modulated(tx, toff, tm, tw, tb, k, s, p, operand=operand, flags=flags)
    grads = dcn_backward_modulated(tx, toff, tm, tw, tg, tb is not None, k, s, p, operand=operand, flags=flags)
    torch.cuda.synchronize()
    return out.cpu().numpy(), tuple(None if t is None else t.cpu().numpy() for t in grads)


def _check(out, grads, ref_out, ref_grads, tol_out=1e-4, tol_g=1e-3, what=""):
    assert rel_err(out, ref_out) < tol_out, (what, "out", rel_err(out, ref_out))
    for nm, a, r in zip(("gx", "goff", "gmask", "gw", "gb"), grads, ref_grads):
        if r is None:
            continue
        assert rel_err(a, r) < tol_g, (what, nm, rel_err(a, r))


def _random_problem(rng, B, C, O, H, W, k=3, s=1, p=1, sigma=1.5, bias=True):
    kh, kw = _lib._pair(k)
    (sh, sw), (ph, pw) = _lib._pair(s), _lib._pair(p)
    Ho, Wo = (H + 2 * ph - kh) // sh + 1, (W + 2 * pw - kw) // sw + 1
    N = kh * kw
    from oracle.make_golden_dcnv2 import dcnv2_mask
    x = rng.standard_normal((B, C, H, W)).astype(np.float32)
    off = (rng.standard_normal((B, 2 * N, Ho, Wo)) * sigma).astype(np.float32)
    mask = dcnv2_mask(rng, (B, N, Ho, Wo))
    w = (rng.standard_normal((O, C, kh, kw)) * np.sqrt(2.0 / (C * N))).astype(np.float32)
    b = rng.standard_normal(O).astype(np.float32) if bias else None
    gout = rng.standard_normal((B, O, Ho, Wo)).astype(np.float32)
    return x, off, mask, w, b, gout


# ---- torchvision fixtures, both kernel families ----------------------------------------------------------------------
TENSOR_PATH = {"dcnv2_b_s2", "dcnv2_e_64", "dcnv2_f_16"}


@pytest.mark.parametrize("flags", [0, FORCE_SIMT])
@pytest.mark.parametrize("name", golden_names("dcnv2_"))
def test_dcnv2_golden(name, flags):
    g = golden(name)
    B, C, O, H, W, k, s, p = _cfg(g)
    if name in TENSOR_PATH and flags == 0:
        assert _path(B, C, O, H, W, k, s, p) == ["umma", "umma"]
    if flags == FORCE_SIMT:
        assert _path(B, C, O, H, W, k, s, p, flags=flags) == ["simt", "simt"]
    out, grads = _run(g["x"], g["off"], g["mask"], g["weight"], g["bias"], g["gout"], k, s, p, flags)
    _check(out, grads, g["out"], (g["gx"], g["goff"], g["gmask"], g["gw"], g["gb"]), what=name)


# ---- every backward branch a DCNv1 shape can take --------------------------------------------------------------------
# (the fourth branch of umma_backward_any, tensor-path data gradient followed by an UNFUSED weight-gradient pass, is not
# reachable in the pixel-row layout: whenever its data-gradient kernel tiles a shape it also fuses the weight gradient,
# since every output-channel group has O <= 256 and its grad_out operand, Wm^T stages and sample buffers fit next to
# the plan ring for every channel count it accepts)
BRANCHES = {
    # name: (B, C, O, H, W, flags, kernels that must run, kernels that must not)
    "fused": (2, 64, 64, 12, 12, 0, {"umma_bwd_data_kernel"}, {"umma_bwd_weight_kernel", "bwd_data_kernel"}),
    "generic_data_umma_wgrad": (2, 192, 64, 10, 10, 0, {"bwd_data_kernel", "umma_bwd_weight_kernel"},
                                {"umma_bwd_data_kernel"}),
    "force_simt": (2, 64, 64, 12, 12, FORCE_SIMT, {"bwd_data_kernel", "bwd_weight_kernel"},
                   {"umma_bwd_data_kernel", "umma_bwd_weight_kernel"}),
}


@pytest.mark.parametrize("branch", sorted(BRANCHES))
def test_backward_branches(branch):
    B, C, O, H, W, flags, must, must_not = BRANCHES[branch]
    rng = np.random.default_rng(11)
    x, off, mask, w, b, gout = _random_problem(rng, B, C, O, H, W)
    ref_out, ref_grads = _tv_ref(x, off, mask, w, b, gout, 1, 1)
    _run(x, off, mask, w, b, gout, 3, 1, 1, flags)   # warm-up outside the profile window
    _lib.profile_begin()
    out, grads = _run(x, off, mask, w, b, gout, 3, 1, 1, flags)
    ran = set(_lib.profile_end())
    assert must <= ran and not (must_not & ran), (branch, sorted(ran))
    _check(out, grads, ref_out, ref_grads, what=branch)


# ---- mask == 1 and mask == 0 -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,flags", [(64, 0), (64, FORCE_SIMT), (16, 0), (4, 0)])
def test_mask_of_ones_is_the_unmodulated_operator(C, flags):
    rng = np.random.default_rng(3)
    x, off, _, w, b, gout = _random_problem(rng, 2, C, 32, 11, 13)
    ones = np.ones((2, 9, 11, 13), np.float32)
    tx, toff, tm, tw, tb, tg = (torch.as_tensor(a).cuda() for a in (x, off, ones, w, b, gout))
    out_m = dcn_forward_modulated(tx, toff, tm, tw, tb, 3, 1, 1, flags=flags)
    out_u = dcn.dcn_forward(tx, toff, tw, tb, 3, 1, 1, dcn.VARIANT_DCNV1, flags=flags)
    assert torch.equal(out_m, out_u)
    gm = dcn_backward_modulated(tx, toff, tm, tw, tg, True, 3, 1, 1, flags=flags)
    gu = dcn.dcn_backward(tx, toff, tw, tg, True, 3, 1, 1, dcn.VARIANT_DCNV1, flags=flags)
    for nm, a, r in zip(("gx", "goff", "gw", "gb"), (gm[0], gm[1], gm[3], gm[4]), gu):
        assert rel_err(a.cpu().numpy(), r.cpu().numpy()) <= 1e-6, nm
    _, ref_grads = _tv_ref(x, off, ones, w, b, gout, 1, 1)
    assert rel_err(gm[2].cpu().numpy(), ref_grads[2]) < 1e-3


@pytest.mark.parametrize("C,flags", [(64, 0), (64, FORCE_SIMT), (16, 0)])
def test_mask_of_zeros_leaves_the_bias(C, flags):
    rng = np.random.default_rng(4)
    x, off, _, w, b, gout = _random_problem(rng, 2, C, 32, 11, 13)
    zeros = np.zeros((2, 9, 11, 13), np.float32)
    out, (gx, goff, gmask, gw, gb) = _run(x, off, zeros, w, b, gout, 3, 1, 1, flags)
    assert np.array_equal(out, np.broadcast_to(b.reshape(1, -1, 1, 1), out.shape))
    assert not gx.any() and not goff.any() and not gw.any()
    _, ref_grads = _tv_ref(x, off, zeros, w, b, gout, 1, 1)
    assert rel_err(gmask, ref_grads[2]) < 1e-3 and rel_err(gb, ref_grads[4]) < 1e-3


# ---- bf16 operands on the ResNet C3 / C4 / C5 shapes; output-channel groups -------------------------------------------
@pytest.mark.parametrize("C,HW", [(128, 56), (256, 28), (512, 14)])
def test_bf16_operands_resnet_shapes(C, HW):
    rng = np.random.default_rng(C)
    B = 2
    x, off, mask, w, b, gout = _random_problem(rng, B, C, C, HW, HW, sigma=1.0)
    assert _path(B, C, C, HW, HW, 3, 1, 1, BF16) == ["umma", "umma"]
    rb = lambda a: torch.as_tensor(a).bfloat16().float().numpy()   # noqa: E731
    ref_out, ref_grads = _tv_ref(rb(x), off, mask, rb(w), b, rb(gout), 1, 1)
    out, grads = _run(x, off, mask, w, b, gout, 3, 1, 1, operand=BF16)
    _check(out, grads, ref_out, ref_grads, tol_out=1e-2, tol_g=2e-2, what=f"bf16 C={C}")


def test_wide_layer_output_channel_groups():
    rng = np.random.default_rng(5)
    x, off, mask, w, b, gout = _random_problem(rng, 2, 64, 512, 9, 10)
    assert _path(2, 64, 512, 9, 10, 3, 1, 1) == ["umma", "umma"]
    ref_out, ref_grads = _tv_ref(x, off, mask, w, b, gout, 1, 1)
    out, grads = _run(x, off, mask, w, b, gout, 3, 1, 1)
    _check(out, grads, ref_out, ref_grads, what="O=512")


# ---- flags -----------------------------------------------------------------------------------------------------------
def test_flags_xt_staged_accum_no_grad_x_relu():
    rng = np.random.default_rng(6)
    x, off, mask, w, b, gout = _random_problem(rng, 2, 64, 64, 12, 12)
    ref_out, ref_grads = _tv_ref(x, off, mask, w, b, gout, 1, 1)
    tx, toff, tm, tw, tb, tg = (torch.as_tensor(a).cuda() for a in (x, off, mask, w, b, gout))
    # XT_STAGED: one workspace from forward to backward
    ws = staged_workspace(tx, tw, 3, 1, 1, dcn.VARIANT_DCNV1)
    assert ws is not None
    out = dcn_forward_modulated(tx, toff, tm, tw, tb, 3, 1, 1, ws=ws)
    grads = dcn_backward_modulated(tx, toff, tm, tw, tg, True, 3, 1, 1, ws=ws, xt_staged=True)
    _check(out.cpu().numpy(), tuple(t.cpu().numpy() for t in grads), ref_out, ref_grads, what="xt_staged")
    # ACCUM_GRAD_X adds into an existing gradient
    base = torch.randn_like(tx)
    acc = base.clone()
    dcn_backward_modulated(tx, toff, tm, tw, tg, True, 3, 1, 1, grad_x=acc)
    assert rel_err((acc - base).cpu().numpy(), ref_grads[0]) < 1e-3
    # NO_GRAD_X: every other gradient unchanged
    g2 = dcn_backward_modulated(tx, toff, tm, tw, tg, True, 3, 1, 1, need_grad_x=False)
    assert g2[0] is None
    _check(out.cpu().numpy(), (None,) + tuple(t.cpu().numpy() for t in g2[1:]), ref_out, (None,) + ref_grads[1:],
           what="no_grad_x")
    # RELU_OUT: fused epilogue on the modulated forward
    for flags in (dcn.FLAG_RELU_OUT, dcn.FLAG_RELU_OUT | FORCE_SIMT):
        outr = dcn_forward_modulated(tx, toff, tm, tw, tb, 3, 1, 1, flags=flags)
        assert rel_err(outr.cpu().numpy(), np.maximum(ref_out, 0)) < 1e-4


# ---- the Python / module interface against live torchvision ----------------------------------------------------------
def test_deform_conv2d_v1_and_module_match_torchvision():
    from torchvision.ops import DeformConv2d, deform_conv2d
    torch.manual_seed(0)
    B, C, O, H, W = 2, 64, 64, 14, 14
    ref = DeformConv2d(C, O, 3, padding=1)
    ours = dcn.TorchvisionDeformConv2d(C, O, 3, padding=1)
    ours.load_state_dict(ref.state_dict())
    ours.cuda()
    x = torch.randn(B, C, H, W)
    off = torch.randn(B, 18, H, W) * 1.5
    mask = torch.sigmoid(torch.randn(B, 9, H, W))
    gout = torch.randn(B, O, H, W)
    leaves = [t.clone().requires_grad_(True) for t in (x, off, mask)]
    out_ref = ref(*leaves)
    out_ref.backward(gout)
    ref_grads = [t.grad for t in leaves] + [ref.weight.grad, ref.bias.grad]
    # module
    mine = [t.cuda().requires_grad_(True) for t in (x, off, mask)]
    out = ours(*mine)
    out.backward(gout.cuda())
    got = [t.grad for t in mine] + [ours.weight.grad, ours.bias.grad]
    assert rel_err(out.detach().cpu().numpy(), out_ref.detach().numpy()) < 1e-4
    for a, r in zip(got, ref_grads):
        assert rel_err(a.cpu().numpy(), r.numpy()) < 1e-3
    # functional, torchvision's positional order, host tensors in and out
    leaves2 = [t.clone().requires_grad_(True) for t in (x, off, ref.weight.detach(), ref.bias.detach(), mask)]
    out2 = dcn.deform_conv2d_v1(leaves2[0], leaves2[1], leaves2[2], leaves2[3], 1, 1, 1, leaves2[4])
    assert out2.device.type == "cpu"
    out2.backward(gout)
    assert rel_err(out2.detach().numpy(), out_ref.detach().numpy()) < 1e-4
    for a, r in zip([leaves2[0].grad, leaves2[1].grad, leaves2[4].grad, leaves2[2].grad, leaves2[3].grad], ref_grads):
        assert rel_err(a.numpy(), r.numpy()) < 1e-3
    # mask=None is DCNv1
    out3 = dcn.deform_conv2d_v1(x.cuda(), off.cuda(), ref.weight.detach().cuda(), ref.bias.detach().cuda(), padding=1)
    assert rel_err(out3.cpu().numpy(), deform_conv2d(x, off, ref.weight, ref.bias, padding=1).detach().numpy()) < 1e-4


# ---- CUDA graph capture ----------------------------------------------------------------------------------------------
def test_cuda_graph_replay_reproduces_eager():
    rng = np.random.default_rng(8)
    x, off, mask, w, b, gout = _random_problem(rng, 2, 64, 64, 12, 12)
    tx, toff, tm, tw, tb, tg = (torch.as_tensor(a).cuda() for a in (x, off, mask, w, b, gout))
    eager_out = dcn_forward_modulated(tx, toff, tm, tw, tb, 3, 1, 1)
    eager = dcn_backward_modulated(tx, toff, tm, tw, tg, True, 3, 1, 1)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                       # warm-up on the capture stream
        dcn_forward_modulated(tx, toff, tm, tw, tb, 3, 1, 1)
        dcn_backward_modulated(tx, toff, tm, tw, tg, True, 3, 1, 1)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out = dcn_forward_modulated(tx, toff, tm, tw, tb, 3, 1, 1)
        g_grads = dcn_backward_modulated(tx, toff, tm, tw, tg, True, 3, 1, 1)
    for a in (g_out,) + g_grads:
        a.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(g_out, eager_out)
    for a, r in zip(g_grads, eager):
        assert rel_err(a.cpu().numpy(), r.cpu().numpy()) <= 1e-6
    dcn.clear_workspaces()


# ---- full size: the cfg2 shape in DCNv1 mode -------------------------------------------------------------------------
def test_full_size_cfg2_shape():
    torch.manual_seed(9)
    B, C, O, H, W = 256, 64, 64, 128, 128
    assert _path(B, C, O, H, W, 3, 1, 1) == ["umma", "umma"]
    x = torch.randn(B, C, H, W, device="cuda")
    off = torch.randn(B, 18, H, W, device="cuda") * 1.5
    mask = torch.sigmoid(torch.randn(B, 9, H, W, device="cuda"))
    w = torch.randn(O, C, 3, 3, device="cuda") * (2.0 / (C * 9)) ** 0.5
    b = torch.randn(O, device="cuda")
    gout = torch.randn(B, O, H, W, device="cuda")
    def rel(a, r):   # tests.util.rel_err on the device: these tensors are GBs
        return float((a.double() - r.double()).abs().max() / r.double().abs().max().clamp_min(1e-30))

    res = {}
    for flags in (0, FORCE_SIMT):
        out = dcn_forward_modulated(x, off, mask, w, b, 3, 1, 1, flags=flags)
        res[flags] = (out,) + dcn_backward_modulated(x, off, mask, w, gout, True, 3, 1, 1, flags=flags)
    names = ("out", "gx", "goff", "gmask", "gw", "gb")
    for nm, a, r in zip(names, res[0], res[FORCE_SIMT]):
        assert rel(a, r) < (1e-4 if nm == "out" else 1e-3), nm
    del res
    # torchvision's own CUDA kernel, where this build of torchvision has one
    from torchvision.ops import deform_conv2d
    try:
        xs = x[:16].clone().requires_grad_(True)
        offs, masks = off[:16].clone().requires_grad_(True), mask[:16].clone().requires_grad_(True)
        ws, bs = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
        tv = deform_conv2d(xs, offs, ws, bs, padding=1, mask=masks)
    except (RuntimeError, NotImplementedError) as e:
        pytest.skip(f"torchvision has no CUDA deform_conv2d here: {e}")
    # the same 16 images through the engine (tensor path)
    out16 = dcn_forward_modulated(x[:16].contiguous(), off[:16].contiguous(), mask[:16].contiguous(), w, b, 3, 1, 1)
    g16 = dcn_backward_modulated(x[:16].contiguous(), off[:16].contiguous(), mask[:16].contiguous(), w, gout[:16].contiguous(),
                                 True, 3, 1, 1)
    tv_grads = torch.autograd.grad(tv, [xs, offs, masks, ws, bs], gout[:16])
    assert rel(out16, tv.detach()) < 1e-4
    for nm, a, r in zip(names[1:], g16, tv_grads):
        assert rel(a, r) < 1e-3, nm
