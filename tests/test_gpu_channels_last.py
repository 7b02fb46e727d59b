"""The channels-last hand-over between engine layers (DESIGN.md §7, "Channels-last contract") against float64.

Inference: `ChainedDeformStages` (dcn_layer_forward_chained), whose forward epilogue writes the consumer layer's framed,
channel-permuted staging copy.  Training: the staged BatchNorm post-op (dcn_bn_relu_forward_staged /
dcn_bn_relu_backward_staged, csrc/dcn_bn.cu) and the framed data gradient (DCN_FLAG_GRAD_X_FRAMED).

The chained cases run batches whose first stage has more tiles than two per SM: the forward kernel is persistent
(one CTA per SM, two TMEM accumulators), so only the third tile of a CTA waits for its accumulator to be released.
Extents cover H*W % 4 != 0 (the unvectorised transposing kernels), partial pixel blocks, every Torch-layout staging
tile (Gt = 64, 32, 16) with Cs > 1, mixed-variant chains, O = 16 and O = 256, and a 1 x 3 kernel.
"""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from jittor_dcn_b200.functional import _run, _storage_tensor, deform_layer
from oracle.torch_chain import chain_forward, out_hw
from tests.util import rel_err

J, T = dcn.VARIANT_JITTOR, dcn.VARIANT_TORCH
CLS = {J: dcn.TorchDeformConv2dJittorSemantics, T: dcn.TorchDeformConv2d}
NAME = {J: "jittor", T: "torch"}


def forward_tiles(B, C, H, W, k, s, p, variant):
    """Tiles of the forward kernel for this layer (make_tiling in csrc/dcn_umma_common.cuh)."""
    Ho, Wo = out_hw(H, W, k, s, p)
    HW = Ho * Wo
    if variant == T:
        G = math.gcd(HW, C)
        Gt = 64 if G % 64 == 0 else (32 if G % 32 == 0 else 16)
        return -(-B * (G // Gt) * (HW // G) // (128 // Gt))
    return B * -(-HW // 128)


def staged_channels(C, Ho, Wo, variant):
    """Position of logical channel c in the staging copy of a layer with input channels C and output extent Ho x Wo
    (Torch layout: c -> (c % Cs) * G + c / Cs, G = gcd(Ho * Wo, C), Cs = C / G; pixel-row layouts: identity)."""
    c = torch.arange(C)
    if variant != T:
        return c
    G = math.gcd(Ho * Wo, C)
    Cs = C // G
    return (c % Cs) * G + c // Cs


def unstage(framed, H, W, perm):
    """[B, H + 3, W + 2, C] staging copy -> [B, C, H, W] in logical channel order."""
    return framed[:, 1:H + 1, 1:W + 1, :][..., perm.to(framed.device)].permute(0, 3, 1, 2)


def _frame_mask(H, W, device):
    mask = torch.ones(H + 3, W + 2, dtype=torch.bool, device=device)
    mask[1:H + 1, 1:W + 1] = False
    return mask


def frame_of(framed, H, W):
    return framed[:, _frame_mask(H, W, framed.device), :]


def _no_tf32(fn):
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        return fn()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ---- A. chained inference ----------------------------------------------------------------------------------------
# name: (stages [(variant, C, O, kernel, stride, padding)], input (H, W), batches)
CHAINS = {
    # the detector's four DCN stages: 32 tiles per image in the first stage
    "detector-torch": ([(T, 16, 32, 3, 2, 1), (T, 32, 64, 3, 2, 1), (T, 64, 128, 3, 2, 1), (T, 128, 256, 3, 2, 1)],
                       (128, 128), (16, 256)),
    "detector-jittor": ([(J, 16, 32, 3, 2, 1), (J, 32, 64, 3, 2, 1), (J, 64, 128, 3, 2, 1), (J, 128, 256, 3, 2, 1)],
                        (128, 128), (16, 256)),
    # 143 pixels: a full and a partial pixel block per image, H*W % 4 != 0
    "odd-extent": ([(J, 64, 64, 3, 1, 1), (J, 64, 64, 3, 1, 1)], (13, 11), (300,)),
    # a pixel-row producer writing a Torch consumer's copy, and a Torch producer writing a pixel-row consumer's
    "mixed": ([(J, 64, 64, 3, 1, 1), (T, 64, 128, 3, 1, 1), (J, 128, 64, 3, 2, 1)], (32, 32), (48,)),
    # Torch consumers: G = 96 (Gt 32), G = 16 with Cs = 3 (Gt 16), G = 64 with Cs = 4
    "torch-gt32": ([(T, 64, 96, 3, 1, 1), (T, 96, 64, 3, 1, 1)], (16, 12), (224,)),
    "torch-gt16-cs3": ([(T, 64, 48, 3, 1, 1), (T, 48, 64, 3, 1, 1)], (20, 20), (96,)),
    "torch-cs4": ([(T, 64, 256, 3, 1, 1), (T, 256, 64, 3, 1, 1)], (8, 8), (640,)),
    # the widest chained producer (O = 256) and the narrowest (O = 16)
    "width-256": ([(J, 64, 256, 3, 1, 1), (J, 256, 64, 3, 1, 1)], (16, 16), (160,)),
    "width-16": ([(T, 32, 16, 3, 1, 1), (T, 16, 32, 3, 1, 1)], (32, 32), (48,)),
    "taps-1x3": ([(J, 64, 64, (1, 3), 1, (0, 1)), (J, 64, 64, (1, 3), 1, (0, 1))], (24, 20), (80,)),
}
CHAIN_CASES = [(name, B) for name, (_, _, batches) in CHAINS.items() for B in batches]


def _stage_shapes(spec, H, W, B):
    shapes = []
    for variant, C, O, k, s, p in spec:
        shapes.append(_lib.make_shape(B, C, O, H, W, k, s, p, variant, _lib.OPERAND_FP32, _lib.FLAG_RELU_OUT))
        H, W = out_hw(H, W, k, s, p)
    return shapes


@pytest.mark.parametrize("name,B", CHAIN_CASES)
def test_chain_cases_run_on_the_tensor_path_with_more_tiles_than_two_per_sm(name, B):
    """Every stage of every chained case is a whole layer on the tensor path, and the first stage has more than
    2 x 148 (the B200's SM count) forward tiles; the GPU test repeats the tile check against the device's own count."""
    spec, (H, W), _ = CHAINS[name]
    for shp in _stage_shapes(spec, H, W, B):
        assert _lib.path_name(shp, _lib.PHASE_LAYER_FORWARD) == "umma", (name, shp.C, shp.O)
    variant, C, _, k, s, p = spec[0]
    assert forward_tiles(B, C, H, W, k, s, p, variant) > 2 * 148


def _make_stages(spec, seed):
    torch.manual_seed(seed)
    stages = []
    for variant, C, O, k, s, p in spec:
        layer = CLS[variant](C, O, k, s, p)
        bn = torch.nn.BatchNorm2d(O)
        with torch.no_grad():                   # live offsets, non-trivial statistics
            layer.offset_conv.weight.normal_(0, 0.01)
            layer.offset_conv.bias.normal_(0, 0.7)
            layer.bias.normal_(0, 0.1)
            bn.weight.normal_(1.0, 0.2)
            bn.bias.normal_(0, 0.3)
            bn.running_mean.normal_(0, 0.3)
            bn.running_var.uniform_(0.5, 1.5)
        stages.append((layer.cuda(), bn.cuda().eval()))
    return stages


def _reference_stages(stages, x):
    """float64 relu(bn_eval(dcn(h, conv2d(h, offset weights)))) stage by stage, on the CPU; -> every stage's output."""
    d = lambda t: None if t is None else t.detach().double().cpu()     # noqa: E731
    h, outs = d(x), []
    for layer, bn in stages:
        off = F.conv2d(h, d(layer.offset_conv.weight), d(layer.offset_conv.bias), layer.stride, layer.padding)
        y = chain_forward(h, off, d(layer.weight), d(layer.bias), variant=NAME[layer.variant],
                          kernel_size=layer.kernel_size, stride=layer.stride, padding=layer.padding)
        y = F.batch_norm(y, d(bn.running_mean), d(bn.running_var), d(bn.weight), d(bn.bias), False, 0.0, bn.eps)
        h = torch.relu(y)
        outs.append(h)
    return outs


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", CHAIN_CASES)
def test_chained_stages_match_the_nchw_layers_and_float64(name, B):
    spec, (H, W), _ = CHAINS[name]
    variant, C, _, k, s, p = spec[0]
    assert forward_tiles(B, C, H, W, k, s, p, variant) > 2 * _sms()
    stages = _make_stages(spec, seed=11)
    torch.manual_seed(12)
    x = torch.randn(B, C, H, W, device="cuda")
    chain = dcn.ChainedDeformStages(stages)

    def run():
        with torch.no_grad():
            _lib.profile_begin()
            out = chain(x)
            torch.cuda.synchronize()
            prof = _lib.profile_end()
            # the same folded layers, one after another through the NCHW whole-layer forward (dcn_layer_forward; not the
            # module forward, which keeps the offset conv on the framework where the layer backward is not covered)
            h = x
            for layer in chain.layers:
                h = deform_layer(h, layer.offset_conv.weight, layer.offset_conv.bias, layer.weight, layer.bias,
                                 layer.kernel_size, layer.stride, layer.padding, layer.variant, layer.engine_flags)
            # the unfolded layers with eval-mode BatchNorm and ReLU as separate modules
            m = x
            for layer, bn in stages:
                m = torch.relu(bn(layer(m)))
            return out, prof, h, m
    out, prof, nchw, modules = _no_tf32(run)
    assert prof["nchw_to_nhwc_kernel"][0] == 1, prof
    assert "nhwc_to_nchw_kernel" not in prof, prof
    assert prof["umma_fwd_kernel"][0] == len(spec), prof
    assert torch.equal(out, nchw)           # same arithmetic: only the layout of the hand-over differs
    assert rel_err(out.cpu().numpy(), modules.cpu().numpy()) < 1e-4
    # float64 on the first and the last images (each image is independent of the others): the last ones are computed
    # by tiles past the second wave of every CTA
    idx = sorted({0, 1, B // 2, B - 3, B - 2, B - 1})
    refs = _reference_stages(stages, x[idx])
    for i, ref in enumerate(refs):
        got = dcn.ChainedDeformStages(stages[:i + 1])(x[idx]) if i < len(refs) - 1 else out[idx]
        err = rel_err(got.cpu().numpy(), ref.numpy())
        print(f"float64 chain {name} B={B} stage {i}: {err:.2e}")
        assert err < 1e-4, (name, B, "stage", i, err)


# ---- B. the staged post-op against float64 -------------------------------------------------------------------------
# (variant, C, H, W, stride) of the consumer layer; its output channel count is 64
CONSUMERS = [
    (J, 16, 13, 11, 1),     # narrow tile, H*W % 4 != 0
    (J, 32, 7, 9, 1),
    (J, 64, 15, 15, 2),
    (T, 48, 20, 20, 1),     # G = 16, Cs = 3
    (T, 96, 16, 12, 1),     # G = 96: Gt = 32
    (T, 192, 16, 16, 1),    # G = 64, Cs = 3
    (T, 256, 8, 8, 1),      # G = 64, Cs = 4
]
CONSUMER_IDS = [f"{NAME[v]}-C{C}-{H}x{W}-s{s}" for v, C, H, W, s in CONSUMERS]
# the Torch C = 96 consumer has no whole-layer backward (dcn_path_name(LAYER_BACKWARD) = "unsupported"), so no
# framed gradient is ever produced for it: parts C and D leave it out
TRAINABLE = [c for c in CONSUMERS if not (c[0] == T and c[1] == 96)]
TRAINABLE_IDS = [i for c, i in zip(CONSUMERS, CONSUMER_IDS) if c in TRAINABLE]
BATCH = 40
MODES = {
    "train": dict(momentum=0.1),
    "train-cumulative": dict(momentum=None),
    "eval": dict(momentum=0.1),
    "no-affine": dict(momentum=0.1, affine=False),
    "no-running-stats": dict(momentum=0.1, track_running_stats=False),
}


def test_consumers_run_on_the_tensor_path():
    for variant, C, H, W, s in CONSUMERS:
        shp = _lib.make_shape(BATCH, C, 64, H, W, 3, s, 1, variant)
        assert _lib.path_name(shp, _lib.PHASE_FORWARD) == "umma"
        assert _lib.path_name(shp, _lib.PHASE_LAYER_FORWARD) == "umma"
        trainable = (variant, C, H, W, s) in TRAINABLE
        assert (_lib.path_name(shp, _lib.PHASE_LAYER_BACKWARD) == "umma") == trainable, (variant, C)


def _consumer(variant, C, s):
    layer = CLS[variant](C, 64, 3, s, 1)
    with torch.no_grad():
        layer.offset_conv.weight.normal_(0, 0.01)
        layer.offset_conv.bias.normal_(0, 0.7)
    return layer.cuda()


def _bn_pair(C, mode):
    ours = dcn.BatchNormReLU2d(C, **MODES[mode])
    with torch.no_grad():
        if ours.affine:
            ours.weight.normal_(1.0, 0.2)
            ours.bias.normal_(0, 0.3)
        if ours.track_running_stats:
            ours.running_mean.normal_(0, 0.3)
            ours.running_var.uniform_(0.5, 1.5)
            ours.num_batches_tracked.fill_(3)          # momentum=None: factor 1 / 4
    ref = torch.nn.BatchNorm2d(C, **MODES[mode]).double()
    ref.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in ours.state_dict().items()})
    training = mode != "eval"
    return ours.cuda().train(training), ref.train(training)


def _staged_workspace_bytes(shp):
    lib = _lib.load()
    return max(lib.dcn_workspace_bytes(ctypes.byref(shp), _lib.PHASE_LAYER_FORWARD),
               lib.dcn_workspace_bytes(ctypes.byref(shp), _lib.PHASE_LAYER_BACKWARD))


def _layer_staging(shp, x):
    """The layer's own staging of NCHW x: the head of a dcn_forward workspace (csrc nchw_to_nhwc)."""
    lib = _lib.load()
    B, C, H, W = x.shape
    Ho, Wo = _lib.output_hw(shp)
    ws = torch.empty(lib.dcn_workspace_bytes(ctypes.byref(shp), _lib.PHASE_FORWARD), dtype=torch.uint8, device="cuda")
    off = torch.zeros(B, 2 * shp.kh * shp.kw, Ho, Wo, device="cuda")
    w = torch.zeros(shp.O, C, shp.kh, shp.kw, device="cuda")
    out = torch.empty(B, shp.O, Ho, Wo, device="cuda")
    _run("dcn_forward", x.device, shp, (x.contiguous(), off, w, None, out), _lib.PHASE_FORWARD, ws)
    return ws[:4 * B * (H + 3) * (W + 2) * C].view(torch.float32).view(B, H + 3, W + 2, C)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("consumer", CONSUMERS, ids=CONSUMER_IDS)
def test_staged_post_op_matches_float64(consumer, mode):
    variant, C, H, W, s = consumer
    torch.manual_seed(21)
    layer = _consumer(variant, C, s)
    shp = _lib.make_shape(BATCH, C, 64, H, W, 3, s, 1, variant)
    Ho, Wo = _lib.output_hw(shp)
    perm = staged_channels(C, Ho, Wo, variant)
    x0 = torch.randn(BATCH, C, H, W, device="cuda") * 1.5 + 0.2
    g0 = torch.randn(BATCH, H + 3, W + 2, C, device="cuda")
    g0[:, _frame_mask(H, W, g0.device), :] = float("nan")      # the frame of a framed gradient is never read
    for need_gx in (True, False):
        torch.manual_seed(22)                            # the same parameters and statistics in both passes
        ours, ref = _bn_pair(C, mode)
        x = x0.clone().requires_grad_(need_gx)
        # the consumer workspace comes from the caching allocator: hand it a NaN-filled block of exactly that size
        need = _staged_workspace_bytes(shp)
        poison = torch.empty(need, dtype=torch.uint8, device="cuda")
        poison.view(torch.float32).fill_(float("nan"))
        poisoned_at = poison.data_ptr()
        del poison
        y = ours.forward_staged(x, layer)
        assert _storage_tensor(y).data_ptr() == poisoned_at, "the staged copy did not land in the NaN-filled block"
        assert tuple(y.shape) == (BATCH, H + 3, W + 2, C)
        x64 = x0.detach().double().cpu().requires_grad_(need_gx)
        ref_y = torch.relu(ref(x64))
        interior = unstage(y.detach(), H, W, perm)
        err = rel_err(interior.cpu().numpy(), ref_y.detach().numpy())
        print(f"float64 post-op {mode} C={C} forward: {err:.2e}")
        assert err < 1e-5, (mode, err)
        assert torch.equal(frame_of(y.detach(), H, W), torch.zeros_like(frame_of(y.detach(), H, W)))
        staging = _layer_staging(shp, ref_y.detach().float().cuda())
        scale = float(ref_y.detach().abs().max())
        assert float((y.detach()[:, 1:H + 1, 1:W + 1] - staging[:, 1:H + 1, 1:W + 1]).abs().max()) <= 1e-6 * scale
        for k, v in ref.state_dict().items():
            mine = ours.state_dict()[k].cpu()
            if k == "num_batches_tracked":
                assert int(mine) == int(v), k
            else:
                assert rel_err(mine.numpy(), v.numpy()) < 1e-5, (mode, k)
        if not y.requires_grad:                          # no affine parameters and no grad_x wanted: nothing to do
            continue
        y.backward(g0)
        leaves = ([x64] if need_gx else []) + ([ref.weight, ref.bias] if ref.affine else [])
        grads = torch.autograd.grad(ref_y, leaves, unstage(g0, H, W, perm).double().cpu())
        got = ([x.grad] if need_gx else []) + ([ours.weight.grad, ours.bias.grad] if ours.affine else [])
        for a, b, what in zip(got, grads, (["grad_x"] if need_gx else []) + ["grad_gamma", "grad_beta"]):
            assert a is not None, what
            err = rel_err(a.cpu().numpy(), b.numpy())
            print(f"float64 post-op {mode} C={C} {what} (grad_x requested: {need_gx}): {err:.2e}")
            assert err < 1e-4, (mode, what, need_gx, err)
        if not need_gx:
            assert x.grad is None


# ---- C. the framed data gradient ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("consumer", TRAINABLE, ids=TRAINABLE_IDS)
def test_framed_grad_x_equals_the_nchw_grad_x(consumer):
    """dcn_layer_backward with DCN_FLAG_GRAD_X_FRAMED writes grad_x as the layer's staging layout; un-permuted, it is
    the NCHW grad_x of the same call without the flag (only the order of the atomics differs)."""
    variant, C, H, W, s = consumer
    lib = _lib.load()
    torch.manual_seed(31)
    layer = _consumer(variant, C, s)
    x = torch.randn(BATCH, C, H, W, device="cuda")
    off = _no_tf32(lambda: F.conv2d(x, layer.offset_conv.weight, layer.offset_conv.bias, layer.stride, layer.padding))
    Ho, Wo = off.shape[2:]
    gout = torch.randn(BATCH, 64, Ho, Wo, device="cuda")
    results = []
    for framed in (False, True):
        shp = _lib.make_shape(BATCH, C, 64, H, W, 3, s, 1, variant, _lib.OPERAND_FP32,
                              _lib.FLAG_GRAD_X_FRAMED if framed else 0)
        ws = torch.empty(lib.dcn_workspace_bytes(ctypes.byref(shp), _lib.PHASE_LAYER_BACKWARD), dtype=torch.uint8,
                         device="cuda")
        if framed:
            gx = torch.full((BATCH, H + 3, W + 2, C), float("nan"), device="cuda")
            assert gx.numel() * 4 <= lib.dcn_staged_input_bytes(ctypes.byref(shp))
        else:
            gx = torch.full((BATCH, C, H, W), float("nan"), device="cuda")
        grads = [torch.empty_like(layer.offset_conv.weight), torch.empty_like(layer.offset_conv.bias),
                 torch.empty_like(layer.weight), torch.empty_like(layer.bias)]
        _run("dcn_layer_backward", x.device, shp,
             (x, off, layer.offset_conv.weight, layer.weight, gout, gx, *grads), _lib.PHASE_LAYER_BACKWARD, ws)
        torch.cuda.synchronize()
        results.append((gx, grads))
    (gx_nchw, g_nchw), (gx_framed, g_framed) = results
    interior = unstage(gx_framed, H, W, staged_channels(C, Ho, Wo, variant))
    assert torch.isfinite(interior).all()
    assert rel_err(interior.cpu().numpy(), gx_nchw.cpu().numpy()) < 1e-5
    for a, b, what in zip(g_framed, g_nchw, ("grad_offset_weight", "grad_offset_bias", "grad_weight", "grad_bias")):
        assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 1e-5, what


# ---- D. end to end ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("consumer", TRAINABLE, ids=TRAINABLE_IDS)
def test_staged_training_step_equals_the_nchw_path(consumer):
    """bn.forward_staged -> layer.forward_staged -> loss against bn(x) -> layer(.) -> loss: loss, output, running
    statistics and every gradient, at the tolerances of the detector's channels-last training step."""
    variant, C, H, W, s = consumer
    torch.manual_seed(41)
    layer_a = _consumer(variant, C, s)
    layer_b = CLS[variant](C, 64, 3, s, 1).cuda()
    layer_b.load_state_dict(layer_a.state_dict())
    bn_a = dcn.BatchNormReLU2d(C).cuda().train()
    with torch.no_grad():
        bn_a.weight.normal_(1.0, 0.2)
        bn_a.bias.normal_(0, 0.3)
    bn_b = dcn.BatchNormReLU2d(C).cuda().train()
    bn_b.load_state_dict(bn_a.state_dict())
    x = torch.randn(BATCH, C, H, W, device="cuda")
    Ho, Wo = out_hw(H, W, 3, s, 1)
    wloss = torch.randn(BATCH, 64, Ho, Wo, device="cuda")

    def step():
        xa = x.clone().requires_grad_(True)
        ya = layer_a(bn_a(xa))
        loss_a = (ya * wloss).sum()
        loss_a.backward()
        xb = x.clone().requires_grad_(True)
        yb = layer_b.forward_staged(bn_b.forward_staged(xb, layer_b), (H, W))
        loss_b = (yb * wloss).sum()
        loss_b.backward()
        return xa, ya, loss_a, xb, yb, loss_b
    xa, ya, loss_a, xb, yb, loss_b = _no_tf32(step)
    assert abs(float(loss_b) - float(loss_a)) < 1e-5 * abs(float(loss_a))
    assert rel_err(yb.detach().cpu().numpy(), ya.detach().cpu().numpy()) < 1e-5
    for (k, v), (_, w) in zip(bn_b.state_dict().items(), bn_a.state_dict().items()):
        if "running_" in k:
            assert rel_err(v.cpu().numpy(), w.cpu().numpy()) < 1e-5, k
    pairs = [("x", xb.grad, xa.grad)] + [
        (k, p.grad, q.grad) for (k, p), (_, q) in zip(list(bn_b.named_parameters()) + list(layer_b.named_parameters()),
                                                      list(bn_a.named_parameters()) + list(layer_a.named_parameters()))]
    for k, p, q in pairs:
        scale = float(q.abs().max())
        if scale < 1e-4:                 # a bias in front of a BatchNorm: round-off of a zero sum on both sides
            assert float(p.abs().max()) < 1e-3, k
        else:
            assert rel_err(p.cpu().numpy(), q.cpu().numpy()) < 2e-4, k
