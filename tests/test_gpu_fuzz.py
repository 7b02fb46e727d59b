"""Shape fuzz: random problems that route to the tensor path, checked against the generic
kernels (which the fixed-shape tests pin to the oracle and the reference goldens).  Exercises the
tile edge cases: partial row tiles, instance counts that do not fill a tile, K not a multiple of
64 / 128, channel permutations (Cs > 1), 16-channel groups, 1x1 and rectangular taps, stride 2,
fused and unfused backward, both layouts, both operand modes.

The DCNv1 / DCNv2 draw (torchvision's operator, with and without `mask`) is checked against
torchvision itself in float64 instead: an independent reference that shares no sampling code
with either kernel family.  It adds per-axis strides and paddings, output-channel groups
(O > 256), integer and half-integer offsets (exact floor ties, samples exactly on the image
border) and masks with exact 0 / 1, negative and > 1 entries."""
import ctypes

import numpy as np
import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from tests.util import rel_err


def _cases(seed, n):
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        C = int(rng.choice([16, 32, 64, 128, 192, 256]))
        O = int(rng.choice([16, 32, 48, 64, 80, 128, 144, 256]))
        k = [(3, 3), (1, 1), (3, 1), (1, 3), (5, 5)][int(rng.integers(0, 5))]
        s = int(rng.choice([1, 2]))
        p = (k[0] // 2, k[1] // 2)
        if rng.random() < 0.6:   # extents with Ho*Wo % 16 == 0 so that the Torch layout tiles (gcd(Ho*Wo, C) % 16)
            H, W = 4 * s * int(rng.integers(2, 9)), 4 * s * int(rng.integers(2, 9))
        else:
            H, W = int(rng.integers(6, 40)), int(rng.integers(6, 40))
        B = int(rng.integers(1, 4))
        variant = int(rng.integers(0, 2))
        out.append((B, C, O, H, W, k, s, p, variant))
    return out


def _rel(a, b):
    den = float(b.double().abs().max())
    return float((a.double() - b.double()).abs().max() / (den if den > 0 else 1.0))


@pytest.mark.gpu
@pytest.mark.parametrize("case", _cases(2026, 90))
def test_fuzz_tensor_path_vs_generic(case):
    B, C, O, H, W, k, s, p, variant = case
    lib = dcn.load()
    shp = dcn.make_shape(B, C, O, H, W, k, s, p, variant)
    Ho, Wo = (H + 2 * p[0] - k[0]) // s + 1, (W + 2 * p[1] - k[1]) // s + 1
    if variant == dcn.VARIANT_JITTOR and min(Ho, Wo) < 2:
        pytest.skip("output extent 1: the reference divides by zero")
    paths = (lib.dcn_path_name(ctypes.byref(shp), 0), lib.dcn_path_name(ctypes.byref(shp), 1))
    if paths == (b"simt", b"simt"):
        pytest.skip("shape does not tile onto the tensor path")
    g = torch.Generator(device="cuda").manual_seed(hash(case) & 0xffff)
    N = k[0] * k[1]
    x = torch.randn(B, C, H, W, device="cuda", generator=g)
    off = torch.randn(B, 2 * N, Ho, Wo, device="cuda", generator=g) * 2.0
    wt = torch.randn(O, C, *k, device="cuda", generator=g) * (2.0 / (C * N)) ** 0.5
    bias = torch.randn(O, device="cuda", generator=g)
    gout = torch.randn(B, O, Ho, Wo, device="cuda", generator=g)
    out_u = dcn.dcn_forward(x, off, wt, bias, k, s, p, variant)
    out_s = dcn.dcn_forward(x, off, wt, bias, k, s, p, variant, flags=dcn.FLAG_FORCE_SIMT)
    assert _rel(out_u, out_s) < 1e-4, ("fwd", paths)
    gu = dcn.dcn_backward(x, off, wt, gout, True, k, s, p, variant)
    gs = dcn.dcn_backward(x, off, wt, gout, True, k, s, p, variant, flags=dcn.FLAG_FORCE_SIMT)
    for a, b, nm in zip(gu, gs, ("gx", "goff", "gw", "gb")):
        assert _rel(a, b) < 1e-3, (nm, paths)


@pytest.mark.gpu
@pytest.mark.parametrize("case", _cases(7, 30))
def test_fuzz_bf16_vs_fp32(case):
    B, C, O, H, W, k, s, p, variant = case
    lib = dcn.load()
    shp = dcn.make_shape(B, C, O, H, W, k, s, p, variant, operand=dcn.OPERAND_BF16)
    Ho, Wo = (H + 2 * p[0] - k[0]) // s + 1, (W + 2 * p[1] - k[1]) // s + 1
    if variant == dcn.VARIANT_JITTOR and min(Ho, Wo) < 2:
        pytest.skip("output extent 1")
    if lib.dcn_path_name(ctypes.byref(shp), 0) != b"umma" or lib.dcn_path_name(ctypes.byref(shp), 1) != b"umma":
        pytest.skip("bf16 needs the tensor path for forward and backward")
    g = torch.Generator(device="cuda").manual_seed(hash(case) & 0xffff)
    N = k[0] * k[1]
    x = torch.randn(B, C, H, W, device="cuda", generator=g).bfloat16()
    off = torch.randn(B, 2 * N, Ho, Wo, device="cuda", generator=g) * 1.5
    wt = (torch.randn(O, C, *k, device="cuda", generator=g) * (2.0 / (C * N)) ** 0.5).bfloat16()
    gout = torch.randn(B, O, Ho, Wo, device="cuda", generator=g).bfloat16()
    out_b = dcn.dcn_forward(x, off, wt, None, k, s, p, variant, operand=dcn.OPERAND_BF16)
    out_f = dcn.dcn_forward(x.float(), off, wt.float(), None, k, s, p, variant)
    assert _rel(out_b, out_f) < 1e-2
    gb_ = dcn.dcn_backward(x, off, wt, gout, True, k, s, p, variant, operand=dcn.OPERAND_BF16)
    gf_ = dcn.dcn_backward(x.float(), off, wt.float(), gout.float(), True, k, s, p, variant)
    for a, b, nm in zip(gb_, gf_, ("gx", "goff", "gw", "gb")):
        assert _rel(a, b) < 2e-2, nm


# ---- DCNv1 / DCNv2 against torchvision -------------------------------------------------------------------------------
FP32, BF16 = dcn.OPERAND_FP32, dcn.OPERAND_BF16
_V1_MACS = 1.2e8   # B*Ho*Wo*N*C*O cap: keeps the float64 CPU reference of one case well under a second


def _v1_cases(seed, n):
    """(B, C, O, H, W, k, s, p, offsets, modulated, operand, data seed).  The channel class (16, 32, 64, >= 128),
    the mask and the operand mode cycle with the case index so that every combination is drawn; offsets are
    "grid" (integers and half-integers) for every third case, else normal with sigma 2."""
    rng = np.random.default_rng(seed)
    kernels = [(3, 3), (1, 1), (3, 1), (1, 3), (5, 5)]
    out = []
    for i in range(n):
        cls, modulated, operand = i % 4, bool((i // 4) % 2), (FP32, BF16)[(i // 8) % 2]
        C = (16, 32, 64, int(rng.choice([128, 192, 256])))[cls]
        O = int(rng.choice([16, 48, 64, 80, 144, 256, 320]))
        while True:
            k = kernels[int(rng.integers(0, len(kernels)))]
            s = (int(rng.choice([1, 2])), int(rng.choice([1, 2])))
            p = (int(rng.integers(0, 3)), int(rng.integers(0, 3)))
            H, W = int(rng.integers(5, 41)), int(rng.integers(5, 41))
            B = int(rng.integers(1, 4))
            if H + 2 * p[0] < k[0] or W + 2 * p[1] < k[1]:
                continue
            Ho, Wo = (H + 2 * p[0] - k[0]) // s[0] + 1, (W + 2 * p[1] - k[1]) // s[1] + 1
            if B * Ho * Wo * k[0] * k[1] * C * O <= _V1_MACS:
                break
        offsets = "grid" if i % 3 == 0 else "normal"
        out.append((B, C, O, H, W, k, s, p, offsets, modulated, operand, seed * 1000 + i))
    return out


V1_CASES = _v1_cases(2027, 96)


def _v1_paths(case):
    B, C, O, H, W, k, s, p, _, _, operand, _ = case
    shp = dcn.make_shape(B, C, O, H, W, k, s, p, dcn.VARIANT_DCNV1, operand)
    return [_lib.path_name(shp, ph) for ph in (_lib.PHASE_FORWARD, _lib.PHASE_BACKWARD)]


def test_fuzz_dcnv1_draw_covers_tensor_path():
    """The DCNv1 / DCNv2 draw reaches the tensor path (both phases) for every channel class x mask x operand mode, and
    with each of the edges it is meant to exercise (no GPU needed: routing is a host decision)."""
    umma = [c for c in V1_CASES if _v1_paths(c) == ["umma", "umma"]]
    seen = {(min(c[1], 128), c[9], c[10]) for c in umma}
    want = {(C, m, op) for C in (16, 32, 64, 128) for m in (False, True) for op in (FP32, BF16)}
    assert want <= seen, sorted(want - seen)
    assert any(2 in c[6] for c in umma), "stride 2"
    assert any(c[6] == (1, 2) or c[6] == (2, 1) for c in umma), "mixed per-axis stride"
    assert any(c[2] > 256 for c in umma), "O > 256 (output-channel groups)"
    assert any(c[7] != (c[5][0] // 2, c[5][1] // 2) for c in umma), "padding != k // 2"
    assert any(c[8] == "grid" for c in umma), "integer offsets"


def _tv_reference(x, off, mask, w, b, gout, s, p):
    """torchvision.ops.deform_conv2d on the CPU in float64: out and the gradients of x, offset, mask, weight, bias."""
    from torchvision.ops import deform_conv2d
    leaves = [t.double().requires_grad_(True) for t in (x, off, w, b)]
    tm = mask.double().requires_grad_(True) if mask is not None else None
    out = deform_conv2d(leaves[0], leaves[1], leaves[2], leaves[3], stride=s, padding=p, mask=tm)
    grads = torch.autograd.grad(out, leaves + ([tm] if tm is not None else []), gout.double())
    gx, goff, gw, gb = grads[:4]
    return out.detach(), (gx, goff, grads[4] if tm is not None else None, gw, gb)


@pytest.mark.gpu
@pytest.mark.parametrize("case", V1_CASES)
def test_fuzz_dcnv1_vs_torchvision(case):
    B, C, O, H, W, k, s, p, offsets, modulated, operand, seed = case
    Ho, Wo = (H + 2 * p[0] - k[0]) // s[0] + 1, (W + 2 * p[1] - k[1]) // s[1] + 1
    N = k[0] * k[1]
    rng = np.random.default_rng(seed)
    x = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32))
    if offsets == "grid":
        off = torch.from_numpy((rng.integers(-4, 5, (B, 2 * N, Ho, Wo)) / 2).astype(np.float32))
    else:
        # on a 2^-10 grid: every sampling coordinate (tap position + offset) is then exact in float32 as in float64.
        # Otherwise a float32 sum can round onto an integer the float64 one stays below, and floor() - hence the
        # corner cell and the coordinate gradient - differs between the kernels and the float64 reference.
        off = torch.from_numpy((np.round(rng.standard_normal((B, 2 * N, Ho, Wo)) * 2048.0) / 1024.0).astype(np.float32))
    from oracle.make_golden_dcnv2 import dcnv2_mask
    mask = torch.from_numpy(dcnv2_mask(rng, (B, N, Ho, Wo))) if modulated else None
    w = torch.from_numpy((rng.standard_normal((O, C, *k)) * np.sqrt(2.0 / (C * N))).astype(np.float32))
    b = torch.from_numpy(rng.standard_normal(O).astype(np.float32))
    gout = torch.from_numpy(rng.standard_normal((B, O, Ho, Wo)).astype(np.float32))
    if operand == BF16:   # the reference sees exactly the operands the kernels get
        x, w, gout = (t.bfloat16().float() for t in (x, w, gout))
        tol_out, tol_g = 1e-2, 2e-2
    else:
        tol_out, tol_g = 1e-4, 1e-3
    ref_out, ref_grads = _tv_reference(x, off, mask, w, b, gout, s, p)
    act = torch.bfloat16 if operand == BF16 else torch.float32
    tx, tw, tg = (t.to(act).cuda() for t in (x, w, gout))
    toff, tb = off.cuda(), b.cuda()
    if modulated:
        tm = mask.cuda()
        out = dcn.dcn_forward_modulated(tx, toff, tm, tw, tb, k, s, p, operand=operand)
        grads = dcn.dcn_backward_modulated(tx, toff, tm, tw, tg, True, k, s, p, operand=operand)
    else:
        out = dcn.dcn_forward(tx, toff, tw, tb, k, s, p, dcn.VARIANT_DCNV1, operand=operand)
        gx, goff, gw, gb = dcn.dcn_backward(tx, toff, tw, tg, True, k, s, p, dcn.VARIANT_DCNV1, operand=operand)
        grads = (gx, goff, None, gw, gb)
    torch.cuda.synchronize()
    what = (_v1_paths(case), case)
    err = rel_err(out.cpu().numpy(), ref_out.numpy())
    assert err < tol_out, ("out", err, what)
    for nm, a, r in zip(("gx", "goff", "gmask", "gw", "gb"), grads, ref_grads):
        if r is None:
            continue
        err = rel_err(a.cpu().numpy(), r.numpy())
        assert err < tol_g, (nm, err, what)
