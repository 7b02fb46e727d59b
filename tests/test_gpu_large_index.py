"""The tensor-path kernels past 2^31 elements.

make_geo bounds every per-tap index space at 2^31 - 1, B*N*Ho*Wo in particular, but grad_offset (B*2N*Ho*Wo
elements) and, for wide layers, x / out / grad_out / grad_x may hold more than 2^31 elements.  Each case runs one
big call whose tail images lie past that line and checks it against plain small calls of the same entry point
(same variant, flags and operand mode; a small call keeps every index below 2^31, and the rest of the suite pins
small calls to the oracle and to torchvision):
  * per-image tensors (out, grad_x, grad_offset, grad_mask) of image 0, the last image wholly below the line, the
    image that straddles it, the first image wholly past it and image B - 1, against the same images run alone;
  * batch reductions (grad_weight, grad_bias) against the float64 sum of the same entry point over chunks of at
    most 4096 images, and — with grad_out zero outside the chosen images, so that the big call's long float32
    accumulations add exact zeros — against the float64 sum of those images' own calls;
  * DCNv1: image B - 1 of the big call against torchvision.ops.deform_conv2d in float64 on the CPU.
The kernel profile of the big calls shows that they ran on the tensor-path kernels, data gradient included.

The cases need tens of GB (at most about 60 GB at the peak, see CASES): each computes what it needs before it
allocates anything and skips when the device has less free memory.
"""
import ctypes
import time
import zlib

import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib

pytestmark = pytest.mark.gpu

LINE = 1 << 31
CHUNK = 4096          # images per call of the reduction reference
MARGIN = 2 << 30      # allocator rounding, CUDA context, the small reference calls

FP32, BF16 = dcn.OPERAND_FP32, dcn.OPERAND_BF16

# name: (B, C, O, H, W, k, p, variant, modulated, operand, tensor that crosses the line)
#   A: grad_offset holds 1.06 * 2^31 elements (C = 16 keeps every other tensor small); images from 34 663 on are
#      past the line, 2 200 of them wholly.  Backward: 20.7 GB of tensors + 19.1 GB of workspace (+ 9.1 GB mask and
#      grad_mask for A-mod).  The fp32 workspace is sized for the generic data gradient's sampling plan too (18.3 GB),
#      which these calls do not use; bf16 operands need 2.4 GB.
#   B: x, out, grad_out and grad_x each hold more than 2^31 elements (staging transposes, forward epilogue, grad_out
#      staging, bias gradient); images from 8 192 on.  Forward 29 GB, backward 31 GB + 27.6 GB workspace.
CASES = {
    "A-dcnv1": (36864, 16, 16, 16, 16, 11, 5, dcn.VARIANT_DCNV1, False, FP32, "goff"),
    "A-torch": (36864, 16, 16, 16, 16, 11, 5, dcn.VARIANT_TORCH, False, FP32, "goff"),
    "A-jittor": (36864, 16, 16, 16, 16, 11, 5, dcn.VARIANT_JITTOR, False, FP32, "goff"),
    "A-mod": (36864, 16, 16, 16, 16, 11, 5, dcn.VARIANT_DCNV1, True, FP32, "goff"),
    "A-bf16": (36864, 16, 16, 16, 16, 11, 5, dcn.VARIANT_DCNV1, True, BF16, "goff"),
    "B-dcnv1": (8320, 64, 64, 64, 64, 3, 1, dcn.VARIANT_DCNV1, False, FP32, "x"),
    "B-torch": (8320, 64, 64, 64, 64, 3, 1, dcn.VARIANT_TORCH, False, FP32, "x"),
}
# kernels (dcn_profile_end names) that must / must not run in the big calls: the generic kernels would compute the
# same answer with 64-bit indices and leave the tensor-path kernels untested
FWD_KERNELS, FWD_GENERIC = {"umma_fwd_kernel"}, {"fwd_kernel", "plan_kernel"}
BWD_KERNELS, BWD_GENERIC = {"umma_bwd_data_kernel"}, {"bwd_data_kernel", "plan_kernel"}


def _images(B, per_image):
    """0, the last image wholly below 2^31, the one straddling it (if any), the first wholly past it, B - 1."""
    last_below = LINE // per_image - 1
    first_past = -(-LINE // per_image)
    assert first_past < B, "the case does not reach past the line"
    picks = {0, last_below, first_past, B - 1}
    if LINE % per_image:
        picks.add(LINE // per_image)
    return sorted(picks)


def _fill(t, gen, kind, a, b=0.0):
    """In-place random fill on the device, 2^28 elements at a time (no temporaries of the big tensor's size)."""
    flat = t.view(-1)
    for i in range(0, flat.numel(), 1 << 28):
        part = flat[i:i + (1 << 28)]
        if kind == "normal":
            part.normal_(0.0, a, generator=gen)
        else:
            part.uniform_(a, b, generator=gen)
    return t


def _rel(a, b):
    a, b = a.double(), b.double()
    den = float(b.abs().max())
    return float((a - b).abs().max()) / (den if den > 0 else 1.0)


class _Span:
    """One entry point (dcn_forward / dcn_backward, or their modulated forms) with fixed shape arguments.
    backward -> (grad_x, grad_offset, grad_mask or None, grad_weight, grad_bias)."""

    def __init__(self, k, p, variant, modulated, operand):
        self.k, self.p, self.variant, self.modulated, self.operand = k, p, variant, modulated, operand

    def forward(self, x, off, mask, w, b):
        if self.modulated:
            return dcn.dcn_forward_modulated(x, off, mask, w, b, self.k, 1, self.p, operand=self.operand)
        return dcn.dcn_forward(x, off, w, b, self.k, 1, self.p, self.variant, operand=self.operand)

    def backward(self, x, off, mask, w, g):
        if self.modulated:
            return dcn.dcn_backward_modulated(x, off, mask, w, g, True, self.k, 1, self.p, operand=self.operand)
        gx, goff, gw, gb = dcn.dcn_backward(x, off, w, g, True, self.k, 1, self.p, self.variant, operand=self.operand)
        return gx, goff, None, gw, gb


def _profiled(fn, *args):
    """fn(*args) -> (its result, the names of the library kernels it launched)."""
    _lib.profile_begin()
    res = fn(*args)
    torch.cuda.synchronize()
    return res, set(_lib.profile_end())


def _tv_image(x, off, mask, w, b, g, k, p):
    """torchvision's CPU operator in float64 on one image: out, grad_x, grad_offset, grad_mask."""
    from torchvision.ops import deform_conv2d
    leaves = [t.cpu().double().requires_grad_(True) for t in (x, off)]
    tm = mask.cpu().double().requires_grad_(True) if mask is not None else None
    out = deform_conv2d(leaves[0], leaves[1], w.cpu().double(), b.cpu().double(), stride=1, padding=p, mask=tm)
    grads = torch.autograd.grad(out, leaves + ([tm] if tm is not None else []), g.cpu().double())
    return out.detach(), grads[0], grads[1], grads[2] if tm is not None else None


@pytest.mark.parametrize("name", list(CASES))
def test_past_2_31_elements(name):
    B, C, O, H, W, k, p, variant, modulated, operand, crossing = CASES[name]
    N = k * k
    shp = dcn.make_shape(B, C, O, H, W, k, 1, p, variant, operand)
    Ho, Wo = _lib.output_hw(shp)
    HW = Ho * Wo
    assert [_lib.path_name(shp, ph) for ph in (_lib.PHASE_FORWARD, _lib.PHASE_BACKWARD)] == ["umma", "umma"]
    per_image = {"goff": 2 * N * HW, "x": C * H * W}[crossing]
    assert B * per_image > LINE
    imgs = _images(B, per_image)

    # ---- memory: everything each phase holds at once, from the shape, before anything is allocated
    lib = dcn.load()
    f4, fa = 4, 2 if operand == BF16 else 4    # float32 / operand element bytes (x, weight, grad_out)
    n_x, n_off, n_mask, n_out = B * C * H * W, B * 2 * N * HW, B * N * HW if modulated else 0, B * O * HW
    small = f4 * (O * C * N + O) * 2
    fwd = fa * n_x + f4 * (n_off + n_mask + n_out) + small + \
        lib.dcn_workspace_bytes(ctypes.byref(shp), _lib.PHASE_FORWARD)
    bwd = (fa + f4) * n_x + f4 * (2 * n_off + 2 * n_mask) + fa * n_out + small + \
        lib.dcn_workspace_bytes(ctypes.byref(shp), _lib.PHASE_BACKWARD)
    need = max(fwd, bwd) + MARGIN
    dcn.clear_workspaces()
    torch.cuda.empty_cache()
    free, total = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"{name} needs {need / 1e9:.1f} GB of device memory, {free / 1e9:.1f} GB free")

    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    span = _Span(k, p, variant, modulated, operand)
    act = torch.bfloat16 if operand == BF16 else torch.float32
    T = {}          # every big tensor lives here only, so that a failure cannot keep it alive
    results = []    # (what, rel_err, tolerance); asserted once everything is freed
    routing = []    # kernels that ran where they should not, or did not run where they should
    try:
        gen = torch.Generator(device="cuda").manual_seed(zlib.crc32(name.encode()))
        T["x"] = _fill(torch.empty(B, C, H, W, device="cuda", dtype=act), gen, "normal", 1.0)
        T["off"] = _fill(torch.empty(B, 2 * N, Ho, Wo, device="cuda"), gen, "normal", 1.5)
        T["mask"] = _fill(torch.empty(B, N, Ho, Wo, device="cuda"), gen, "uniform", -0.25, 1.25) if modulated else None
        w = _fill(torch.empty(O, C, k, k, device="cuda", dtype=act), gen, "normal", (2.0 / (C * N)) ** 0.5)
        bias = _fill(torch.empty(O, device="cuda"), gen, "normal", 1.0)

        def img(key, i):
            return None if T[key] is None else T[key][i:i + 1]

        # ---- forward: the chosen images of the big call against the same images alone
        T["out"], ran = _profiled(span.forward, T["x"], T["off"], T["mask"], w, bias)
        routing += [f"forward: {n} did not run" for n in sorted(FWD_KERNELS - ran)]
        routing += [f"forward: {n} ran" for n in sorted(FWD_GENERIC & ran)]
        out_img = {i: T["out"][i:i + 1].clone() for i in imgs}
        del T["out"]
        dcn.clear_workspaces()
        torch.cuda.empty_cache()
        for i in imgs:
            ref = span.forward(img("x", i), img("off", i), img("mask", i), w, bias)
            results.append((f"out[{i}]", _rel(out_img[i], ref), 1e-5))

        # ---- backward
        T["gout"] = _fill(torch.empty(B, O, Ho, Wo, device="cuda", dtype=act), gen, "normal", 1.0)
        (T["gx"], T["goff"], T["gmask"], gw, gb), ran = _profiled(span.backward, T["x"], T["off"], T["mask"], w,
                                                                  T["gout"])
        routing += [f"backward: {n} did not run" for n in sorted(BWD_KERNELS - ran)]
        routing += [f"backward: {n} ran" for n in sorted(BWD_GENERIC & ran)]
        names = ("gx", "goff", "gmask")
        big_img = {(nm, i): img(nm, i).clone() for nm in names if T[nm] is not None for i in imgs}
        del T["gx"], T["goff"], T["gmask"]
        torch.cuda.empty_cache()
        gw_imgs = torch.zeros(gw.shape, dtype=torch.float64, device="cuda")   # the chosen images' own reductions
        gb_imgs = torch.zeros(gb.shape, dtype=torch.float64, device="cuda")
        for i in imgs:
            ref = span.backward(img("x", i), img("off", i), img("mask", i), w, img("gout", i))
            for nm, r in zip(names, ref[:3]):
                if r is not None:
                    results.append((f"{nm}[{i}]", _rel(big_img[(nm, i)], r), 1e-5))
            gw_imgs += ref[3].double()
            gb_imgs += ref[4].double()
        # batch reductions: float64 sum of the same entry point over chunks of images
        gw_ref = torch.zeros(gw.shape, dtype=torch.float64, device="cuda")
        gb_ref = torch.zeros(gb.shape, dtype=torch.float64, device="cuda")
        for c0 in range(0, B, CHUNK):
            sl = slice(c0, min(B, c0 + CHUNK))
            T["part"] = span.backward(T["x"][sl], T["off"][sl], None if T["mask"] is None else T["mask"][sl], w,
                                      T["gout"][sl])
            gw_ref += T["part"][3].double()
            gb_ref += T["part"][4].double()
            del T["part"]
        # grad_weight sums B*Ho*Wo products in float32 accumulators that each CTA carries over all of its tiles, so its
        # rounding error grows with the batch: 5e-4 .. 1.4e-3 against the chunked sum on a B200.  At this tolerance the
        # check catches a lost batch tail, not one lost image (~5e-3 of max |grad_weight| in case A) or tile: the
        # check below does.
        results.append(("grad_weight", _rel(gw, gw_ref), 3e-3))
        results.append(("grad_bias", _rel(gb, gb_ref), 1e-4))
        # the same reductions with grad_out zero outside the chosen images: every other image adds exact zeros, so the
        # big call must reproduce the chosen images' own sum to float32 rounding, whatever its accumulation length
        keep = {i: img("gout", i).clone() for i in imgs}
        T["gout"].zero_()
        for i in imgs:
            T["gout"][i:i + 1] = keep[i]
        T["part"] = span.backward(T["x"], T["off"], T["mask"], w, T["gout"])
        results.append(("grad_weight, chosen images", _rel(T["part"][3], gw_imgs), 1e-5))
        results.append(("grad_bias, chosen images", _rel(T["part"][4], gb_imgs), 1e-5))
        del T["part"]

        # ---- DCNv1: the last image against torchvision in float64
        if variant == dcn.VARIANT_DCNV1:
            i = B - 1
            ref = _tv_image(img("x", i), img("off", i), img("mask", i), w, bias, img("gout", i), k, p)
            got = (out_img[i], big_img[("gx", i)], big_img[("goff", i)], big_img.get(("gmask", i)))
            tols = (1e-2, 2e-2, 2e-2, 2e-2) if operand == BF16 else (1e-4, 1e-3, 1e-3, 1e-3)
            for nm, a, r, tol in zip(("out", "gx", "goff", "gmask"), got, ref, tols):
                if r is not None:
                    results.append((f"torchvision {nm}[{i}]", _rel(a.cpu(), r), tol))
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
    finally:
        T.clear()
        dcn.clear_workspaces()
        torch.cuda.empty_cache()
    print(f"\n[{name}] {torch.cuda.get_device_name()} ({total / 2**30:.1f} GiB): B={B} C={C} O={O} {H}x{W} k={k} "
          f"images {imgs}: need {need / 1e9:.1f} GB, peak {peak / 1e9:.1f} GB, {time.perf_counter() - t0:.1f} s")
    for what, err, tol in results:
        print(f"  {what:24s} rel_err {err:.3g}  (<= {tol:g})")
    for what in routing:
        print(f"  routing: {what}")
    bad = [(what, err) for what, err, tol in results if not err <= tol]
    assert not routing and not bad, f"{name}: {routing} {bad}"
