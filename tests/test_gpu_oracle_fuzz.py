"""Seeded fuzz of the reference's two operators (VARIANT_TORCH, VARIANT_JITTOR) on every kernel path, against the
float64 C oracle (oracle/dcn_oracle.c).

The oracle replays the reference's fp32 coordinate chain bit-exactly (test_gpu_parity.py::test_corners_bit_exact*) and
accumulates every sum in double, so it shares nothing with the engine but the chain's definition: no coordinate code,
no bias-gradient kernel, no staging copy, no Python wrapper.  The draw routes to each of the engine's kernel families:

  * Torch layout on the tensor path (tcgen05): G = gcd(Ho*Wo, C) of 16, 32 and 64 channels per sampling point, so
    each tile width Gt; more channels than one sampling point's class holds (Cs = C / G > 1, the channel-permuted
    staging copy); partial last tiles; the fused weight gradient (O <= 128, or <= 256 with bf16 operands) and the
    separate weight-gradient kernel (fp32, 128 < O <= 256); output-channel groups (O > 256);
  * Jittor layout on the tensor path: 16, 32, 64 and >= 128 channels, pixel counts that leave a partial 128-pixel
    tile, output-channel groups, and C = 192 whose data gradient runs on the generic kernel;
  * the Torch layout's materialised-sample + GEMM path (G not a multiple of 16) and the generic SIMT kernels;

with per-axis strides and paddings, rectangular kernels, fp32 and bf16 operands, and offsets that are normal, exact
integers and half-integers (floor ties, samples exactly on the border), all zero, or normal with outliers far enough
out that every corner lies outside the image (the frame-only block of dcn_umma_common.cuh:xt_corner_base).  Some cases
also set a flag: the ReLU epilogue, accumulation into a given grad_x, no grad_x, or a backward that reuses the
forward's staged input.

Tolerances are those of test_gpu_parity.py: fp32 1e-4 forward, 1e-3 gradients; bf16 operands (DESIGN.md §4) are
checked against the oracle on the bf16-rounded x, weight and grad_out at 1e-2 / 2e-2."""
import math

import numpy as np
import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from jittor_dcn_b200.functional import staged_workspace
from oracle import dcn_oracle as orc
from tests.util import rel_err

TORCH, JITTOR = dcn.VARIANT_TORCH, dcn.VARIANT_JITTOR
FP32, BF16 = dcn.OPERAND_FP32, dcn.OPERAND_BF16
RELU, ACCUM, NO_GX, STAGED = dcn.FLAG_RELU_OUT, dcn.FLAG_ACCUM_GRAD_X, dcn.FLAG_NO_GRAD_X, _lib.FLAG_XT_STAGED
KERNELS = [(3, 3), (1, 1), (3, 1), (1, 3), (5, 5), (3, 5)]
OFFSETS = ("normal", "grid", "zero", "far")
FLAGS = (RELU, ACCUM, NO_GX, STAGED)
# Torch layout: the tile width Gt that G = gcd(Ho*Wo, C) gives (make_tiling), or, for G not a multiple of 16, the
# materialised-sample + GEMM path (C, O >= 32 and K = C*kh*kw >= 256: dcn_gemm_path.cu) or else the SIMT kernels
TORCH_CLASSES = (16, 32, 64, "gemm", "simt")
# Jittor layout: the channels (48: no pixel-row tiling, SIMT; 192: tensor-path forward and weight gradient, data
# gradient on the SIMT kernel because a 128-column lane block does not hold whole taps)
JITTOR_C = ((16,), (32,), (64,), (128, 256), (48, 192))
_MACS = 2e8   # B*Ho*Wo*kh*kw*C*O cap: the oracle's backward is a single-threaded float64 loop of that many MACs x 2


def _out_hw(H, W, k, s, p):
    return (H + 2 * p[0] - k[0]) // s[0] + 1, (W + 2 * p[1] - k[1]) // s[1] + 1


def _gt_of(G):
    """Tile width Gt of the Torch layout for G = gcd(Ho*Wo, C) (make_tiling), None when it does not tile."""
    return 64 if G % 64 == 0 else 32 if G % 32 == 0 else 16 if G % 16 == 0 else None


def _torch_class(C, O, Ho, Wo, k):
    Gt = _gt_of(math.gcd(Ho * Wo, C))
    if Gt:
        return Gt
    return "gemm" if C >= 32 and O >= 32 and C * k[0] * k[1] >= 256 else "simt"


def _cases(seed, n):
    """(B, C, O, H, W, k, s, p, variant, operand, (offset mode, sigma), flag, data seed).  Variant, operand, offset mode
    and the extent / channel class cycle with the case index, so that every combination of them is drawn (the Jittor
    classes with two channel counts take one in each 80-case cycle); kernel, strides, paddings, extents, batch and O are
    drawn within the class.  About one case in five sets one of FLAGS, drawn independently of the cycled axes."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        variant, operand = (TORCH, JITTOR)[i % 2], (FP32, BF16)[(i // 2) % 2]
        mode, cls = OFFSETS[(i // 4) % 4], (i // 16) % 5
        flag = int(rng.choice(FLAGS)) if rng.random() < 0.2 else 0
        while True:
            if variant == TORCH:
                want = TORCH_CLASSES[cls]
                C = int(rng.choice([c for c in (16, 32, 48, 64, 128, 192, 256) if isinstance(want, str) or
                                    c % want == 0]))
            else:
                C = JITTOR_C[cls][(i // 80) % len(JITTOR_C[cls])]
            O = int(rng.choice([16, 48, 64, 80, 128, 144, 256, 272, 320, 512]))
            k = KERNELS[int(rng.integers(0, len(KERNELS)))]
            s = (int(rng.integers(1, 3)), int(rng.integers(1, 3)))
            p = (int(rng.integers(0, 3)), int(rng.integers(0, 3)))
            H, W = int(rng.integers(3, 41)), int(rng.integers(3, 41))
            B = int(rng.integers(1, 4))
            Ho, Wo = _out_hw(H, W, k, s, p)
            if min(Ho, Wo) < 2:   # the Jittor variant divides by Ho - 1 and Wo - 1; kept out of both for symmetry
                continue
            if variant == TORCH and _torch_class(C, O, Ho, Wo, k) != want:
                continue
            if B * Ho * Wo * k[0] * k[1] * C * O <= _MACS:
                break
        sigma = float(rng.choice([0.5, 2.0, 4.0])) if mode == "normal" else (2.0 if mode == "far" else 0.0)
        out.append((B, C, O, H, W, k, s, p, variant, operand, (mode, sigma), flag, seed * 1000 + i))
    return out


CASES = _cases(2028, 150)
_FLAG_NAMES = {0: "", RELU: "-relu", ACCUM: "-accum", NO_GX: "-nogx", STAGED: "-staged"}


def _case_id(case):
    B, C, O, H, W, k, s, p, variant, operand, (mode, sigma), flag, seed = case
    return (f"{seed % 1000:03d}-{'torch' if variant == TORCH else 'jittor'}-{'bf16' if operand == BF16 else 'fp32'}"
            f"-B{B}C{C}O{O}-{H}x{W}-k{k[0]}{k[1]}-s{s[0]}{s[1]}-p{p[0]}{p[1]}-{mode}{sigma:g}{_FLAG_NAMES[flag]}")


# ---- routes: what the host runs for a case ---------------------------------------------------------------------------
def _paths(case):
    """(forward, backward) kernel family the host picks: "umma", "gemm" or "simt" (dcn_path_name)."""
    B, C, O, H, W, k, s, p, variant, operand = case[:10]
    shp = dcn.make_shape(B, C, O, H, W, k, s, p, variant, operand)
    return _lib.path_name(shp, _lib.PHASE_FORWARD), _lib.path_name(shp, _lib.PHASE_BACKWARD)


def _o_groups(O):
    """Output-channel group sizes of a tensor-path launch (dcn_umma_host.cu:o_groups): O <= 256 per launch."""
    if O <= 256:
        return [O]
    n = -(-O // 256)
    size = (-(-O // n) + 15) // 16 * 16
    return [min(size, O - o0) for o0 in range(0, O, size)]


def _route(case):
    """The tensor path's decisions for a case, restated from DESIGN.md §3 / §4 and make_tiling:
    Torch tiling (G, Gt, Cs, Rt, number of class instances), output-channel groups, whether the data gradient runs on
    the tcgen05 kernel and, per group, whether that kernel also forms the weight gradient (fused)."""
    B, C, O, H, W, k, s, p, variant, operand = case[:10]
    Ho, Wo = _out_hw(H, W, k, s, p)
    r = dict(groups=_o_groups(O), HW=Ho * Wo)
    if variant == TORCH:
        G = math.gcd(Ho * Wo, C)
        Gt = _gt_of(G)
        r.update(G=G, Gt=Gt, Cs=C // G, Rt=128 // Gt if Gt else None,
                 num_inst=B * (G // Gt) * (Ho * Wo // G) if Gt else None, data_umma=True)
        # the fused kernel keeps the grad_out images of a whole tile and the weight-gradient accumulators on chip:
        # O <= 128 in fp32, O <= 256 with bf16 operands (one image per operand instead of hi / lo)
        r["fused"] = [o <= (256 if operand == BF16 else 128) for o in r["groups"]]
    else:
        # a pixel-row lane block of 128 columns holds whole taps; the fused kernel then covers O <= 256
        r["data_umma"] = C % 128 == 0 or C in (16, 32, 64)
        r["fused"] = [r["data_umma"]] * len(r["groups"])
    return r


def _classes(case):
    """Labels of the routes and edges a case exercises (test_oracle_fuzz_draw_covers_every_route)."""
    B, C, O, H, W, k, s, p, variant, operand, (mode, _), flag, _ = case
    fwd, bwd = _paths(case)
    r = _route(case)
    out = {f"offsets {mode}"}
    if fwd == bwd == "umma":
        out.add(f"flag {flag} on umma")
        if s[0] != s[1]:
            out.add("umma mixed stride")
        if p != (k[0] // 2, k[1] // 2):
            out.add("umma padding != k // 2")
        if k[0] != k[1]:
            out.add("umma rectangular kernel")
        if variant == TORCH:
            out.add(f"torch umma Gt={r['Gt']}")
            if r["Cs"] > 1:
                out.add("torch umma Cs > 1")
            if r["num_inst"] % r["Rt"]:
                out.add("torch umma partial last tile")
            if operand == FP32 and O <= 128:
                out.add("torch umma fp32 fused wgrad")
            if operand == FP32 and 128 < O <= 256:
                out.add("torch umma fp32 unfused wgrad")
            if operand == BF16 and 128 < O <= 256:
                out.add("torch umma bf16 fused wgrad 128 < O <= 256")
            if O > 256:
                out.add("torch umma O > 256")
        else:
            out.add(f"jittor umma C={min(C, 128)}")
            if r["HW"] % 128:
                out.add("jittor umma Ho*Wo % 128 != 0")
            if O > 256:
                out.add("jittor umma O > 256")
            if not r["data_umma"]:
                out.add("jittor umma generic data gradient")
    if variant == TORCH and fwd == bwd == "gemm":
        out.add(f"torch gemm {'bf16' if operand == BF16 else 'fp32'}")
    if fwd == bwd == "simt" and operand == FP32:
        out.add(f"{'torch' if variant == TORCH else 'jittor'} simt fp32")
    return out


WANTED = ({f"torch umma Gt={g}" for g in (16, 32, 64)} |
          {"torch umma Cs > 1", "torch umma partial last tile", "torch umma fp32 fused wgrad",
           "torch umma fp32 unfused wgrad", "torch umma bf16 fused wgrad 128 < O <= 256", "torch umma O > 256"} |
          {f"jittor umma C={c}" for c in (16, 32, 64, 128)} |
          {"jittor umma Ho*Wo % 128 != 0", "jittor umma O > 256", "jittor umma generic data gradient"} |
          {"torch gemm fp32", "torch gemm bf16", "torch simt fp32", "jittor simt fp32"} |
          {"umma mixed stride", "umma padding != k // 2", "umma rectangular kernel"} |
          {f"offsets {m}" for m in OFFSETS} | {f"flag {f} on umma" for f in FLAGS})


def test_oracle_fuzz_draw_covers_every_route():
    """The draw reaches every kernel path and tiling class it is meant to test (no GPU needed: routing is a host
    decision).  test_routes_match_the_kernels_that_ran checks the restated rules against the launched kernels."""
    seen = set().union(*(_classes(c) for c in CASES))
    assert WANTED <= seen, sorted(WANTED - seen)
    # flags on both layouts' tensor path, where they change what the kernels do
    for flag in FLAGS:
        assert {c[8] for c in CASES if c[11] == flag and _paths(c) == ("umma", "umma")} == {TORCH, JITTOR}, flag


# ---- the comparison --------------------------------------------------------------------------------------------------
def _bf16_round(a):
    return torch.from_numpy(a).bfloat16().float().numpy()


def _inputs(case):
    """x, offset, weight, bias, grad_out (float32 numpy); x / weight / grad_out bf16-rounded for bf16 operands."""
    B, C, O, H, W, k, s, p, variant, operand, (mode, sigma), flag, seed = case
    Ho, Wo = _out_hw(H, W, k, s, p)
    N = k[0] * k[1]
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, C, H, W)).astype(np.float32)
    if mode == "grid":
        off = (rng.integers(-8, 9, (B, 2 * N, Ho, Wo)) / 2).astype(np.float32)
    else:
        off = (rng.standard_normal((B, 2 * N, Ho, Wo)) * sigma).astype(np.float32)
    if mode == "far":
        off.reshape(-1)[::97] *= 1e3
    w = (rng.standard_normal((O, C, *k)) * np.sqrt(2.0 / (C * N))).astype(np.float32)
    b = rng.standard_normal(O).astype(np.float32)
    gout = rng.standard_normal((B, O, Ho, Wo)).astype(np.float32)
    if operand == BF16:
        x, w, gout = _bf16_round(x), _bf16_round(w), _bf16_round(gout)
    return x, off, w, b, gout


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_fuzz_against_the_oracle(case):
    B, C, O, H, W, k, s, p, variant, operand, offsets, flag, seed = case
    x, off, w, b, gout = _inputs(case)
    sh = orc.make_shape(B, C, O, H, W, k, s, p, variant)
    ref_out = orc.forward(sh, x, off, w, b)
    ref = orc.backward(sh, x, off, w, gout)
    tol_out, tol_g = (1e-2, 2e-2) if operand == BF16 else (1e-4, 1e-3)
    paths = _paths(case)
    act = torch.bfloat16 if operand == BF16 else torch.float32
    tx, tw, tg = (torch.from_numpy(a).cuda().to(act) for a in (x, w, gout))
    toff, tb = torch.from_numpy(off).cuda(), torch.from_numpy(b).cuda()
    geo = dict(kernel_size=k, stride=s, padding=p, variant=variant, operand=operand)

    def check(name, got, exp, tol):
        err = rel_err(got.cpu().numpy() if isinstance(got, torch.Tensor) else got, exp)
        assert err < tol, f"{name}: error {err:.3g} >= {tol:g} on paths {paths} for case {_case_id(case)}"

    def check_grads(tag, grads, skip=()):
        for nm, got, exp in zip(("gx", "goff", "gw", "gb"), grads, ref):
            if nm not in skip:
                check(f"{tag}{nm}", got, exp, tol_g)

    out = dcn.dcn_forward(tx, toff, tw, tb, **geo)
    check("out", out, ref_out, tol_out)
    grads = dcn.dcn_backward(tx, toff, tw, tg, True, **geo)
    check_grads("", grads)

    # Flags.  The backward's float atomics (grad_x, grad_offset, the weight gradient's per-CTA partial sums) land in
    # an order that varies between two identical calls, so a flagged call is held to the plain one at 2e-5 relative
    # (fp32 reassociation), besides the oracle.  The forward has no atomics: it is compared bitwise.
    def same(tag, a, bb):
        err = rel_err(a.cpu().numpy(), bb.cpu().numpy())
        assert err < 2e-5, f"{tag}: {err:.3g} from the plain call on paths {paths} for case {_case_id(case)}"

    if flag == RELU:
        out_r = dcn.dcn_forward(tx, toff, tw, tb, flags=RELU, **geo)
        check("relu out", out_r, np.maximum(ref_out, 0), tol_out)
        assert torch.equal(out_r, out.clamp_min(0)), \
            f"relu out is not max(out, 0) on paths {paths} for case {_case_id(case)}"
    elif flag == ACCUM:
        base = torch.from_numpy(np.random.default_rng(seed + 1).standard_normal(x.shape).astype(np.float32)).cuda()
        acc = base.clone()
        got = dcn.dcn_backward(tx, toff, tw, tg, True, grad_x=acc, **geo)
        assert got[0] is acc, f"grad_x is not the given tensor on paths {paths} for case {_case_id(case)}"
        check("accumulated gx - prefill", (acc.double() - base.double()).cpu().numpy(), ref[0], tol_g)
        check_grads("accum ", got, skip=("gx",))
    elif flag == NO_GX:
        got = dcn.dcn_backward(tx, toff, tw, tg, True, need_grad_x=False, **geo)
        assert got[0] is None, f"grad_x returned on paths {paths} for case {_case_id(case)}"
        check_grads("no-gx ", got, skip=("gx",))
        for nm, a, bb in zip(("goff", "gw", "gb"), got[1:], grads[1:]):
            same(f"no-gx {nm}", a, bb)
    elif flag == STAGED:
        ws = staged_workspace(tx, tw, k, s, p, variant, operand)
        if ws is not None:   # both phases keep the staged input at the workspace head: umma / umma or gemm / gemm
            ws.fill_(0xff)   # only the forward's own staging makes the buffer valid
        out_s = dcn.dcn_forward(tx, toff, tw, tb, ws=ws, **geo)
        got = dcn.dcn_backward(tx, toff, tw, tg, True, ws=ws, xt_staged=True, **geo)
        assert torch.equal(out_s, out), \
            f"staged forward differs from the plain one on paths {paths} for case {_case_id(case)}"
        check_grads("staged ", got)
        for nm, a, bb in zip(("gx", "goff", "gw", "gb"), got, grads):
            same(f"staged {nm}", a, bb)


@pytest.mark.gpu
@pytest.mark.parametrize("operand", [FP32, BF16], ids=["fp32", "bf16"])
def test_relu_out_on_the_gemm_path(operand):
    """Regression: the Torch layout's GEMM path (gcd(Ho*Wo, C) = 4 here) ignored DCN_FLAG_RELU_OUT and returned the
    output before the ReLU.  Found by the fuzz above (case 140)."""
    case = (2, 64, 64, 10, 10, (3, 3), (1, 1), (1, 1), TORCH, operand, ("normal", 2.0), RELU, 7)
    assert _paths(case) == ("gemm", "gemm")
    x, off, w, b, gout = _inputs(case)
    ref_out = orc.forward(orc.make_shape(2, 64, 64, 10, 10, 3, 1, 1, TORCH), x, off, w, b)
    act = torch.bfloat16 if operand == BF16 else torch.float32
    out = dcn.dcn_forward(torch.from_numpy(x).cuda().to(act), torch.from_numpy(off).cuda(),
                          torch.from_numpy(w).cuda().to(act), torch.from_numpy(b).cuda(), 3, 1, 1, TORCH, operand,
                          flags=RELU)
    assert rel_err(out.cpu().numpy(), np.maximum(ref_out, 0)) < (1e-2 if operand == BF16 else 1e-4)


# ---- routes against the launched kernels -----------------------------------------------------------------------------
ROUTE_CLASSES = ["torch umma fp32 fused wgrad", "torch umma fp32 unfused wgrad",
                 "torch umma bf16 fused wgrad 128 < O <= 256", "torch umma O > 256", "jittor umma C=16",
                 "jittor umma C=128", "jittor umma O > 256", "jittor umma generic data gradient", "torch gemm fp32",
                 "torch gemm bf16", "torch simt fp32", "jittor simt fp32"]


def _launched(fn):
    _lib.profile_begin()
    try:
        fn()
    finally:
        res = _lib.profile_end()
    return {name: n for name, (n, _) in res.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("label", ROUTE_CLASSES)
def test_routes_match_the_kernels_that_ran(label):
    """The first case of each route class, under the engine's launch profiler: the kernels the host launched agree
    with the class _route / _classes put it in."""
    case = next(c for c in CASES if label in _classes(c))
    B, C, O, H, W, k, s, p, variant, operand = case[:10]
    x, off, w, b, gout = _inputs(case)
    act = torch.bfloat16 if operand == BF16 else torch.float32
    tx, tw, tg = (torch.from_numpy(a).cuda().to(act) for a in (x, w, gout))
    toff, tb = torch.from_numpy(off).cuda(), torch.from_numpy(b).cuda()
    geo = dict(kernel_size=k, stride=s, padding=p, variant=variant, operand=operand)
    dcn.dcn_backward(tx, toff, tw, tg, True, **geo)   # warm-up: workspace allocation happens outside the profile
    fwd = _launched(lambda: dcn.dcn_forward(tx, toff, tw, tb, **geo))
    bwd = _launched(lambda: dcn.dcn_backward(tx, toff, tw, tg, True, **geo))
    torch.cuda.synchronize()
    paths, r = _paths(case), _route(case)
    what = (label, _case_id(case), paths, r, fwd, bwd)
    if paths[0] == "umma":
        assert fwd.get("umma_fwd_kernel") == len(r["groups"]), what
    if paths[1] == "umma":
        unfused = sum(not f for f in r["fused"])
        assert bwd.get("umma_bwd_weight_kernel", 0) == unfused, what
        assert bwd.get("umma_bwd_data_kernel", 0) == (len(r["groups"]) if r["data_umma"] else 0), what
        assert ("bwd_data_kernel" in bwd) == (not r["data_umma"]), what
    if "gemm" in paths:
        assert paths == ("gemm", "gemm"), what
        assert "cublas_gemm_fwd" in fwd, what
        assert "cublas_gemm_bwd_data" in bwd and "cublas_gemm_bwd_weight" in bwd, what
    if paths == ("simt", "simt"):
        assert "fwd_kernel" in fwd and "bwd_data_kernel" in bwd, what
        assert not any(n.startswith(("umma_", "cublas_")) for n in (*fwd, *bwd)), what
