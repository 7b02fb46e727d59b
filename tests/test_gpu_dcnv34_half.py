"""DCNv3 and DCNv4 on bfloat16 and float16 operands.  Inputs are drawn in float32 and rounded to the dtype; the half
kernels must then be the float32 kernels on the widened tensors, rounded once: out, grad_offset, grad_mask and
grad_offset_mask bit for bit, grad_input up to the order of its float atomics.  This runs on the LIVE tables of
test_gpu_dcnv3.py (softmax on and off) and test_gpu_dcnv4.py and on the dcnv3_* / dcnv4_* fixtures.  Also: one check
per dtype against the float64 references, the DCNv4 row layout in half types (NaN padding, +0.0 gradient padding, rows
that start 2-byte aligned), determinism, the `need` subsets, the kernel names, CUDA-graph replay, both modules under
autocast and after .half(), and a bfloat16 offset_mask past 2^31 elements (byte offsets past 2^32)."""
import contextlib

import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from jittor_dcn_b200 import functional as fn
from jittor_dcn_b200 import dcnv3 as dcnv3_module
from jittor_dcn_b200 import dcnv4 as dcnv4_module
from oracle import dcnv3_reference, dcnv4_reference
from tests import test_gpu_dcnv3 as v3
from tests import test_gpu_dcnv4 as v4
from tests.util import golden, golden_names, rel_err

pytestmark = pytest.mark.gpu

DTYPES = [torch.bfloat16, torch.float16]
SUFFIX = {torch.bfloat16: "_bf16", torch.float16: "_f16"}


def _round(dtype, *ts):
    return [t.to(dtype) for t in ts]


def _gx_tol(dtype):
    """grad_input of two calls in a half type: float32 sums in different atomic orders, each rounded once, may land one
    ulp apart."""
    return torch.finfo(dtype).eps + 1e-5


def _v3_pair(x, off, m, gout, geo, softmax, need=(True, True, True)):
    """[(out, grads) of the half call, (out, grads) of the float32 call on the widened tensors, grad_input of the half
    operands in the float32 buffer the kernels accumulate into (or None)], on the GPU."""
    h = [t.cuda() for t in (x, off, m, gout)]
    f = [t.float() for t in h]
    res = []
    for a in (h, f):
        out = dcn.dcn_v3_forward(*a[:3], *geo, softmax_mask=softmax)
        grads = dcn.dcn_v3_backward(*a, *geo, softmax_mask=softmax, need=need)
        res.append((out, grads))
    gx32 = None
    if need[0]:
        shp, xd, offd, md = fn._dcnv3_inputs(*h[:3], *geo[:10], softmax)
        gx32 = torch.empty(xd.shape, dtype=torch.float32, device=xd.device)
        fn._run("dcn_v3_backward_typed", xd.device, shp,
                (fn._CORE_OPERANDS[xd.dtype], float(geo[10]), xd, offd, md, h[3], gx32, None, None))
    torch.cuda.synchronize()
    return res + [gx32]


def _v4_pair(x, om, gout, geo, rc, need=(True, True)):
    h = [t.cuda() for t in (x, om, gout)]
    f = [t.float() for t in h]
    res = []
    for a in (h, f):
        out = dcn.dcn_v4_forward(*a[:2], *geo, remove_center=rc)
        grads = dcn.dcn_v4_backward(*a, *geo, remove_center=rc, need=need)
        res.append((out, grads))
    gx32 = None
    if need[0]:
        shp, xd, omd = fn._dcnv4_inputs(*h[:2], *geo[:10], rc)
        gx32 = torch.empty(xd.shape, dtype=torch.float32, device=xd.device)
        fn._run("dcn_v4_backward_typed", xd.device, shp,
                (fn._CORE_OPERANDS[xd.dtype], float(geo[10]), xd, omd, h[2], gx32, None))
    torch.cuda.synchronize()
    return res + [gx32]


def _assert_float32_bits(half, full, gx32, dtype):
    """out and the coordinate-side gradients: the float32 results rounded to dtype.  grad_input: the float32 buffer
    within 1e-5 of the float32 call's (atomic order only), and what comes back, that buffer rounded once."""
    (ho, hg), (fo, fg) = half, full
    assert ho.dtype == dtype and torch.equal(ho, fo.to(dtype))
    if hg[0] is not None:
        assert hg[0].dtype == dtype
        assert rel_err(gx32.cpu().numpy(), fg[0].cpu().numpy()) <= 1e-5
        assert rel_err(hg[0].float().cpu().numpy(), fg[0].cpu().numpy()) <= _gx_tol(dtype)
    for h, f in zip(hg[1:], fg[1:]):
        if h is not None:
            assert h.dtype == dtype and torch.equal(h, f.to(dtype))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("softmax", [False, True])
@pytest.mark.parametrize("name", list(v3.LIVE))
def test_dcnv3_is_the_float32_kernel_rounded(name, softmax, dtype):
    N, H, W, geo = v3.LIVE[name]
    ts = _round(dtype, *v3._inputs(N, H, W, geo, seed=list(v3.LIVE).index(name)))
    _assert_float32_bits(*_v3_pair(*ts, geo, softmax), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", list(v4.LIVE))
def test_dcnv4_is_the_float32_kernel_rounded(name, dtype):
    """gc16_3x3 (G = 4, K = 9) and gc16_s2_d2_g3 (G = 3, K = 9) have group rows of 27 elements: in a half type every
    other group starts only 2-byte aligned."""
    N, H, W, geo, rc = v4.LIVE[name]
    ts = _round(dtype, *v4._inputs(N, H, W, geo, rc, seed=list(v4.LIVE).index(name)))
    half, full, gx32 = _v4_pair(*ts, geo, rc)
    _assert_float32_bits(half, full, gx32, dtype)
    K, _ = dcnv4_reference.points(geo[0], geo[1], rc)
    assert v4._padding_is_plus_zero(half[1][1].float().cpu(), geo[8], K)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", golden_names("dcnv3_") + golden_names("dcnv4_"))
def test_fixture_inputs_are_the_float32_kernel_rounded(name, dtype):
    g = golden(name)
    t = {k: torch.as_tensor(v) for k, v in g.items()}
    geo = tuple(int(v) for v in g["geo"]) + (float(g["offset_scale"]),)
    if name.startswith("dcnv3_"):
        ts = _round(dtype, t["input"], t["offset"], t["mask"], t["grad_out"])
        _assert_float32_bits(*_v3_pair(*ts, geo, bool(g["softmax"])), dtype)
    else:
        rc = bool(g["remove_center"])
        ts = _round(dtype, t["input"], t["offset_mask"], t["grad_out"])
        half, full, gx32 = _v4_pair(*ts, geo, rc)
        _assert_float32_bits(half, full, gx32, dtype)
        K, _ = dcnv4_reference.points(geo[0], geo[1], rc)
        assert v4._padding_is_plus_zero(half[1][1].float().cpu(), geo[8], K)


def _tolerance(dtype, f32_tol):
    """One rounding to dtype of a result whose float32 error is within f32_tol of max |ref|: at most half an ulp, u = eps/2
    relative to the element (2^-8 for bfloat16, 2^-11 for float16), so at most u * max |ref|, plus f32_tol."""
    return torch.finfo(dtype).eps / 2 + f32_tol


@pytest.mark.parametrize("dtype", DTYPES)
def test_against_the_float64_references(dtype):
    N, H, W, geo = v3.LIVE["gc32_3x5"]
    x, off, m, gout = _round(dtype, *v3._inputs(N, H, W, geo, seed=41))
    (out, grads), _, _ = _v3_pair(x, off, m, gout, geo, True)
    ref = dcnv3_reference.reference(x.float(), off.float(), m.float(), geo, gout.float(), softmax_mask=True)
    assert rel_err(out.float().cpu().numpy(), ref[0].numpy()) <= _tolerance(dtype, 1e-4)
    for got, exp, nm in zip(grads, ref[1:], v3.GRAD_NAMES):
        assert rel_err(got.float().cpu().numpy(), exp.numpy()) <= _tolerance(dtype, 1e-3), nm
    N, H, W, geo, rc = v4.LIVE["gc16_s2_d2_g3"]
    x, om, gout = _round(dtype, *v4._inputs(N, H, W, geo, rc, seed=42))
    (out, grads), _, _ = _v4_pair(x, om, gout, geo, rc)
    ref = dcnv4_reference.reference(x.float(), om.float(), geo, gout.float(), remove_center=rc)
    assert rel_err(out.float().cpu().numpy(), ref[0].numpy()) <= _tolerance(dtype, 1e-4)
    for got, exp, nm in zip(grads, ref[1:], ("grad_input", "grad_offset_mask")):
        assert rel_err(got.float().cpu().numpy(), exp.numpy()) <= _tolerance(dtype, 1e-3), nm


@pytest.mark.parametrize("dtype", DTYPES)
def test_dcnv4_nan_in_the_half_padding_reaches_nothing(dtype):
    N, H, W, geo, rc = v4.LIVE["gc16_s2_d2_g3"]
    x, om, gout = _round(dtype, *v4._inputs(N, H, W, geo, rc, seed=31))
    K, _ = dcnv4_reference.points(geo[0], geo[1], rc)
    used = 3 * geo[8] * K
    assert om[..., used:].isnan().all()
    zero = om.clone()
    zero[..., used:] = 0.0
    (out_nan, g_nan), _, _ = _v4_pair(x, om, gout, geo, rc)
    (out_zero, g_zero), _, _ = _v4_pair(x, zero, gout, geo, rc)
    assert torch.isfinite(out_nan).all() and torch.isfinite(g_nan[0]).all() and torch.isfinite(g_nan[1]).all()
    assert torch.equal(out_nan, out_zero) and torch.equal(g_nan[1], g_zero[1])
    assert v4._padding_is_plus_zero(g_nan[1].float().cpu(), geo[8], K)


@pytest.mark.parametrize("dtype", DTYPES)
def test_coordinate_gradients_are_deterministic_and_need_computes_only_what_it_names(dtype):
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0)
    x, off, m, gout = _round(dtype, *v3._inputs(4, 28, 28, geo, seed=11))
    (_, a), _, _ = _v3_pair(x, off, m, gout, geo, True)
    (_, b), _, _ = _v3_pair(x, off, m, gout, geo, True)
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    for i in range(3):
        need = tuple(k == i for k in range(3))
        (_, g), _, _ = _v3_pair(x, off, m, gout, geo, True, need=need)
        assert all((t is None) == (k != i) for k, t in enumerate(g))
        if i > 0:
            assert torch.equal(g[i], a[i])
    x, om, gout = _round(dtype, *v4._inputs(4, 28, 28, geo, True, seed=12))
    (_, a), _, _ = _v4_pair(x, om, gout, geo, True)
    (_, b), _, _ = _v4_pair(x, om, gout, geo, True)
    assert torch.equal(a[1], b[1])
    for need in ((True, False), (False, True)):
        (_, g), _, _ = _v4_pair(x, om, gout, geo, True, need=need)
        assert all((t is None) == (not n) for t, n in zip(g, need))
        if need[1]:
            assert torch.equal(g[1], a[1])


@pytest.mark.parametrize("dtype", DTYPES)
def test_one_half_kernel_launch_per_call(dtype):
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 2, 16, 1.0)
    x, off, m, gout = (t.cuda() for t in _round(dtype, *v3._inputs(1, 6, 6, geo, seed=23)))
    xo, om, go4 = (t.cuda() for t in _round(dtype, *v4._inputs(1, 6, 6, geo, False, seed=24)))
    _lib.profile_begin()
    before = dcn.load().dcn_launch_count()
    dcn.dcn_v3_forward(x, off, m, *geo, softmax_mask=True)
    dcn.dcn_v3_backward(x, off, m, gout, *geo, softmax_mask=True)
    dcn.dcn_v4_forward(xo, om, *geo)
    dcn.dcn_v4_backward(xo, om, go4, *geo)
    torch.cuda.synchronize()
    launched = dcn.load().dcn_launch_count() - before
    prof = _lib.profile_end()
    s = SUFFIX[dtype]
    assert {k: v[0] for k, v in prof.items()} == {f"dcnv3_fwd_kernel{s}": 1, f"dcnv3_bwd_kernel{s}": 1,
                                                   f"dcnv4_fwd_kernel{s}": 1, f"dcnv4_bwd_kernel{s}": 1}
    assert launched == 4


def test_bf16_forward_and_backward_capture_and_replay():
    dtype = torch.bfloat16
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0)
    x, om, gout = _round(dtype, *v4._inputs(2, 12, 12, geo, True, seed=17))
    sx, so = (t.cuda().requires_grad_(True) for t in (x, om))
    sg = gout.cuda()

    def step():
        out = dcn.dcnv4_core(sx, so, *geo, remove_center=True)
        return (out,) + torch.autograd.grad(out, [sx, so], sg)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    for seed in (21, 22):
        x, om, gout = _round(dtype, *v4._inputs(2, 12, 12, geo, True, seed=seed))
        with torch.no_grad():
            sx.copy_(x.cuda())
            so.copy_(om.cuda())
            sg.copy_(gout.cuda())
        graph.replay()
        torch.cuda.synchronize()
        (out, grads), _, _ = _v4_pair(x, om, gout, geo, True)
        assert torch.equal(static[0], out) and torch.equal(static[2], grads[1])
        assert rel_err(static[1].float().cpu().numpy(), grads[0].float().cpu().numpy()) <= _gx_tol(dtype)


class _Float32Core:
    """The parent's composition, rebuilt: the core on float32 copies, its output cast back to the operands' dtype."""

    def __init__(self, fn):
        self.fn = fn

    def apply(self, *args):
        with torch.autocast(device_type="cuda", enabled=False):
            out = self.fn.apply(*(a.float() if torch.is_tensor(a) else a for a in args))
        return out.to(args[0].dtype)


def _module_run(m, inp, gout, autocast_dtype):
    x = inp.clone().requires_grad_(True)
    for p in m.parameters():
        p.grad = None
    _lib.profile_begin()
    with torch.autocast("cuda", dtype=autocast_dtype) if autocast_dtype else contextlib.nullcontext():
        out = m(x)
    out.backward(gout.to(out.dtype))
    torch.cuda.synchronize()
    prof = _lib.profile_end()
    return out.detach(), x.grad, [p.grad.clone() for p in m.parameters()], prof


def _check_module(mod, fn_name, m, inp, gout, autocast_dtype, dtype, monkeypatch):
    out, gx, gp, prof = _module_run(m, inp, gout, autocast_dtype)
    s = SUFFIX[dtype]
    kern = "dcnv3" if fn_name == "DCNv3Function" else "dcnv4"
    assert set(prof) == {f"{kern}_fwd_kernel{s}", f"{kern}_bwd_kernel{s}"}, prof
    with monkeypatch.context() as mp:
        mp.setattr(mod, fn_name, _Float32Core(getattr(mod, fn_name)))
        out_p, gx_p, gp_p, prof_p = _module_run(m, inp, gout, autocast_dtype)
    assert set(prof_p) == {f"{kern}_fwd_kernel", f"{kern}_bwd_kernel"}, prof_p
    assert out.dtype == out_p.dtype == dtype and torch.equal(out, out_p)
    assert rel_err(gx.float().cpu().numpy(), gx_p.float().cpu().numpy()) <= 1e-2
    for (name, _), a, b in zip(m.named_parameters(), gp, gp_p):
        assert rel_err(a.float().cpu().numpy(), b.float().cpu().numpy()) <= 1e-2, name


@pytest.mark.parametrize("dtype", DTYPES)
def test_dcnv3_module_runs_the_half_kernels_under_autocast(dtype, monkeypatch):
    m, _ = v3._module_pair(dict(channels=64, group=4), seed=1)
    m = m.cuda()
    inp = torch.randn(2, 12, 12, 64, device="cuda")
    gout = torch.randn(2, 12, 12, 64, device="cuda")
    _check_module(dcnv3_module, "DCNv3Function", m, inp, gout, dtype, dtype, monkeypatch)


@pytest.mark.parametrize("dtype", DTYPES)
def test_dcnv4_module_runs_the_half_kernels_under_autocast(dtype, monkeypatch):
    m, _ = v4._module_pair(dict(channels=64, group=4, dw_kernel_size=3), seed=1)
    m = m.cuda()
    inp = torch.randn(2, 144, 64, device="cuda")
    gout = torch.randn(2, 144, 64, device="cuda")
    _check_module(dcnv4_module, "DCNv4Function", m, inp, gout, dtype, dtype, monkeypatch)


def test_modules_after_half_run_the_f16_kernels(monkeypatch):
    m3, _ = v3._module_pair(dict(channels=64, group=4), seed=2)
    inp = torch.randn(2, 12, 12, 64, device="cuda").half()
    _check_module(dcnv3_module, "DCNv3Function", m3.cuda().half(), inp, torch.randn_like(inp), None, torch.float16,
                  monkeypatch)
    m4, _ = v4._module_pair(dict(channels=64, group=4), seed=2)
    inp = torch.randn(2, 144, 64, device="cuda").half()
    _check_module(dcnv4_module, "DCNv4Function", m4.cuda().half(), inp, torch.randn_like(inp), None, torch.float16,
                  monkeypatch)


def test_dcnv4_module_without_pointwise_keeps_the_float32_core_under_autocast():
    """x is the float32 input itself and offset_mask comes from a bf16 linear layer: mixed, so float32 copies."""
    m, _ = v4._module_pair(dict(channels=64, group=2, without_pointwise=True), seed=3)
    inp = torch.randn(2, 144, 64, device="cuda")
    out, _, _, prof = _module_run(m.cuda(), inp, torch.randn_like(inp), torch.bfloat16)
    assert set(prof) == {"dcnv4_fwd_kernel", "dcnv4_bwd_kernel"} and out.dtype == torch.float32


def test_bf16_offset_mask_past_2_31_elements():
    """test_gpu_dcnv4.py's 2^31-element offset_mask in bfloat16: image 8192 of offset_mask starts at element 2^31, byte
    2^32.  The images around the line and the last one must equal the same call on them alone, and the float32 kernel
    on the widened last image."""
    N, H, W, G, Gc = 8200, 64, 64, 1, 64
    geo = (3, 7, 1, 1, 1, 3, 1, 1, G, Gc, 1.0)
    Cm = dcnv4_reference.row_floats(3, 7, G, False)
    assert Cm == 64 and 8192 * H * W * Cm == 2 ** 31
    # bf16 x, out, grad_out, offset_mask, grad_offset_mask; float32 grad_input and its bf16 copy
    nbytes = N * H * W * (G * Gc * (2 * 3 + 4 + 2) + Cm * 2 * 2)
    need = nbytes + (2 << 30)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2**30:.0f} GiB free, have {free / 2**30:.0f}")
    torch.manual_seed(0)
    x = torch.randn(N, H, W, G * Gc, device="cuda").bfloat16()
    om = torch.randn(N, H, W, Cm, device="cuda")
    om[..., :42] = torch.round(om[..., :42] * 1536) / 1024
    om[..., 63] = float("nan")                          # the one padding column
    om = om.bfloat16()
    out = dcn.dcn_v4_forward(x, om, *geo)
    gout = torch.randn_like(out)
    grads = dcn.dcn_v4_backward(x, om, gout, *geo)
    torch.cuda.synchronize()
    for i in (0, 8191, 8192, 8193, N - 1):
        s = slice(i, i + 1)
        o1 = dcn.dcn_v4_forward(x[s], om[s], *geo)
        g1 = dcn.dcn_v4_backward(x[s], om[s], gout[s], *geo)
        assert torch.equal(out[s], o1), i
        assert torch.equal(grads[1][s], g1[1]), i
        assert rel_err(grads[0][s].float().cpu().numpy(), g1[0].float().cpu().numpy()) <= _gx_tol(torch.bfloat16), i
    assert bool((grads[1][..., 63] == 0).all())
    half, full, gx32 = _v4_pair(x[-1:], om[-1:], gout[-1:], geo, False)
    _assert_float32_bits(half, full, gx32, torch.bfloat16)
    assert torch.equal(out[-1:], half[0]) and torch.equal(grads[1][-1:], half[1][1])
    del x, om, out, gout, grads
    torch.cuda.empty_cache()
