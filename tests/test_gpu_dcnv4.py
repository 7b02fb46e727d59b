"""DCNv4 on the GPU: csrc/dcn_dcnv3.cu's dcnv4 kernels against the dcnv4_* fixtures and against the float64 reference
evaluated live on the CPU (out <= 1e-4, each gradient <= 1e-3 of max |ref|) over channels per group, kernels from 1x1 to
7x7, remove_center, strides, dilations, paddings, offset scales and padded rows; bitwise equality with the DCNv3 kernels
on the unpacked tensors; NaN in the padding columns; the determinism of grad_offset_mask; each subset of gradients;
CUDA-graph replay; the kernel names; the module against the restated reference in fp32 and under bf16 autocast; and an
offset_mask past 2^31 elements.  Offsets are drawn on a 2^-10 grid: every fp32 coordinate of the kernels is then
exact, and floor() picks the cell the float64 reference picks."""
import ctypes

import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from oracle import dcnv3_reference, dcnv4_reference
from tests.util import golden, golden_names, rel_err

pytestmark = pytest.mark.gpu


def _inputs(N, H, W, geo, rc, seed, spread=1.5):
    """input, offset_mask (NaN in the padding columns), grad_out on the CPU."""
    kh, kw, sh, sw, ph, pw, dh, dw, G, Gc, _ = geo
    Ho, Wo = dcnv3_reference.out_extent(H, W, kh, kw, sh, sw, ph, pw, dh, dw)
    K, _ = dcnv4_reference.points(kh, kw, rc)
    Cm = dcnv4_reference.row_floats(kh, kw, G, rc)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, H, W, G * Gc, generator=g)
    off = torch.round(torch.randn(N, Ho, Wo, G, 2 * K, generator=g) * spread * 1024) / 1024
    m = torch.randn(N, Ho, Wo, G, K, generator=g)
    om = torch.full((N, Ho, Wo, Cm), float("nan"))
    om[..., :3 * G * K] = torch.cat([off, m], -1).reshape(N, Ho, Wo, 3 * G * K)
    gout = torch.randn(N, Ho, Wo, G * Gc, generator=g)
    return x, om, gout


def _engine(x, om, gout, geo, rc, need=(True, True)):
    xc, omc = x.cuda(), om.cuda()
    out = dcn.dcn_v4_forward(xc, omc, *geo, remove_center=rc)
    grads = dcn.dcn_v4_backward(xc, omc, gout.cuda(), *geo, remove_center=rc, need=need)
    torch.cuda.synchronize()
    return out.cpu(), [None if t is None else t.cpu() for t in grads]


def _check(out, grads, ref):
    assert rel_err(out.numpy(), ref[0].numpy()) <= 1e-4
    for got, exp, name in zip(grads, ref[1:], ("grad_input", "grad_offset_mask")):
        assert rel_err(got.numpy(), exp.numpy()) <= 1e-3, name


def _padding_is_plus_zero(gom, G, K):
    pad = gom[..., 3 * G * K:]
    return bool((pad == 0).all()) and not bool(torch.signbit(pad).any())


@pytest.mark.parametrize("name", golden_names("dcnv4_"))
def test_against_the_fixtures(name):
    g = golden(name)
    t = {k: torch.as_tensor(v) for k, v in g.items()}
    geo = tuple(int(v) for v in g["geo"]) + (float(g["offset_scale"]),)
    rc = bool(g["remove_center"])
    out, grads = _engine(t["input"], t["offset_mask"], t["grad_out"], geo, rc)
    _check(out, grads, [t[k] for k in ("out", "grad_input", "grad_offset_mask")])
    K, _ = dcnv4_reference.points(geo[0], geo[1], rc)
    assert _padding_is_plus_zero(grads[1], geo[8], K)


LIVE = {
    #  name               N  H   W   (kh, kw, sh, sw, ph, pw, dh, dw, G, Gc, os)          remove_center
    "gc16_3x3":          (2, 12, 13, (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0),    False),   # Cm 112
    "gc16_3x3_rc":       (2, 12, 13, (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0),    True),    # Cm 96
    "gc32_5x5_rc":       (1, 10, 14, (5, 5, 1, 1, 2, 2, 1, 1, 2, 32, 1.0),    True),    # K 24
    "gc64_7x7":          (1, 11, 9, (7, 7, 1, 1, 3, 3, 1, 1, 2, 64, 0.5),     False),   # K 49: 294 -> 296
    "gc64_7x7_rc":       (1, 11, 9, (7, 7, 1, 1, 3, 3, 1, 1, 1, 64, 1.0),     True),    # K 48
    "gc128_1x1_p0":      (2, 7, 8, (1, 1, 1, 1, 0, 0, 1, 1, 1, 128, 2.0),     False),   # K 1: 3 -> 8
    "gc256_3x3_s2":      (1, 9, 10, (3, 3, 2, 2, 1, 1, 1, 1, 1, 256, 1.0),    False),   # 27 -> 32
    "gc16_s2_d2_g3":     (2, 15, 14, (3, 3, 2, 1, 2, 0, 2, 2, 3, 16, 2.0),    False),   # 81 -> 88
    "gc32_d2_os05_rc":   (1, 12, 12, (3, 3, 1, 2, 0, 1, 2, 1, 5, 32, 0.5),    True),    # 120
    "gc64_5x3_s2_rc":    (2, 10, 11, (5, 3, 2, 2, 2, 1, 1, 2, 2, 64, 1.0),    True),    # K 14: 84 -> 88
    "gc256_5x5_d2":      (1, 13, 12, (5, 5, 1, 1, 4, 4, 2, 2, 2, 256, 1.5),   False),   # 150 -> 152
    "gc128_3x5_rc_os2":  (1, 9, 11, (3, 5, 1, 1, 1, 2, 1, 1, 3, 128, 2.0),    True),    # K 14: 126 -> 128
}


@pytest.mark.parametrize("name", list(LIVE))
def test_against_the_live_float64_reference(name):
    N, H, W, geo, rc = LIVE[name]
    x, om, gout = _inputs(N, H, W, geo, rc, seed=list(LIVE).index(name))
    out, grads = _engine(x, om, gout, geo, rc)
    _check(out, grads, dcnv4_reference.reference(x, om, geo, gout, remove_center=rc))
    K, _ = dcnv4_reference.points(geo[0], geo[1], rc)
    assert _padding_is_plus_zero(grads[1], geo[8], K)


@pytest.mark.parametrize("name", [n for n in LIVE if not LIVE[n][4] and LIVE[n][3][0] * LIVE[n][3][1] <= 32])
def test_bitwise_equal_to_dcnv3_on_the_unpacked_tensors(name):
    """Same chain, same summation order: out and grad_offset_mask unpacked are the DCNv3 kernels' bits (the cases
    without remove_center that DCNv3's kernels take: at most 32 points)."""
    N, H, W, geo, _ = LIVE[name]
    kh, kw, G = geo[0], geo[1], geo[8]
    P = kh * kw
    x, om, gout = _inputs(N, H, W, geo, False, seed=100 + list(LIVE).index(name))
    out4, (gx4, gom4) = _engine(x, om, gout, geo, False)
    off, m = dcnv4_reference.unpack(om, kh, kw, G, False)
    args = [t.contiguous().cuda() for t in (x, off, m)]
    out3 = dcn.dcn_v3_forward(*args, *geo)
    gx3, goff3, gm3 = dcn.dcn_v3_backward(*args, gout.cuda(), *geo)
    assert torch.equal(out4, out3.cpu())
    rows = gom4[..., :3 * G * P].reshape(gom4.shape[:3] + (G, 3 * P))
    assert torch.equal(rows[..., :2 * P].reshape(goff3.shape), goff3.cpu())
    assert torch.equal(rows[..., 2 * P:].reshape(gm3.shape), gm3.cpu())
    assert rel_err(gx4.numpy(), gx3.cpu().numpy()) <= 1e-5


def test_nan_in_the_padding_changes_nothing():
    N, H, W, geo, rc = LIVE["gc16_s2_d2_g3"]
    x, om, gout = _inputs(N, H, W, geo, rc, seed=31)
    K, _ = dcnv4_reference.points(geo[0], geo[1], rc)
    used = 3 * geo[8] * K
    assert om.shape[-1] - used == 7
    zero = om.clone()
    zero[..., used:] = 0.0
    out_nan, g_nan = _engine(x, om, gout, geo, rc)
    out_zero, g_zero = _engine(x, zero, gout, geo, rc)
    assert torch.isfinite(out_nan).all() and torch.isfinite(g_nan[0]).all() and torch.isfinite(g_nan[1]).all()
    assert torch.equal(out_nan, out_zero) and torch.equal(g_nan[1], g_zero[1])
    assert rel_err(g_nan[0].numpy(), g_zero[0].numpy()) <= 1e-5
    # the gradient buffer starts as NaN garbage too: every padding column is written with +0.0
    xc, omc = x.cuda(), om.cuda()
    gom = torch.full_like(omc, float("nan"))
    shp, xd, omd = dcn.functional._dcnv4_inputs(xc, omc, *geo[:10], rc)
    go = gout.cuda()
    rc_ = _lib.load().dcn_v4_backward(ctypes.byref(shp), geo[10], xd.data_ptr(), omd.data_ptr(), go.data_ptr(),
                                      None, gom.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc_ == 0
    torch.cuda.synchronize()
    assert torch.equal(gom.cpu(), g_nan[1]) and _padding_is_plus_zero(gom.cpu(), geo[8], K)


@pytest.mark.parametrize("rc", [False, True])
def test_grad_offset_mask_is_deterministic(rc):
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0)
    x, om, gout = _inputs(4, 28, 28, geo, rc, seed=11)
    _, a = _engine(x, om, gout, geo, rc)
    _, b = _engine(x, om, gout, geo, rc)
    assert torch.equal(a[1], b[1])


@pytest.mark.parametrize("rc", [False, True])
def test_gradients_one_at_a_time(rc):
    geo = (3, 5, 1, 1, 1, 2, 1, 1, 2, 16, 1.0)
    x, om, gout = _inputs(2, 10, 11, geo, rc, seed=5)
    ref = dcnv4_reference.reference(x, om, geo, gout, remove_center=rc)
    _, full = _engine(x, om, gout, geo, rc)
    for need in ((True, False), (False, True)):
        _, grads = _engine(x, om, gout, geo, rc, need=need)
        for k in range(2):
            if not need[k]:
                assert grads[k] is None
            else:
                assert rel_err(grads[k].numpy(), ref[1 + k].numpy()) <= 1e-3
        if need[1]:                                 # plain stores: the same bits with or without grad_input
            assert torch.equal(grads[1], full[1])
    assert dcn.dcn_v4_backward(x.cuda(), om.cuda(), gout.cuda(), *geo, remove_center=rc, need=(False, False)) == \
        (None, None)
    # through autograd: only what is asked for
    xa, oma = x.cuda().requires_grad_(True), om.cuda()
    (gxa,) = torch.autograd.grad(dcn.dcnv4_core(xa, oma, *geo, remove_center=rc), [xa], gout.cuda())
    assert rel_err(gxa.cpu().numpy(), ref[1].numpy()) <= 1e-3


def test_cuda_graph_capture_and_replay():
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0)
    x, om, gout = _inputs(2, 12, 12, geo, True, seed=17)
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
        x, om, gout = _inputs(2, 12, 12, geo, True, seed=seed)
        with torch.no_grad():
            sx.copy_(x.cuda())
            so.copy_(om.cuda())
            sg.copy_(gout.cuda())
        graph.replay()
        torch.cuda.synchronize()
        ref = dcnv4_reference.reference(x, om, geo, gout, remove_center=True)
        _check(static[0].detach().cpu(), [t.cpu() for t in static[1:]], ref)


def test_kernel_names_through_the_profiler():
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 2, 16, 1.0)
    x, om, gout = _inputs(1, 6, 6, geo, False, seed=23)
    _lib.profile_begin()
    before = dcn.load().dcn_launch_count()
    _engine(x, om, gout, geo, False)
    launched = dcn.load().dcn_launch_count() - before
    prof = _lib.profile_end()
    assert prof["dcnv4_fwd_kernel"][0] == 1 and prof["dcnv4_bwd_kernel"][0] == 1
    assert "dcnv3_fwd_kernel" not in prof and launched == 2


def _module_pair(cfg, seed=0):
    torch.manual_seed(seed)
    m = dcn.DCNv4(**cfg)
    ref = dcnv4_reference.DCNv4Ref(**cfg)
    with torch.no_grad():                                   # trained-looking parameters, identical in both
        for (_, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
            p.add_(0.05 * torch.randn_like(p))
            q.copy_(p)
    return m, ref.double()


@pytest.mark.parametrize("cfg", [dict(channels=64, group=4),
                                 dict(channels=128, group=4, kernel_size=5, pad=2, offset_scale=0.5, dw_kernel_size=3,
                                      center_feature_scale=True, remove_center=True),
                                 dict(channels=96, group=3, dilation=2, pad=2, output_bias=False),
                                 dict(channels=64, group=2, without_pointwise=True, remove_center=True)])
def test_module_against_the_restated_reference(cfg):
    m, ref = _module_pair(cfg)
    N, H, W, C = 2, 13, 13, cfg["channels"]
    inp = torch.randn(N, H * W, C)
    gout = torch.randn(N, H * W, C)
    m = m.cuda()
    xd = inp.cuda().requires_grad_(True)
    out = m(xd)
    out.backward(gout.cuda())
    xr = inp.double().requires_grad_(True)
    exp = ref(xr)
    exp.backward(gout.double())
    assert out.shape == (N, H * W, C)
    assert rel_err(out.detach().cpu().numpy(), exp.detach().numpy()) <= 1e-4
    assert rel_err(xd.grad.cpu().numpy(), xr.grad.numpy()) <= 1e-3
    for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        assert rel_err(p.grad.cpu().numpy(), q.grad.numpy()) <= 1e-3, name


def test_module_with_a_rectangular_shape():
    m, ref = _module_pair(dict(channels=64, group=4, dw_kernel_size=3), seed=2)
    inp = torch.randn(2, 9 * 14, 64)
    out = m.cuda()(inp.cuda(), shape=(9, 14))
    exp = ref(inp.double(), shape=(9, 14))
    assert rel_err(out.detach().cpu().numpy(), exp.detach().numpy()) <= 1e-4


def test_module_under_bf16_autocast():
    """Both modules on the GPU under the same bf16 autocast, each with its core on float32 operands: the linear layers
    run in bf16 in both, so what differs is the core.  Tolerances are those of bf16 storage."""
    cfg = dict(channels=64, group=4, dw_kernel_size=3)
    m, ref = _module_pair(cfg, seed=1)
    m, ref = m.cuda(), ref.float().cuda()
    ref.core_fp32 = True
    inp = torch.randn(2, 144, 64, device="cuda")
    gout = torch.randn(2, 144, 64, device="cuda")
    xd, xr = inp.clone().requires_grad_(True), inp.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = m(xd)
        exp = ref(xr)
    assert out.dtype == exp.dtype == torch.bfloat16
    out.backward(gout)
    exp.backward(gout)
    assert rel_err(out.detach().float().cpu().numpy(), exp.detach().float().cpu().numpy()) <= 2e-2
    assert rel_err(xd.grad.cpu().numpy(), xr.grad.cpu().numpy()) <= 2e-2
    for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        assert torch.isfinite(p.grad).all(), name
        assert rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()) <= 3e-2, name


def test_offset_mask_past_2_31_elements():
    """N*Ho*Wo*Cm = 8200*64*64*64 > 2^31 while N*Ho*Wo*G = 33.6M (G = 1, a 3x7 kernel: K = 21, Cm = 64): image 8192
    of offset_mask starts exactly at element 2^31.  The images around the line and the last one must equal the same
    call on them alone, and the last one the float64 reference."""
    N, H, W, G, Gc = 8200, 64, 64, 1, 64
    geo = (3, 7, 1, 1, 1, 3, 1, 1, G, Gc, 1.0)
    Cm = dcnv4_reference.row_floats(3, 7, G, False)
    assert Cm == 64 and N * H * W * Cm > 2 ** 31 and 8192 * H * W * Cm == 2 ** 31
    floats = N * H * W * (G * Gc * 4 + Cm * 2)          # x, out, grad_out, grad_x; offset_mask and its gradient
    need = 4 * floats + (2 << 30)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2**30:.0f} GiB free, have {free / 2**30:.0f}")
    torch.manual_seed(0)
    x = torch.randn(N, H, W, G * Gc, device="cuda")
    om = torch.randn(N, H, W, Cm, device="cuda")
    om[..., :42] = torch.round(om[..., :42] * 1536) / 1024
    om[..., 63] = float("nan")                          # the one padding column
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
        assert rel_err(grads[0][s].cpu().numpy(), g1[0].cpu().numpy()) <= 1e-5, i
    assert bool((grads[1][..., 63] == 0).all())
    ref = dcnv4_reference.reference(x[-1:].cpu(), om[-1:].cpu(), geo, gout[-1:].cpu())
    _check(out[-1:].cpu(), [g[-1:].cpu() for g in grads], ref)
    del x, om, out, gout, grads
    torch.cuda.empty_cache()
