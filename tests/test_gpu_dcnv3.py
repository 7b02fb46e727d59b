"""DCNv3 on the GPU: csrc/dcn_dcnv3.cu against the dcnv3_* fixtures and against the float64 reference evaluated live on
the CPU (out <= 1e-4, each gradient <= 1e-3 of max |ref|) over channels per group, kernels, strides, dilations,
paddings and offset scales; the fused softmax against a separate one, the gradients one at a time, the determinism of
grad_offset and grad_mask, CUDA-graph replay, the kernel names, the drop-in module against the restated reference in
fp32 and under bf16 autocast, and one input past 2^31 elements.  Offsets are drawn on a 2^-10 grid: every fp32
coordinate of the kernels is then exact, and floor() picks the cell the float64 reference picks."""
import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from oracle import dcnv3_reference
from tests.util import golden, golden_names, rel_err

pytestmark = pytest.mark.gpu

GRAD_NAMES = ("grad_input", "grad_offset", "grad_mask")


def _inputs(N, H, W, geo, seed, spread=1.5):
    kh, kw, sh, sw, ph, pw, dh, dw, G, Gc, _ = geo
    Ho, Wo = dcnv3_reference.out_extent(H, W, kh, kw, sh, sw, ph, pw, dh, dw)
    P = kh * kw
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, H, W, G * Gc, generator=g)
    off = torch.round(torch.randn(N, Ho, Wo, G * P * 2, generator=g) * spread * 1024) / 1024
    m = torch.randn(N, Ho, Wo, G * P, generator=g)
    gout = torch.randn(N, Ho, Wo, G * Gc, generator=g)
    return x, off, m, gout


def _engine(x, off, m, gout, geo, softmax=False, need=(True, True, True)):
    args = [t.cuda() for t in (x, off, m)]
    out = dcn.dcn_v3_forward(*args, *geo, softmax_mask=softmax)
    grads = dcn.dcn_v3_backward(*args, gout.cuda(), *geo, softmax_mask=softmax, need=need)
    torch.cuda.synchronize()
    return out.cpu(), [None if t is None else t.cpu() for t in grads]


def _check(out, grads, ref):
    assert rel_err(out.numpy(), ref[0].numpy()) <= 1e-4
    for got, exp, name in zip(grads, ref[1:], GRAD_NAMES):
        assert rel_err(got.numpy(), exp.numpy()) <= 1e-3, name


@pytest.mark.parametrize("name", golden_names("dcnv3_"))
def test_against_the_fixtures(name):
    g = golden(name)
    t = {k: torch.as_tensor(v) for k, v in g.items()}
    geo = tuple(int(v) for v in g["geo"]) + (float(g["offset_scale"]),)
    out, grads = _engine(t["input"], t["offset"], t["mask"], t["grad_out"], geo, softmax=bool(g["softmax"]))
    _check(out, grads, [t[k] for k in ("out",) + GRAD_NAMES])


LIVE = {
    #  name            N  H   W   (kh, kw, sh, sw, ph, pw, dh, dw, G, Gc, os)
    "gc16_3x3":       (2, 12, 13, (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0)),
    "gc32_3x5":       (1, 10, 14, (3, 5, 1, 1, 1, 2, 1, 1, 2, 32, 1.0)),
    "gc64_5x5_p2":    (1, 11, 9, (5, 5, 1, 1, 2, 2, 1, 1, 2, 64, 0.5)),
    "gc128_1x1_p0":   (2, 7, 8, (1, 1, 1, 1, 0, 0, 1, 1, 1, 128, 2.0)),
    "gc256_3x3_s2":   (1, 9, 10, (3, 3, 2, 2, 1, 1, 1, 1, 1, 256, 1.0)),
    "gc16_s2_d2":     (2, 15, 14, (3, 3, 2, 1, 2, 0, 2, 2, 3, 16, 2.0)),
    "gc32_d2_os05":   (1, 12, 12, (3, 3, 1, 2, 0, 1, 2, 1, 4, 32, 0.5)),
    "gc64_5x3_s2":    (2, 10, 11, (5, 3, 2, 2, 2, 1, 1, 2, 2, 64, 1.0)),
}


@pytest.mark.parametrize("softmax", [False, True])
@pytest.mark.parametrize("name", list(LIVE))
def test_against_the_live_float64_reference(name, softmax):
    N, H, W, geo = LIVE[name]
    x, off, m, gout = _inputs(N, H, W, geo, seed=list(LIVE).index(name))
    out, grads = _engine(x, off, m, gout, geo, softmax=softmax)
    _check(out, grads, dcnv3_reference.reference(x, off, m, geo, gout, softmax_mask=softmax))


def test_fused_softmax_equals_a_separate_one():
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 4, 32, 1.0)
    x, off, logits, gout = _inputs(2, 14, 15, geo, seed=3)
    G, P = 4, 9
    lg = logits.cuda().requires_grad_(True)
    soft = torch.softmax(lg.view(2, 14, 15, G, P), -1).reshape(lg.shape)
    xs, offs = x.cuda(), off.cuda()
    sep = dcn.dcn_v3_forward(xs, offs, soft.detach(), *geo)
    _, _, gm_sep = dcn.dcn_v3_backward(xs, offs, soft.detach(), gout.cuda(), *geo)
    (gl_sep,) = torch.autograd.grad(soft, [lg], gm_sep)
    fused, (gx, goff, gl) = _engine(x, off, logits, gout, geo, softmax=True)
    assert rel_err(fused.numpy(), sep.cpu().numpy()) <= 1e-5
    assert rel_err(gl.numpy(), gl_sep.cpu().numpy()) <= 1e-4


@pytest.mark.parametrize("softmax", [False, True])
def test_gradients_one_at_a_time(softmax):
    geo = (3, 5, 1, 1, 1, 2, 1, 1, 2, 16, 1.0)
    x, off, m, gout = _inputs(2, 10, 11, geo, seed=5)
    ref = dcnv3_reference.reference(x, off, m, geo, gout, softmax_mask=softmax)
    _, full = _engine(x, off, m, gout, geo, softmax)
    for i in range(3):
        need = tuple(k == i for k in range(3))
        _, grads = _engine(x, off, m, gout, geo, softmax, need=need)
        for k, got in enumerate(grads):
            if k != i:
                assert got is None
        assert rel_err(grads[i].numpy(), ref[1 + i].numpy()) <= 1e-3, GRAD_NAMES[i]
        if i > 0:                                   # plain stores: the same bits with or without the other gradients
            assert torch.equal(grads[i], full[i])


@pytest.mark.parametrize("softmax", [False, True])
def test_offset_and_mask_gradients_are_deterministic(softmax):
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0)
    x, off, m, gout = _inputs(4, 28, 28, geo, seed=11)
    _, a = _engine(x, off, m, gout, geo, softmax)
    _, b = _engine(x, off, m, gout, geo, softmax)
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


def test_cuda_graph_capture_and_replay():
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0)
    x, off, m, gout = _inputs(2, 12, 12, geo, seed=17)
    sx, so, sm = (t.cuda().requires_grad_(True) for t in (x, off, m))
    sg = gout.cuda()

    def step():
        out = dcn.dcnv3_core(sx, so, sm, *geo, softmax_mask=True)
        return (out,) + torch.autograd.grad(out, [sx, so, sm], sg)

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
        x, off, m, gout = _inputs(2, 12, 12, geo, seed=seed)
        with torch.no_grad():
            sx.copy_(x.cuda())
            so.copy_(off.cuda())
            sm.copy_(m.cuda())
            sg.copy_(gout.cuda())
        graph.replay()
        torch.cuda.synchronize()
        ref = dcnv3_reference.reference(x, off, m, geo, gout, softmax_mask=True)
        _check(static[0].detach().cpu(), [t.cpu() for t in static[1:]], ref)


def test_kernel_names_through_the_profiler():
    geo = (3, 3, 1, 1, 1, 1, 1, 1, 2, 16, 1.0)
    x, off, m, gout = _inputs(1, 6, 6, geo, seed=23)
    _lib.profile_begin()
    before = dcn.load().dcn_launch_count()
    _engine(x, off, m, gout, geo)
    launched = dcn.load().dcn_launch_count() - before
    prof = _lib.profile_end()
    assert prof["dcnv3_fwd_kernel"][0] == 1 and prof["dcnv3_bwd_kernel"][0] == 1
    assert launched == 2


def _module_pair(cfg, seed=0):
    torch.manual_seed(seed)
    m = dcn.DCNv3(**cfg)
    ref = dcnv3_reference.DCNv3Ref(**cfg)
    with torch.no_grad():                                   # trained-looking parameters, identical in both
        for (_, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
            p.add_(0.05 * torch.randn_like(p))
            q.copy_(p)
    return m, ref.double()


@pytest.mark.parametrize("cfg", [dict(channels=64, group=4),
                                 dict(channels=128, group=4, kernel_size=5, pad=2, offset_scale=0.5,
                                      center_feature_scale=True),
                                 dict(channels=96, group=3, dilation=2, pad=2)])
def test_module_against_the_restated_reference(cfg):
    m, ref = _module_pair(cfg)
    N, H, W, C = 2, 14, 13, cfg["channels"]
    inp = torch.randn(N, H, W, C)
    gout = torch.randn(N, H, W, C)
    m = m.cuda()
    xd = inp.cuda().requires_grad_(True)
    out = m(xd)
    out.backward(gout.cuda())
    xr = inp.double().requires_grad_(True)
    exp = ref(xr)
    exp.backward(gout.double())
    assert rel_err(out.detach().cpu().numpy(), exp.detach().numpy()) <= 1e-4
    assert rel_err(xd.grad.cpu().numpy(), xr.grad.numpy()) <= 1e-3
    for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        assert rel_err(p.grad.cpu().numpy(), q.grad.numpy()) <= 1e-3, name


def test_module_under_bf16_autocast():
    """Both modules on the GPU under the same bf16 autocast, each with its core on float32 operands: the linear layers
    and the depthwise conv run in bf16 in both, so what differs is the core (the kernels with the softmax fused, against
    the composition with a bf16-rounded softmax).  Tolerances are those of bf16 storage."""
    cfg = dict(channels=64, group=4)
    m, ref = _module_pair(cfg, seed=1)
    m, ref = m.cuda(), ref.float().cuda()
    ref.core_fp32 = True
    inp = torch.randn(2, 12, 12, 64, device="cuda")
    gout = torch.randn(2, 12, 12, 64, device="cuda")
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


def test_input_past_2_31_elements():
    """N*H*W*C = 8200*64*64*64 > 2^31: image 8192 starts exactly at element 2^31.  The images around the line and
    the last one must equal the same call on them alone."""
    N, H, W, G, Gc = 8200, 64, 64, 4, 16
    geo = (3, 3, 1, 1, 1, 1, 1, 1, G, Gc, 1.0)
    per_img = H * W * G * Gc
    assert N * per_img > 2 ** 31 and 8192 * per_img == 2 ** 31
    floats = N * H * W * (G * Gc * 4 + G * 9 * 3 * 2)        # x, out, grad_out, grad_x; offset, mask and their grads
    need = 4 * floats + (2 << 30)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2**30:.0f} GiB free, have {free / 2**30:.0f}")
    torch.manual_seed(0)
    x = torch.randn(N, H, W, G * Gc, device="cuda")
    off = torch.round(torch.randn(N, H, W, G * 9 * 2, device="cuda") * 1536) / 1024
    m = torch.randn(N, H, W, G * 9, device="cuda")
    out = dcn.dcn_v3_forward(x, off, m, *geo, softmax_mask=True)
    gout = torch.randn_like(out)
    grads = dcn.dcn_v3_backward(x, off, m, gout, *geo, softmax_mask=True)
    torch.cuda.synchronize()
    for i in (0, 8191, 8192, 8193, N - 1):
        s = slice(i, i + 1)
        o1 = dcn.dcn_v3_forward(x[s], off[s], m[s], *geo, softmax_mask=True)
        g1 = dcn.dcn_v3_backward(x[s], off[s], m[s], gout[s], *geo, softmax_mask=True)
        assert torch.equal(out[s], o1), i
        assert torch.equal(grads[1][s], g1[1]) and torch.equal(grads[2][s], g1[2]), i
        assert rel_err(grads[0][s].cpu().numpy(), g1[0].cpu().numpy()) <= 1e-5, i
    ref = dcnv3_reference.reference(x[-1:].cpu(), off[-1:].cpu(), m[-1:].cpu(), geo, gout[-1:].cpu(),
                                    softmax_mask=True)
    _check(out[-1:].cpu(), [g[-1:].cpu() for g in grads], ref)
    del x, off, m, out, gout, grads
    torch.cuda.empty_cache()
