"""DCNv4 without a GPU: the C ABI's refusals and messages, the symbols, the Python entry points' argument checks, the
module's interface, state-dict keys and initialisation, the dcnv4_* fixtures, and the oracle: DCNv4's reference is
DCNv3's on the unpacked offset_mask."""
import ctypes
import os
import re
import tempfile

import numpy as np
import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from oracle import dcnv3_reference, dcnv4_reference, make_golden, make_golden_dcnv4
from tests.util import golden, golden_names

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["N", "H", "W", "G", "Gc", "kh", "kw", "sh", "sw", "ph", "pw", "dh", "dw", "flags"]
RC = 2


def _shape(**kw):
    d = dict(N=2, H=16, W=16, G=4, Gc=16, kh=3, kw=3, sh=1, sw=1, ph=1, pw=1, dh=1, dw=1, flags=0)
    d.update(kw)
    return dcn.DcnV3Shape(*(d[f] for f in FIELDS))


@pytest.fixture
def ptrs():
    buf = ctypes.create_string_buffer(1 << 12)
    base = (ctypes.addressof(buf) + 255) // 256 * 256
    yield ctypes.c_void_p(base), ctypes.c_void_p(base + 4)
    del buf


def _fwd(lib, s, args):
    return lib.dcn_v4_forward(ctypes.byref(s) if s is not None else None, 1.0, *args, None)


def _bwd(lib, s, args):
    return lib.dcn_v4_backward(ctypes.byref(s) if s is not None else None, 1.0, *args, None)


FWD_ARGS = ("input", "offset_mask", "out")
BWD_ARGS = ("input", "offset_mask", "grad_out", "grad_input", "grad_offset_mask")


def test_header_declares_the_flag_and_the_two_calls():
    text = open(os.path.join(ROOT, "include", "dcn_b200.h")).read()
    assert re.search(r"DCN_V4_FLAG_REMOVE_CENTER = 2\b", text) and _lib.DCN_V4_FLAG_REMOVE_CENTER == RC
    assert dcn.DCN_V4_FLAG_REMOVE_CENTER == RC
    for name in ("dcn_v4_forward", "dcn_v4_backward"):
        assert re.search(rf"DCN_API int {name}\(const DcnV3Shape\* s", text), name
        assert name in _lib.EXPORTS and hasattr(dcn.load(), name)
    lib = dcn.load()
    assert len(lib.dcn_v4_forward.argtypes) == 6 and len(lib.dcn_v4_backward.argtypes) == 8
    assert lib.dcn_version() == 100


@pytest.mark.parametrize("i", range(len(FWD_ARGS)))
def test_forward_rejects_null_and_misaligned_pointers_by_name(ptrs, i):
    lib = dcn.load()
    ok, bad = ptrs
    args = [ok] * len(FWD_ARGS)
    args[i] = None
    assert _fwd(lib, _shape(), args) == -2
    assert lib.dcn_last_error().decode().endswith(f"{FWD_ARGS[i]} is NULL")
    args[i] = bad
    assert _fwd(lib, _shape(), args) == -3
    assert lib.dcn_last_error().decode().startswith(f"{FWD_ARGS[i]} (")


@pytest.mark.parametrize("i", range(len(BWD_ARGS)))
def test_backward_rejects_null_and_misaligned_pointers_by_name(ptrs, i):
    lib = dcn.load()
    ok, bad = ptrs
    args = [ok] * len(BWD_ARGS)
    args[i] = bad
    assert _bwd(lib, _shape(), args) == -3
    assert lib.dcn_last_error().decode().startswith(f"{BWD_ARGS[i]} (")
    args[i] = None
    if i >= 3:
        return          # the two gradients are optional (NULL: not computed); this call would launch
    assert _bwd(lib, _shape(), args) == -2
    assert lib.dcn_last_error().decode().endswith(f"{BWD_ARGS[i]} is NULL")


def test_backward_with_no_gradient_requested_does_nothing(ptrs):
    ok, _ = ptrs
    assert _bwd(dcn.load(), _shape(), [ok] * 3 + [None] * 2) == 0


def test_null_shape_is_refused(ptrs):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, None, [ok] * 3) == -2 and b"DcnV3Shape is NULL" in lib.dcn_last_error()
    assert _bwd(lib, None, [ok] * 5) == -2 and b"DcnV3Shape is NULL" in lib.dcn_last_error()


@pytest.mark.parametrize("kw, msg", [
    (dict(H=0), b"bad shape"),
    (dict(ph=-1), b"bad shape"),
    (dict(H=2, ph=0), b"empty output Ho=0 Wo=16"),
    (dict(N=1 << 10, H=1024, W=2048, G=1, ph=1), b"N*Ho*Wo*G = 2147483648 exceeds the limit 2^31 - 1"),
    (dict(kh=1, kw=1, ph=0, pw=0, flags=RC), b"K = 0 points: a 1 x 1 kernel with remove_center has none"),
    (dict(G=1 << 20, kh=31, kw=31, ph=15, pw=15, N=1, H=1, W=1), b"Cm = ceil(3*G*K / 8)*8 = 3023044608 exceeds"),
])
def test_bad_shapes(ptrs, kw, msg):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, _shape(**kw), [ok] * 3) == -1 and msg in lib.dcn_last_error()
    assert _bwd(lib, _shape(**kw), [ok] * 5) == -1 and msg in lib.dcn_last_error()


@pytest.mark.parametrize("kw, msg", [
    (dict(Gc=8), b"Gc = 8 channels per group is not supported (Gc in {16, 32, 64, 128, 256})"),
    (dict(Gc=512), b"Gc = 512 channels per group is not supported"),
    (dict(flags=1), b"unknown flags 0x1 (only DCN_V4_FLAG_REMOVE_CENTER = 2 is defined; DCNv4 has no softmax)"),
    (dict(flags=4 | RC), b"unknown flags 0x4"),
    (dict(kh=2, kw=3, flags=RC), b"remove_center needs an odd kernel, got 2 x 3 (no centre point)"),
    (dict(kh=3, kw=4, flags=RC), b"remove_center needs an odd kernel, got 3 x 4"),
])
def test_limits_are_unsupported_with_a_message(ptrs, kw, msg):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, _shape(**kw), [ok] * 3) == -6 and msg in lib.dcn_last_error()
    assert _bwd(lib, _shape(**kw), [ok] * 5) == -6 and msg in lib.dcn_last_error()


def test_checks_run_shape_then_pointers_then_support(ptrs):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, _shape(Gc=8, H=0), [ok] * 3) == -1                 # a bad shape wins over support
    assert _fwd(lib, _shape(Gc=8, kh=1, kw=1, ph=0, pw=0, flags=RC), [ok] * 3) == -1    # K = 0 is a shape
    assert _fwd(lib, _shape(Gc=8), [None] + [ok] * 2) == -2             # a NULL pointer wins over support
    assert _fwd(lib, _shape(kh=2, flags=RC), [None] + [ok] * 2) == -2
    for Gc in (16, 32, 64, 128, 256):                                   # what is covered passes up to the pointers
        for kh, kw in ((1, 1), (3, 3), (5, 5), (7, 7), (3, 5), (4, 8), (9, 9)):
            for flags in (0, RC):
                if flags and (kh % 2 == 0 or kw % 2 == 0 or kh * kw == 1):
                    continue
                s = _shape(Gc=Gc, kh=kh, kw=kw, ph=4, pw=4, flags=flags)
                assert _fwd(lib, s, [None] + [ok] * 2) == -2, (Gc, kh, kw, flags)


def test_dcnv3_keeps_refusing_the_new_flag(ptrs):
    lib = dcn.load()
    ok, _ = ptrs
    assert lib.dcn_v3_forward(ctypes.byref(_shape(flags=RC)), 1.0, ok, ok, ok, ok, None) == -6
    assert b"unknown flags 0x2" in lib.dcn_last_error()


GEO = dict(kernel_h=3, kernel_w=3, stride_h=1, stride_w=1, pad_h=1, pad_w=1, dilation_h=1, dilation_w=1, group=2,
           group_channels=16, offset_scale=1.0)


def _cpu_inputs(N=1, H=5, W=6, G=2, Gc=16, Cm=56):
    return torch.zeros(N, H, W, G * Gc), torch.zeros(N, H, W, Cm)


def _args(x, om, **kw):
    g = dict(GEO, **kw)
    return (x, om) + tuple(g.values())


@pytest.mark.parametrize("kh, kw, G, rc, Cm", [(3, 3, 2, False, 56), (3, 3, 3, False, 88), (3, 3, 4, True, 96),
                                               (5, 5, 2, True, 144), (7, 7, 1, False, 152), (1, 1, 8, False, 24)])
def test_row_width(kh, kw, G, rc, Cm):
    assert dcn.dcnv4_row_floats(kh, kw, G, rc) == Cm == dcnv4_reference.row_floats(kh, kw, G, rc)


def test_functional_refuses_cpu_and_non_fp32_inputs():
    x, om = _cpu_inputs()
    with pytest.raises(ValueError, match="dcnv4: input must be a CUDA tensor: there is no CPU path"):
        dcn.dcnv4_core(*_args(x, om))
    with pytest.raises(ValueError, match="input must be a float32 tensor, got torch.float16"):
        dcn.dcnv4_core(*_args(x.half(), om))
    with pytest.raises(ValueError, match="offset_mask must be a float32 tensor, got torch.float64"):
        dcn.DCNv4Function.apply(*_args(x, om.double()), 256, False)
    with pytest.raises(ValueError, match="offset_mask must be a float32 tensor, got torch.bfloat16"):
        dcn.dcn_v4_forward(*_args(x, om.bfloat16()))


def test_functional_checks_shapes_before_the_device(monkeypatch):
    """Shape checks run on metadata; here the device check is bypassed to reach them without a GPU."""
    from jittor_dcn_b200 import functional as fn
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    x, om = _cpu_inputs()
    cases = [
        (_args(x[0], om), False, "input must be \\[N, H, W, group\\*group_channels\\]"),
        (_args(x, om, group=4), False, "input has 32 channels, group\\*group_channels = 4\\*16 = 64"),
        (_args(x, om[..., :54]), False,
         "offset_mask has 54 floats per pixel, expected Cm = ceil\\(3\\*group\\*K / 8\\)\\*8 = ceil\\(3\\*2\\*9 / 8\\)\\*8 = 56"),
        (_args(x, om), True, "offset_mask has 56 floats per pixel, expected Cm = .* = ceil\\(3\\*2\\*8 / 8\\)\\*8 = 48 \\(K = 3\\*3 - 1, remove_center\\)"),
        (_args(x, om[:, :2]), False, "offset_mask shape \\(1, 2, 6, 56\\) != \\(1, 5, 6, 56\\)"),
        (_args(x, om, kernel_h=2, pad_h=0), True, "remove_center needs an odd kernel, got 2 x 3"),
        (_args(x, om, kernel_h=1, kernel_w=1, pad_h=0, pad_w=0), True, "a 1 x 1 kernel with remove_center has no points"),
        (_args(x, om, kernel_h=7, pad_h=0), False, "empty output"),
        (_args(x, om, stride_w=0), False, "stride_w = 0 is out of range"),
        (_args(x, om, kernel_w=3.0), False, "kernel_w must be an int"),
    ]
    for args, rc, msg in cases:
        with pytest.raises(ValueError, match=msg):
            fn._dcnv4_inputs(*args[:12], rc)
    shp, _, _ = fn._dcnv4_inputs(*_args(x, om[..., :48])[:12], True)      # the valid remove_center call
    assert (shp.kh, shp.kw, shp.G, shp.Gc, shp.flags) == (3, 3, 2, 16, RC)


STATE_KEYS = ["offset_mask.weight", "offset_mask.bias", "value_proj.weight", "value_proj.bias", "output_proj.weight",
              "output_proj.bias"]


def test_module_interface_and_state_dict():
    m = dcn.DCNv4()
    assert (m.channels, m.kernel_size, m.stride, m.pad, m.dilation, m.group, m.group_channels, m.offset_scale,
            m.dw_kernel_size, m.center_feature_scale, m.remove_center, m.without_pointwise, m.K) == \
        (64, 3, 1, 1, 1, 4, 16, 1.0, None, False, 0, False, 36)
    assert list(m.state_dict()) == STATE_KEYS
    assert tuple(m.offset_mask.weight.shape) == (112, 64)          # 3*4*9 = 108 -> 112
    m2 = dcn.DCNv4(channels=96, group=3, kernel_size=5, pad=2, dw_kernel_size=3, center_feature_scale=True,
                   remove_center=True, output_bias=False)
    assert list(m2.state_dict()) == ["center_feature_scale_proj_weight", "center_feature_scale_proj_bias",
                                     "offset_mask_dw.weight", "offset_mask_dw.bias", "offset_mask.weight",
                                     "offset_mask.bias", "value_proj.weight", "value_proj.bias", "output_proj.weight"]
    assert m2.K == 3 * 24 and tuple(m2.offset_mask.weight.shape) == (216, 96)
    assert tuple(m2.offset_mask_dw.weight.shape) == (96, 1, 3, 3) and m2.output_proj.bias is None
    assert list(dcn.DCNv4(without_pointwise=True).state_dict()) == STATE_KEYS[:2]
    for cfg in (dict(), dict(channels=96, group=3, kernel_size=5, dw_kernel_size=3, center_feature_scale=True,
                             remove_center=True, output_bias=False), dict(without_pointwise=True)):
        ours, ref = dcn.DCNv4(**cfg), dcnv4_reference.DCNv4Ref(**cfg)
        assert [(k, tuple(v.shape)) for k, v in ours.state_dict().items()] == \
            [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
    with pytest.raises(ValueError, match="channels must be divisible by group, but got 100 and 8"):
        dcn.DCNv4(channels=100, group=8)
    with pytest.raises(ValueError, match="channels // group = 24 channels per group is not supported"):
        dcn.DCNv4(channels=96, group=4)
    with pytest.raises(ValueError, match="remove_center needs an odd kernel_size, got 4"):
        dcn.DCNv4(kernel_size=4, remove_center=True)


@pytest.mark.parametrize("cfg", [dict(), dict(channels=128, kernel_size=5, group=8, dw_kernel_size=3,
                                              center_feature_scale=True, remove_center=True)])
def test_module_initialisation_equals_the_reference_under_one_seed(cfg):
    torch.manual_seed(7)
    m = dcn.DCNv4(**cfg)
    torch.manual_seed(7)
    ref = dcnv4_reference.DCNv4Ref(**cfg)
    for (k, a), (_, b) in zip(m.state_dict().items(), ref.state_dict().items()):
        assert torch.equal(a, b), k
    assert float(m.offset_mask.weight.detach().abs().max()) == 0.0
    assert float(m.offset_mask.bias.detach().abs().max()) == 0.0
    for lin in (m.value_proj, m.output_proj):
        assert float(lin.bias.detach().abs().max()) == 0.0 and float(lin.weight.detach().abs().max()) > 0.0
        bound = (6.0 / (lin.in_features + lin.out_features)) ** 0.5       # xavier_uniform_
        assert float(lin.weight.detach().abs().max()) <= bound


def test_dcnv4_fixtures_cover_the_required_cases():
    names = golden_names("dcnv4_")
    assert names == sorted(make_golden_dcnv4.DCNV4)
    kernels, strides, dils, scales, rcs, padded, outside, border = set(), set(), set(), set(), set(), 0, 0, 0
    for n in names:
        g = golden(n)
        kh, kw, sh, sw, ph, pw, dh, dw, G, gc = (int(v) for v in g["geo"])
        os_, rc = float(g["offset_scale"]), bool(g["remove_center"])
        kernels.add((kh, kw)), strides.update((sh, sw)), dils.update((dh, dw)), scales.add(os_), rcs.add(rc)
        K, _ = dcnv4_reference.points(kh, kw, rc)
        om = g["offset_mask"]
        assert om.shape[-1] == dcnv4_reference.row_floats(kh, kw, G, rc)
        assert np.isnan(om[..., 3 * G * K:]).all() and not np.isnan(om[..., :3 * G * K]).any()
        assert (g["grad_offset_mask"][..., 3 * G * K:] == 0).all()
        padded += om.shape[-1] - 3 * G * K
        N, H, W, _ = g["input"].shape
        Ho, Wo = dcnv3_reference.out_extent(H, W, kh, kw, sh, sw, ph, pw, dh, dw)
        off, _ = dcnv4_reference.unpack(torch.as_tensor(om).double(), kh, kw, G, rc)
        x, y = dcnv3_reference.sample_coordinates(Ho, Wo, off, kh, kw, sh, sw, ph, pw, dh, dw, G, os_)
        x, y = x.numpy(), y.numpy()
        outside += int(((x < -1) | (x > W) | (y < -1) | (y > H)).sum())
        border += int(((x == 0) | (x == W - 1) | (y == 0) | (y == H - 1) | (x == -1) | (y == -1)).sum())
    assert {(3, 3), (5, 5)} <= kernels and 2 in strides and 2 in dils and any(s != 1.0 for s in scales)
    assert rcs == {True, False} and padded > 0 and outside > 0 and border > 0
    assert any(golden(n)["offset_mask"].shape[-1] - 3 * int(golden(n)["geo"][8]) * 9 >= 7 for n in names)  # 81 -> 88


def test_dcnv4_fixtures_regenerate():
    """Inputs, geometry and switches regenerate bit for bit.  So do the float64 results on a host like the one that
    made them; a CPU of another vector width may sum the float64 reference in another order, which 1e-12 covers."""
    prev = torch.get_num_threads()
    torch.set_num_threads(make_golden.GOLDEN_CPU_THREADS)
    try:
        with tempfile.TemporaryDirectory() as d:
            make_golden_dcnv4.make_dcnv4(d)
            for n in make_golden_dcnv4.DCNV4:
                new, old = dict(np.load(os.path.join(d, n + ".npz"))), golden(n)
                assert sorted(new) == sorted(old)
                for k in old:
                    assert new[k].dtype == old[k].dtype and new[k].shape == old[k].shape, (n, k)
                    if old[k].dtype == np.float64 and old[k].ndim:
                        den = max(float(np.abs(old[k]).max()), 1e-30)
                        assert float(np.abs(new[k] - old[k]).max()) / den <= 1e-12, (n, k)
                    else:
                        assert new[k].tobytes() == old[k].tobytes(), (n, k)
    finally:
        torch.set_num_threads(prev)


@pytest.mark.parametrize("geo", [
    (3, 3, 1, 1, 1, 1, 1, 1, 2, 4, 1.0),
    (3, 5, 2, 1, 0, 2, 2, 1, 3, 3, 0.5),      # rectangular kernel and padding, G*3K = 135 -> Cm 136
    (2, 3, 1, 2, 1, 0, 1, 2, 2, 2, 2.0),      # even kernel extent
])
def test_reference_without_remove_center_is_dcnv3_on_the_hand_unpacked_tensors(geo):
    kh, kw, sh, sw, ph, pw, dh, dw, G, Gc, os_ = geo
    N, H, W = 2, 6, 7
    Ho, Wo = dcnv3_reference.out_extent(H, W, kh, kw, sh, sw, ph, pw, dh, dw)
    P = kh * kw
    Cm = dcnv4_reference.row_floats(kh, kw, G, False)
    gen = torch.Generator().manual_seed(sum(geo[:10]))
    x = torch.randn(N, H, W, G * Gc, generator=gen, dtype=torch.float64)
    om = torch.randn(N, Ho, Wo, Cm, generator=gen, dtype=torch.float64)
    om[..., 3 * G * P:] = float("nan")
    gout = torch.randn(N, Ho, Wo, G * Gc, generator=gen, dtype=torch.float64)
    rows = om[..., :3 * G * P].reshape(N, Ho, Wo, G, 3 * P)            # by hand: [(dx, dy) * P, m * P] per group
    off = rows[..., :2 * P].reshape(N, Ho, Wo, G * P * 2)
    m = rows[..., 2 * P:].reshape(N, Ho, Wo, G * P)
    out4, gx4, gom4 = dcnv4_reference.reference(x, om, geo, gout)
    out3, gx3, goff3, gm3 = dcnv3_reference.reference(x, off, m, geo, gout)
    assert torch.equal(out4, out3) and torch.equal(gx4, gx3)
    g = gom4[..., :3 * G * P].reshape(N, Ho, Wo, G, 3 * P)
    assert torch.equal(g[..., :2 * P].reshape(goff3.shape), goff3)
    assert torch.equal(g[..., 2 * P:].reshape(gm3.shape), gm3)
    assert (gom4[..., 3 * G * P:] == 0).all()
    comp = dcnv4_reference.dcnv4_core_pytorch(x, om, *geo)              # and the grid_sample composition agrees
    assert float((comp - out4).abs().max()) <= 1e-12 * float(out4.abs().max())


@pytest.mark.parametrize("kh, kw", [(3, 3), (5, 5), (3, 5), (5, 3), (7, 7)])
def test_remove_center_is_dcnv3_with_the_centre_point_at_mask_zero(kh, kw):
    """remove_center: the K = kh*kw - 1 points are DCNv3's grid points without the centre, in the same x-major order;
    the centre point's gradients are dropped."""
    G, Gc, N, H, W = 2, 3, 1, 7, 8
    geo = (kh, kw, 1, 1, kh // 2, kw // 2, 1, 1, G, Gc, 1.0)
    K, c = dcnv4_reference.points(kh, kw, True)
    assert c == (kw // 2) * kh + kh // 2 and K == kh * kw - 1
    P = kh * kw
    i, j = divmod(c, kh)                                                 # x-major: p = i*kh + j
    assert (i, j) == (kw // 2, kh // 2)
    Cm = dcnv4_reference.row_floats(kh, kw, G, True)
    gen = torch.Generator().manual_seed(kh * 10 + kw)
    x = torch.randn(N, H, W, G * Gc, generator=gen, dtype=torch.float64)
    om = torch.randn(N, H, W, Cm, generator=gen, dtype=torch.float64)
    gout = torch.randn(N, H, W, G * Gc, generator=gen, dtype=torch.float64)
    rows = om[..., :3 * G * K].reshape(N, H, W, G, 3 * K)
    off = torch.zeros(N, H, W, G, P, 2, dtype=torch.float64)
    m = torch.zeros(N, H, W, G, P, dtype=torch.float64)
    keep = [p for p in range(P) if p != c]
    off[..., keep, :] = rows[..., :2 * K].reshape(N, H, W, G, K, 2)
    m[..., keep] = rows[..., 2 * K:]
    out4, gx4, gom4 = dcnv4_reference.reference(x, om, geo, gout, remove_center=True)
    out3, gx3, goff3, gm3 = dcnv3_reference.reference(x, off.reshape(N, H, W, -1), m.reshape(N, H, W, -1), geo, gout)
    assert torch.equal(out4, out3) and torch.equal(gx4, gx3)
    g = gom4[..., :3 * G * K].reshape(N, H, W, G, 3 * K)
    assert torch.equal(g[..., :2 * K].reshape(N, H, W, G, K, 2), goff3.reshape(N, H, W, G, P, 2)[..., keep, :])
    assert torch.equal(g[..., 2 * K:], gm3.reshape(N, H, W, G, P)[..., keep])
