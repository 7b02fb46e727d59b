"""DCNv3 without a GPU: the C ABI's refusals and messages, the DcnV3Shape mirror, the Python entry points' argument
checks, the drop-in module's interface and initialisation, the dcnv3_* fixtures, and the oracle's consistency: the
grid_sample restatement, the pixel-coordinate reference, a per-point loop and the MSDA reference at one level agree."""
import ctypes
import os
import re
import tempfile

import numpy as np
import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from oracle import dcnv3_reference, make_golden, make_golden_dcnv3, msda_reference
from tests.util import golden, golden_names

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["N", "H", "W", "G", "Gc", "kh", "kw", "sh", "sw", "ph", "pw", "dh", "dw", "flags"]


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
    return lib.dcn_v3_forward(ctypes.byref(s) if s is not None else None, 1.0, *args, None)


def _bwd(lib, s, args):
    return lib.dcn_v3_backward(ctypes.byref(s) if s is not None else None, 1.0, *args, None)


FWD_ARGS = ("input", "offset", "mask", "out")
BWD_ARGS = ("input", "offset", "mask", "grad_out", "grad_input", "grad_offset", "grad_mask")


def test_shape_struct_matches_header():
    text = open(os.path.join(ROOT, "include", "dcn_b200.h")).read()
    body = re.search(r"typedef struct DcnV3Shape \{(.*?)\} DcnV3Shape;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [n.strip() for decl in re.findall(r"int32_t ([^;]+);", body) for n in decl.split(",")]
    assert names == [f[0] for f in _lib.DcnV3Shape._fields_] == FIELDS
    assert ctypes.sizeof(_lib.DcnV3Shape) == 56
    assert re.search(r"DCN_V3_FLAG_SOFTMAX_MASK = 1\b", text) and _lib.DCN_V3_FLAG_SOFTMAX_MASK == 1


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
    if i >= 4:
        return          # the three gradients are optional (NULL: not computed); this call would launch
    assert _bwd(lib, _shape(), args) == -2
    assert lib.dcn_last_error().decode().endswith(f"{BWD_ARGS[i]} is NULL")


def test_backward_with_no_gradient_requested_does_nothing(ptrs):
    ok, _ = ptrs
    assert _bwd(dcn.load(), _shape(), [ok] * 4 + [None] * 3) == 0


def test_null_shape_is_refused(ptrs):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, None, [ok] * 4) == -2 and b"DcnV3Shape is NULL" in lib.dcn_last_error()
    assert _bwd(lib, None, [ok] * 7) == -2 and b"DcnV3Shape is NULL" in lib.dcn_last_error()


@pytest.mark.parametrize("field, value", [(f, v) for f in ("N", "H", "W", "G", "Gc", "kh", "kw", "sh", "sw", "dh", "dw")
                                          for v in (0, -1)] + [("ph", -1), ("pw", -1)])
def test_out_of_range_geometry_is_a_bad_shape(ptrs, field, value):
    lib = dcn.load()
    ok, _ = ptrs
    s = _shape(**{field: value})
    assert _fwd(lib, s, [ok] * 4) == -1 and b"bad shape" in lib.dcn_last_error()
    assert _bwd(lib, s, [ok] * 7) == -1 and b"bad shape" in lib.dcn_last_error()


@pytest.mark.parametrize("kw, msg", [
    (dict(H=2, ph=0), b"empty output Ho=0 Wo=16"),
    (dict(W=4, pw=0, dw=2), b"empty output Ho=16 Wo=0"),
    (dict(N=1 << 10, H=1024, W=2048, G=1, ph=1), b"N*Ho*Wo*G = 2147483648 exceeds the limit 2^31 - 1"),
    (dict(N=1 << 10, H=1024, W=2048, G=1, kh=5, ph=0, kw=5, pw=0), b"N*H*W = 2147483648 exceeds the limit 2^31 - 1"),
])
def test_output_extent_and_index_limits(ptrs, kw, msg):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, _shape(**kw), [ok] * 4) == -1 and msg in lib.dcn_last_error()
    assert _bwd(lib, _shape(**kw), [ok] * 7) == -1 and msg in lib.dcn_last_error()


@pytest.mark.parametrize("kw, msg", [
    (dict(Gc=8), b"Gc = 8 channels per group is not supported (Gc in {16, 32, 64, 128, 256})"),
    (dict(Gc=48), b"Gc = 48 channels per group is not supported"),
    (dict(Gc=512), b"Gc = 512 channels per group is not supported"),
    (dict(kh=7, kw=5, ph=3, pw=2), b"P = kh*kw = 35 points exceeds the limit P <= 32"),
    (dict(flags=2), b"unknown flags 0x2 (only DCN_V3_FLAG_SOFTMAX_MASK = 1 is defined)"),
    (dict(flags=3), b"unknown flags 0x2"),
])
def test_limits_are_unsupported_with_a_message(ptrs, kw, msg):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, _shape(**kw), [ok] * 4) == -6 and msg in lib.dcn_last_error()
    assert _bwd(lib, _shape(**kw), [ok] * 7) == -6 and msg in lib.dcn_last_error()


def test_checks_run_shape_then_pointers_then_support(ptrs):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, _shape(Gc=8, H=0), [ok] * 4) == -1                 # a bad shape wins over support
    assert _fwd(lib, _shape(Gc=8), [None] + [ok] * 3) == -2             # a NULL pointer wins over support
    for Gc in (16, 32, 64, 128, 256):                                   # what is covered passes up to the pointers
        for kh, kw in ((1, 1), (3, 3), (5, 5), (3, 5), (4, 8)):
            for flags in (0, 1):
                assert _fwd(lib, _shape(Gc=Gc, kh=kh, kw=kw, ph=2, pw=2, flags=flags), [None] + [ok] * 3) == -2


GEO = dict(kernel_h=3, kernel_w=3, stride_h=1, stride_w=1, pad_h=1, pad_w=1, dilation_h=1, dilation_w=1, group=2,
           group_channels=16, offset_scale=1.0)


def _cpu_inputs(N=1, H=5, W=6, G=2, Gc=16, P=9):
    return torch.zeros(N, H, W, G * Gc), torch.zeros(N, H, W, G * P * 2), torch.zeros(N, H, W, G * P)


def _args(x, off, m, **kw):
    g = dict(GEO, **kw)
    return (x, off, m) + tuple(g.values())


def test_functional_refuses_cpu_and_non_fp32_inputs():
    x, off, m = _cpu_inputs()
    with pytest.raises(ValueError, match="input must be a CUDA tensor: there is no CPU path"):
        dcn.dcnv3_core(*_args(x, off, m))
    with pytest.raises(ValueError, match="input must be a float32 tensor, got torch.float16"):
        dcn.dcnv3_core(*_args(x.half(), off, m))
    with pytest.raises(ValueError, match="offset must be a float32 tensor, got torch.float64"):
        dcn.DCNv3Function.apply(*_args(x, off.double(), m), 256)
    with pytest.raises(ValueError, match="mask must be a float32 tensor"):
        dcn.dcnv3_core(*_args(x, off, m.bfloat16()))
    with pytest.raises(ValueError, match="remove_center=True is not supported"):
        dcn.DCNv3Function.apply(*_args(x, off, m), 256, True)


def test_functional_checks_shapes_before_the_device(monkeypatch):
    """Shape checks run on metadata; here the device check is bypassed to reach them without a GPU."""
    from jittor_dcn_b200 import functional as fn
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    x, off, m = _cpu_inputs()
    cases = [
        (_args(x[0], off, m), "input must be \\[N, H, W, group\\*group_channels\\]"),
        (_args(x, off, m, group=4), "input has 32 channels, group\\*group_channels = 4\\*16 = 64"),
        (_args(x, off[..., :-2], m), "offset shape"),
        (_args(x, off, m[:, :1]), "mask shape"),
        (_args(x, off, m, kernel_h=7, pad_h=0), "empty output"),
        (_args(x, off, m, stride_w=0), "stride_w = 0 is out of range"),
        (_args(x, off, m, pad_h=-1), "pad_h = -1 is out of range"),
        (_args(x, off, m, kernel_w=3.0), "kernel_w must be an int"),
    ]
    for args, msg in cases:
        with pytest.raises(ValueError, match=msg):
            fn._dcnv3_inputs(*args[:13], False)


def test_module_interface_and_state_dict():
    m = dcn.DCNv3()
    assert (m.channels, m.kernel_size, m.dw_kernel_size, m.stride, m.pad, m.dilation, m.group, m.group_channels,
            m.offset_scale, m.center_feature_scale) == (64, 3, 3, 1, 1, 1, 4, 16, 1.0, False)
    assert list(m.state_dict()) == ["dw_conv.0.weight", "dw_conv.0.bias", "dw_conv.1.1.weight", "dw_conv.1.1.bias",
                                    "offset.weight", "offset.bias", "mask.weight", "mask.bias", "input_proj.weight",
                                    "input_proj.bias", "output_proj.weight", "output_proj.bias"]
    for cfg in (dict(), dict(channels=128, kernel_size=5, group=8, center_feature_scale=True, dw_kernel_size=3)):
        ours, ref = dcn.DCNv3(**cfg), dcnv3_reference.DCNv3Ref(**cfg)
        assert [(k, tuple(v.shape)) for k, v in ours.state_dict().items()] == \
            [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
    m2 = dcn.DCNv3(channels=128, kernel_size=5, group=8, center_feature_scale=True)
    assert list(m2.state_dict())[:2] == ["center_feature_scale_proj_weight", "center_feature_scale_proj_bias"]
    assert tuple(m2.offset.weight.shape) == (8 * 25 * 2, 128) and tuple(m2.mask.weight.shape) == (8 * 25, 128)
    assert isinstance(dcn.DCNv3(norm_layer="BN").dw_conv[1][0], torch.nn.BatchNorm2d)
    assert isinstance(dcn.DCNv3(act_layer="ReLU").dw_conv[2], torch.nn.ReLU)
    with pytest.raises(ValueError, match="channels must be divisible by group, but got 100 and 8"):
        dcn.DCNv3(channels=100, group=8)
    with pytest.warns(UserWarning):
        dcn.DCNv3(channels=48, group=4)


@pytest.mark.parametrize("cfg", [dict(), dict(channels=128, kernel_size=5, group=8, center_feature_scale=True)])
def test_module_initialisation_equals_the_reference_under_one_seed(cfg):
    torch.manual_seed(7)
    m = dcn.DCNv3(**cfg)
    torch.manual_seed(7)
    ref = dcnv3_reference.DCNv3Ref(**cfg)
    for (k, a), (_, b) in zip(m.state_dict().items(), ref.state_dict().items()):
        assert torch.equal(a, b), k
    for lin in (m.offset, m.mask):
        assert float(lin.weight.detach().abs().max()) == 0.0 and float(lin.bias.detach().abs().max()) == 0.0
    assert float(m.input_proj.bias.detach().abs().max()) == 0.0 and float(m.input_proj.weight.detach().abs().max()) > 0.0


def test_dcnv3_fixtures_cover_the_required_cases():
    names = golden_names("dcnv3_")
    assert names == sorted(make_golden_dcnv3.DCNV3)
    Gc, kernels, strides, dils, scales, softmax, outside, border = set(), set(), set(), set(), set(), set(), 0, 0
    for n in names:
        g = golden(n)
        kh, kw, sh, sw, ph, pw, dh, dw, G, gc = (int(v) for v in g["geo"])
        os_ = float(g["offset_scale"])
        Gc.add(gc), kernels.add((kh, kw)), strides.update((sh, sw)), dils.update((dh, dw)), scales.add(os_)
        softmax.add(bool(g["softmax"]))
        N, H, W, _ = g["input"].shape
        Ho, Wo = dcnv3_reference.out_extent(H, W, kh, kw, sh, sw, ph, pw, dh, dw)
        x, y = dcnv3_reference.sample_coordinates(Ho, Wo, torch.as_tensor(g["offset"]).double(), kh, kw, sh, sw, ph,
                                                  pw, dh, dw, G, os_)
        x, y = x.numpy(), y.numpy()
        outside += int(((x < -1) | (x > W) | (y < -1) | (y > H)).sum())
        border += int(((x == 0) | (x == W - 1) | (y == 0) | (y == H - 1) | (x == -1) | (y == -1)).sum())
    assert {16, 32} <= Gc and {(3, 3), (3, 5)} <= kernels and 2 in strides and 2 in dils
    assert any(s != 1.0 for s in scales) and softmax == {True, False} and outside > 0 and border > 0


def test_dcnv3_fixtures_regenerate_within_1e_6():
    prev = torch.get_num_threads()
    torch.set_num_threads(make_golden.GOLDEN_CPU_THREADS)
    try:
        with tempfile.TemporaryDirectory() as d:
            make_golden_dcnv3.make_dcnv3(d)
            for n in make_golden_dcnv3.DCNV3:
                new, old = dict(np.load(os.path.join(d, n + ".npz"))), golden(n)
                assert sorted(new) == sorted(old)
                for k in old:
                    if old[k].dtype.kind == "f":
                        den = max(float(np.abs(old[k]).max()), 1e-30)
                        assert float(np.abs(new[k] - old[k]).max()) / den <= 1e-6, (n, k)
                    else:
                        assert np.array_equal(new[k], old[k]), (n, k)
    finally:
        torch.set_num_threads(prev)


@pytest.mark.parametrize("geo", [
    (3, 3, 1, 1, 1, 1, 1, 1, 2, 4, 1.0),
    (3, 5, 2, 1, 0, 2, 2, 1, 1, 3, 0.5),      # rectangular kernel and padding: pins the x-major order
    (2, 3, 1, 2, 1, 0, 1, 2, 2, 2, 2.0),      # even kernel extent: hw / hh rounded down
])
def test_oracle_restatements_agree(geo):
    """grid_sample composition == pixel-coordinate reference == per-point loop == MSDA reference at L = 1."""
    kh, kw, sh, sw, ph, pw, dh, dw, G, Gc, os_ = geo
    N, H, W = 2, 6, 7
    Ho, Wo = dcnv3_reference.out_extent(H, W, kh, kw, sh, sw, ph, pw, dh, dw)
    P = kh * kw
    gen = torch.Generator().manual_seed(sum(geo[:10]))
    x = torch.randn(N, H, W, G * Gc, generator=gen, dtype=torch.float64)
    off = torch.randn(N, Ho, Wo, G * P * 2, generator=gen, dtype=torch.float64) * 1.5
    m = torch.randn(N, Ho, Wo, G * P, generator=gen, dtype=torch.float64)
    comp = dcnv3_reference.dcnv3_core_pytorch(x, off, m, *geo)
    pix = dcnv3_reference.dcnv3_core_pixels(x, off, m, *geo)
    loop = dcnv3_reference.points_loop(x, off, m, *geo)
    xs, ys = dcnv3_reference.sample_coordinates(Ho, Wo, off, kh, kw, sh, sw, ph, pw, dh, dw, G, os_)
    loc = torch.stack(((xs + 0.5) / W, (ys + 0.5) / H), -1).reshape(N, Ho * Wo, G, 1, P, 2)
    ms = msda_reference.ms_deform_attn_core_pytorch(x.reshape(N, H * W, G, Gc), [(H, W)], loc,
                                                    m.reshape(N, Ho * Wo, G, 1, P)).reshape(N, Ho, Wo, G * Gc)
    for other in (pix, loop, ms):
        assert float((comp - other).abs().max()) <= 1e-12 * float(comp.abs().max())
    # the softmax switch of the reference is InternImage's per-group softmax of the logits
    soft = torch.softmax(m.reshape(N, Ho, Wo, G, P), -1).reshape(m.shape)
    assert torch.allclose(dcnv3_reference.reference(x, off, m, geo, softmax_mask=True),
                          dcnv3_reference.dcnv3_core_pytorch(x, off, soft, *geo), rtol=0, atol=1e-12)
