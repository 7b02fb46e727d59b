"""The whole modulated layer (mmcv's ModulatedDeformConv2dPack) without a GPU: argument checks of the three C calls
(and of the three unmodulated layer calls that share their implementation), the shapes the layer path covers, and the
module's interface and initialisation."""
import ctypes
import math

import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib

FWD, BWD = _lib.PHASE_LAYER_FORWARD_MODULATED, _lib.PHASE_LAYER_BACKWARD_MODULATED
FLAVOURS = (True, False)   # modulated: dcn_*_modulated; False: dcn_offset_conv_forward / dcn_layer_forward / _backward


def _buffers():
    buf = ctypes.create_string_buffer(1 << 16)
    base = (ctypes.addressof(buf) + 255) // 256 * 256
    return buf, base, ctypes.c_void_p(base)


def _shape(variant=dcn.VARIANT_DCNV1, operand=dcn.OPERAND_FP32, flags=0):
    return dcn.make_shape(2, 64, 64, 12, 12, 3, 1, 1, variant, operand, flags)


def _calls(lib, s, x=None, offset=None, mask=None, gwoff=None, ws_bytes=1 << 15, ok=None, modulated=True):
    """(name, rc) of the three calls of one layer flavour with every pointer valid except those given, one call per
    item, so that dcn_last_error() is that call's."""
    p = lambda v: ok if v is None else v
    if modulated:
        yield "offset_conv", lib.dcn_offset_conv_forward_modulated(ctypes.byref(s), p(x), ok, None, p(offset), p(mask),
                                                                   ok, ws_bytes, None)
        yield "forward", lib.dcn_layer_forward_modulated(ctypes.byref(s), p(x), ok, None, ok, None, p(offset), p(mask),
                                                         ok, ok, ws_bytes, None)
        yield "backward", lib.dcn_layer_backward_modulated(ctypes.byref(s), p(x), p(offset), p(mask), ok, ok, ok, ok,
                                                           p(gwoff), None, ok, None, ok, ws_bytes, None)
    else:
        yield "offset_conv", lib.dcn_offset_conv_forward(ctypes.byref(s), p(x), ok, None, p(offset), ok, ws_bytes, None)
        yield "forward", lib.dcn_layer_forward(ctypes.byref(s), p(x), ok, None, ok, None, p(offset), ok, ok, ws_bytes,
                                               None)
        yield "backward", lib.dcn_layer_backward(ctypes.byref(s), p(x), p(offset), ok, ok, ok, ok, p(gwoff), None, ok,
                                                 None, ok, ws_bytes, None)


@pytest.mark.parametrize("modulated, arg", [(True, "x"), (True, "offset"), (True, "mask"), (False, "x"),
                                             (False, "offset")], ids=["x", "offset", "mask", "plain-x", "plain-offset"])
def test_layer_calls_reject_null_and_misaligned_pointers_by_name(modulated, arg):
    lib = dcn.load()
    buf, base, ok = _buffers()
    s = _shape()
    for ptr, code, text in ((ctypes.c_void_p(0), -2, f"{arg} is NULL"), (ctypes.c_void_p(base + 4), -3, arg)):
        for name, rc in _calls(lib, s, ok=ok, modulated=modulated, **{arg: ptr}):
            assert rc == code, (name, rc)
            assert text.encode() in lib.dcn_last_error(), (name, lib.dcn_last_error())
    del buf


def test_layer_backward_rejects_a_bad_grad_offset_weight():
    lib = dcn.load()
    buf, base, ok = _buffers()
    s = _shape()
    for modulated in FLAVOURS:
        rc = dict(_calls(lib, s, ok=ok, gwoff=ctypes.c_void_p(0), modulated=modulated))["backward"]
        assert rc == -2 and b"grad_offset_weight is NULL" in lib.dcn_last_error(), modulated
        rc = dict(_calls(lib, s, ok=ok, gwoff=ctypes.c_void_p(base + 8), modulated=modulated))["backward"]
        assert rc == -3 and b"grad_offset_weight" in lib.dcn_last_error(), modulated
    del buf


@pytest.mark.parametrize("variant", [dcn.VARIANT_TORCH, dcn.VARIANT_JITTOR])
def test_layer_calls_refuse_the_reference_variants(variant):
    lib = dcn.load()
    buf, base, ok = _buffers()
    s = _shape(variant=variant)
    for name, rc in _calls(lib, s, ok=ok):
        assert rc == -6, name
        assert b"DCN_VARIANT_DCNV1" in lib.dcn_last_error(), name
    for ph in (FWD, BWD):
        assert _lib.path_name(s, ph) == "unsupported"
        assert lib.dcn_workspace_bytes(ctypes.byref(s), ph) == 0
    del buf


def test_layer_calls_refuse_bf16_operands():
    lib = dcn.load()
    buf, base, ok = _buffers()
    s = _shape(operand=dcn.OPERAND_BF16)
    for name, rc in _calls(lib, s, ok=ok):
        assert rc == -6, name
        assert b"fp32 operands only" in lib.dcn_last_error(), name
    del buf


def test_layer_calls_refuse_a_workspace_that_is_too_small():
    lib = dcn.load()
    buf, base, ok = _buffers()
    s = _shape()
    for modulated in FLAVOURS:
        for name, rc in _calls(lib, s, ok=ok, ws_bytes=16, modulated=modulated):
            assert rc == -4, (name, modulated)
            assert b"workspace" in lib.dcn_last_error(), (name, modulated)
    del buf


def test_force_simt_and_uncovered_shapes_answer_unsupported():
    lib = dcn.load()
    buf, base, ok = _buffers()
    for s in (_shape(flags=dcn.FLAG_FORCE_SIMT), dcn.make_shape(2, 4, 16, 12, 12, 3, 1, 1, dcn.VARIANT_DCNV1)):
        assert [_lib.path_name(s, ph) for ph in (FWD, BWD)] == ["unsupported", "unsupported"]
        rc = lib.dcn_layer_forward_modulated(ctypes.byref(s), ok, ok, None, ok, None, ok, ok, ok, ok, 1 << 15, None)
        assert rc == -6 and b"DCN_PHASE_LAYER_FORWARD_MODULATED" in lib.dcn_last_error()
        assert [_lib.path_name(s, ph) for ph in (_lib.PHASE_LAYER_FORWARD, _lib.PHASE_LAYER_BACKWARD)] == \
            ["unsupported", "unsupported"]
        rc = lib.dcn_layer_forward(ctypes.byref(s), ok, ok, None, ok, None, ok, ok, ok, 1 << 15, None)
        assert rc == -6 and b"DCN_PHASE_LAYER_FORWARD)" in lib.dcn_last_error()
    del buf


# (B, C, O, H, W, kernel, stride, padding): ResNet C3-C5 (O = 512 runs as output-channel groups), cfg2 in DCNv1 mode,
# the 16 / 32-channel layers of the warp-MMA kernels, a 1 x 3 kernel (3N = 9)
COVERED = [
    (8, 128, 128, 28, 28, 3, 1, 1), (8, 128, 128, 56, 56, 3, 2, 1),
    (8, 256, 256, 14, 14, 3, 1, 1), (8, 256, 256, 28, 28, 3, 2, 1),
    (8, 512, 512, 7, 7, 3, 1, 1), (8, 512, 512, 14, 14, 3, 2, 1),
    (256, 64, 64, 128, 128, 3, 1, 1),
    (8, 16, 16, 32, 32, 3, 1, 1), (8, 32, 32, 32, 32, 3, 2, 1),
    (8, 64, 64, 16, 16, (1, 3), 1, 1),
]


@pytest.mark.parametrize("shape", COVERED)
def test_required_shapes_run_on_the_layer_path(shape):
    B, C, O, H, W, k, s, p = shape
    shp = dcn.make_shape(B, C, O, H, W, k, s, p, dcn.VARIANT_DCNV1)
    assert [_lib.path_name(shp, ph) for ph in (FWD, BWD)] == ["umma", "umma"]
    assert all(dcn.load().dcn_workspace_bytes(ctypes.byref(shp), ph) > 0 for ph in (FWD, BWD))
    assert dcn.modulated_layer_supported((B, C, H, W), O, k, s, p)
    assert not dcn.modulated_layer_supported((B, C, H, W), O, k, s, p, flags=dcn.FLAG_FORCE_SIMT)


def test_module_interface_and_state_dict():
    m = dcn.ModulatedDeformConv2dPack(16, 32, 3, stride=2, padding=1)
    assert (m.in_channels, m.out_channels, m.kernel_size, m.stride, m.padding, m.dilation, m.groups,
            m.deform_groups) == (16, 32, (3, 3), (2, 2), (1, 1), (1, 1), 1, 1)
    assert m.engine_offset_conv is True and m.keep_staged_input is False
    assert list(m.state_dict()) == ["weight", "bias", "conv_offset.weight", "conv_offset.bias"]
    assert tuple(m.weight.shape) == (32, 16, 3, 3) and tuple(m.bias.shape) == (32,)
    assert tuple(m.conv_offset.weight.shape) == (27, 16, 3, 3) and tuple(m.conv_offset.bias.shape) == (27,)
    c = m.conv_offset
    assert (c.kernel_size, c.stride, c.padding, c.dilation, c.groups) == ((3, 3), (2, 2), (1, 1), (1, 1), 1)
    assert m.extra_repr() == "16, 32, kernel_size=(3, 3), stride=(2, 2), padding=(1, 1)"
    nb = dcn.ModulatedDeformConv2dPack(8, 4, (1, 3))
    assert nb.bias is not None and list(dict(nb.named_parameters())) == ["weight", "bias", "conv_offset.weight",
                                                                         "conv_offset.bias"]
    assert tuple(nb.conv_offset.weight.shape) == (9, 8, 1, 3)
    nob = dcn.ModulatedDeformConv2dPack(8, 4, 3, padding=1, bias=False)
    assert nob.bias is None and list(nob.state_dict()) == ["weight", "conv_offset.weight", "conv_offset.bias"]
    assert nob.extra_repr() == "8, 4, kernel_size=(3, 3), stride=(1, 1), padding=(1, 1), bias=False"
    # a checkpoint of the same keys loads unchanged
    m2 = dcn.ModulatedDeformConv2dPack(16, 32, 3, stride=2, padding=1)
    m2.load_state_dict(m.state_dict())
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))


def test_module_initialisation_follows_mmcv():
    torch.manual_seed(3)
    m = dcn.ModulatedDeformConv2dPack(64, 48, 3, padding=1)
    bound = 1.0 / math.sqrt(64 * 9)
    w = m.weight.detach()
    assert w.abs().max() <= bound and w.abs().max() > 0.9 * bound and w.std() > 0.5 * bound / math.sqrt(3)
    assert torch.count_nonzero(m.bias) == 0
    assert torch.count_nonzero(m.conv_offset.weight) == 0 and torch.count_nonzero(m.conv_offset.bias) == 0


@pytest.mark.parametrize("kw, what", [(dict(dilation=2), "dilation"), (dict(groups=2), "groups"),
                                      (dict(deform_groups=2), "deform_groups")])
def test_module_refuses_what_the_engine_does_not_run(kw, what):
    with pytest.raises(ValueError, match=what):
        dcn.ModulatedDeformConv2dPack(8, 16, 3, padding=1, **kw)


def test_module_falls_back_to_the_composition_on_the_cpu():
    # no CUDA tensor: the layer path is not taken, the composition's span has no CPU path and says so
    m = dcn.ModulatedDeformConv2dPack(4, 8, 3, padding=1)
    assert not m._whole_layer_on_engine(torch.zeros(1, 4, 6, 6))
    if not torch.cuda.is_available():
        with pytest.raises(dcn.DcnError, match="CUDA"):
            m(torch.zeros(1, 4, 6, 6))


def test_offset_weight_shape_is_checked():
    x = torch.zeros(1, 4, 6, 6)
    with pytest.raises(ValueError, match="3N outputs"):
        dcn.dcn_layer_forward_modulated(x, torch.zeros(18, 4, 3, 3), None, torch.zeros(8, 4, 3, 3), None)
