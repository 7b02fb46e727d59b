"""DCNv3 / DCNv4 on bfloat16 and float16 operands without a GPU: the dtype rule of the Python entry points (one shared
dtype of float32, bfloat16 or float16; a mixed call names the first tensor that is not float32) and the typed C calls'
operand check, which comes after the pointer checks and returns the untyped calls' status for everything else."""
import ctypes
import itertools
import os
import re

import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["N", "H", "W", "G", "Gc", "kh", "kw", "sh", "sw", "ph", "pw", "dh", "dw", "flags"]
GEO = dict(kernel_h=3, kernel_w=3, stride_h=1, stride_w=1, pad_h=1, pad_w=1, dilation_h=1, dilation_w=1, group=2,
           group_channels=16, offset_scale=1.0)
HALF = (torch.bfloat16, torch.float16)
DTYPES = (torch.float32, torch.bfloat16, torch.float16, torch.float64)


def _v3_inputs(dtypes):
    return [torch.zeros(s, dtype=d) for s, d in zip([(1, 5, 6, 32), (1, 5, 6, 36), (1, 5, 6, 18)], dtypes)]


def _v4_inputs(dtypes):
    Cm = dcn.dcnv4_row_floats(3, 3, 2)
    return [torch.zeros(s, dtype=d) for s, d in zip([(1, 5, 6, 32), (1, 5, 6, Cm)], dtypes)]


CALLS = {
    "dcnv3_core": (3, ("input", "offset", "mask"), lambda t: dcn.dcnv3_core(*t, *GEO.values())),
    "DCNv3Function": (3, ("input", "offset", "mask"), lambda t: dcn.DCNv3Function.apply(*t, *GEO.values(), 256)),
    "dcn_v3_forward": (3, ("input", "offset", "mask"), lambda t: dcn.dcn_v3_forward(*t, *GEO.values())),
    "dcn_v3_backward": (3, ("input", "offset", "mask"),
                        lambda t: dcn.dcn_v3_backward(*t, torch.zeros(1, 5, 6, 32, dtype=t[0].dtype), *GEO.values())),
    "dcnv4_core": (2, ("input", "offset_mask"), lambda t: dcn.dcnv4_core(*t, *GEO.values())),
    "DCNv4Function": (2, ("input", "offset_mask"), lambda t: dcn.DCNv4Function.apply(*t, *GEO.values(), 256, False)),
    "dcn_v4_forward": (2, ("input", "offset_mask"), lambda t: dcn.dcn_v4_forward(*t, *GEO.values())),
    "dcn_v4_backward": (2, ("input", "offset_mask"),
                        lambda t: dcn.dcn_v4_backward(*t, torch.zeros(1, 5, 6, 32, dtype=t[0].dtype), *GEO.values())),
}


def _inputs(call, dtypes):
    return (_v3_inputs if CALLS[call][0] == 3 else _v4_inputs)(dtypes)


@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("call", list(CALLS))
def test_one_half_dtype_passes_the_dtype_check(call, dtype):
    """All-bf16 or all-fp16 CPU tensors get past the dtype check and stop at the device check."""
    n, _, fn = CALLS[call]
    with pytest.raises(ValueError, match="input must be a CUDA tensor: there is no CPU path"):
        fn(_inputs(call, [dtype] * n))


@pytest.mark.parametrize("call", list(CALLS))
def test_mixed_dtypes_name_the_first_tensor_that_is_not_float32(call):
    n, names, fn = CALLS[call]
    for dtypes in itertools.product(DTYPES[:3], repeat=n):
        if len(set(dtypes)) == 1:
            continue
        first = next(i for i, d in enumerate(dtypes) if d != torch.float32)
        msg = (f"{names[first]} must be a float32 tensor, got {dtypes[first]} "
               r"\(.* must share one dtype: float32, bfloat16 or float16\)")
        with pytest.raises(ValueError, match=msg):
            fn(_inputs(call, dtypes))


@pytest.mark.parametrize("call", list(CALLS))
def test_float64_is_refused(call):
    n, _, fn = CALLS[call]
    with pytest.raises(ValueError, match="input must be a float32 tensor, got torch.float64"):
        fn(_inputs(call, [torch.float64] * n))


def test_a_non_tensor_is_named():
    x, off, m = _v3_inputs([torch.bfloat16] * 3)
    with pytest.raises(ValueError, match="mask must be a float32 tensor, got list"):
        dcn.dcn_v3_forward(x, off, [0.0], *GEO.values())


# ---- the typed C calls ---------------------------------------------------------------------------------------------
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


# name -> (pointer arguments, index of the first optional one or None)
TYPED = {"dcn_v3_forward": (4, None), "dcn_v3_backward": (7, 4), "dcn_v4_forward": (3, None),
         "dcn_v4_backward": (5, 3)}


def _untyped(name, s, args):
    return getattr(dcn.load(), name)(ctypes.byref(s) if s is not None else None, 1.0, *args, None)


def _typed(name, s, operand, args):
    return getattr(dcn.load(), name + "_typed")(ctypes.byref(s) if s is not None else None, operand, 1.0, *args, None)


def test_header_declares_the_operand_and_the_four_calls():
    text = open(os.path.join(ROOT, "include", "dcn_b200.h")).read()
    assert re.search(r"DCN_OPERAND_FP16 = 2\b", text) and _lib.OPERAND_FP16 == dcn.OPERAND_FP16 == 2
    for name in TYPED:
        assert re.search(rf"DCN_API int {name}_typed\(const DcnV3Shape\* s, int32_t operand, float offset_scale",
                         text), name
        assert name + "_typed" in _lib.EXPORTS and hasattr(dcn.load(), name + "_typed")


@pytest.mark.parametrize("operand", [3, -1])
@pytest.mark.parametrize("name", list(TYPED))
def test_an_unknown_operand_is_unsupported(ptrs, name, operand):
    ok, _ = ptrs
    n, _ = TYPED[name]
    assert _typed(name, _shape(), operand, [ok] * n) == -6
    assert lib_error() == (f"{name}_typed: unknown operand {operand} (DCN_OPERAND_FP32 = 0, DCN_OPERAND_BF16 = 1 or "
                           "DCN_OPERAND_FP16 = 2)")


def lib_error():
    return dcn.load().dcn_last_error().decode()


@pytest.mark.parametrize("operand", [0, 1, 2, 3, -1])
@pytest.mark.parametrize("name", list(TYPED))
def test_pointer_and_shape_checks_come_first_with_the_untyped_status(ptrs, name, operand):
    ok, bad = ptrs
    n, optional = TYPED[name]
    for i in range(n):
        args = [ok] * n
        args[i] = bad
        assert _typed(name, _shape(), operand, args) == _untyped(name, _shape(), args) == -3
        args[i] = None
        if optional is None or i < optional:
            assert _typed(name, _shape(), operand, args) == _untyped(name, _shape(), args) == -2
            assert lib_error().endswith(" is NULL")
    assert _typed(name, None, operand, [ok] * n) == _untyped(name, None, [ok] * n) == -2
    assert _typed(name, _shape(N=0), operand, [ok] * n) == _untyped(name, _shape(N=0), [ok] * n) == -1


@pytest.mark.parametrize("name", list(TYPED))
def test_the_operand_is_checked_after_the_flags(ptrs, name):
    """An unknown flag and an unknown operand together: the flag is named, as in the untyped call."""
    ok, _ = ptrs
    n, _ = TYPED[name]
    assert _typed(name, _shape(flags=8), 3, [ok] * n) == _untyped(name, _shape(flags=8), [ok] * n) == -6
    assert "unknown flags 0x8" in lib_error()
    assert _typed(name, _shape(Gc=24), 3, [ok] * n) == -6 and "Gc = 24" in lib_error()


@pytest.mark.parametrize("name", ["dcn_v3_backward", "dcn_v4_backward"])
@pytest.mark.parametrize("operand", [0, 1, 2])
def test_backward_with_no_gradient_requested_does_nothing(ptrs, name, operand):
    ok, _ = ptrs
    n, optional = TYPED[name]
    assert _typed(name, _shape(), operand, [ok] * optional + [None] * (n - optional)) == 0


def test_a_dcn_shape_still_refuses_operand_2():
    lib = dcn.load()
    s = dcn.make_shape(2, 64, 64, 12, 12, 3, 1, 1, dcn.VARIANT_TORCH, 2)
    assert lib.dcn_workspace_bytes(ctypes.byref(s), 0) == 0
    h, w = ctypes.c_int32(), ctypes.c_int32()
    assert lib.dcn_output_hw(ctypes.byref(s), ctypes.byref(h), ctypes.byref(w)) == -6
    assert "unknown operand mode 2" in lib_error() and "DCNv3 / DCNv4" in lib_error()
