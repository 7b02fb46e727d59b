"""CPU-side checks of the drop-in boundary: the shared library loads, exports exactly the
symbols include/dcn_b200.h declares, and rejects bad arguments before touching a GPU."""
import ctypes
import os
import re

import pytest

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "dcn_b200.h")).read()
    return sorted(set(re.findall(r"DCN_API[^;(]*?\b(dcn_\w+)\s*\(", text)))


def test_header_and_binding_list_the_same_symbols():
    assert _declared() == sorted(_lib.EXPORTS)


def test_library_loads_and_exports_every_declared_symbol():
    lib = dcn.load()
    for name in _declared():
        assert hasattr(lib, name), name
    assert lib.dcn_version() == 100


def test_shape_struct_matches_header():
    text = open(os.path.join(ROOT, "include", "dcn_b200.h")).read()
    body = re.search(r"typedef struct DcnShape \{(.*?)\} DcnShape;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [n.strip() for decl in re.findall(r"int32_t ([^;]+);", body) for n in decl.split(",")]
    assert names == [f[0] for f in _lib.DcnShape._fields_]
    assert ctypes.sizeof(_lib.DcnShape) == 4 * len(names)


def test_output_extent_follows_the_offset_conv():
    # deform_conv.py:34-35
    for (H, W, k, s, p), exp in [((128, 128, 3, 2, 1), (64, 64)), ((17, 23, 3, 1, 1), (17, 23)),
                                 ((20, 28, 3, 2, 1), (10, 14)), ((9, 11, (1, 3), 1, (0, 1)), (9, 11)),
                                 ((6, 6, 1, 1, 0), (6, 6))]:
        assert _lib.output_hw(dcn.make_shape(1, 2, 3, H, W, k, s, p)) == exp


def test_bad_shapes_are_rejected_without_a_gpu():
    lib = dcn.load()
    bad = [dcn.make_shape(0, 4, 8, 10, 10), dcn.make_shape(1, 4, 8, 1, 10, 3, 1, 0),
           dcn.make_shape(1, 4, 8, 10, 10, 3, 0, 1), dcn.make_shape(1, 4, 8, 10, 10, variant=7),
           dcn.make_shape(4, 4096, 8, 1024, 1024)]
    for s in bad:
        assert lib.dcn_workspace_bytes(ctypes.byref(s), 0) == 0
        assert lib.dcn_output_hw(ctypes.byref(s), None, None) == -1
        assert b"bad shape" in lib.dcn_last_error()


def test_null_and_misaligned_pointers_are_rejected_without_a_gpu():
    lib = dcn.load()
    s = dcn.make_shape(1, 4, 8, 10, 10)
    buf = ctypes.create_string_buffer(1 << 16)
    base = (ctypes.addressof(buf) + 255) // 256 * 256
    ok = ctypes.c_void_p(base)
    rc = lib.dcn_forward(ctypes.byref(s), None, ok, ok, None, ok, ok, 1 << 15, None)
    assert rc == -2 and b"x is NULL" in lib.dcn_last_error()
    rc = lib.dcn_forward(ctypes.byref(s), ok, ctypes.c_void_p(base + 4), ok, None, ok, ok, 1 << 15, None)
    assert rc == -3 and b"offset" in lib.dcn_last_error()
    rc = lib.dcn_forward(ctypes.byref(s), ok, ok, ok, None, ok, ok, 16, None)
    assert rc == -4 and b"workspace" in lib.dcn_last_error()
    rc = lib.dcn_backward(ctypes.byref(s), ok, ok, ok, ok, None, ok, ok, None, ok, 1 << 15, None)
    assert rc == -2 and b"grad_x" in lib.dcn_last_error()
    assert lib.dcn_status_string(-4) == b"workspace too small"


def test_framed_grad_x_is_refused_where_no_kernel_writes_it_without_a_gpu():
    """DCN_FLAG_GRAD_X_FRAMED asks for grad_x in the consumer's framed channels-last layout, which only the tensor-path
    data gradient writes, and writes by overwriting.  Every backward entry point refuses the flag, before any CUDA call,
    where another data gradient would run and for the pair with DCN_FLAG_ACCUM_GRAD_X.  (Otherwise NCHW values, or a
    sum, would land in a buffer the caller reads as framed.)  A workspace of 0 bytes: the refusal comes before the
    workspace check, so nothing could be launched."""
    lib = dcn.load()
    buf = ctypes.create_string_buffer(1 << 12)
    ok = ctypes.c_void_p((ctypes.addressof(buf) + 255) // 256 * 256)
    framed = _lib.FLAG_GRAD_X_FRAMED

    def backward(s):
        return lib.dcn_backward(ctypes.byref(s), ok, ok, ok, ok, ok, ok, ok, None, ok, 0, None)

    def backward_modulated(s):
        return lib.dcn_backward_modulated(ctypes.byref(s), ok, ok, ok, ok, ok, ok, ok, ok, ok, None, ok, 0, None)

    def layer_backward(s):
        return lib.dcn_layer_backward(ctypes.byref(s), ok, ok, ok, ok, ok, ok, ok, None, ok, None, ok, 0, None)

    def layer_backward_modulated(s):
        return lib.dcn_layer_backward_modulated(ctypes.byref(s), ok, ok, ok, ok, ok, ok, ok, ok, None, ok, None, ok, 0,
                                                None)

    def refused(call, s, why):
        assert call(s) == -6, (call.__name__, lib.dcn_last_error())
        msg = lib.dcn_last_error()
        assert b"DCN_FLAG_GRAD_X_FRAMED" in msg and why in msg, (call.__name__, msg)

    on_gemm = _lib.make_shape(2, 512, 512, 14, 14, 3, 1, 1, dcn.VARIANT_TORCH, dcn.OPERAND_FP32, framed)  # C5-like
    assert _lib.path_name(on_gemm, 1) == "gemm"
    on_simt = _lib.make_shape(2, 5, 8, 9, 13, 3, 1, 1, dcn.VARIANT_TORCH, dcn.OPERAND_FP32, framed)
    assert _lib.path_name(on_simt, 1) == "simt"
    # tensor-path backward whose fp32 data gradient still runs on the generic kernel (the fall-back inside it)
    on_fallback = _lib.make_shape(2, 192, 16, 8, 8, 3, 1, 1, dcn.VARIANT_JITTOR, dcn.OPERAND_FP32, framed)
    assert _lib.path_name(on_fallback, 1) == "umma"
    forced = _lib.make_shape(2, 64, 64, 16, 16, 3, 1, 1, dcn.VARIANT_JITTOR, dcn.OPERAND_FP32,
                             framed | _lib.FLAG_FORCE_SIMT)
    for s in (on_gemm, on_simt, on_fallback, forced):
        refused(backward, s, b"tensor path")
    refused(backward_modulated, _lib.make_shape(2, 5, 8, 9, 13, 3, 1, 1, dcn.VARIANT_DCNV1, dcn.OPERAND_FP32, framed),
            b"tensor path")
    # the ACCUM pair, on a shape where every call runs on the tensor path
    for variant, calls in ((dcn.VARIANT_JITTOR, (backward, layer_backward)),
                           (dcn.VARIANT_DCNV1, (backward_modulated, layer_backward_modulated))):
        s = _lib.make_shape(2, 64, 64, 16, 16, 3, 1, 1, variant, dcn.OPERAND_FP32, framed | _lib.FLAG_ACCUM_GRAD_X)
        assert _lib.path_name(s, 1) == "umma" and _lib.path_name(s, 4 if variant == dcn.VARIANT_JITTOR else 6) == "umma"
        for call in calls:
            refused(call, s, b"DCN_FLAG_ACCUM_GRAD_X")
        # without ACCUM the same calls pass the flag check and stop at the empty workspace
        s.flags = framed
        for call in calls:
            assert call(s) == -4, (call.__name__, lib.dcn_last_error())


def test_module_keeps_the_reference_interface():
    """ctor signature, attributes, parameter names/shapes and init of train.py:70-93."""
    m = dcn.TorchDeformConv2d(16, 32, 3, 2, 1)
    assert (m.in_channels, m.out_channels, m.kernel_size, m.stride, m.padding, m.N) == \
        (16, 32, (3, 3), (2, 2), (1, 1), 9)
    sd = m.state_dict()
    assert list(sd) == ["weight", "bias", "offset_conv.weight", "offset_conv.bias"]
    assert tuple(sd["weight"].shape) == (32, 16, 3, 3) and tuple(sd["bias"].shape) == (32,)
    assert tuple(sd["offset_conv.weight"].shape) == (18, 16, 3, 3)
    assert float(sd["offset_conv.weight"].abs().max()) == 0.0 and float(sd["bias"].abs().max()) == 0.0
    std = float(sd["weight"].std())
    assert abs(std - (2.0 / (16 * 9)) ** 0.5) < 0.02
    m2 = dcn.TorchDeformConv2d(4, 8, (1, 3), (1, 1), (0, 1), bias=False)
    assert m2.bias is None and m2.N == 3 and list(m2.state_dict()) == ["weight", "offset_conv.weight", "offset_conv.bias"]


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    m = dcn.TorchDeformConv2d(2, 2)
    with pytest.raises(dcn.DcnError):
        m(torch.zeros(1, 2, 4, 4))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "jittor_dcn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("no CPU fallback", ""), os.path.join(dirpath, f)


def test_library_reads_no_environment():
    """Which kernel and launch plan runs depends on the shape alone, never on the process environment."""
    csrc = os.path.join(ROOT, "jittor_dcn_b200", "csrc")
    for f in os.listdir(csrc):
        if f.endswith((".cu", ".cuh", ".h", ".cpp")):
            assert "getenv" not in open(os.path.join(csrc, f)).read(), f


def test_detector_harness_keeps_reference_parameter_names():
    """state_dict keys/shapes of train.py:142-175 (435,862 parameters, SURVEY 2 #6)."""
    from jittor_dcn_b200.detector import EDNetDetection
    from tests.util import golden
    m = EDNetDetection()
    g = golden("detector_eval")
    ref = {k[3:]: v for k, v in g.items() if k.startswith("sd.")}
    sd = m.state_dict()
    assert list(sd) == list(ref)
    for k in sd:
        assert tuple(sd[k].shape) == tuple(ref[k].shape), k
    assert sum(p.numel() for p in m.parameters()) == 435862


def test_wide_layers_dispatch_to_output_channel_groups_without_a_gpu():
    """O > 256 (ResNet-50 C5, BASELINE configs[3]) stays on the tensor path for the pixel-row layouts; the Torch
    layout follows gcd(Ho*Wo, C); bf16 storage never turns a shape away (generic kernels on widened copies)."""
    lib = dcn.load()

    def path(shape_args, variant, operand, phase):
        s = dcn.make_shape(*shape_args, 3, 1, 1, variant, operand)
        return lib.dcn_path_name(ctypes.byref(s), phase), lib.dcn_workspace_bytes(ctypes.byref(s), phase)

    c5 = (128, 512, 512, 14, 14)
    for operand in (dcn.OPERAND_FP32, dcn.OPERAND_BF16):
        for phase in (0, 1):
            for variant in (dcn.VARIANT_JITTOR, dcn.VARIANT_DCNV1):
                name, ws = path(c5, variant, operand, phase)
                assert name == b"umma" and ws > 0
            # gcd(196, 512) = 4 channels per sampling point: too few for the fused kernels; the samples are materialised
            # once and the contractions run as plain GEMMs (csrc/dcn_gemm_path.cu)
            name, ws = path(c5, dcn.VARIANT_TORCH, operand, phase)
            assert name == b"gemm" and ws > 0
    # groups are sized by the largest one: the workspace of O = 512 equals that of its 256-channel group for
    # everything but the per-group weight / grad_out images, so it can never be smaller
    for phase in (0, 1):
        assert path(c5, dcn.VARIANT_JITTOR, dcn.OPERAND_FP32, phase)[1] >= \
            path((128, 512, 256, 14, 14), dcn.VARIANT_JITTOR, dcn.OPERAND_FP32, phase)[1]
    # O must split into multiples of 16
    assert path((1, 64, 264, 8, 8), dcn.VARIANT_JITTOR, dcn.OPERAND_FP32, 0)[0] == b"simt"
    assert path((1, 64, 768, 8, 8), dcn.VARIANT_JITTOR, dcn.OPERAND_FP32, 0)[0] == b"umma"


def test_bn_relu_abi_rejects_bad_arguments_without_a_gpu():
    lib = dcn.load()
    buf = ctypes.create_string_buffer(1 << 16)
    base = (ctypes.addressof(buf) + 255) // 256 * 256
    ok = ctypes.c_void_p(base)
    need = lib.dcn_bn_workspace_bytes(32)
    assert need >= 2 * 32 * 8 + 2 * 32 * 4 and lib.dcn_bn_workspace_bytes(0) == 0
    f = ctypes.c_float
    assert lib.dcn_bn_relu_forward(0, 32, 64, 1, ok, ok, ok, ok, ok, f(0.1), f(1e-5), ok, ok, ok, need, None) == -1
    assert lib.dcn_bn_relu_forward(4, 32, 64, 1, None, ok, ok, ok, ok, f(0.1), f(1e-5), ok, ok, ok, need, None) == -2
    assert lib.dcn_bn_relu_forward(4, 32, 64, 1, ok, ok, ok, ok, ok, f(0.1), f(1e-5), ok, ok, ok, 8, None) == -4
    # eval mode reads the running statistics: they must be there
    assert lib.dcn_bn_relu_forward(4, 32, 64, 0, ok, ok, ok, None, None, f(0.1), f(1e-5), ok, ok, ok, need, None) == -2
    assert lib.dcn_bn_relu_backward(4, 32, 64, 1, ok, None, ok, ok, ok, ok, ok, need, None) == -2
    assert lib.dcn_bn_relu_backward(4, 32, 64, 1, ok, ctypes.c_void_p(base + 4), ok, ok, ok, ok, ok, need, None) == -3


def test_bn_relu_module_keeps_the_batchnorm_interface():
    """Same parameters, buffers, state-dict keys and defaults as tnn.BatchNorm2d (train.py:146-159), so that the
    reference's checkpoints load unchanged; like it, training mode refuses one value per channel."""
    import torch
    ref = torch.nn.BatchNorm2d(16)
    ours = dcn.BatchNormReLU2d(16)
    assert list(ours.state_dict()) == list(ref.state_dict())
    assert (ours.eps, ours.momentum, ours.affine, ours.track_running_stats) == \
        (ref.eps, ref.momentum, ref.affine, ref.track_running_stats)
    ours.load_state_dict(ref.state_dict())
    with pytest.raises(ValueError):
        ours(torch.zeros(1, 16, 1, 1))
    with pytest.raises(ValueError):
        ours(torch.zeros(2, 16, 4))


def test_round2_entry_points_validate_their_arguments_without_a_gpu():
    """Chained / staged / RoI entry points (SURVEY 8f.2, 8f.4) refuse bad descriptions before touching CUDA."""
    lib = dcn.load()
    buf = ctypes.create_string_buffer(1 << 12)
    ok = ctypes.c_void_p((ctypes.addressof(buf) + 255) // 256 * 256)
    f = ctypes.c_float
    prod = dcn.make_shape(2, 16, 32, 32, 32, 3, 2, 1, dcn.VARIANT_TORCH)           # -> [2, 32, 16, 16]
    good = dcn.make_shape(2, 32, 64, 16, 16, 3, 2, 1, dcn.VARIANT_TORCH)
    bad = dcn.make_shape(2, 32, 64, 20, 16, 3, 2, 1, dcn.VARIANT_TORCH)            # wrong input extent
    assert lib.dcn_staged_input_bytes(ctypes.byref(good)) >= 2 * (16 + 3) * (16 + 2) * 32 * 4
    rc = lib.dcn_layer_forward_chained(ctypes.byref(prod), ctypes.byref(bad), ok, ok, ok, ok, ok, ok, ok, ok, 1 << 30, None)
    assert rc == -1 and b"consumer" in lib.dcn_last_error()
    rc = lib.dcn_layer_forward_chained(ctypes.byref(prod), ctypes.byref(good), None, ok, ok, ok, ok, ok, ok, ok, 1 << 30, None)
    assert rc == -2                                                               # x is NULL
    rc = lib.dcn_layer_forward_chained(ctypes.byref(prod), ctypes.byref(good), ok, ok, ok, ok, ok, ok, ok, ok, 16, None)
    assert rc == -4                                                               # workspace too small
    odd = dcn.make_shape(2, 5, 7, 9, 13, 3, 1, 1, dcn.VARIANT_TORCH)               # consumer on the generic kernels
    rc = lib.dcn_bn_relu_forward_staged(ctypes.byref(odd), 1, ok, ok, ok, ok, ok, f(0.1), f(1e-5), ok, ok, ok, 1 << 20, None)
    assert rc == -6
    rc = lib.dcn_bn_relu_backward_staged(ctypes.byref(good), 1, ok, None, ok, ok, ok, ok, ok, 1 << 20, None)
    assert rc == -2
    assert lib.dcn_roi_pool_forward(7, 1, 4, 8, 8, 2, ok, ok, ok, f(1.0), f(0.1), 0, ok, None) == -1
    assert lib.dcn_roi_pool_forward(0, 1, 4, 8, 8, 2, None, ok, ok, f(1.0), f(0.1), 0, ok, None) == -2
    assert lib.dcn_roi_pool_forward(0, 1, 4, 8, 8, 0, ok, ok, ok, f(1.0), f(0.1), 0, ok, None) == 0       # no rois: nothing to do
    for cls in (dcn.DeformRoIPool, dcn.DeformPSRoIPool):
        with pytest.raises(ValueError):
            cls(7)
    # the detector's conv1 (csrc/dcn_stem.cu): extents, supported set, pointers
    assert lib.dcn_stem_conv_forward(0, 1, 16, 8, 8, ok, ok, ok, ok, None) == -1
    assert lib.dcn_stem_conv_forward(2, 1, 24, 8, 8, ok, ok, ok, ok, None) == -6 and b"O in {16, 32}" in lib.dcn_last_error()
    assert lib.dcn_stem_conv_forward(2, 1, 16, 8, 6, ok, ok, ok, ok, None) == -6           # W % 4
    assert lib.dcn_stem_conv_forward(2, 5, 16, 8, 8, ok, ok, ok, ok, None) == -6           # Cin > 4
    assert lib.dcn_stem_conv_forward(2, 1, 16, 8, 8, None, ok, ok, ok, None) == -2
    assert lib.dcn_stem_conv_backward(2, 1, 16, 8, 8, ok, ok, None, ok, None) == -2
    # path names of the three kernel families
    for shape, name in (((256, 64, 64, 128, 128), b"umma"), ((128, 512, 512, 14, 14), b"gemm"), ((3, 5, 7, 9, 13), b"simt")):
        s = dcn.make_shape(*shape, 3, 1, 1, dcn.VARIANT_TORCH)
        assert lib.dcn_path_name(ctypes.byref(s), 0) == name and lib.dcn_path_name(ctypes.byref(s), 1) == name


def test_stem_conv_module_is_a_drop_in_on_cpu():
    """StemConv2d (the detector's conv1) keeps nn.Conv2d's parameters and, without a CUDA input, its kernels too."""
    import torch
    import torch.nn as nn
    torch.manual_seed(0)
    ref, eng = nn.Conv2d(1, 16, 3, 1, 1), dcn.StemConv2d(1, 16, 3, 1, 1)
    assert [(k, tuple(v.shape)) for k, v in eng.state_dict().items()] == [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
    eng.load_state_dict(ref.state_dict())
    x = torch.randn(2, 1, 12, 16)
    assert torch.equal(eng(x), ref(x))
    from jittor_dcn_b200.functional import stem_conv_supported
    assert not stem_conv_supported(x, eng.weight)                      # CPU tensor
