"""ctypes binding of libdcn_b200.so (the C ABI in include/dcn_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# DCN_B200_LIB=dbg selects the debug build (python -m jittor_dcn_b200.build --debug: device-side bounds and
# pipeline-agreement checks, csrc/dcn_common.cuh) — for test runs only
LIB_PATH = os.path.join(HERE, "libdcn_b200_dbg.so" if os.environ.get("DCN_B200_LIB") == "dbg" else "libdcn_b200.so")

VARIANT_JITTOR = 0   # deform_conv.py:56-81
VARIANT_TORCH = 1    # train.py:95-140
VARIANT_DCNV1 = 2    # standard DCNv1 (torchvision.ops.deform_conv2d semantics), SURVEY 8f.3
OPERAND_FP32 = 0
OPERAND_BF16 = 1
FLAG_ACCUM_GRAD_X = 1 << 0
FLAG_FORCE_SIMT = 1 << 1
FLAG_NO_GRAD_X = 1 << 2
FLAG_RELU_OUT = 1 << 3     # forward epilogue stores max(acc + bias, 0) (SURVEY 8f.2)
FLAG_XT_STAGED = 1 << 4
FLAG_GRAD_X_FRAMED = 1 << 6   # grad_x = the framed channels-last accumulator itself (training hand-over, SURVEY 8f.2)
PHASE_FORWARD, PHASE_BACKWARD, PHASE_CORNERS = 0, 1, 2
PHASE_LAYER_FORWARD, PHASE_LAYER_BACKWARD = 3, 4   # offset conv + DCN span (dcn_layer_*)
# offset-and-mask conv + modulated DCN span (dcn_layer_*_modulated)
PHASE_LAYER_FORWARD_MODULATED, PHASE_LAYER_BACKWARD_MODULATED = 5, 6
ROI_POOL, PSROI_POOL = 0, 1                        # dcn_roi_pool_* kind (deform_conv.py:83 / :160)


class DcnShape(ctypes.Structure):
    """Mirror of include/dcn_b200.h:DcnShape."""
    _fields_ = [(n, ctypes.c_int32) for n in
                ("B", "C", "O", "H", "W", "kh", "kw", "sh", "sw", "ph", "pw",
                 "variant", "operand", "flags")]


class DcnMsdaShape(ctypes.Structure):
    """Mirror of include/dcn_b200.h:DcnMsdaShape (multi-scale deformable attention)."""
    _fields_ = [(n, ctypes.c_int32) for n in ("B", "S", "Q", "M", "D", "L", "P", "flags")]


class DcnV3Shape(ctypes.Structure):
    """Mirror of include/dcn_b200.h:DcnV3Shape (DCNv3, InternImage's core)."""
    _fields_ = [(n, ctypes.c_int32) for n in ("N", "H", "W", "G", "Gc", "kh", "kw", "sh", "sw", "ph", "pw", "dh", "dw",
                                              "flags")]


DCN_V3_FLAG_SOFTMAX_MASK = 1
DCN_V4_FLAG_REMOVE_CENTER = 2

# export name -> (restype, argtypes) of every symbol include/dcn_b200.h declares; load() applies it, and
# tests/test_binding_table.py checks it against the header's prototypes
_i32, _f32, _sz, _vp, _str = ctypes.c_int32, ctypes.c_float, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_char_p
_i32p, _vpp = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_void_p)
_shp, _msp, _v3p = ctypes.POINTER(DcnShape), ctypes.POINTER(DcnMsdaShape), ctypes.POINTER(DcnV3Shape)
BINDINGS = {
    "dcn_version": (_i32, []),
    "dcn_last_error": (_str, []),
    "dcn_status_string": (_str, [_i32]),
    "dcn_output_hw": (_i32, [_shp, _i32p, _i32p]),
    "dcn_workspace_bytes": (_sz, [_shp, _i32]),
    "dcn_path_name": (_str, [_shp, _i32]),
    "dcn_launch_count": (ctypes.c_uint64, []),
    "dcn_launch_count_reset": (None, []),
    "dcn_profile_begin": (_i32, []),
    "dcn_profile_end": (_i32, [_str, _sz]),
    "dcn_forward": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_backward": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_forward_modulated": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_backward_modulated": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_offset_conv_forward": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_layer_forward": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_layer_backward": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_offset_conv_forward_modulated": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_layer_forward_modulated": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_layer_backward_modulated": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                            _vp]),
    "dcn_staged_input_bytes": (_sz, [_shp]),
    "dcn_staged_input_clear": (_i32, [_shp, _vp, _vp]),
    "dcn_layer_forward_chained": (_i32, [_shp, _shp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_bn_relu_forward_staged": (_i32, [_shp, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _sz, _vp]),
    "dcn_bn_relu_backward_staged": (_i32, [_shp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_debug_corners": (_i32, [_shp, _vp, _vp, _vp, _vp, _vp]),
    "dcn_roi_pool_forward": (_i32, [_i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _f32, _f32, _i32, _vp, _vp]),
    "dcn_roi_pool_backward": (_i32, [_i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _f32, _f32, _i32, _vp, _vp,
                                     _vp, _vp]),
    "dcn_msda_forward": (_i32, [_msp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dcn_msda_backward": (_i32, [_msp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dcn_v3_forward": (_i32, [_v3p, _f32, _vp, _vp, _vp, _vp, _vp]),
    "dcn_v3_backward": (_i32, [_v3p, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dcn_v4_forward": (_i32, [_v3p, _f32, _vp, _vp, _vp, _vp]),
    "dcn_v4_backward": (_i32, [_v3p, _f32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dcn_stem_conv_forward": (_i32, [_i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "dcn_stem_conv_backward": (_i32, [_i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "dcn_bn_workspace_bytes": (_sz, [_i32]),
    "dcn_bn_relu_forward": (_i32, [_i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _sz,
                                   _vp]),
    "dcn_bn_relu_backward": (_i32, [_i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dcn_comm_unique_id": (_i32, [_vp]),
    "dcn_comm_init": (_i32, [_i32, _i32, _vp, _vpp]),
    "dcn_allreduce_sum_f32": (_i32, [_vp, _vp, _sz, _f32, _vp]),
    "dcn_comm_destroy": (_i32, [_vp]),
    "dcn_p2p_handle_bytes": (_sz, []),
    "dcn_p2p_create": (_i32, [_i32, _i32, _sz, _vpp]),
    "dcn_p2p_local_handle": (_i32, [_vp, _vp]),
    "dcn_p2p_connect": (_i32, [_vp, _vp]),
    "dcn_p2p_allreduce_sum_f32": (_i32, [_vp, _vp, _sz, _f32, _vp]),
    "dcn_p2p_destroy": (_i32, [_vp]),
}
EXPORTS = tuple(BINDINGS)


class DcnError(RuntimeError):
    pass


_lib = None


def load():
    """Loads the engine; raises if it has not been built (python -m jittor_dcn_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DcnError(
            f"{LIB_PATH} is missing: the CUDA engine is not built and there is no CPU fallback. "
            "Run `python -m jittor_dcn_b200.build` (needs nvcc).")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in BINDINGS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        lib = load()
        raise DcnError(f"{what} failed: {lib.dcn_status_string(rc).decode()} ({rc}): "
                       f"{lib.dcn_last_error().decode()}")


def profile_begin():
    check(load().dcn_profile_begin(), "dcn_profile_begin")


def profile_end():
    """-> {kernel name: (launches, total_ms)} for everything launched since profile_begin."""
    buf = ctypes.create_string_buffer(1 << 14)
    check(load().dcn_profile_end(buf, len(buf)), "dcn_profile_end")
    res = {}
    for line in buf.value.decode().splitlines():
        name, cnt, ms = line.rsplit(" ", 2)
        res[name] = (int(cnt), float(ms))
    return res


def _pair(v):
    return (int(v[0]), int(v[1])) if isinstance(v, (tuple, list)) else (int(v), int(v))


def make_shape(B, C, O, H, W, kernel_size=3, stride=1, padding=1, variant=VARIANT_TORCH,
               operand=OPERAND_FP32, flags=0):
    (kh, kw), (sh, sw), (ph, pw) = _pair(kernel_size), _pair(stride), _pair(padding)
    return DcnShape(B, C, O, H, W, kh, kw, sh, sw, ph, pw, variant, operand, flags)


def path_name(shape, phase):
    """Which kernel family runs: "umma" (tcgen05 kernels) or "simt" (generic CUDA-core kernels) for this problem / phase."""
    return load().dcn_path_name(ctypes.byref(shape), phase).decode()


def output_hw(shape):
    h, w = ctypes.c_int32(), ctypes.c_int32()
    check(load().dcn_output_hw(ctypes.byref(shape), ctypes.byref(h), ctypes.byref(w)), "dcn_output_hw")
    return h.value, w.value
