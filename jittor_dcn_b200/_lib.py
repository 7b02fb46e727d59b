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

# every symbol include/dcn_b200.h declares (tests/test_abi.py checks the two lists agree)
EXPORTS = (
    "dcn_version", "dcn_last_error", "dcn_status_string", "dcn_output_hw", "dcn_workspace_bytes",
    "dcn_path_name", "dcn_launch_count", "dcn_launch_count_reset", "dcn_profile_begin",
    "dcn_profile_end", "dcn_forward", "dcn_backward", "dcn_forward_modulated", "dcn_backward_modulated",
    "dcn_debug_corners", "dcn_comm_unique_id", "dcn_comm_init", "dcn_allreduce_sum_f32",
    "dcn_comm_destroy", "dcn_bn_workspace_bytes", "dcn_bn_relu_forward", "dcn_bn_relu_backward",
    "dcn_offset_conv_forward", "dcn_layer_forward", "dcn_layer_backward",
    "dcn_p2p_handle_bytes", "dcn_p2p_create", "dcn_p2p_local_handle", "dcn_p2p_connect",
    "dcn_p2p_allreduce_sum_f32", "dcn_p2p_destroy", "dcn_roi_pool_forward", "dcn_roi_pool_backward",
    "dcn_staged_input_bytes", "dcn_staged_input_clear", "dcn_layer_forward_chained",
    "dcn_bn_relu_forward_staged", "dcn_bn_relu_backward_staged", "dcn_stem_conv_forward", "dcn_stem_conv_backward",
    "dcn_offset_conv_forward_modulated", "dcn_layer_forward_modulated", "dcn_layer_backward_modulated",
    "dcn_msda_forward", "dcn_msda_backward", "dcn_v3_forward", "dcn_v3_backward", "dcn_v4_forward", "dcn_v4_backward",
)


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
    vp, sz, i32p = ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_int32)
    shp = ctypes.POINTER(DcnShape)
    lib.dcn_version.restype = ctypes.c_int
    lib.dcn_last_error.restype = ctypes.c_char_p
    lib.dcn_status_string.restype = ctypes.c_char_p
    lib.dcn_status_string.argtypes = [ctypes.c_int]
    lib.dcn_output_hw.argtypes = [shp, i32p, i32p]
    lib.dcn_workspace_bytes.restype = sz
    lib.dcn_workspace_bytes.argtypes = [shp, ctypes.c_int]
    lib.dcn_path_name.restype = ctypes.c_char_p
    lib.dcn_path_name.argtypes = [shp, ctypes.c_int]
    lib.dcn_launch_count.restype = ctypes.c_uint64
    lib.dcn_launch_count_reset.restype = None
    lib.dcn_profile_end.argtypes = [ctypes.c_char_p, sz]
    lib.dcn_forward.argtypes = [shp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_backward.argtypes = [shp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_forward_modulated.argtypes = [shp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_backward_modulated.argtypes = [shp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_debug_corners.argtypes = [shp, vp, vp, vp, vp, vp]
    lib.dcn_offset_conv_forward.argtypes = [shp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_layer_forward.argtypes = [shp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_layer_backward.argtypes = [shp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_offset_conv_forward_modulated.argtypes = [shp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_layer_forward_modulated.argtypes = [shp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_layer_backward_modulated.argtypes = [shp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    msp = ctypes.POINTER(DcnMsdaShape)
    lib.dcn_msda_forward.argtypes = [msp, vp, vp, vp, vp, vp, vp, vp]
    lib.dcn_msda_backward.argtypes = [msp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    v3p, f32 = ctypes.POINTER(DcnV3Shape), ctypes.c_float
    lib.dcn_v3_forward.argtypes = [v3p, f32, vp, vp, vp, vp, vp]
    lib.dcn_v3_backward.argtypes = [v3p, f32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.dcn_v4_forward.argtypes = [v3p, f32, vp, vp, vp, vp]
    lib.dcn_v4_backward.argtypes = [v3p, f32, vp, vp, vp, vp, vp, vp]
    lib.dcn_comm_unique_id.argtypes = [vp]
    lib.dcn_comm_init.argtypes = [ctypes.c_int, ctypes.c_int, vp, ctypes.POINTER(vp)]
    lib.dcn_allreduce_sum_f32.argtypes = [vp, vp, sz, ctypes.c_float, vp]
    lib.dcn_comm_destroy.argtypes = [vp]
    lib.dcn_p2p_handle_bytes.restype = sz
    lib.dcn_p2p_create.argtypes = [ctypes.c_int, ctypes.c_int, sz, ctypes.POINTER(vp)]
    lib.dcn_p2p_local_handle.argtypes = [vp, vp]
    lib.dcn_p2p_connect.argtypes = [vp, vp]
    lib.dcn_p2p_allreduce_sum_f32.argtypes = [vp, vp, sz, ctypes.c_float, vp]
    lib.dcn_p2p_destroy.argtypes = [vp]
    i32, f32 = ctypes.c_int32, ctypes.c_float
    lib.dcn_bn_workspace_bytes.restype = sz
    lib.dcn_bn_workspace_bytes.argtypes = [i32]
    lib.dcn_bn_relu_forward.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp, vp, f32, f32, vp, vp, vp, sz, vp]
    lib.dcn_bn_relu_backward.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_bn_relu_forward_staged.argtypes = [shp, i32, vp, vp, vp, vp, vp, f32, f32, vp, vp, vp, sz, vp]
    lib.dcn_bn_relu_backward_staged.argtypes = [shp, i32, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_staged_input_bytes.restype = sz
    lib.dcn_staged_input_bytes.argtypes = [shp]
    lib.dcn_staged_input_clear.argtypes = [shp, vp, vp]
    lib.dcn_layer_forward_chained.argtypes = [shp, shp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.dcn_roi_pool_forward.argtypes = [i32, i32, i32, i32, i32, i32, vp, vp, vp, f32, f32, i32, vp, vp]
    lib.dcn_roi_pool_backward.argtypes = [i32, i32, i32, i32, i32, i32, vp, vp, vp, f32, f32, i32, vp, vp, vp, vp]
    lib.dcn_stem_conv_forward.argtypes = [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.dcn_stem_conv_backward.argtypes = [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp]
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
