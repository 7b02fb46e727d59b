"""Multi-scale deformable attention without a GPU: the C ABI's refusals and messages, the DcnMsdaShape mirror, the
Python entry points' argument checks, the drop-in module's interface and initialisation, and the msda_* fixtures."""
import ctypes
import os
import re
import tempfile

import numpy as np
import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from oracle import make_golden, make_golden_msda, msda_reference
from tests.util import golden, golden_names

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _shape(B=2, S=100, Q=10, M=8, D=32, L=4, P=4, flags=0):
    return dcn.DcnMsdaShape(B, S, Q, M, D, L, P, flags)


@pytest.fixture
def ptrs():
    buf = ctypes.create_string_buffer(1 << 12)
    base = (ctypes.addressof(buf) + 255) // 256 * 256
    yield ctypes.c_void_p(base), ctypes.c_void_p(base + 4)
    del buf


def _fwd(lib, s, args):
    return lib.dcn_msda_forward(ctypes.byref(s) if s is not None else None, *args, None)


def _bwd(lib, s, args):
    return lib.dcn_msda_backward(ctypes.byref(s) if s is not None else None, *args, None)


FWD_ARGS = ("value", "spatial_shapes", "level_start_index", "sampling_locations", "attention_weights", "out")
BWD_ARGS = ("value", "spatial_shapes", "level_start_index", "sampling_locations", "attention_weights", "grad_out",
            "grad_value", "grad_sampling_locations", "grad_attention_weights")


def test_shape_struct_matches_header():
    text = open(os.path.join(ROOT, "include", "dcn_b200.h")).read()
    body = re.search(r"typedef struct DcnMsdaShape \{(.*?)\} DcnMsdaShape;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [n.strip() for decl in re.findall(r"int32_t ([^;]+);", body) for n in decl.split(",")]
    assert names == [f[0] for f in _lib.DcnMsdaShape._fields_] == ["B", "S", "Q", "M", "D", "L", "P", "flags"]
    assert ctypes.sizeof(_lib.DcnMsdaShape) == 32


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
    if BWD_ARGS[i].startswith("grad_") and BWD_ARGS[i] != "grad_out":
        return          # the three gradients are optional (NULL: not computed); this call would launch
    assert _bwd(lib, _shape(), args) == -2
    assert lib.dcn_last_error().decode().endswith(f"{BWD_ARGS[i]} is NULL")


def test_backward_with_no_gradient_requested_does_nothing(ptrs):
    ok, _ = ptrs
    assert _bwd(dcn.load(), _shape(), [ok] * 6 + [None] * 3) == 0


def test_null_shape_is_refused(ptrs):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, None, [ok] * 6) == -2 and b"DcnMsdaShape is NULL" in lib.dcn_last_error()
    assert _bwd(lib, None, [ok] * 9) == -2 and b"DcnMsdaShape is NULL" in lib.dcn_last_error()


@pytest.mark.parametrize("field", ["B", "S", "Q", "M", "D", "L", "P"])
@pytest.mark.parametrize("value", [0, -1])
def test_non_positive_extents_are_bad_shapes(ptrs, field, value):
    lib = dcn.load()
    ok, _ = ptrs
    s = _shape()
    setattr(s, field, value)
    assert _fwd(lib, s, [ok] * 6) == -1 and b"bad shape" in lib.dcn_last_error()
    assert _bwd(lib, s, [ok] * 9) == -1 and b"bad shape" in lib.dcn_last_error()


def test_index_space_limit(ptrs):
    lib = dcn.load()
    ok, _ = ptrs
    s = _shape(B=1 << 10, Q=1 << 18, M=8)        # B*Q*M = 2^31
    assert _fwd(lib, s, [ok] * 6) == -1 and b"B*Q*M = 2147483648 exceeds the limit 2^31 - 1" in lib.dcn_last_error()


@pytest.mark.parametrize("kw, msg", [
    (dict(flags=1), b"flags must be 0 (reserved), got 1"),
    (dict(D=8), b"D = 8 channels per head is not supported (D in {16, 32, 64, 128, 256})"),
    (dict(D=48), b"D = 48 channels per head is not supported"),
    (dict(D=512), b"D = 512 channels per head is not supported"),
    (dict(L=17), b"L = 17 levels exceeds the limit L <= 16"),
    (dict(P=33), b"P = 33 points exceeds the limit P <= 32"),
])
def test_limits_are_unsupported_with_a_message(ptrs, kw, msg):
    lib = dcn.load()
    ok, _ = ptrs
    assert _fwd(lib, _shape(**kw), [ok] * 6) == -6 and msg in lib.dcn_last_error()
    assert _bwd(lib, _shape(**kw), [ok] * 9) == -6 and msg in lib.dcn_last_error()


def test_required_coverage_passes_validation_up_to_the_pointers(ptrs):
    """D in {16, 32, 64, 128}, L in 1..5, P in 1..8 pass the shape checks (a NULL pointer is the next refusal)."""
    lib = dcn.load()
    ok, _ = ptrs
    for D in (16, 32, 64, 128, 256):
        for L in (1, 5):
            for P in (1, 4, 8):
                assert _fwd(lib, _shape(D=D, L=L, P=P), [None] + [ok] * 5) == -2


def _cpu_inputs(B=1, M=2, D=32, Q=3, levels=((4, 5), (2, 3)), P=2):
    L = len(levels)
    S = sum(h * w for h, w in levels)
    ss = torch.tensor(levels, dtype=torch.int64)
    return (torch.zeros(B, S, M, D), ss, msda_reference.level_start_index_of(ss), torch.zeros(B, Q, M, L, P, 2),
            torch.zeros(B, Q, M, L, P))


def test_functional_refuses_cpu_and_non_fp32_inputs():
    v, ss, lsi, loc, aw = _cpu_inputs()
    with pytest.raises(ValueError, match="value must be a CUDA tensor: there is no CPU path"):
        dcn.ms_deform_attn(v, ss, lsi, loc, aw)
    with pytest.raises(ValueError, match="value must be a float32 tensor, got torch.float16"):
        dcn.ms_deform_attn(v.half(), ss, lsi, loc, aw)
    with pytest.raises(ValueError, match="sampling_locations must be a float32 tensor, got torch.float64"):
        dcn.MSDeformAttnFunction.apply(v, ss, lsi, loc.double(), aw, 64)
    with pytest.raises(ValueError, match="attention_weights must be a float32 tensor"):
        dcn.ms_deform_attn(v, ss, lsi, loc, aw.bfloat16())


def test_functional_checks_shapes_before_the_device(monkeypatch):
    """Shape checks run on metadata; here the device check is bypassed to reach them without a GPU."""
    from jittor_dcn_b200 import functional as fn
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    v, ss, lsi, loc, aw = _cpu_inputs()
    cases = [
        ((v[0], ss, lsi, loc, aw), "value must be \\[B, S, M, D\\]"),
        ((v, ss.float(), lsi, loc, aw), "spatial_shapes must be an integer tensor"),
        ((v, ss, lsi.bool(), loc, aw), "level_start_index must be an integer tensor"),
        ((v, ss[:, :1], lsi, loc, aw), "spatial_shapes must be \\[L, 2\\]"),
        ((v, ss, lsi[:1], loc, aw), "level_start_index shape"),
        ((v, ss, lsi, loc[..., 0], aw), "sampling_locations must be \\[B, Q, M, L, P, 2\\]"),
        ((v, ss, lsi, loc[:, :, :1], aw), "sampling_locations shape"),
        ((v, ss, lsi, loc, aw[..., :1]), "attention_weights shape"),
    ]
    for args, msg in cases:
        with pytest.raises(ValueError, match=msg):
            fn._msda_inputs(*args)


def test_module_interface_and_state_dict():
    m = dcn.MSDeformAttn()
    assert (m.d_model, m.n_levels, m.n_heads, m.n_points, m.im2col_step) == (256, 4, 8, 4, 64)
    ref = msda_reference.MSDeformAttnRef()
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == \
        [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
    assert list(m.state_dict()) == [f"{mod}.{p}" for mod in ("sampling_offsets", "attention_weights", "value_proj",
                                                            "output_proj") for p in ("weight", "bias")]
    m2 = dcn.MSDeformAttn(d_model=64, n_levels=5, n_heads=4, n_points=8)
    assert tuple(m2.sampling_offsets.weight.shape) == (4 * 5 * 8 * 2, 64)
    with pytest.raises(ValueError, match="d_model must be divisible by n_heads, but got 100 and 8"):
        dcn.MSDeformAttn(d_model=100)
    with pytest.warns(UserWarning):
        dcn.MSDeformAttn(d_model=48, n_heads=4)


@pytest.mark.parametrize("cfg", [(256, 4, 8, 4), (64, 5, 4, 8), (32, 1, 1, 1)])
def test_module_initialisation_equals_the_reference_under_one_seed(cfg):
    torch.manual_seed(7)
    m = dcn.MSDeformAttn(*cfg)
    torch.manual_seed(7)
    ref = msda_reference.MSDeformAttnRef(*cfg)
    for (k, a), (_, b) in zip(m.state_dict().items(), ref.state_dict().items()):
        assert torch.equal(a, b), k
    # the rotating grid, scaled by i + 1 per point; zero offset weights and attention weights
    d_model, L, M, P = cfg
    bias = m.sampling_offsets.bias.detach().view(M, L, P, 2)
    assert torch.allclose(bias[:, :, P - 1], bias[:, :, 0] * P)
    assert float(m.sampling_offsets.weight.detach().abs().max()) == 0.0
    assert float(m.attention_weights.weight.detach().abs().max()) == 0.0


def test_module_refuses_a_bad_reference_point_form():
    m = dcn.MSDeformAttn(d_model=32, n_levels=1, n_heads=1, n_points=1)
    ss = torch.tensor([[2, 2]])
    with pytest.raises(ValueError, match="Last dim of reference_points must be 2 or 4, but get 3 instead"):
        m(torch.zeros(1, 3, 32), torch.zeros(1, 3, 1, 3), torch.zeros(1, 4, 32), ss, torch.tensor([0]))


def test_msda_fixtures_cover_the_required_cases():
    names = golden_names("msda_")
    assert names == sorted(make_golden_msda.MSDA)
    D, P, L, square, outside, border, neg, unnormalised = set(), set(), set(), [], False, False, False, False
    for n in names:
        g = golden(n)
        D.add(g["value"].shape[3])
        P.add(int(g["P"]))
        L.add(g["spatial_shapes"].shape[0])
        square += [h == w for h, w in g["spatial_shapes"]]
        loc, aw = g["sampling_locations"], g["attention_weights"]
        outside |= bool(((loc < 0) | (loc > 1)).any())
        border |= bool((loc == 0).any() and (loc == 1).any())
        neg |= bool((aw < 0).any())
        unnormalised |= not np.allclose(aw.sum((-1, -2)), 1)
    assert {32, 64} <= D and {1, 4} <= P and 1 in L and max(L) > 1 and not all(square)
    assert outside and border and neg and unnormalised


def test_msda_fixtures_regenerate_within_1e_6():
    prev = torch.get_num_threads()
    torch.set_num_threads(make_golden.GOLDEN_CPU_THREADS)
    try:
        with tempfile.TemporaryDirectory() as d:
            make_golden_msda.make_msda(d)
            for n in make_golden_msda.MSDA:
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
