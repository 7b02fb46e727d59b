"""Modulated deformable convolution (DCNv2) without a GPU: argument checks of the C ABI and of the Python entry
points, the torchvision-compatible module, and the dcnv2_* fixtures against torchvision."""
import ctypes
import os
import tempfile

import numpy as np
import pytest
import torch

import jittor_dcn_b200 as dcn
from oracle import make_golden, make_golden_dcnv2
from tests.util import golden, golden_names


@pytest.fixture
def golden_threads():
    """torch's CPU kernels split their sums by thread: the fixtures were made at make_golden.GOLDEN_CPU_THREADS."""
    prev = torch.get_num_threads()
    torch.set_num_threads(make_golden.GOLDEN_CPU_THREADS)
    yield
    torch.set_num_threads(prev)


def _buffers():
    buf = ctypes.create_string_buffer(1 << 16)
    base = (ctypes.addressof(buf) + 255) // 256 * 256
    return buf, base, ctypes.c_void_p(base)


def test_modulated_abi_rejects_bad_pointers_without_a_gpu():
    lib = dcn.load()
    s = dcn.make_shape(1, 4, 8, 10, 10, 3, 1, 1, dcn.VARIANT_DCNV1)
    buf, base, ok = _buffers()
    bad = ctypes.c_void_p(base + 4)
    ws = 1 << 15
    rc = lib.dcn_forward_modulated(ctypes.byref(s), ok, ok, None, ok, None, ok, ok, ws, None)
    assert rc == -2 and b"mask is NULL" in lib.dcn_last_error()
    rc = lib.dcn_forward_modulated(ctypes.byref(s), ok, ok, bad, ok, None, ok, ok, ws, None)
    assert rc == -3 and b"mask" in lib.dcn_last_error()
    rc = lib.dcn_backward_modulated(ctypes.byref(s), ok, ok, None, ok, ok, ok, ok, ok, ok, None, ok, ws, None)
    assert rc == -2 and b"mask is NULL" in lib.dcn_last_error()
    rc = lib.dcn_backward_modulated(ctypes.byref(s), ok, ok, ok, ok, ok, ok, ok, None, ok, None, ok, ws, None)
    assert rc == -2 and b"grad_mask is NULL" in lib.dcn_last_error()
    rc = lib.dcn_backward_modulated(ctypes.byref(s), ok, ok, ok, ok, ok, ok, ok, bad, ok, None, ok, ws, None)
    assert rc == -3 and b"grad_mask" in lib.dcn_last_error()
    # the remaining pointers behave as in dcn_forward / dcn_backward
    rc = lib.dcn_forward_modulated(ctypes.byref(s), None, ok, ok, ok, None, ok, ok, ws, None)
    assert rc == -2 and b"x is NULL" in lib.dcn_last_error()
    rc = lib.dcn_backward_modulated(ctypes.byref(s), ok, ok, ok, ok, ok, None, ok, ok, ok, None, ok, ws, None)
    assert rc == -2 and b"grad_x" in lib.dcn_last_error()
    del buf


@pytest.mark.parametrize("variant", [dcn.VARIANT_TORCH, dcn.VARIANT_JITTOR])
def test_modulated_abi_refuses_the_reference_variants(variant):
    lib = dcn.load()
    s = dcn.make_shape(1, 4, 8, 10, 10, 3, 1, 1, variant)
    buf, base, ok = _buffers()
    assert lib.dcn_forward_modulated(ctypes.byref(s), ok, ok, ok, ok, None, ok, ok, 1 << 15, None) == -6
    assert b"DCN_VARIANT_DCNV1" in lib.dcn_last_error()
    assert lib.dcn_backward_modulated(ctypes.byref(s), ok, ok, ok, ok, ok, ok, ok, ok, ok, None, ok, 1 << 15,
                                      None) == -6
    del buf


@pytest.mark.parametrize("C", [4, 64])   # generic kernels / tensor path
def test_modulated_abi_workspace_is_that_of_the_unmodulated_calls(C):
    lib = dcn.load()
    s = dcn.make_shape(2, C, 64, 12, 12, 3, 1, 1, dcn.VARIANT_DCNV1)
    buf, base, ok = _buffers()
    for phase in (0, 1):
        need = lib.dcn_workspace_bytes(ctypes.byref(s), phase)
        assert need > 16
    rc = lib.dcn_forward_modulated(ctypes.byref(s), ok, ok, ok, ok, None, ok, ok, 16, None)
    assert rc == -4 and b"workspace" in lib.dcn_last_error()
    rc = lib.dcn_backward_modulated(ctypes.byref(s), ok, ok, ok, ok, ok, ok, ok, ok, ok, None, ok, 16, None)
    assert rc == -4 and b"workspace" in lib.dcn_last_error()
    del buf


def test_deform_conv2d_v1_validates_its_arguments_without_a_gpu():
    x = torch.zeros(2, 4, 9, 11)
    w = torch.zeros(6, 4, 3, 3)
    off = torch.zeros(2, 18, 9, 11)
    with pytest.raises(ValueError, match="dilation"):
        dcn.deform_conv2d_v1(x, off, w, padding=1, dilation=2)
    with pytest.raises(ValueError, match=r"\(2, 18, 9, 11\)"):        # two offset groups
        dcn.deform_conv2d_v1(x, torch.zeros(2, 36, 9, 11), w, padding=1)
    with pytest.raises(ValueError, match=r"\(2, 9, 9, 11\)"):
        dcn.deform_conv2d_v1(x, off, w, padding=1, mask=torch.zeros(2, 18, 9, 11))
    with pytest.raises(ValueError, match=r"\(2, 9, 7, 9\)"):           # padding 0: 7 x 9 outputs
        dcn.deform_conv2d_v1(x, torch.zeros(2, 18, 7, 9), w, mask=torch.zeros(2, 9, 9, 11))
    # torchvision's positional order: (input, offset, weight, bias, stride, padding, dilation, mask)
    with pytest.raises(ValueError, match="dilation"):
        dcn.deform_conv2d_v1(x, off, w, None, 1, 1, (1, 2), None)


def test_torchvision_module_matches_torchvision_deform_conv2d():
    from torchvision.ops import DeformConv2d
    for args, kw in (((8, 16, 3), {}), ((8, 16, (1, 3)), dict(stride=2, padding=(0, 1), bias=False)),
                     ((3, 5, 3), dict(padding=1))):
        torch.manual_seed(7)
        ref = DeformConv2d(*args, **kw)
        torch.manual_seed(7)
        ours = dcn.TorchvisionDeformConv2d(*args, **kw)
        rs, os_ = ref.state_dict(), ours.state_dict()
        assert list(rs) == list(os_)
        for k in rs:
            assert rs[k].shape == os_[k].shape and torch.equal(rs[k], os_[k]), k
        for a in ("in_channels", "out_channels", "kernel_size", "stride", "padding", "dilation", "groups"):
            assert getattr(ref, a) == getattr(ours, a), a
        ours.load_state_dict(rs)          # checkpoints load unchanged
    with pytest.raises(ValueError, match="dilation"):
        dcn.TorchvisionDeformConv2d(8, 16, 3, dilation=2)
    with pytest.raises(ValueError, match="groups"):
        dcn.TorchvisionDeformConv2d(8, 16, 3, groups=2)


def test_dcnv2_fixtures_regenerate_from_torchvision(golden_threads):
    names = golden_names("dcnv2_")
    assert names == sorted(make_golden_dcnv2.DCNV2)
    with tempfile.TemporaryDirectory() as tmp:
        make_golden_dcnv2.make_dcnv2(np.random.default_rng(make_golden_dcnv2.SEED), out_dir=tmp)
        for name in names:
            ref = golden(name)
            new = dict(np.load(os.path.join(tmp, name + ".npz")))
            assert sorted(ref) == sorted(new), name
            for k in ref:
                a, b = np.asarray(new[k], np.float64), np.asarray(ref[k], np.float64)
                den = max(np.abs(b).max(), 1e-30)
                assert np.abs(a - b).max() / den <= 1e-6, (name, k)


def test_dcnv2_fixtures_cover_the_mask_edge_values():
    m = np.concatenate([golden(n)["mask"].ravel() for n in golden_names("dcnv2_")])
    assert (m == 0).any() and (m == 1).any() and (m < 0).any() and (m > 1).any()
