"""Pins the CPU oracle (oracle/dcn_oracle.c, oracle/torch_chain.py) to outputs of the
UNMODIFIED reference held in tests/golden/ (made by oracle/make_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import dcn_oracle as orc
from oracle import torch_chain
from tests.util import golden, golden_names, rel_err, shape_from_cfg, stencil_from_corners


@pytest.mark.parametrize("name", golden_names("stencil_"))
def test_corner_indices_and_weights_bit_exact(name):
    """Sampling indices and corner weights must match the reference bit for bit."""
    g = golden(name)
    s = shape_from_cfg(g["cfg"], orc.VARIANT_TORCH)
    y0, x0, w4, _ = orc.corners(s, g["off"])
    st = stencil_from_corners(y0, x0, w4, s.H, s.W)          # [B,N,Ho,Wo,HW]
    ref = g["S"].transpose(0, 4, 2, 3, 1)                    # S[B,C=HW,Ho,Wo,N] -> [B,N,Ho,Wo,HW]
    assert ref.shape == st.shape
    assert np.array_equal(st.view(np.uint32) & 0x7FFFFFFF, ref.view(np.uint32) & 0x7FFFFFFF), \
        f"{(st != ref).sum()} stencil entries differ"


@pytest.mark.parametrize("S,n_low", [(128, 10), (64, 15), (56, 7), (28, 2), (14, 3), (32, 0)])
def test_roundtrip_wobble_bit_exact(S, n_low):
    """Zero offsets: w -> /(S-1)*2-1 -> (+1)*((S-1)/2) is not the identity in float32;
    the oracle must floor low exactly where the reference does (SURVEY.md A.3)."""
    g = golden(f"wobble_{S}")
    s = orc.make_shape(1, 1, 1, S, S, 3, 1, 1, orc.VARIANT_TORCH)
    off = np.zeros((1, 18, S, S), np.float32)
    y0, x0, w4, fxy = orc.corners(s, off)
    # rows probe: outputs (h=0, w=t) read input row ~t at column 0
    for probe, yy, ww in (("rows", y0[0, 0, 0, :], w4[0, 0, 0, :, :]),
                          ("cols", x0[0, 0, :, 0], w4[0, 0, :, 0, :])):
        exp = np.zeros((S, S), np.float32)
        for t in range(S):
            lo = ww[t, 0]                                    # nw weight = (1-f) * 1
            hi = ww[t, 2] if probe == "rows" else ww[t, 1]   # sw (rows) / ne (cols) = f * 1
            if 0 <= yy[t] < S:
                exp[t, yy[t]] = lo
            if 0 <= yy[t] + 1 < S:
                exp[t, yy[t] + 1] = hi
        assert np.array_equal(exp, g[probe]), probe
    # known answer from the survey probe: how many integer coordinates floor one lower
    assert int((y0[0, 0, 0, :] != np.arange(S)).sum()) == n_low
    ref_low = int(sum(1 for t in range(S) if g["rows"][t, t] != 1.0 and t > 0 and g["rows"][t, t - 1] != 0))
    assert ref_low == n_low


@pytest.mark.parametrize("name", golden_names("layer_") + golden_names("umma_") + golden_names("gemm_"))
def test_c_oracle_matches_reference_layer(name):
    g = golden(name)
    s = shape_from_cfg(g["cfg"], orc.VARIANT_TORCH)
    out = orc.forward(s, g["x"], g["off"], g["weight"], g.get("bias"))
    assert rel_err(out, g["out"]) < 2e-6
    gx, goff, gw, gb = orc.backward(s, g["x"], g["off"], g["weight"], g["gout"])
    assert rel_err(gx, g["gx"]) < 5e-6
    assert rel_err(goff, g["goff"]) < 5e-6
    assert rel_err(gw, g["gw"]) < 5e-6
    if "gb" in g:
        assert rel_err(gb, g["gb"]) < 5e-6


@pytest.fixture
def golden_cpu_threads():
    """torch's CPU convolution and GEMM kernels split their sums by thread, so a golden made by a multi-threaded CPU run
    is reproduced bit for bit only at the thread count it was made with (oracle/make_golden.py: GOLDEN_CPU_THREADS)."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", golden_names("layer_") + golden_names("umma_") + golden_names("gemm_"))
def test_torch_chain_is_bitwise_the_reference(name, golden_cpu_threads):
    """Same torch ops in the same order => identical bits (forward and autograd)."""
    g = golden(name)
    B, C, O, H, W, kh, kw, sh, sw, ph, pw = (int(v) for v in g["cfg"])
    t = {k: torch.as_tensor(v) for k, v in g.items() if k != "cfg"}
    out, grads = torch_chain.chain_forward_backward(
        t["x"], t["off"], t["weight"], t.get("bias"), t["gout"], variant="torch",
        kernel_size=(kh, kw), stride=(sh, sw), padding=(ph, pw))
    assert torch.equal(out, t["out"])
    assert torch.equal(grads[0], t["gx"])
    assert torch.equal(grads[1], t["goff"])
    assert rel_err(grads[2].numpy(), g["gw"]) < 1e-6   # mm blocking may differ with thread count


@pytest.mark.parametrize("name", golden_names("jittor_"))
def test_c_oracle_jittor_variant_matches_transliteration(name):
    """Jittor variant: parity UNPINNED (no jittor here) — checked against the torch
    transliteration of deform_conv.py:30-81 only."""
    g = golden(name)
    s = shape_from_cfg(g["cfg"], orc.VARIANT_JITTOR)
    if s.H + 2 * s.ph - s.kh < s.sh or s.W + 2 * s.pw - s.kw < s.sw:
        pytest.skip("H_out or W_out == 1: the reference divides by zero (deform_conv.py:37-38)")
    out = orc.forward(s, g["x"], g["off"], g["weight"], g.get("bias"))
    assert rel_err(out, g["out"]) < 2e-6
    gx, goff, gw, gb = orc.backward(s, g["x"], g["off"], g["weight"], g["gout"])
    assert rel_err(gx, g["gx"]) < 5e-6
    assert rel_err(goff, g["goff"]) < 5e-6
    assert rel_err(gw, g["gw"]) < 5e-6


def test_sample_tensor_layout():
    """dcn_oracle_sample returns the [B,C,Ho,Wo,N] tensor of train.py:129."""
    g = golden("stencil_s1_6x7")
    s = shape_from_cfg(g["cfg"], orc.VARIANT_TORCH)
    x = np.zeros((s.B, s.C, s.H, s.W), np.float32)
    for c in range(s.C):
        x[:, c, c // s.W, c % s.W] = 1.0
    S = orc.sample(s, x, g["off"])
    assert np.array_equal(S, g["S"])


# ---- DCN_VARIANT_DCNV1: the oracle against torchvision.ops.deform_conv2d's own outputs ----------
@pytest.mark.parametrize("name", golden_names("dcnv1_stencil_"))
def test_dcnv1_corners_bit_exact_vs_torchvision(name):
    g = golden(name)
    s = shape_from_cfg(g["cfg"], orc.VARIANT_DCNV1)
    y0, x0, w4, _ = orc.corners(s, g["off"])
    st = stencil_from_corners(y0, x0, w4, s.H, s.W)
    ref = g["S"].transpose(0, 4, 2, 3, 1)
    assert np.array_equal(st.view(np.uint32) & 0x7FFFFFFF, ref.view(np.uint32) & 0x7FFFFFFF)


@pytest.mark.parametrize("name", [n for n in golden_names("dcnv1_") if "stencil" not in n])
def test_dcnv1_oracle_matches_torchvision(name):
    g = golden(name)
    s = shape_from_cfg(g["cfg"], orc.VARIANT_DCNV1)
    out = orc.forward(s, g["x"], g["off"], g["weight"], g["bias"])
    assert rel_err(out, g["out"]) < 2e-6
    gx, goff, gw, gb = orc.backward(s, g["x"], g["off"], g["weight"], g["gout"])
    assert rel_err(gx, g["gx"]) < 5e-6
    assert rel_err(goff, g["goff"]) < 5e-6
    assert rel_err(gw, g["gw"]) < 5e-6
    assert rel_err(gb, g["gb"]) < 5e-6


def test_harness_detector_with_the_chain_port_reproduces_the_reference_training_step(golden_cpu_threads):
    """The harness detector topology (jittor_dcn_b200/detector.py) with its DCN layers replaced by the CPU port of
    the reference's op chain (oracle/torch_chain.py) and the framework's BatchNorm2d + ReLU is the reference
    detector restated: one training step (train mode, loss of train.py:242-248) must reproduce the golden made by
    the UNMODIFIED reference (oracle/make_golden.py:make_detector_train_golden) — same torch build, same kernels.
    Pins the harness topology / loss recipe and the port that bench.py times as the CPU baseline."""
    import torch
    from jittor_dcn_b200.detector import EDNetDetection, detection_loss
    from oracle import torch_chain
    g, ev = golden("detector_train_step"), golden("detector_eval")
    torch.manual_seed(0)
    m = EDNetDetection(dcn_cls=torch_chain.ChainLayer, fused_bn_relu=False).train()
    m.load_state_dict({k[3:]: torch.as_tensor(v) for k, v in ev.items() if k.startswith("sd.")})
    cls, bbox = m(torch.as_tensor(g["x"]))
    loss = detection_loss(cls, bbox, torch.as_tensor(g["labels"]), torch.as_tensor(g["boxes"]))
    loss.backward()
    assert abs(float(loss) - float(g["loss"])) <= 1e-6 * abs(float(g["loss"]))
    assert rel_err(cls.detach().numpy(), g["cls"]) < 1e-5
    assert rel_err(bbox.detach().numpy(), g["bbox"]) < 1e-5
    for k, v in m.state_dict().items():
        if "running_" in k:
            assert rel_err(v.numpy(), g["buf." + k]) < 1e-6, k
    for k, p in m.named_parameters():
        if "grad." + k in g and float(np.abs(g["grad." + k]).max()) > 1e-3:
            assert rel_err(p.grad.numpy(), g["grad." + k]) < 1e-4, k
