"""Generates tests/golden/*.npz from the UNMODIFIED reference.  TEST INFRA; run in the build
container only (needs /root/reference):

    python -m oracle.make_golden

The reference has no tests, golden vectors or seeds of its own (SURVEY.md 4), so these
fixtures — outputs of the reference's own ``TorchDeformConv2d`` (train.py:70-140, loaded
verbatim by oracle/ref_loader.py) on seeded inputs — are what pins the oracle.

Fixture kinds
  stencil_*  : sampling geometry, BIT-EXACT.  The input has one one-hot channel per pixel and
               the weight matrix is the K x K identity, so ``out`` IS the sample tensor
               (a product with 1.0 and sums with 0.0 are exact in any GEMM order) and every
               value is one corner weight sitting at that corner's pixel.
  wobble_*   : the float32 normalise -> un-normalise round trip at zero offsets
               (SURVEY.md 0.6 / A.3) for S in {128,64,56,32,28,14}, again through one-hot
               channels, bit-exact.
  layer_*    : forward + the four autograd gradients on small random problems.
  dcnv1_*    : DCN_VARIANT_DCNV1 (standard DCNv1, not a reference operator): outputs of
               torchvision.ops.deform_conv2d itself, incl. bit-exact stencil probes.
  jittor_*   : same problems through the torch transliteration of deform_conv.py
               (oracle/torch_chain.py, variant="jittor") — NOT a run of the reference
               (jittor is not installable here); pins the C oracle's Jittor variant to the
               transliteration only.
"""
import os
import sys

import numpy as np
import torch
import torch.nn as tnn

from . import ref_loader, torch_chain

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")
# torch's CPU kernels split their sums by thread: the goldens in tests/golden/ were made with 8 threads, and
# tests/test_oracle_golden.py runs its bitwise torch comparisons at that count to reproduce them on any host
GOLDEN_CPU_THREADS = 8


def _save(name, **arrays):
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


def _cfg(**kw):
    return np.array([kw[k] for k in ("B", "C", "O", "H", "W", "kh", "kw", "sh", "sw", "ph", "pw")],
                    np.int32)


def _sample_tensor_from_identity_run(C, H, W, k, s, p, x, off):
    """Runs the reference layer with Wm = I and returns S[B,C,Ho,Wo,N] recovered from out."""
    kh, kw = torch_chain._pair(k)
    N = kh * kw
    K = C * N
    B = x.shape[0]
    Ho, Wo = torch_chain.out_hw(H, W, k, s, p)
    weight = np.eye(K, dtype=np.float32).reshape(K, C, kh, kw)
    res = ref_loader.run_reference_layer(C, K, k, s, p, x, off, weight, None)
    out = res["out"]  # [B, K, Ho, Wo];  out[b, j, r] = S_b.flat[r*K + j]   (train.py:129-136)
    S = out.reshape(B, K, Ho * Wo).transpose(0, 2, 1).reshape(B, C, Ho, Wo, N)
    return np.ascontiguousarray(S)


def make_stencils(rng):
    for name, (H, W, k, s, p, sigma) in {
        "stencil_s1_6x7": (6, 7, 3, 1, 1, 1.5),
        "stencil_s2_9x8": (9, 8, 3, 2, 1, 2.0),
        "stencil_s1_5x5_far": (5, 5, 3, 1, 1, 6.0),
        "stencil_k1x3_4x6": (4, 6, (1, 3), 1, (0, 1), 1.0),
    }.items():
        kh, kw = torch_chain._pair(k)
        sh, sw = torch_chain._pair(s)
        ph, pw = torch_chain._pair(p)
        N = kh * kw
        C = H * W
        B = 2
        Ho, Wo = torch_chain.out_hw(H, W, k, s, p)
        x = np.zeros((B, C, H, W), np.float32)
        for c in range(C):
            x[:, c, c // W, c % W] = 1.0
        off = (rng.standard_normal((B, 2 * N, Ho, Wo)) * sigma).astype(np.float32)
        off[0, :, 0, :] = 0.0                      # the reference's init state (zero offsets)
        off[1, :, -1, :] = np.round(off[1, :, -1, :])  # integer offsets (fx = 0 corner cases)
        S = _sample_tensor_from_identity_run(C, H, W, k, s, p, x, off)
        _save(name, cfg=_cfg(B=B, C=C, O=C * N, H=H, W=W, kh=kh, kw=kw, sh=sh, sw=sw, ph=ph, pw=pw),
              off=off, S=S)


def make_wobble():
    """Zero offsets, square S x S, stride 1: output (h=0, w=t) samples input (row~t, col 0).

    Channel c is one-hot at pixel (row c, col 0); column 0 round-trips exactly (ix = 0), so
    S[0, c, 0, t, n] is the pure row weight: (1-fy) at c = y0 and fy at c = y0+1.
    """
    for S_ in (128, 64, 56, 32, 28, 14):
        x = np.zeros((1, S_, S_, S_), np.float32)
        for c in range(S_):
            x[0, c, c, 0] = 1.0
        off = np.zeros((1, 18, S_, S_), np.float32)
        smp = _sample_tensor_from_identity_run(S_, S_, S_, 3, 1, 1, x, off)
        rows = smp[0, :, 0, :, 0].T.copy()  # [t, c]
        # second direction: one-hot at (row 0, col c); outputs (h=t, w=0)
        x2 = np.zeros_like(x)
        for c in range(S_):
            x2[0, c, 0, c] = 1.0
        smp2 = _sample_tensor_from_identity_run(S_, S_, S_, 3, 1, 1, x2, off)
        cols = smp2[0, :, :, 0, 0].T.copy()  # [t, c]
        _save(f"wobble_{S_}", S=np.int32(S_), rows=rows, cols=cols)


LAYERS = {
    #  name            B  C   O   H   W   k       s  p       sigma bias
    "layer_a_s1":     (2, 4,  8,  10, 10, 3,      1, 1,      1.5, True),
    "layer_b_nonsq":  (2, 3,  5,  17, 23, 3,      1, 1,      1.0, True),
    "layer_c_s2":     (1, 4,  8,  20, 28, 3,      2, 1,      2.0, True),
    "layer_d_det0":   (2, 16, 32, 16, 16, 3,      2, 1,      0.0, True),   # zero offsets = init state
    "layer_e_far":    (1, 2,  3,  8,  8,  3,      1, 1,      6.0, True),   # mostly out of bounds
    "layer_f_k1x3":   (1, 3,  4,  9,  11, (1, 3), 1, (0, 1), 1.0, True),
    "layer_g_nobias": (2, 4,  6,  7,  9,  3,      1, 1,      1.0, False),
    "layer_h_k1":     (2, 5,  7,  6,  6,  1,      1, 0,      1.0, True),
    "layer_i_wide":   (1, 8,  4,  6,  6,  3,      1, 1,      1.0, True),   # Ho*Wo < C: rows span channels
}


# Reference goldens that ROUTE TO THE TENSOR PATH (dcn_path_name == "umma" for both phases and all three coordinate
# modes; tests/test_gpu_parity.py asserts the routing): every Torch-layout tiling class (Gt x Rt = 64x2, 32x4, 16x8),
# two channel chunks per sampling point, partial last tiles, a stride-2 layer, live offsets.
UMMA_LAYERS = {
    #  name          B  C    O   H   W   k  s  p  sigma bias     Torch-layout tiling
    "umma_a_64x2":  (3, 64,  64, 16, 16, 3, 1, 1, 1.5, True),   # G = 64: Gt 64, Rt 2, 6 full tiles
    "umma_b_32x4":  (3, 32,  48, 12, 8,  3, 1, 1, 2.0, True),   # G = 32: Gt 32, Rt 4, R = 3: 9 instances, partial tile
    "umma_c_16x8":  (2, 64,  32, 12, 12, 3, 1, 1, 1.0, True),   # G = 16: Gt 16, Rt 8, Cs = 4, R = 9: partial tile
    "umma_d_chunk": (1, 128, 64, 16, 16, 3, 1, 1, 2.5, False),  # G = 128: two 64-channel chunks per sampling point
    "umma_e_s2":    (2, 32,  64, 32, 32, 3, 2, 1, 2.0, True),   # stride 2 (detector conv3 shape at 32 x 32)
}


# layer fixtures whose Torch-layout shapes run on the materialised-sample + GEMM path (csrc/dcn_gemm_path.cu,
# dcn_path_name == "gemm": gcd(Ho*Wo, C) not a multiple of 16, C >= 32, O >= 32, K >= 256)
GEMM_LAYERS = {
    "gemm_a_c5like": (2, 64, 48, 14, 14, 3, 1, 1, 1.5, True),    # gcd(196, 64) = 4, the C5 situation
    "gemm_b_gcd24":  (2, 96, 40, 10, 12, 3, 1, 1, 2.0, False),   # gcd(120, 96) = 24
    "gemm_c_s2":     (2, 48, 32, 19, 21, 3, 2, 1, 1.0, True),    # stride 2: Ho*Wo = 110, gcd(110, 48) = 2
}


def make_layers(rng, layers=None):
    for name, (B, C, O, H, W, k, s, p, sigma, has_bias) in (layers or LAYERS).items():
        kh, kw = torch_chain._pair(k)
        sh, sw = torch_chain._pair(s)
        ph, pw = torch_chain._pair(p)
        N = kh * kw
        Ho, Wo = torch_chain.out_hw(H, W, k, s, p)
        x = rng.standard_normal((B, C, H, W)).astype(np.float32)
        off = (rng.standard_normal((B, 2 * N, Ho, Wo)) * sigma).astype(np.float32)
        weight = (rng.standard_normal((O, C, kh, kw)) * np.sqrt(2.0 / (C * N))).astype(np.float32)
        bias = rng.standard_normal((O,)).astype(np.float32) if has_bias else None
        gout = rng.standard_normal((B, O, Ho, Wo)).astype(np.float32)
        ref = ref_loader.run_reference_layer(C, O, k, s, p, x, off, weight, bias, gout)
        arrays = dict(cfg=_cfg(B=B, C=C, O=O, H=H, W=W, kh=kh, kw=kw, sh=sh, sw=sw, ph=ph, pw=pw),
                      x=x, off=off, weight=weight, gout=gout, **ref)
        if has_bias:
            arrays["bias"] = bias
        _save(name, **arrays)
        # Jittor-variant transliteration (NOT a reference run)
        tb = None if bias is None else torch.as_tensor(bias)
        out, grads = torch_chain.chain_forward_backward(
            torch.as_tensor(x), torch.as_tensor(off), torch.as_tensor(weight), tb,
            torch.as_tensor(gout), variant="jittor", kernel_size=k, stride=s, padding=p)
        jar = dict(arrays)
        jar.update(out=out.numpy(), gx=grads[0].numpy(), goff=grads[1].numpy(), gw=grads[2].numpy())
        if has_bias:
            jar["gb"] = grads[3].numpy()
        _save("jittor_" + (name[len("layer_"):] if name.startswith("layer_") else name), **jar)


def make_module_golden():
    """Whole module incl. a LIVE offset conv (weights N(0,0.01), bias N(0,1)): state_dict in,
    output + parameter gradients out — the drop-in test for the module boundary."""
    torch.manual_seed(1234)
    cls = ref_loader.load_reference_classes(("TorchDeformConv2d",))["TorchDeformConv2d"]
    m = cls(8, 16, 3, 2, 1)
    with torch.no_grad():
        m.offset_conv.weight.normal_(0, 0.01)
        m.offset_conv.bias.normal_(0, 1.0)
        m.bias.normal_(0, 0.1)
    x = torch.randn(2, 8, 24, 24, requires_grad=True)
    out = m(x)
    gout = torch.randn_like(out)
    out.backward(gout)
    arrays = {"sd." + k: v.detach().numpy() for k, v in m.state_dict().items()}
    arrays.update({"grad." + k: p.grad.numpy() for k, p in m.named_parameters()})
    _save("module_live_offsets", x=x.detach().numpy(), out=out.detach().numpy(), gout=gout.numpy(),
          gx=x.grad.numpy(), **arrays)


# Whole-module fixtures whose shapes run the WHOLE layer on the engine (offset conv as a plain mode of the tcgen05
# kernels + DCN span, dcn_layer_forward / dcn_layer_backward): outputs of the unmodified reference module.
MODULE_UMMA = {
    #  name               C    O   H   W   s
    "module_umma_s1":    (64,  64, 16, 16, 1),
    "module_umma_s2":    (32,  64, 32, 32, 2),    # detector conv3 channel counts, stride 2
    "module_umma_c128":  (128, 32, 12, 12, 1),    # Torch layout: 16 channels per sampling point, Cs = 8
    "module_umma_c16":   (16,  32, 32, 32, 2),    # detector conv2 channel counts
}


def make_module_umma_goldens():
    cls = ref_loader.load_reference_classes(("TorchDeformConv2d",))["TorchDeformConv2d"]
    for i, (name, (C, O, H, W, s_)) in enumerate(MODULE_UMMA.items()):
        torch.manual_seed(777 + i)
        m = cls(C, O, 3, s_, 1)
        with torch.no_grad():
            m.offset_conv.weight.normal_(0, 0.02)
            m.offset_conv.bias.normal_(0, 1.0)
            m.bias.normal_(0, 0.1)
        x = torch.randn(2, C, H, W, requires_grad=True)
        out = m(x)
        gout = torch.randn_like(out)
        out.backward(gout)
        with torch.no_grad():
            offset = m.offset_conv(x)
        arrays = {"sd." + k: v.detach().numpy() for k, v in m.state_dict().items()}
        arrays.update({"grad." + k: p.grad.numpy() for k, p in m.named_parameters()})
        _save(name, cfg=np.array([C, O, H, W, s_], np.int32), x=x.detach().numpy(), out=out.detach().numpy(),
              gout=gout.numpy(), gx=x.grad.numpy(), offset=offset.numpy(), **arrays)


def make_detector_golden():
    """One forward of the reference's toy detector (train.py:142-175) in eval mode."""
    torch.manual_seed(4321)
    cls = ref_loader.load_reference_classes()["TorchEDNetDetection"]
    m = cls().eval()
    with torch.no_grad():
        for mod in (m.conv2, m.conv3, m.conv4, m.conv5):
            mod.offset_conv.weight.normal_(0, 0.02)
            mod.offset_conv.bias.normal_(0, 0.7)
        x = torch.zeros(2, 1, 128, 128)
        x[0, 0, 10:38, 50:78] = torch.rand(28, 28)
        x[1, 0, 90:118, 3:31] = torch.rand(28, 28)
        cls_logits, bbox = m(x)
    arrays = {"sd." + k: v.numpy() for k, v in m.state_dict().items()}
    _save("detector_eval", x=x.numpy(), cls=cls_logits.numpy(), bbox=bbox.numpy(), **arrays)


def make_detector_train_golden():
    """One TRAINING step's forward + backward of the unmodified reference detector (train.py:142-175 in train
    mode, i.e. BatchNorm with batch statistics; loss recipe of train.py:195-199, 242-248): loss, heads,
    BatchNorm running statistics after the step and the parameter gradients.  Initial weights = the state dict
    stored in detector_eval.npz.  The four large DCN weight gradients are stored as their norm and their
    projection on a fixed random direction (keeps the fixture small)."""
    torch.manual_seed(97)
    cls = ref_loader.load_reference_classes()["TorchEDNetDetection"]
    m = cls()
    ev = dict(np.load(os.path.join(OUT, "detector_eval.npz")))
    m.load_state_dict({k[3:]: torch.as_tensor(v) for k, v in ev.items() if k.startswith("sd.")})
    m.train()
    B = 6
    x = torch.zeros(B, 1, 128, 128)
    pos = torch.randint(0, 101, (B, 2))
    for i in range(B):
        px, py = int(pos[i, 0]), int(pos[i, 1])
        x[i, 0, py:py + 28, px:px + 28] = torch.rand(28, 28)
    labels = torch.randint(0, 10, (B,))
    boxes = torch.stack([pos[:, 0], pos[:, 1], pos[:, 0] + 28, pos[:, 1] + 28], 1).float() / 128.0
    cls_out, bbox_out = m(x)
    cls_loss = tnn.CrossEntropyLoss()(cls_out, labels)
    diff = torch.abs(bbox_out - boxes)                                   # train.py:195-199, beta = 1
    bbox_loss = torch.where(diff < 1.0, 0.5 * diff * diff / 1.0, diff - 0.5).mean()
    total = cls_loss + 5.0 * bbox_loss                                   # train.py:247
    total.backward()
    arrays = {"x": x.numpy(), "labels": labels.numpy(), "boxes": boxes.numpy(), "loss": np.float32(total.item()),
              "cls": cls_out.detach().numpy(), "bbox": bbox_out.detach().numpy()}
    for k, v in m.state_dict().items():
        if "running_" in k or "num_batches" in k:
            arrays["buf." + k] = v.numpy()
    g = torch.Generator().manual_seed(5)
    for k, p_ in m.named_parameters():
        gr = p_.grad
        if gr.numel() > 20000:
            d = torch.randn(gr.shape, generator=g)
            arrays["gproj." + k] = np.array([float(gr.norm()), float((gr * d).sum()), float(d.norm())], np.float64)
        else:
            arrays["grad." + k] = gr.numpy()
    _save("detector_train_step", **arrays)


DCNV1 = {
    #  name             B  C   O   H   W   k       s  p       sigma
    "dcnv1_a_s1":      (2, 4,  6,  9,  11, 3,      1, 1,      1.5),
    "dcnv1_b_s2":      (2, 16, 32, 16, 16, 3,      2, 1,      2.0),   # tiles onto the tensor path
    "dcnv1_c_far":     (1, 3,  4,  8,  8,  3,      1, 1,      6.0),
    "dcnv1_d_k1x3":    (1, 4,  5,  7,  10, (1, 3), 1, (0, 1), 1.0),
    "dcnv1_e_64":      (1, 64, 64, 12, 12, 3,      1, 1,      1.0),   # tensor path, one tap per K block
}


def make_dcnv1(rng):
    """Standard DCNv1 (DCN_VARIANT_DCNV1): outputs of torchvision.ops.deform_conv2d itself (CPU)."""
    from torchvision.ops import deform_conv2d
    for name, (B, C, O, H, W, k, s, p, sigma) in DCNV1.items():
        kh, kw = torch_chain._pair(k)
        sh, sw = torch_chain._pair(s)
        ph, pw = torch_chain._pair(p)
        N = kh * kw
        Ho, Wo = torch_chain.out_hw(H, W, k, s, p)
        x = torch.as_tensor(rng.standard_normal((B, C, H, W)).astype(np.float32)).requires_grad_(True)
        off = torch.as_tensor((rng.standard_normal((B, 2 * N, Ho, Wo)) * sigma).astype(np.float32)).requires_grad_(True)
        wt = torch.as_tensor((rng.standard_normal((O, C, kh, kw)) * np.sqrt(2.0 / (C * N))).astype(np.float32)).requires_grad_(True)
        bias = torch.as_tensor(rng.standard_normal((O,)).astype(np.float32)).requires_grad_(True)
        gout = torch.as_tensor(rng.standard_normal((B, O, Ho, Wo)).astype(np.float32))
        out = deform_conv2d(x, off, wt, bias, stride=(sh, sw), padding=(ph, pw))
        gx, goff, gw, gb = torch.autograd.grad(out, [x, off, wt, bias], gout)
        _save(name, cfg=_cfg(B=B, C=C, O=O, H=H, W=W, kh=kh, kw=kw, sh=sh, sw=sw, ph=ph, pw=pw),
              x=x.detach().numpy(), off=off.detach().numpy(), weight=wt.detach().numpy(), bias=bias.detach().numpy(),
              gout=gout.numpy(), out=out.detach().numpy(), gx=gx.numpy(), goff=goff.numpy(), gw=gw.numpy(),
              gb=gb.numpy())
    # sampling geometry, bit-exact: one-hot channels and identity weights, so out IS the column matrix
    for name, (H, W, k, s, p, sigma) in {"dcnv1_stencil_s1": (6, 7, 3, 1, 1, 1.5),
                                         "dcnv1_stencil_s2": (9, 8, 3, 2, 1, 2.5)}.items():
        N, C, B = 9, H * W, 2
        Ho, Wo = torch_chain.out_hw(H, W, k, s, p)
        x = torch.zeros(B, C, H, W)
        for c in range(C):
            x[:, c, c // W, c % W] = 1.0
        off = torch.as_tensor((rng.standard_normal((B, 2 * N, Ho, Wo)) * sigma).astype(np.float32))
        off[0, :, 0, :] = 0.0
        off[1, :, -1, :] = torch.round(off[1, :, -1, :])
        wt = torch.eye(C * N).reshape(C * N, C, 3, 3)        # out[b, c*N + n, p] = column (c, n) of pixel p
        out = deform_conv2d(x, off, wt, None, stride=s, padding=p)
        S = out.reshape(B, C, N, Ho, Wo).permute(0, 1, 3, 4, 2).contiguous()   # [B, C, Ho, Wo, N]
        _save(name, cfg=_cfg(B=B, C=C, O=C * N, H=H, W=W, kh=3, kw=3, sh=s, sw=s, ph=p, pw=p),
              off=off.numpy(), S=S.numpy())


def main():
    assert ref_loader.available(), "needs /root/reference (build container only)"
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(GOLDEN_CPU_THREADS)
    if "--only-module-umma" in sys.argv:
        make_module_umma_goldens()
        return 0
    if "--only-gemm" in sys.argv:
        make_layers(np.random.default_rng(20261020), GEMM_LAYERS)   # own generator: added in round 2
        return 0
    make_layers(np.random.default_rng(20261019), UMMA_LAYERS)   # own generator: added in round 2
    make_module_umma_goldens()
    if "--only-umma" in sys.argv:
        return 0
    rng = np.random.default_rng(20261018)
    make_stencils(rng)
    make_layers(rng)
    make_module_golden()
    make_detector_golden()
    make_detector_train_golden()
    make_wobble()
    make_dcnv1(np.random.default_rng(4242))
    with open(os.path.join(OUT, "PROVENANCE.txt"), "w") as fh:
        fh.write("made by: python -m oracle.make_golden\n"
                 f"torch {torch.__version__}, numpy {np.__version__}\n"
                 "reference: x-y20/jittor-dcn train.py:70-175 loaded verbatim via ast "
                 "(oracle/ref_loader.py)\n"
                 "stencil_*, wobble_*, layer_*, umma_*, module_*, detector_* (eval forward, one training step): outputs of "
                 "the unmodified reference\n"
                 "umma_*: layer fixtures whose shapes run on the tcgen05 path (dcn_path_name == umma, forward and "
                 "backward, all coordinate modes): " + ", ".join(UMMA_LAYERS) + "\n"
                 "module_umma_*: whole-module fixtures (live offset conv) whose shapes run offset conv + DCN span on "
                 "the engine (dcn_layer_forward / dcn_layer_backward)\n"
                 "layer_*: layer_d_det0 runs on the tcgen05 path, the other eight on the generic kernels\n"
                 "jittor_*: torch transliteration of deform_conv.py:30-81 "
                 "(oracle/torch_chain.py) - parity unpinned\n"
                 "dcnv1_*: outputs of torchvision.ops.deform_conv2d (CPU) for DCN_VARIANT_DCNV1\n")


if __name__ == "__main__":
    sys.exit(main())
