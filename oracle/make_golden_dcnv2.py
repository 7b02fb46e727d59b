"""Generates tests/golden/dcnv2_*.npz: the modulated form of DCN_VARIANT_DCNV1 (DCNv2, torchvision's ``mask=``).
TEST INFRA.  Needs torchvision only (no reference checkout):

    python -m oracle.make_golden_dcnv2

Every fixture holds the seeded inputs (x, offset, mask, weight, bias, grad_out) and what torchvision's CPU
``deform_conv2d(..., mask=)`` returns for them: the output and the gradients of x, offset, mask, weight and bias.
Masks mix sigmoid(normal) with exact 0, exact 1, negative and > 1 values: the operator applies no range.  Like the
other fixtures they are made at oracle/make_golden.py's GOLDEN_CPU_THREADS (torch's CPU kernels split their sums by
thread), and tests/golden/PROVENANCE_dcnv2.txt records the versions.
"""
import os
import sys

import numpy as np
import torch

from . import torch_chain
from .make_golden import GOLDEN_CPU_THREADS, OUT, _cfg

DCNV2 = {
    #  name             B  C   O   H   W   k       s  p       sigma
    "dcnv2_a_s1":      (2, 4,  6,  9,  11, 3,      1, 1,      1.5),   # generic kernels
    "dcnv2_b_s2":      (2, 32, 32, 15, 16, 3,      2, 1,      2.0),   # stride 2, tensor path
    "dcnv2_c_k1x3":    (1, 4,  5,  7,  10, (1, 3), 1, (0, 1), 1.0),   # 1 x 3, non-square padding
    "dcnv2_d_far":     (1, 3,  4,  8,  8,  3,      1, 1,      6.0),   # most samples leave the image
    "dcnv2_e_64":      (1, 64, 64, 12, 12, 3,      1, 1,      1.0),   # tensor path, one tap per K block
    "dcnv2_f_16":      (2, 16, 32, 10, 9,  3,      1, 1,      1.5),   # tensor path, 16 channels per sampling point
}
SEED = 20261021


def dcnv2_mask(rng, shape):
    """sigmoid(normal) with exact 0, exact 1, negative and > 1 entries mixed in: the operator applies no range."""
    m = 1.0 / (1.0 + np.exp(-rng.standard_normal(shape)))
    pick = rng.random(shape)
    m[pick < 0.08] = 0.0
    m[(pick >= 0.08) & (pick < 0.16)] = 1.0
    neg = (pick >= 0.16) & (pick < 0.22)
    m[neg] = -rng.random(int(neg.sum())) - 0.05
    big = (pick >= 0.22) & (pick < 0.28)
    m[big] = 1.0 + 2.0 * rng.random(int(big.sum())) + 0.05
    return m.astype(np.float32)


def make_dcnv2(rng, out_dir=OUT):
    """torchvision.ops.deform_conv2d with ``mask`` (CPU): forward and the gradients of x, offset, mask, weight, bias."""
    from torchvision.ops import deform_conv2d
    os.makedirs(out_dir, exist_ok=True)
    for name, (B, C, O, H, W, k, s, p, sigma) in DCNV2.items():
        kh, kw = torch_chain._pair(k)
        sh, sw = torch_chain._pair(s)
        ph, pw = torch_chain._pair(p)
        N = kh * kw
        Ho, Wo = torch_chain.out_hw(H, W, k, s, p)
        x = torch.as_tensor(rng.standard_normal((B, C, H, W)).astype(np.float32)).requires_grad_(True)
        off = torch.as_tensor((rng.standard_normal((B, 2 * N, Ho, Wo)) * sigma).astype(np.float32)).requires_grad_(True)
        mask = torch.as_tensor(dcnv2_mask(rng, (B, N, Ho, Wo))).requires_grad_(True)
        wt = torch.as_tensor((rng.standard_normal((O, C, kh, kw)) * np.sqrt(2.0 / (C * N))).astype(np.float32)).requires_grad_(True)
        bias = torch.as_tensor(rng.standard_normal((O,)).astype(np.float32)).requires_grad_(True)
        gout = torch.as_tensor(rng.standard_normal((B, O, Ho, Wo)).astype(np.float32))
        out = deform_conv2d(x, off, wt, bias, stride=(sh, sw), padding=(ph, pw), mask=mask)
        gx, goff, gmask, gw, gb = torch.autograd.grad(out, [x, off, mask, wt, bias], gout)
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, cfg=_cfg(B=B, C=C, O=O, H=H, W=W, kh=kh, kw=kw, sh=sh, sw=sw, ph=ph, pw=pw),
                            x=x.detach().numpy(), off=off.detach().numpy(), mask=mask.detach().numpy(),
                            weight=wt.detach().numpy(), bias=bias.detach().numpy(), gout=gout.numpy(),
                            out=out.detach().numpy(), gx=gx.numpy(), goff=goff.numpy(), gmask=gmask.numpy(),
                            gw=gw.numpy(), gb=gb.numpy())
        print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


def main():
    import torchvision
    torch.set_num_threads(GOLDEN_CPU_THREADS)
    make_dcnv2(np.random.default_rng(SEED))
    with open(os.path.join(OUT, "PROVENANCE_dcnv2.txt"), "w") as fh:
        fh.write("made by: python -m oracle.make_golden_dcnv2\n"
                 f"torch {torch.__version__}, torchvision {torchvision.__version__}, numpy {np.__version__}, "
                 f"{GOLDEN_CPU_THREADS} CPU threads, seed {SEED}\n"
                 "dcnv2_*: outputs and the five gradients (x, offset, mask, weight, bias) of "
                 "torchvision.ops.deform_conv2d(..., mask=) (CPU) for the modulated DCN_VARIANT_DCNV1 calls "
                 "(dcn_forward_modulated / dcn_backward_modulated); masks mix sigmoid(normal) with exact 0, exact 1, "
                 "negative and > 1 values: " + ", ".join(DCNV2) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
