"""Generates tests/golden/dcnv3_*.npz: the DCNv3 core (InternImage's ops_dcnv3).  TEST INFRA.  Needs torch only:

    python -m oracle.make_golden_dcnv3

Every fixture holds seeded float32 inputs (input, offset, mask, grad_out), the geometry, the softmax switch and,
evaluated in float64 on the CPU from those very values, the output of oracle/dcnv3_reference.py's grid_sample
composition and the autograd gradients of input, offset and mask (of the logits when the softmax is on).  Offsets are
drawn on a 2^-10 grid, so that every fp32 coordinate of the kernels is exact; some move samples outside the image and
some put them exactly on its border (an integer coordinate 0 or H - 1 / W - 1, and -1 / W, where only one corner
row or column remains).  Made at oracle/make_golden.py's GOLDEN_CPU_THREADS; tests/golden/PROVENANCE_dcnv3.txt
records the versions.
"""
import os
import sys

import numpy as np
import torch

from . import dcnv3_reference
from .make_golden import GOLDEN_CPU_THREADS, OUT

# geo = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels, os)
DCNV3 = {
    #  name                 N  H   W   geo                                         softmax
    "dcnv3_a_3x3":         (2, 9, 11, (3, 3, 1, 1, 1, 1, 1, 1, 2, 16, 1.0),    False),
    "dcnv3_b_3x5_softmax": (1, 8, 10, (3, 5, 1, 1, 1, 2, 1, 1, 2, 32, 1.0),    True),
    "dcnv3_c_s2_d2_os":    (2, 13, 12, (3, 3, 2, 2, 2, 1, 2, 2, 3, 16, 0.5),   True),
    "dcnv3_d_edges":       (1, 7, 9, (3, 5, 1, 2, 1, 2, 2, 1, 2, 32, 2.0),     False),
}
SEED = 20261021


def make_case(rng, N, H, W, geo, softmax, edges):
    kh, kw, sh, sw, ph, pw, dh, dw, G, Gc, os_ = geo
    Ho, Wo = dcnv3_reference.out_extent(H, W, kh, kw, sh, sw, ph, pw, dh, dw)
    P = kh * kw
    x = rng.standard_normal((N, H, W, G * Gc)).astype(np.float32)
    off = np.round(rng.normal(0, 1.5, (N, Ho, Wo, G * P * 2)) * 1024) / 1024
    if edges:   # pin some samples onto the border lines and past them: coordinate -> off
        xs, ys = dcnv3_reference.sample_coordinates(Ho, Wo, torch.zeros(N, Ho, Wo, G * P * 2), kh, kw, sh, sw, ph, pw,
                                                    dh, dw, G, os_)
        o = off.reshape(N, Ho, Wo, G, P, 2)
        for c, base, ext in ((0, xs.numpy(), W), (1, ys.numpy(), H)):
            targets = rng.choice(np.array([-1.0, 0.0, ext - 1.0, float(ext), -2.5, ext + 1.5]), o.shape[:-1])
            pick = rng.random(o.shape[:-1]) < 0.25
            o[..., c] = np.where(pick, (targets - base) / os_, o[..., c])
        off = o.reshape(N, Ho, Wo, G * P * 2)
    off = off.astype(np.float32)
    mask = rng.standard_normal((N, Ho, Wo, G * P)).astype(np.float32)
    gout = rng.standard_normal((N, Ho, Wo, G * Gc)).astype(np.float32)
    out, gx, goff, gm = dcnv3_reference.reference(x, off, mask, geo, gout, softmax_mask=softmax)
    return dict(input=x, offset=off, mask=mask, grad_out=gout, geo=np.array(geo[:10], np.int64),
                offset_scale=np.float64(os_), softmax=np.bool_(softmax), out=out.numpy(), grad_input=gx.numpy(),
                grad_offset=goff.numpy(), grad_mask=gm.numpy())


def make_dcnv3(out_dir=OUT):
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(SEED)
    for name, (N, H, W, geo, softmax) in DCNV3.items():
        arrays = make_case(rng, N, H, W, geo, softmax, edges=name.endswith("edges"))
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **arrays)
        print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


def main():
    torch.set_num_threads(GOLDEN_CPU_THREADS)
    make_dcnv3()
    with open(os.path.join(OUT, "PROVENANCE_dcnv3.txt"), "w") as fh:
        fh.write("made by: python -m oracle.make_golden_dcnv3\n"
                 f"torch {torch.__version__}, numpy {np.__version__}, {GOLDEN_CPU_THREADS} CPU threads, seed {SEED}\n"
                 "dcnv3_*: float32 inputs and, in float64 on the CPU, the output and the gradients of input, offset "
                 "and mask (the mask logits where softmax is set) of InternImage's grid_sample composition "
                 "(oracle/dcnv3_reference.py) for dcn_v3_forward / dcn_v3_backward: " + ", ".join(DCNV3) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
