"""Generates tests/golden/dcnv4_*.npz: the DCNv4 core.  TEST INFRA.  Needs torch only:

    python -m oracle.make_golden_dcnv4

Every fixture holds seeded float32 inputs (input, offset_mask, grad_out), the geometry, the remove_center switch and,
evaluated in float64 on the CPU from those very values, the output of oracle/dcnv4_reference.py (DCNv3's
pixel-coordinate reference on the unpacked offset_mask) and the autograd gradients of input and offset_mask.  The
padding columns of offset_mask hold NaN (they must never be read); their gradient is 0.  Offsets are drawn on a 2^-10
grid, so that every fp32 coordinate of the kernels is exact; in the edges case some move samples outside the image and
some put them exactly on its border.  Made at oracle/make_golden.py's GOLDEN_CPU_THREADS;
tests/golden/PROVENANCE_dcnv4.txt records the versions.
"""
import os
import sys

import numpy as np
import torch

from . import dcnv3_reference, dcnv4_reference
from .make_golden import GOLDEN_CPU_THREADS, OUT

# geo = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels, os)
DCNV4 = {
    #  name                 N  H   W   geo                                         remove_center   Cm
    "dcnv4_a_3x3":         (2, 9, 11, (3, 3, 1, 1, 1, 1, 1, 1, 2, 16, 1.0),    False),         # 54 -> 56
    "dcnv4_b_5x5_rc":      (1, 10, 9, (5, 5, 1, 1, 2, 2, 1, 1, 2, 32, 1.0),    True),          # K 24: 144
    "dcnv4_c_s2_d2_os":    (2, 13, 12, (3, 3, 2, 2, 2, 1, 2, 2, 4, 16, 0.5),   False),         # 108 -> 112
    "dcnv4_d_edges_rc":    (1, 7, 9, (3, 5, 1, 2, 1, 2, 2, 1, 2, 32, 2.0),     True),          # K 14: 84 -> 88
    "dcnv4_e_pad_g3":      (1, 8, 10, (3, 3, 1, 1, 1, 1, 1, 1, 3, 16, 1.0),    False),         # 81 -> 88
}
SEED = 20261022


def make_case(rng, N, H, W, geo, remove_center, edges):
    kh, kw, sh, sw, ph, pw, dh, dw, G, Gc, os_ = geo
    Ho, Wo = dcnv3_reference.out_extent(H, W, kh, kw, sh, sw, ph, pw, dh, dw)
    K, c = dcnv4_reference.points(kh, kw, remove_center)
    Cm = dcnv4_reference.row_floats(kh, kw, G, remove_center)
    x = rng.standard_normal((N, H, W, G * Gc)).astype(np.float32)
    off = np.round(rng.normal(0, 1.5, (N, Ho, Wo, G, K, 2)) * 1024) / 1024
    if edges:   # pin some samples onto the border lines and past them: coordinate -> off
        xs, ys = dcnv3_reference.sample_coordinates(Ho, Wo, torch.zeros(N, Ho, Wo, G * kh * kw * 2), kh, kw, sh, sw,
                                                    ph, pw, dh, dw, G, os_)
        keep = [p for p in range(kh * kw) if p != c]     # the grid points of the K samples
        for ci, base, ext in ((0, xs.numpy()[..., keep], W), (1, ys.numpy()[..., keep], H)):
            targets = rng.choice(np.array([-1.0, 0.0, ext - 1.0, float(ext), -2.5, ext + 1.5]), off.shape[:-1])
            pick = rng.random(off.shape[:-1]) < 0.25
            off[..., ci] = np.where(pick, (targets - base) / os_, off[..., ci])
    mask = rng.standard_normal((N, Ho, Wo, G, K))
    om = np.full((N, Ho, Wo, Cm), np.nan, np.float32)
    om[..., :3 * G * K] = np.concatenate([off.reshape(N, Ho, Wo, G, 2 * K), mask], -1).reshape(N, Ho, Wo, 3 * G * K)
    gout = rng.standard_normal((N, Ho, Wo, G * Gc)).astype(np.float32)
    out, gx, gom = dcnv4_reference.reference(x, om, geo, gout, remove_center=remove_center)
    return dict(input=x, offset_mask=om, grad_out=gout, geo=np.array(geo[:10], np.int64),
                offset_scale=np.float64(os_), remove_center=np.bool_(remove_center), out=out.numpy(),
                grad_input=gx.numpy(), grad_offset_mask=gom.numpy())


def make_dcnv4(out_dir=OUT):
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(SEED)
    for name, (N, H, W, geo, rc) in DCNV4.items():
        arrays = make_case(rng, N, H, W, geo, rc, edges="edges" in name)
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **arrays)
        print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


def main():
    torch.set_num_threads(GOLDEN_CPU_THREADS)
    make_dcnv4()
    with open(os.path.join(OUT, "PROVENANCE_dcnv4.txt"), "w") as fh:
        fh.write("made by: python -m oracle.make_golden_dcnv4\n"
                 f"torch {torch.__version__}, numpy {np.__version__}, {GOLDEN_CPU_THREADS} CPU threads, seed {SEED}\n"
                 "dcnv4_*: float32 inputs (NaN in the padding columns of offset_mask) and, in float64 on the CPU, the "
                 "output and the gradients of input and offset_mask of DCNv3's pixel-coordinate reference on the "
                 "unpacked offset_mask (oracle/dcnv4_reference.py) for dcn_v4_forward / dcn_v4_backward: "
                 + ", ".join(DCNV4) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
