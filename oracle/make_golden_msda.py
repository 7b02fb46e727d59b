"""Generates tests/golden/msda_*.npz: multi-scale deformable attention (Deformable DETR's MSDeformAttn core).
TEST INFRA.  Needs torch only:

    python -m oracle.make_golden_msda

Every fixture holds seeded float32 inputs (value, spatial_shapes, level_start_index, sampling_locations,
attention_weights, grad_out) and, evaluated in float64 on the CPU from those very values, the output of
oracle/msda_reference.py's grid_sample composition and the autograd gradients of value, sampling_locations and
attention_weights.  Locations are drawn around [0, 1] with some outside it and some exactly on 0 and 1; attention
weights include negative values and do not sum to one.  Coordinates x*W - 0.5 within 1e-3 of an integer are moved
away: there the derivative is one-sided and a float32 kernel may take the other side.  Made at oracle/make_golden.py's
GOLDEN_CPU_THREADS; tests/golden/PROVENANCE_msda.txt records the versions.
"""
import os
import sys

import numpy as np
import torch

from . import msda_reference
from .make_golden import GOLDEN_CPU_THREADS, OUT

MSDA = {
    #  name            B  M  D   Q   levels (H, W)                 P
    "msda_a_one":     (2, 2, 32, 10, ((9, 13),), 4),                     # one non-square level
    "msda_b_multi":   (1, 4, 64, 12, ((8, 8), (4, 6), (2, 3)), 1),       # three levels, one point
    "msda_c_edges":   (2, 2, 32, 16, ((6, 10), (3, 5)), 4),              # outside [0, 1], borders, odd weights
}
SEED = 20261022


def _away_from_pixels(loc, spatial_shapes, eps=1e-3):
    """Moves any coordinate loc*W - 0.5 (resp. loc*H - 0.5) that lies within eps of an integer by 2*eps pixels."""
    L = len(spatial_shapes)
    for l, (H, W) in enumerate(spatial_shapes):
        for c, ext in ((0, W), (1, H)):
            v = loc[:, :, :, l, :, c].astype(np.float64) * ext - 0.5
            near = np.abs(v - np.round(v)) < eps
            v[near] += 2 * eps
            loc[:, :, :, l, :, c] = ((v + 0.5) / ext).astype(np.float32)
    assert L == loc.shape[3]
    return loc


def make_case(rng, B, M, D, Q, levels, P, edges):
    L = len(levels)
    S = sum(h * w for h, w in levels)
    value = rng.standard_normal((B, S, M, D)).astype(np.float32)
    loc = rng.uniform(-0.1, 1.1, (B, Q, M, L, P, 2)).astype(np.float32)
    aw = rng.standard_normal((B, Q, M, L, P)).astype(np.float32)     # negative, not summing to one
    if edges:
        flat = loc.reshape(-1)
        pick = rng.random(flat.shape)
        flat[pick < 0.05] = 0.0
        flat[(pick >= 0.05) & (pick < 0.10)] = 1.0
        far = (pick >= 0.10) & (pick < 0.20)
        flat[far] = rng.choice([-0.6, -0.3, 1.3, 1.7], int(far.sum())).astype(np.float32)
    loc = _away_from_pixels(loc, levels)
    grad_out = rng.standard_normal((B, Q, M * D)).astype(np.float32)
    ss = np.array(levels, np.int64)
    lsi = msda_reference.level_start_index_of(ss).numpy()
    out, gv, gl, ga = msda_reference.reference(value, ss, loc, aw, grad_out)
    return dict(value=value, spatial_shapes=ss, level_start_index=lsi, sampling_locations=loc, attention_weights=aw,
                grad_out=grad_out, out=out.numpy(), grad_value=gv.numpy(), grad_sampling_locations=gl.numpy(),
                grad_attention_weights=ga.numpy(), P=np.int64(P))


def make_msda(out_dir=OUT):
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(SEED)
    for name, (B, M, D, Q, levels, P) in MSDA.items():
        arrays = make_case(rng, B, M, D, Q, levels, P, edges=name.endswith("edges"))
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **arrays)
        print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


def main():
    torch.set_num_threads(GOLDEN_CPU_THREADS)
    make_msda()
    with open(os.path.join(OUT, "PROVENANCE_msda.txt"), "w") as fh:
        fh.write("made by: python -m oracle.make_golden_msda\n"
                 f"torch {torch.__version__}, numpy {np.__version__}, {GOLDEN_CPU_THREADS} CPU threads, seed {SEED}\n"
                 "msda_*: float32 inputs and, in float64 on the CPU, the output and the gradients of value, "
                 "sampling_locations and attention_weights of Deformable DETR's grid_sample composition "
                 "(oracle/msda_reference.py) for dcn_msda_forward / dcn_msda_backward: " + ", ".join(MSDA) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
