"""The DCNv3 core (csrc/dcn_dcnv3.cu) against InternImage's grid_sample composition.

    python tools/bench_dcnv3.py [--steps 20] [--warmup 3] [--rounds 3] [--out profiles/r3_bench_dcnv3.json]

Arms, per workload, median ms of the forward (no autograd) and of forward + backward (the gradients of input, offset
and mask):
  engine        dcnv3_core with the mask softmax fused (dcnv3_fwd_kernel / dcnv3_bwd_kernel), as the DCNv3 module runs it
  composition   softmax + dcnv3_core_pytorch (F.grid_sample, fp32) on the same GPU — the only GPU yardstick that
                builds offline; InternImage's ops_dcnv3 extension is not built for sm_100a
Workloads, fp32, 3x3 kernel, stride 1, padding 1, offset_scale 1: the four InternImage-T stages at 224^2 and batch 128,
one detection-resolution stage (200 x 336 x 64, G = 4, batch 2) and one Gc = 32 stage (InternImage-H style, C = 320,
G = 10).  Offsets are normal draws of about 1 px; mask logits are normal draws.  CUDA events around each call after
warm-up; the arms alternate in rounds in one process.  Kernel times come from a separate dcn_profile_* pass.  Each
kernel's share of the HBM floor is its compulsory bytes (computed below from the shapes) over 7.7 TB/s, divided by its
measured time.  The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import jittor_dcn_b200 as dcn  # noqa: E402
from jittor_dcn_b200 import _lib  # noqa: E402
from oracle.dcnv3_reference import dcnv3_core_pytorch  # noqa: E402
from tools.bench_msda import card, timed  # noqa: E402

WORKLOADS = {
    #  name           N    H    W    C    G
    "t_stage1":     (128, 56, 56, 64, 4),
    "t_stage2":     (128, 28, 28, 128, 8),
    "t_stage3":     (128, 14, 14, 256, 16),
    "t_stage4":     (128, 7, 7, 512, 32),
    "det_stage1":   (2, 200, 336, 64, 4),
    "h_gc32":       (16, 56, 56, 320, 10),
}
K = 3
HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def compulsory_bytes(N, H, W, C, G):
    """fp32 bytes each kernel must move at least once (Ho = H, Wo = W at 3x3 / stride 1 / padding 1)."""
    P = K * K
    pix, x = N * H * W, N * H * W * C * 4
    offset, mask = pix * G * P * 2 * 4, pix * G * P * 4
    fwd = x + offset + mask + x                              # read input, offset, mask; write out
    bwd = x + offset + mask + x + (x + x) + offset + mask    # read input, offset, mask, grad_out; grad_input RMW;
    return fwd, bwd                                          # write grad_offset, grad_mask


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the arms per workload")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: these are GPU timings")
    torch.manual_seed(0)
    res = {"card": card(),
           "method": f"median of {args.steps} CUDA-event timed calls after {args.warmup} warm-up calls, "
                     f"{args.rounds} alternating rounds per arm (median over rounds); fp32; 3x3, stride 1, pad 1, "
                     "offset_scale 1, mask softmax fused (engine) / F.softmax before the core (composition)",
           "hbm_floor_note": "hbm_floor_share = compulsory bytes / 7.7e12 B/s / kernel time; compulsory bytes are "
                             "computed from the shapes (fwd: input, offset, mask read, out written; bwd: input, "
                             "offset, mask, grad_out read, grad_input read and written once, grad_offset and "
                             "grad_mask written)",
           "workloads": {}}
    for name in args.workloads.split(","):
        N, H, W, C, G = WORKLOADS[name]
        Gc, P = C // G, K * K
        geo = (K, K, 1, 1, 1, 1, 1, 1, G, Gc, 1.0)
        x = torch.randn(N, H, W, C, device="cuda")
        off = torch.randn(N, H, W, G * P * 2, device="cuda")
        logits = torch.randn(N, H, W, G * P, device="cuda")
        gout = torch.randn(N, H, W, C, device="cuda")
        xr, orr, lr = (t.clone().requires_grad_(True) for t in (x, off, logits))

        def comp(a, b, c):
            soft = torch.softmax(c.view(N, H, W, G, P), -1).view(N, H, W, G * P)
            return dcnv3_core_pytorch(a, b, soft, *geo)

        def engine_fwd():
            with torch.no_grad():
                dcn.dcnv3_core(x, off, logits, *geo, softmax_mask=True)

        def engine_fwd_bwd():
            torch.autograd.grad(dcn.dcnv3_core(xr, orr, lr, *geo, softmax_mask=True), [xr, orr, lr], gout)

        def comp_fwd():
            with torch.no_grad():
                comp(x, off, logits)

        def comp_fwd_bwd():
            torch.autograd.grad(comp(xr, orr, lr), [xr, orr, lr], gout)

        arms = {"engine_fwd": engine_fwd, "engine_fwd_bwd": engine_fwd_bwd,
                "composition_fwd": comp_fwd, "composition_fwd_bwd": comp_fwd_bwd}
        with torch.no_grad():   # same results first: the fp32 composition on the GPU against the engine
            ref = comp(x, off, logits)
            diff = float((dcn.dcnv3_core(x, off, logits, *geo, softmax_mask=True) - ref).abs().max())
            diff_rel = diff / float(ref.abs().max())
            del ref
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        rounds = {k: [] for k in arms}
        for _ in range(args.rounds):
            for k, fn in arms.items():
                rounds[k].append(timed(fn, args.steps))
        entry = {"shape": dict(N=N, H=H, W=W, C=C, G=G, Gc=Gc, kernel=K),
                 "max_abs_diff_engine_vs_composition_fwd": diff,
                 "max_rel_diff_engine_vs_composition_fwd": diff_rel}
        for k, v in rounds.items():
            entry[k + "_ms"] = sorted(v)[len(v) // 2]
        for k in ("fwd", "fwd_bwd"):
            entry[f"composition_over_engine_{k}"] = entry[f"composition_{k}_ms"] / entry[f"engine_{k}_ms"]
        _lib.profile_begin()    # per-kernel times: a separate pass, the event profiler adds host work
        for _ in range(args.steps):
            engine_fwd_bwd()
        torch.cuda.synchronize()
        prof = _lib.profile_end()
        entry["kernels_ms_per_call"] = {k: v[1] / v[0] for k, v in prof.items()}
        fwd_b, bwd_b = compulsory_bytes(N, H, W, C, G)
        entry["compulsory_bytes"] = {"dcnv3_fwd_kernel": fwd_b, "dcnv3_bwd_kernel": bwd_b}
        entry["hbm_floor_share"] = {}
        for k, b in entry["compulsory_bytes"].items():
            t = entry["kernels_ms_per_call"].get(k)
            if t:
                entry["hbm_floor_share"][k] = b / HBM_BYTES_PER_S / (t * 1e-3)
        res["workloads"][name] = entry
        print(json.dumps({name: entry}), flush=True)
        del x, off, logits, gout, xr, orr, lr, arms
        torch.cuda.empty_cache()
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
