"""The DCNv4 core (csrc/dcn_dcnv3.cu, dcnv4_*_kernel) against the ways to run DCNv4 without it.

    python tools/bench_dcnv4.py [--steps 20] [--warmup 3] [--rounds 3] [--out profiles/r3_bench_dcnv4.json]

Arms, per workload, median ms of the forward (no autograd) and of forward + backward (the gradients of input and
offset_mask):
  engine          dcnv4_core on the packed offset_mask (dcnv4_fwd_kernel / dcnv4_bwd_kernel)
  unpack_dcnv3    offset_mask unpacked into DCNv3's offset / mask by framework ops (with remove_center, the centre point
                  reinserted at offset 0 and mask 0), then the engine's dcnv3_core: what a user can do without DCNv4
  unpack_pytorch  the same unpacking, then InternImage's grid_sample composition (dcnv3_core_pytorch, fp32)
Workloads, fp32, stride 1, offset_scale 1: the four FlashInternImage-T stages at 224^2 and batch 128 (C = 64 / 128 /
256 / 512, Gc = 16, 3x3), one detection-resolution stage (200 x 336 x 64, batch 2), stage 1 with remove_center, and
stage 2 with a 5x5 kernel.  Offsets are normal draws of about 1 px, mask values normal draws.  CUDA events around each
call after warm-up; the arms alternate in rounds in one process.  Kernel times come from a separate dcn_profile_* pass.
Each kernel's share of the HBM floor is its compulsory bytes (computed below from the shapes) over 7.7 TB/s, divided by
its measured time.  The card's name and power limit are read in the same run and written beside the numbers.
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
from oracle.dcnv4_reference import unpack  # noqa: E402
from tools.bench_msda import card, timed  # noqa: E402

WORKLOADS = {
    #  name              N    H    W    C    G   kernel  remove_center
    "t_stage1":        (128, 56, 56, 64, 4, 3, False),
    "t_stage2":        (128, 28, 28, 128, 8, 3, False),
    "t_stage3":        (128, 14, 14, 256, 16, 3, False),
    "t_stage4":        (128, 7, 7, 512, 32, 3, False),
    "det_stage1":      (2, 200, 336, 64, 4, 3, False),
    "t_stage1_rc":     (128, 56, 56, 64, 4, 3, True),
    "t_stage2_5x5":    (128, 28, 28, 128, 8, 5, False),
}
HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def compulsory_bytes(N, H, W, C, Cm):
    """fp32 bytes each kernel must move at least once (Ho = H, Wo = W: stride 1, padding kernel // 2)."""
    x, om = N * H * W * C * 4, N * H * W * Cm * 4
    fwd = x + om + x                           # read input, offset_mask; write out
    bwd = x + om + x + (x + x) + om            # read input, offset_mask, grad_out; grad_input RMW; write grad_om
    return fwd, bwd


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
                     f"{args.rounds} alternating rounds per arm (median over rounds); fp32; stride 1, "
                     "pad kernel // 2, offset_scale 1; the unpack arms include the framework ops that unpack",
           "hbm_floor_note": "hbm_floor_share = compulsory bytes / 7.7e12 B/s / kernel time; compulsory bytes are "
                             "computed from the shapes (fwd: input, offset_mask read, out written; bwd: input, "
                             "offset_mask, grad_out read, grad_input read and written once, grad_offset_mask written)",
           "workloads": {}}
    for name in args.workloads.split(","):
        N, H, W, C, G, k, rc = WORKLOADS[name]
        Gc = C // G
        geo = (k, k, 1, 1, k // 2, k // 2, 1, 1, G, Gc, 1.0)
        Cm = dcn.dcnv4_row_floats(k, k, G, rc)
        x = torch.randn(N, H, W, C, device="cuda")
        om = torch.randn(N, H, W, Cm, device="cuda")
        gout = torch.randn(N, H, W, C, device="cuda")
        xr, omr = (t.clone().requires_grad_(True) for t in (x, om))

        def engine(a, b):
            return dcn.dcnv4_core(a, b, *geo, remove_center=rc)

        def unpack_dcnv3(a, b):
            off, m = unpack(b, k, k, G, rc)
            return dcn.dcnv3_core(a, off, m, *geo)

        def unpack_pytorch(a, b):
            off, m = unpack(b, k, k, G, rc)
            return dcnv3_core_pytorch(a, off, m, *geo)

        arms = {}
        for arm, f in (("engine", engine), ("unpack_dcnv3", unpack_dcnv3), ("unpack_pytorch", unpack_pytorch)):
            def fwd(f=f):
                with torch.no_grad():
                    f(x, om)

            def fwd_bwd(f=f):
                torch.autograd.grad(f(xr, omr), [xr, omr], gout)

            arms[arm + "_fwd"], arms[arm + "_fwd_bwd"] = fwd, fwd_bwd
        entry = {"shape": dict(N=N, H=H, W=W, C=C, G=G, Gc=Gc, kernel=k, remove_center=rc, Cm=Cm)}
        with torch.no_grad():   # same results first
            ref = engine(x, om)
            for arm, f in (("unpack_dcnv3", unpack_dcnv3), ("unpack_pytorch", unpack_pytorch)):
                diff = float((f(x, om) - ref).abs().max())
                entry[f"max_abs_diff_engine_vs_{arm}_fwd"] = diff
                entry[f"max_rel_diff_engine_vs_{arm}_fwd"] = diff / float(ref.abs().max())
            del ref
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        rounds = {a: [] for a in arms}
        for _ in range(args.rounds):
            for a, fn in arms.items():
                rounds[a].append(timed(fn, args.steps))
        for a, v in rounds.items():
            entry[a + "_ms"] = sorted(v)[len(v) // 2]
        for a in ("unpack_dcnv3", "unpack_pytorch"):
            for p in ("fwd", "fwd_bwd"):
                entry[f"{a}_over_engine_{p}"] = entry[f"{a}_{p}_ms"] / entry[f"engine_{p}_ms"]
        _lib.profile_begin()    # per-kernel times: a separate pass, the event profiler adds host work
        for _ in range(args.steps):
            arms["engine_fwd_bwd"]()
        torch.cuda.synchronize()
        prof = _lib.profile_end()
        entry["kernels_ms_per_call"] = {kn: v[1] / v[0] for kn, v in prof.items()}
        fwd_b, bwd_b = compulsory_bytes(N, H, W, C, Cm)
        entry["compulsory_bytes"] = {"dcnv4_fwd_kernel": fwd_b, "dcnv4_bwd_kernel": bwd_b}
        entry["hbm_floor_share"] = {}
        for kn, b in entry["compulsory_bytes"].items():
            t = entry["kernels_ms_per_call"].get(kn)
            if t:
                entry["hbm_floor_share"][kn] = b / HBM_BYTES_PER_S / (t * 1e-3)
        res["workloads"][name] = entry
        print(json.dumps({name: entry}), flush=True)
        del x, om, gout, xr, omr, arms
        torch.cuda.empty_cache()
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
