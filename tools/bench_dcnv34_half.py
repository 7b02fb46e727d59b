"""The DCNv3 / DCNv4 cores on bfloat16 and float16 operands against the float32 composition they replace.

    python tools/bench_dcnv34_half.py [--steps 20] [--warmup 3] [--rounds 3] [--out profiles/r3_bench_dcnv34_half.json]

Workloads: those of tools/bench_dcnv3.py (3x3, mask softmax fused) and tools/bench_dcnv4.py, each in bf16 and fp16.
Arms, per workload and dtype, median ms of the forward (no autograd) and of forward + backward (the gradients of input
and offset / mask, or offset_mask):
  half_core   the core on the half tensors (dcnv{3,4}_{fwd,bwd}_kernel_bf16 / _f16)
  cast_fp32   what the DCNv3 / DCNv4 modules did on half tensors before: .float() copies, the float32 core, then
              .to(dtype) of the output
Also per arm: the kernels' times from a separate dcn_profile_* pass of forward + backward, the peak memory of forward +
backward (torch.cuda.max_memory_allocated after a reset, with the inputs already allocated), and the largest output
difference between the arms (0 expected: the half kernels are the float32 kernels on widened operands, rounded once).
Each kernel's HBM-floor share is its compulsory bytes, with 2-byte operands and the float32 grad_input, over 7.7 TB/s,
divided by its measured time.  The card's name and power limit are read in the same run and written beside the
numbers.
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
from tools import bench_dcnv3, bench_dcnv4  # noqa: E402
from tools.bench_msda import card, timed  # noqa: E402

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}


def workloads():
    """name -> (family, N, H, W, C, G, kernel, remove_center, floats per pixel of the offset tensors)."""
    out = {}
    for name, (N, H, W, C, G) in bench_dcnv3.WORKLOADS.items():
        k = bench_dcnv3.K
        out["v3_" + name] = ("v3", N, H, W, C, G, k, False, G * k * k * 3)
    for name, (N, H, W, C, G, k, rc) in bench_dcnv4.WORKLOADS.items():
        out["v4_" + name] = ("v4", N, H, W, C, G, k, rc, dcn.dcnv4_row_floats(k, k, G, rc))
    return out


def compulsory_bytes(N, H, W, C, Co, elem):
    """Bytes each kernel must move at least once (Ho = H, Wo = W): input, the offset tensors (Co elements per pixel),
    out, grad_out, grad_offset tensors at `elem` bytes; grad_input float32, read and written once."""
    x, o, gx = N * H * W * C * elem, N * H * W * Co * elem, N * H * W * C * 4
    fwd = x + o + x                     # read input, offsets; write out
    bwd = x + o + x + 2 * gx + o        # read input, offsets, grad_out; grad_input RMW; write the offsets' gradient
    return fwd, bwd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the arms per workload")
    ap.add_argument("--workloads", default=",".join(workloads()))
    ap.add_argument("--dtypes", default=",".join(DTYPES))
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: these are GPU timings")
    torch.manual_seed(0)
    res = {"card": card(),
           "method": f"median of {args.steps} CUDA-event timed calls after {args.warmup} warm-up calls, "
                     f"{args.rounds} alternating rounds per arm (median over rounds); stride 1, pad kernel // 2, "
                     "offset_scale 1; DCNv3 with the mask softmax fused; cast_fp32 includes its casts",
           "peak_memory_note": "max_memory_allocated during one forward + backward, minus what was allocated before it",
           "hbm_floor_note": "hbm_floor_share = compulsory bytes / 7.7e12 B/s / kernel time; compulsory bytes: 2-byte "
                             "input, offsets, out, grad_out and offsets' gradient, float32 grad_input read and "
                             "written once",
           "workloads": {}}
    table = workloads()
    for name in args.workloads.split(","):
        fam, N, H, W, C, G, k, rc, Co = table[name]
        Gc = C // G
        geo = (k, k, 1, 1, k // 2, k // 2, 1, 1, G, Gc, 1.0)
        for dname in args.dtypes.split(","):
            dtype = DTYPES[dname]
            x = torch.randn(N, H, W, C, device="cuda").to(dtype)
            gout = torch.randn(N, H, W, C, device="cuda").to(dtype)
            if fam == "v3":
                P = k * k
                offs = [torch.randn(N, H, W, G * P * 2, device="cuda").to(dtype),
                        torch.randn(N, H, W, G * P, device="cuda").to(dtype)]

                def core(*t):
                    return dcn.dcnv3_core(*t, *geo, softmax_mask=True)
            else:
                offs = [torch.randn(N, H, W, Co, device="cuda").to(dtype)]

                def core(*t):
                    return dcn.dcnv4_core(*t, *geo, remove_center=rc)

            def cast_fp32(*t):
                return core(*(a.float() for a in t)).to(dtype)

            leaves = [t.clone().requires_grad_(True) for t in [x] + offs]
            arms = {}
            for arm, f in (("half_core", core), ("cast_fp32", cast_fp32)):
                def fwd(f=f):
                    with torch.no_grad():
                        f(x, *offs)

                def fwd_bwd(f=f):
                    torch.autograd.grad(f(*leaves), leaves, gout)

                arms[arm + "_fwd"], arms[arm + "_fwd_bwd"] = fwd, fwd_bwd
            entry = {"shape": dict(family=fam, dtype=dname, N=N, H=H, W=W, C=C, G=G, Gc=Gc, kernel=k,
                                   remove_center=rc, offset_elements_per_pixel=Co)}
            with torch.no_grad():
                entry["max_abs_diff_half_core_vs_cast_fp32_fwd"] = float(
                    (core(x, *offs).float() - cast_fp32(x, *offs).float()).abs().max())
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
            for p in ("fwd", "fwd_bwd"):
                entry[f"cast_fp32_over_half_core_{p}"] = entry[f"cast_fp32_{p}_ms"] / entry[f"half_core_{p}_ms"]
            for arm in ("half_core", "cast_fp32"):
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                arms[arm + "_fwd_bwd"]()
                torch.cuda.synchronize()
                entry[f"{arm}_peak_bytes_fwd_bwd"] = torch.cuda.max_memory_allocated() - base
                _lib.profile_begin()    # per-kernel times: a separate pass, the event profiler adds host work
                for _ in range(args.steps):
                    arms[arm + "_fwd_bwd"]()
                torch.cuda.synchronize()
                prof = _lib.profile_end()
                entry[f"{arm}_kernels_ms_per_call"] = {kn: v[1] / v[0] for kn, v in prof.items()}
            entry["peak_bytes_saved_fwd_bwd"] = (entry["cast_fp32_peak_bytes_fwd_bwd"]
                                                 - entry["half_core_peak_bytes_fwd_bwd"])
            fwd_b, bwd_b = compulsory_bytes(N, H, W, C, Co, 2)
            sfx = "_bf16" if dtype == torch.bfloat16 else "_f16"
            kf, kb = f"dcnv{fam[1]}_fwd_kernel{sfx}", f"dcnv{fam[1]}_bwd_kernel{sfx}"
            entry["compulsory_bytes"] = {kf: fwd_b, kb: bwd_b}
            entry["hbm_floor_share"] = {}
            for kn, b in entry["compulsory_bytes"].items():
                t = entry["half_core_kernels_ms_per_call"].get(kn)
                if t:
                    entry["hbm_floor_share"][kn] = b / HBM_BYTES_PER_S / (t * 1e-3)
            res["workloads"][f"{name}_{dname}"] = entry
            print(json.dumps({f"{name}_{dname}": entry}), flush=True)
            del x, gout, offs, leaves, arms
            torch.cuda.empty_cache()
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
