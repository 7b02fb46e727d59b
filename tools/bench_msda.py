"""Multi-scale deformable attention (csrc/dcn_msda.cu) against Deformable DETR's grid_sample composition.

    python tools/bench_msda.py [--steps 20] [--warmup 3] [--rounds 3] [--out profiles/r3_bench_msda.json]

Arms, per workload, median ms of the forward (no autograd) and of forward + backward (the gradients of value,
sampling_locations and attention_weights):
  engine        ms_deform_attn (msda_fwd_kernel / msda_bwd_kernel)
  composition   ms_deform_attn_core_pytorch (F.grid_sample per level, fp32) on the same GPU — the only GPU yardstick
                that builds offline; the Deformable DETR / mmcv CUDA extensions are not built for sm_100a
Workloads, fp32, M = 8 heads of D = 32 channels: the encoder of Deformable DETR on an 800 x 1333 image (strides 8-64),
DINO's decoder (900 queries) on the same value tensor, and Mask2Former's pixel decoder (3 levels, batch 8).  Locations
are reference points plus offsets of about 2 px on each level; weights are a softmax of normal draws.  CUDA events
around each call after warm-up; the arms alternate in rounds in one process.  Kernel times come from a separate
dcn_profile_* pass.  The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import jittor_dcn_b200 as dcn  # noqa: E402
from jittor_dcn_b200 import _lib  # noqa: E402
from oracle.msda_reference import level_start_index_of, ms_deform_attn_core_pytorch  # noqa: E402

DETR_LEVELS = ((100, 167), (50, 84), (25, 42), (13, 21))
WORKLOADS = {
    #  name          B  levels                               Q (None: = S)  P
    "detr_enc":   (4, DETR_LEVELS, None, 4),
    "dino_dec":   (4, DETR_LEVELS, 900, 4),
    "m2f_pixdec": (8, ((64, 128), (32, 64), (16, 32)), None, 4),
}
M, D = 8, 32
RED_RATE = 1.5e12   # measured coalesced red.global.add rate, L2-resident target (profiles/r2_red_probe.txt)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (v.strip() for v in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:   # the numbers stay usable; say why the card is unknown
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unavailable ({e})"}


def timed(fn, steps):
    ms = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    return ms[len(ms) // 2]


def inputs(B, levels, Q, P):
    L = len(levels)
    ss = torch.tensor(levels, dtype=torch.int64)
    S = int(ss.prod(1).sum())
    Q = S if Q is None else Q
    value = torch.randn(B, S, M, D, device="cuda")
    ref = torch.rand(B, Q, 1, L, 1, 2, device="cuda")
    wh = ss.flip(1).to("cuda", torch.float32)[None, None, None, :, None, :]     # (W_l, H_l)
    loc = ref + 2.0 * torch.randn(B, Q, M, L, P, 2, device="cuda") / wh
    aw = torch.randn(B, Q, M, L * P, device="cuda").softmax(-1).view(B, Q, M, L, P)
    return value, ss.cuda(), level_start_index_of(ss).cuda(), loc, aw, torch.randn(B, Q, M * D, device="cuda")


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
                     f"{args.rounds} alternating rounds per arm (median over rounds); fp32; M = {M}, D = {D}",
           "red_floor_note": "grad_value_red_floor_ms = B*Q*M*L*P*4*D adds at the measured 1.5e12 adds/s L2 atomic "
                             "rate: an estimate from shapes, not measured",
           "workloads": {}}
    for name in args.workloads.split(","):
        B, levels, Q, P = WORKLOADS[name]
        value, ss, lsi, loc, aw, gout = inputs(B, levels, Q, P)
        S, Q, L = value.shape[1], loc.shape[1], len(levels)
        shapes = [tuple(v) for v in levels]
        vr, lr, ar = (t.clone().requires_grad_(True) for t in (value, loc, aw))

        def engine_fwd():
            with torch.no_grad():
                dcn.ms_deform_attn(value, ss, lsi, loc, aw)

        def engine_fwd_bwd():
            torch.autograd.grad(dcn.ms_deform_attn(vr, ss, lsi, lr, ar), [vr, lr, ar], gout)

        def comp_fwd():
            with torch.no_grad():
                ms_deform_attn_core_pytorch(value, shapes, loc, aw)

        def comp_fwd_bwd():
            torch.autograd.grad(ms_deform_attn_core_pytorch(vr, shapes, lr, ar), [vr, lr, ar], gout)

        arms = {"engine_fwd": engine_fwd, "engine_fwd_bwd": engine_fwd_bwd,
                "composition_fwd": comp_fwd, "composition_fwd_bwd": comp_fwd_bwd}
        # same results first: the composition in fp32 on the GPU against the engine
        with torch.no_grad():
            diff = float((dcn.ms_deform_attn(value, ss, lsi, loc, aw) -
                          ms_deform_attn_core_pytorch(value, shapes, loc, aw)).abs().max())
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        rounds = {k: [] for k in arms}
        for _ in range(args.rounds):
            for k, fn in arms.items():
                rounds[k].append(timed(fn, args.steps))
        entry = {"shape": dict(B=B, S=S, Q=Q, M=M, D=D, L=L, P=P, levels=shapes),
                 "max_abs_diff_engine_vs_composition_fwd": diff}
        for k, v in rounds.items():
            entry[k + "_ms"] = sorted(v)[len(v) // 2]
        for k in ("fwd", "fwd_bwd"):
            entry[f"composition_over_engine_{k}"] = entry[f"composition_{k}_ms"] / entry[f"engine_{k}_ms"]
        # per-kernel times (a separate pass: the event profiler adds host work)
        _lib.profile_begin()
        for _ in range(args.steps):
            engine_fwd_bwd()
        torch.cuda.synchronize()
        prof = _lib.profile_end()
        entry["kernels_ms_per_call"] = {k: v[1] / v[0] for k, v in prof.items()}
        reds = B * Q * M * L * P * 4 * D
        entry["grad_value_red_count"] = reds
        entry["grad_value_red_floor_ms"] = reds / RED_RATE * 1e3
        entry["grad_value_bytes"] = B * S * M * D * 4
        fwd_bytes = 4 * (B * S * M * D + B * Q * M * L * P * 3 + B * Q * M * D)
        entry["fwd_algorithmic_hbm_bytes"] = fwd_bytes
        fk = entry["kernels_ms_per_call"].get("msda_fwd_kernel")
        if fk:
            entry["fwd_kernel_algorithmic_GBps"] = fwd_bytes / (fk * 1e-3) / 1e9
        res["workloads"][name] = entry
        print(json.dumps({name: entry}), flush=True)
        del value, loc, aw, gout, vr, lr, ar, arms
        torch.cuda.empty_cache()
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
