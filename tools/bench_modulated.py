"""Modulated (DCNv2) against unmodulated DCNv1 on the engine, and torchvision's CUDA deform_conv2d(mask=) as a yardstick.

    python tools/bench_modulated.py [--steps 20] [--warmup 5] [--out profiles/bench_modulated.json]

Per shape: median ms of fwd+bwd and of the forward alone, CUDA events around each call after warm-up, unmodulated and
modulated calls alternating in the same process.  Shapes: the cfg2 shape in DCNv1 mode (fp32) and the ResNet-50 C3 / C4
/ C5 layers at batch 128 with bf16 operands (ResNet-DCNv2 backbones); torchvision on the cfg2 and C4 shapes (fp32,
its only mode).  The card's name and power limit are read in the same run and written beside the numbers.
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
from jittor_dcn_b200.functional import dcn_backward_modulated, dcn_forward_modulated  # noqa: E402

SHAPES = {
    #  name              B    C    O    H    operand           torchvision yardstick
    "cfg2_dcnv1_fp32": (256, 64, 64, 128, dcn.OPERAND_FP32, True),
    "c3_bf16":         (128, 128, 128, 56, dcn.OPERAND_BF16, False),
    "c4_bf16":         (128, 256, 256, 28, dcn.OPERAND_BF16, True),
    "c5_bf16":         (128, 512, 512, 14, dcn.OPERAND_BF16, False),
}


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of unmodulated / modulated per shape")
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: these are GPU timings")
    torch.manual_seed(0)
    res = {"card": card(), "method": f"median of {args.steps} CUDA-event timed calls after {args.warmup} warm-up "
                                     f"calls, {args.rounds} alternating rounds per arm (median over rounds)",
           "shapes": {}}
    for name, (B, C, O, H, operand, tv) in SHAPES.items():
        act = torch.bfloat16 if operand == dcn.OPERAND_BF16 else torch.float32
        x = torch.randn(B, C, H, H, device="cuda").to(act)
        off = torch.randn(B, 18, H, H, device="cuda")
        mask = torch.sigmoid(torch.randn(B, 9, H, H, device="cuda"))
        w = (torch.randn(O, C, 3, 3, device="cuda") * (2.0 / (C * 9)) ** 0.5).to(act)
        b = torch.randn(O, device="cuda")
        gout = torch.randn(B, O, H, H, device="cuda").to(act)
        arms = {
            "unmodulated_fwd": lambda: dcn.dcn_forward(x, off, w, b, 3, 1, 1, dcn.VARIANT_DCNV1, operand),
            "modulated_fwd": lambda: dcn_forward_modulated(x, off, mask, w, b, 3, 1, 1, operand),
            "unmodulated_fwd_bwd": lambda: (dcn.dcn_forward(x, off, w, b, 3, 1, 1, dcn.VARIANT_DCNV1, operand),
                                            dcn.dcn_backward(x, off, w, gout, True, 3, 1, 1, dcn.VARIANT_DCNV1,
                                                             operand)),
            "modulated_fwd_bwd": lambda: (dcn_forward_modulated(x, off, mask, w, b, 3, 1, 1, operand),
                                          dcn_backward_modulated(x, off, mask, w, gout, True, 3, 1, 1, operand)),
        }
        if tv:
            from torchvision.ops import deform_conv2d
            xf, wf = x.float().requires_grad_(True), w.float().requires_grad_(True)
            offg, maskg, bg = off.clone().requires_grad_(True), mask.clone().requires_grad_(True), b.clone().requires_grad_(True)
            goutf = gout.float()
            try:
                deform_conv2d(xf[:1], offg[:1], wf, bg, padding=1, mask=maskg[:1])

                def tv_fwd():
                    with torch.no_grad():
                        return deform_conv2d(xf, offg, wf, bg, padding=1, mask=maskg)

                def tv_fwd_bwd():
                    o = deform_conv2d(xf, offg, wf, bg, padding=1, mask=maskg)
                    return torch.autograd.grad(o, [xf, offg, maskg, wf, bg], goutf)

                arms["torchvision_cuda_fwd"] = tv_fwd
                arms["torchvision_cuda_fwd_bwd"] = tv_fwd_bwd
            except (RuntimeError, NotImplementedError) as e:
                res["shapes"].setdefault(name, {})["torchvision_cuda"] = f"not available: {e}"
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        rounds = {k: [] for k in arms}
        for _ in range(args.rounds):
            for k, fn in arms.items():
                rounds[k].append(timed(fn, args.steps))
        entry = res["shapes"].setdefault(name, {})
        entry["shape"] = dict(B=B, C=C, O=O, H=H, W=H, k=3, s=1, p=1,
                              operand="bf16" if operand == dcn.OPERAND_BF16 else "fp32")
        entry["path"] = [dcn._lib.path_name(dcn.make_shape(B, C, O, H, H, 3, 1, 1, dcn.VARIANT_DCNV1, operand), ph)
                         for ph in (0, 1)]
        for k, v in rounds.items():
            entry[k + "_ms"] = sorted(v)[len(v) // 2]
        entry["modulated_over_unmodulated_fwd_bwd"] = entry["modulated_fwd_bwd_ms"] / entry["unmodulated_fwd_bwd_ms"]
        entry["modulated_over_unmodulated_fwd"] = entry["modulated_fwd_ms"] / entry["unmodulated_fwd_ms"]
        del x, off, mask, w, b, gout, arms
        dcn.clear_workspaces()
        torch.cuda.empty_cache()
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
