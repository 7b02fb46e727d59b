"""The whole modulated layer (ModulatedDeformConv2dPack) as one engine node against the two-node composition.

    python tools/bench_modulated_layer.py [--steps 10] [--warmup 3] [--rounds 3] [--out profiles/r3_bench_modulated_layer.json]

Arms, per shape, median ms of the forward (no autograd) and of forward + backward:
  one_node      ModulatedDeformConv2dPack on the engine's layer path (offset-and-mask conv, sigmoid, modulated span)
  two_node      the same module with engine_offset_conv = False: framework conv + chunk / cat / sigmoid + the engine's
                modulated span (the framework's default cuDNN settings; cudnn.allow_tf32 is recorded)
  torchvision   framework conv + chunk / cat / sigmoid + torchvision.ops.deform_conv2d(mask=), where this torchvision
                build has a CUDA kernel
Shapes: those of tools/bench_modulated.py, all in fp32 (the layer path's operand mode).  CUDA events around each call
after warm-up; the arms alternate in rounds in the same process.  The card's name and power limit are read in the same
run and written beside the numbers.
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import jittor_dcn_b200 as dcn  # noqa: E402

SHAPES = {
    #  name    B    C    O    H
    "cfg2": (256, 64, 64, 128),
    "c3":   (128, 128, 128, 56),
    "c4":   (128, 256, 256, 28),
    "c5":   (128, 512, 512, 14),
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


def tv_layer(m):
    from torchvision.ops import deform_conv2d

    def run(x):
        o1, o2, ml = torch.chunk(m.conv_offset(x), 3, dim=1)
        return deform_conv2d(x, torch.cat((o1, o2), dim=1), m.weight, m.bias, m.stride, m.padding,
                             mask=torch.sigmoid(ml))
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the arms per shape")
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: these are GPU timings")
    torch.manual_seed(0)
    res = {"card": card(),
           "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
           "note": "two_node and torchvision run the framework convolution with the framework's default settings",
           "method": f"median of {args.steps} CUDA-event timed calls after {args.warmup} warm-up calls, "
                     f"{args.rounds} alternating rounds per arm (median over rounds); fp32",
           "shapes": {}}
    for name in args.shapes.split(","):
        B, C, O, H = SHAPES[name]
        one = dcn.ModulatedDeformConv2dPack(C, O, 3, padding=1).cuda()
        with torch.no_grad():
            one.conv_offset.weight.normal_(0.0, 0.5 / (C * 9) ** 0.5)
            one.conv_offset.bias.uniform_(-0.5, 0.5)
        two = copy.deepcopy(one)
        two.engine_offset_conv = False
        x = torch.randn(B, C, H, H, device="cuda").requires_grad_(True)
        gout = torch.randn(B, O, H, H, device="cuda")
        layers = {"one_node": one, "two_node": two}
        entry = res["shapes"].setdefault(name, {})
        entry["shape"] = dict(B=B, C=C, O=O, H=H, W=H, k=3, s=1, p=1, operand="fp32")
        entry["layer_path"] = one._whole_layer_on_engine(x)
        try:
            run = tv_layer(two)
            run(x[:1].detach())
            layers["torchvision"] = run
        except (RuntimeError, NotImplementedError) as e:
            entry["torchvision"] = f"not available: {e}"

        def fwd(f):
            def go():
                with torch.no_grad():
                    f(x)
            return go

        def fwd_bwd(f, params):
            def go():
                torch.autograd.grad(f(x), [x] + params, gout)
            return go

        arms = {}
        for k, f in layers.items():
            params = list((two if k == "torchvision" else f).parameters())
            arms[k + "_fwd"] = fwd(f)
            arms[k + "_fwd_bwd"] = fwd_bwd(f, params)
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        rounds = {k: [] for k in arms}
        for _ in range(args.rounds):
            for k, fn in arms.items():
                rounds[k].append(timed(fn, args.steps))
        for k, v in rounds.items():
            entry[k + "_ms"] = sorted(v)[len(v) // 2]
        for k in ("fwd", "fwd_bwd"):
            entry[f"two_node_over_one_node_{k}"] = entry[f"two_node_{k}_ms"] / entry[f"one_node_{k}_ms"]
        print(json.dumps({name: entry}), flush=True)
        del one, two, x, gout, layers, arms
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
