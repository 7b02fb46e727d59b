#!/usr/bin/env python
"""bench.py — DeformConv2d fwd+bwd images/sec on B200 (the metric of BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2|cfg3|det2|det5]
                    [--variant torch|jittor] [--impl ours|reference] [--dump-outputs DIR]
    torchrun ... bench.py --gpus N ...            (N > 1, one rank per GPU, NCCL)

A "step" is one pass of the hot path (engine forward + backward through the C ABI,
dcn_forward + dcn_backward, offsets supplied) over one batch of synthetic input.  At N > 1
every rank works on its own batch of the same size (weak scaling along the batch dimension,
the only natural sharding — SURVEY.md 8e) and the step ends with ONE all-reduce of the flat
weight/bias/offset-conv gradient bucket.

JSON keys (one line, rank 0): see the task contract; `value` = device-resident inputs,
`e2e` = the same metric through the module API (`TorchDeformConv2d.forward/backward`) with
HOST input buffers (pinned H2D of x every step, D2H of the parameter gradients),
`roofline` = dominant kernel against MEASURED_PEAKS.json, `cpu_baseline` = the reference's op
chain (oracle/torch_chain.py, same torch CPU kernels as the reference) on this host's cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (description, B per GPU, C, O, H, W, k, s, p)
    "cfg2": ("DeformConv2d 64->64 3x3 s1 p1, 128x128, batch 256 per GPU (BASELINE configs[1] shape), fwd+bwd",
             256, 64, 64, 128, 128, 3, 1, 1),
    "cfg3": ("DeformConv2d 256->256 3x3 s1 p1, 28x28, batch 64 per GPU (BASELINE configs[2]), fwd+bwd",
             64, 256, 256, 28, 28, 3, 1, 1),
    "det2": ("detector conv2 16->32 3x3 s2 p1, 128x128, batch 1024 per GPU (BASELINE configs[4] layer), fwd+bwd",
             1024, 16, 32, 128, 128, 3, 2, 1),
    "det3": ("detector conv3 32->64 3x3 s2 p1, 64x64, batch 1024 per GPU (BASELINE configs[4] layer), fwd+bwd",
             1024, 32, 64, 64, 64, 3, 2, 1),
    "det4": ("detector conv4 64->128 3x3 s2 p1, 32x32, batch 1024 per GPU (BASELINE configs[4] layer), fwd+bwd",
             1024, 64, 128, 32, 32, 3, 2, 1),
    "det5": ("detector conv5 128->256 3x3 s2 p1, 16x16, batch 1024 per GPU (BASELINE configs[4] layer), fwd+bwd",
             1024, 128, 256, 16, 16, 3, 2, 1),
    "c3": ("ResNet-50 C3 DCN layer 128->128 3x3 s1 p1, 56x56, batch 128 per GPU (BASELINE configs[3] layer), fwd+bwd",
           128, 128, 128, 56, 56, 3, 1, 1),
    "c4": ("ResNet-50 C4 DCN layer 256->256 3x3 s1 p1, 28x28, batch 128 per GPU (BASELINE configs[3] layer), fwd+bwd",
           128, 256, 256, 28, 28, 3, 1, 1),
    "c5": ("ResNet-50 C5 DCN layer 512->512 3x3 s1 p1, 14x14, batch 128 per GPU (BASELINE configs[3] layer; O = 512 "
           "runs as two output-channel groups), fwd+bwd",
           128, 512, 512, 14, 14, 3, 1, 1),
}
# BASELINE configs[3]: the 13 DCN layers of ResNet-50's C3-C5 stages (SURVEY 8d config 4), interleaved so that no
# layer finds its own inputs still in L2
STACK_ORDER = ["c3", "c4", "c5", "c4", "c3", "c4", "c5", "c4", "c3", "c4", "c5", "c4", "c3"]
STACK_DESC = ("stack: DCN ResNet-50 C3-C5 stage stack, 13 independent DeformConv2d layers fwd+bwd (4x 128->128 @56x56, "
              "6x 256->256 @28x28, 3x 512->512 @14x14), batch 128 per GPU (BASELINE configs[3])")
# BASELINE configs[4]: whole toy-detector training step, global batch 1024 sharded over the GPUs
DETECTOR_DESC = ("detector: data-parallel DCN detector training step (train.py:142-175 topology, 4 DeformConv2d "
                 "layers), 1x128x128 synthetic canvases, global batch 1024 sharded over the GPUs, Adam, one "
                 "gradient all-reduce (BASELINE configs[4])")


_JSON_OUT = None


def claim_stdout():
    """stdout carries exactly ONE JSON line: everything else that libraries write to file descriptor 1 (NCCL prints its
    version banner there) is sent to stderr; the JSON line goes to the original descriptor."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS) + ["detector", "stack"])
    ap.add_argument("--global-batch", type=int, default=1024, help="detector workload: global batch")
    ap.add_argument("--variant", default="torch", choices=["torch", "jittor"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--operand", default="fp32", choices=["fp32", "bf16"],
                    help="fp32 (reference parity, bf16 hi/lo split on the tensor cores) or bf16 storage of "
                         "x / weight / grad_out with fp32 accumulation (BASELINE configs[3])")
    ap.add_argument("--offset-sigma", type=float, default=2.0,
                    help="std (pixels) of the synthetic live offsets (SURVEY 8d)")
    ap.add_argument("--scope", default="span", choices=["span", "layer"],
                    help="single-layer workloads: 'span' = dcn_forward + dcn_backward with offsets supplied "
                         "(deform_conv.py:62-81 / train.py:102-140); 'layer' = the whole module on the engine, companion "
                         "offset conv included (dcn_layer_forward + dcn_layer_backward, SURVEY 8f.1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--force-simt", action="store_true")
    ap.add_argument("--no-graph", action="store_true",
                    help="detector workload: launch the training step eagerly instead of replaying its CUDA graph")
    ap.add_argument("--nccl-allreduce", action="store_true",
                    help="detector workload: exchange the gradient bucket with dcn_allreduce_sum_f32 (NCCL, eager "
                         "launches) instead of the one-kernel peer-memory all-reduce inside the step's CUDA graph")
    ap.add_argument("--no-detector-dp", action="store_true",
                    help="default workload: skip the extra detector_dp measurement (BASELINE configs[4])")
    ap.add_argument("--nchw-between-layers", action="store_true",
                    help="detector workload: keep NCHW activations between the DCN layers (round-1 data flow) instead of the "
                         "channels-last hand-over between every post-op and the next layer (SURVEY 8f.2)")
    ap.add_argument("--stock-bn", action="store_true",
                    help="detector workload: the framework's BatchNorm2d + ReLU instead of the engine's fused post-op")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="single-layer workloads: write what the last timed step computed on rank 0 (output and "
                         "gradients) as DIR/<name>.npy in float32, at most 64 MB in all: a larger array as a fixed, seeded "
                         "sample of its elements")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BUDGET_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays):
    """Writes each tensor of `arrays` ({name: tensor}) as out_dir/<name>.npy in float32.  Every file gets an equal share
    of DUMP_BUDGET_BYTES; an array larger than its share is stored as a fixed sample, the flattened array's elements at
    sorted(numpy.random.default_rng(0).choice(numel, share, replace=False)), so that runs with the same arguments store
    the same positions and two builds can be compared element for element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = (DUMP_BUDGET_BYTES // len(arrays) - 256) // 4          # elements; 256 bytes per file for the .npy header
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > share:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), share, replace=False))
            t = t.reshape(-1)[torch.as_tensor(idx, device=t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], bf16_burst=p["bf16_tflops"], bf16_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "samples": len(sm),
                "reasons": sorted(reasons)}


def layer_bytes_flops(B, C, O, H, W, Ho, Wo, N, act_bytes=4):
    """Algorithmic work (SURVEY.md 8d), per launch of each role; act_bytes = 2 in bf16 operand mode
    for x, weight and grad_out (out and all gradients stay float32)."""
    K = C * N
    x, off, out, wgt = act_bytes * B * C * H * W, 4 * B * 2 * N * Ho * Wo, 4 * B * O * Ho * Wo, act_bytes * O * K
    flops = 2.0 * B * Ho * Wo * K * O
    return {
        "fwd": dict(bytes=x + off + out + wgt, flops=flops),
        "bwd_data": dict(bytes=out + x + off + wgt + x + off, flops=flops),   # read gout,x,off,W; write gx,goff
        "bwd_weight": dict(bytes=out + x + off + wgt, flops=flops),           # read gout,x,off; write gW
        "bwd": dict(bytes=out + 2 * x + 2 * off + 2 * wgt, flops=2 * flops),  # SURVEY 8d backward total
    }


KERNEL_ROLE = {"fwd_kernel": "fwd", "bwd_data_kernel": "bwd_data", "bwd_weight_kernel": "bwd_weight",
               "umma_fwd_kernel": "fwd", "umma_bwd_data_kernel": "bwd_data",
               "umma_bwd_weight_kernel": "bwd_weight"}


def cpu_reference_step(wl, variant, micro_b, with_offset_conv, seed=0):
    """One fwd+bwd of the reference's op chain on `micro_b` samples; returns a callable."""
    import torch
    from oracle import torch_chain
    _, B, C, O, H, W, k, s, p = wl
    torch.manual_seed(seed)
    layer = torch_chain.ChainLayer(C, O, k, s, p, True, variant)
    with torch.no_grad():
        layer.weight.normal_(0, (2.0 / (C * k * k)) ** 0.5)
        layer.offset_conv.weight.normal_(0, 0.01)
        layer.offset_conv.bias.normal_(0, 1.0)
    x = torch.randn(micro_b, C, H, W)
    Ho, Wo = torch_chain.out_hw(H, W, k, s, p)
    gout = torch.randn(micro_b, O, Ho, Wo)
    off = torch.randn(micro_b, 2 * k * k, Ho, Wo) * 2.0

    def step_layer():
        xi = x.clone().requires_grad_(True)
        out = layer(xi)
        out.backward(gout)
        layer.zero_grad(set_to_none=True)

    def step_span():
        torch_chain.chain_forward_backward(x, off, layer.weight, layer.bias, gout, variant=variant,
                                           kernel_size=k, stride=s, padding=p)

    return step_layer if with_offset_conv else step_span


def time_cpu(fn, budget_s, min_runs=2, max_runs=7):
    fn()  # warm-up
    times, t_all = [], time.perf_counter()
    while len(times) < min_runs or (len(times) < max_runs and time.perf_counter() - t_all < budget_s):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return statistics.median(times), len(times)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on this box's host
    cores.  /root/reference cannot travel, so this is its op chain restated with the same
    torch CPU kernels (oracle/torch_chain.py; pinned bit-for-bit to the unmodified reference
    in tests/test_oracle_golden.py): kind = "port"."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    wl = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    micro_b = 8 if args.workload in ("cfg2",) else 16
    step = cpu_reference_step(wl, args.variant, micro_b, with_offset_conv=True)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    n = 0
    # bounded: K steps, but never more than ~150 s in total
    while n < args.steps and (n < 2 or time.perf_counter() - t0 < 150):
        step()
        n += 1
    dt = (time.perf_counter() - t0) / n
    value = micro_b / dt
    sample = f"{n} steps of {micro_b} samples (micro-batch of the {wl[1]}-sample workload; samples are independent)"
    line = {
        "impl": "reference", "metric": "DeformConv2d fwd+bwd images/sec", "value": value, "unit": "images/s",
        "n_gpus": args.gpus, "steps": n, "warmup": min(args.warmup, 2), "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": args.workload + ": " + wl[0], "variant": args.variant,
                                        "cpu_micro_batch": micro_b, "includes_offset_conv": True},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def measure_detector(args, world, rank, local_rank, dev, steps, warmup, want_e2e=True, sample_clocks=True):
    """BASELINE configs[4]: the reference's toy detector (4 DCN layers on the engine — offset conv included —, relu(bn(x))
    on the engine, the rest stock torch CUDA ops) trained data-parallel: global batch sharded over the ranks (STRONG
    scaling), Adam lr 1e-3 wd 1e-4, loss CE + 5*smoothL1 (train.py:187-199,247), ONE all-reduce of the flat
    435,862-float gradient bucket.  The exchange is the engine's one-kernel peer-memory all-reduce (dcn_p2p_*), which a
    CUDA graph can record, so the WHOLE step — forward, backward, exchange, Adam — is replayed as one graph at every
    N.  The process group must already exist for world > 1.  Returns a dict (rank 0: complete; others: timing only)."""
    import torch
    import torch.distributed as dist
    import jittor_dcn_b200 as dcn
    from jittor_dcn_b200 import _lib, dp
    from jittor_dcn_b200.detector import EDNetDetection, detection_loss, synthetic_canvases

    lib = dcn.load()
    b0, b1 = dp.shard_range(args.global_batch, rank, world)
    B = b1 - b0
    torch.manual_seed(0)                                   # replicated weights
    cls = dcn.TorchDeformConv2d if args.variant == "torch" else dcn.TorchDeformConv2dJittorSemantics
    model = EDNetDetection(dcn_cls=cls, fused_bn_relu=not args.stock_bn,
                           channels_last=not args.nchw_between_layers and not args.stock_bn).to(dev)
    with torch.no_grad():                                  # live offsets (the reference starts at zero)
        for m in model.modules():
            if isinstance(m, dcn.TorchDeformConv2d):
                m.offset_conv.weight.normal_(0, 0.01)
                m.offset_conv.bias.normal_(0, 1.0)
    use_graph = not args.no_graph
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-4, capturable=use_graph)
    x, labels, boxes = synthetic_canvases(B, torch.Generator().manual_seed(100 + rank), dev)
    x_host = x.cpu().pin_memory()
    bucket = dp.GradBucket(model.parameters())
    comm, comm_kind = None, "none"
    if world > 1:
        if args.nccl_allreduce:
            comm = dp.DcnComm(rank, world, dev)
            comm_kind = "dcn_allreduce_sum_f32 (NCCL, one flat bucket of %d floats)" % bucket.numel
            use_graph = False          # a captured NCCL collective hung on the 2-GPU box (round 1): eager launches
        else:
            comm = dp.DcnP2P(rank, world, dev, bucket.numel)
            comm_kind = ("dcn_p2p_allreduce_sum_f32 (ONE kernel over NVLink peer memory, one flat bucket of %d "
                         "floats; recorded in the step's CUDA graph)" % bucket.numel)
    weight = dp.shard_weight(args.global_batch, rank, world) if world > 1 else None
    stream = torch.cuda.current_stream(dev)

    def train_step():
        loss = detection_loss(*model(x), labels, boxes)
        loss.backward()
        if comm is not None:
            dp.allreduce_gradients(bucket, comm, weight=weight)
        opt.step()
        return loss

    def eager_step(from_host=False):
        if from_host:
            x.copy_(x_host, non_blocking=True)
        opt.zero_grad(set_to_none=True)
        return train_step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # Per-kernel table and launch count of ONE step, taken eagerly (a replayed graph launches the very same
    # kernels, but neither the library's launch counter nor its event pairs see a replay).
    for _ in range(3):
        eager_step()
    barrier()
    lib.dcn_launch_count_reset()
    _lib.profile_begin()
    eager_step()
    barrier()
    launches_per_step = int(lib.dcn_launch_count())
    prof = _lib.profile_end()

    # The step is launch-bound at small per-GPU batches (batch 16: ~150 launches for ~1 ms of kernels; 8 GPUs at
    # global batch 1024: 6.2 ms eager for 2.6 ms of kernels), so the whole training step is captured once and replayed;
    # inputs live in static buffers.  thread_local capture mode: torch's NCCL watchdog thread (the process group only
    # serves barriers / rendez-vous here) must not invalidate the capture.
    graph, graph_note, static_loss = None, "eager launches", None
    if use_graph:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(stream)
            with torch.cuda.stream(side):
                for _ in range(2):
                    eager_step()
            stream.wait_stream(side)
            barrier()
            opt.zero_grad(set_to_none=True)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                static_loss = train_step()
            graph_note = "whole training step%s replayed as one CUDA graph" % (
                " (gradient all-reduce included)" if comm is not None else "")
        except Exception as e:  # noqa: BLE001 - report and fall back to eager launches
            graph, graph_note = None, f"eager launches (graph capture failed: {type(e).__name__}: {e})"[:300]
            barrier()
            opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-4)

    def step(from_host=False):
        if graph is None:
            return eager_step(from_host)
        if from_host:
            x.copy_(x_host, non_blocking=True)
        graph.replay()
        return static_loss

    for _ in range(max(warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank) if (rank == 0 and sample_clocks) else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1) / steps
    clocks = sampler.stop() if sampler else None
    e2e_s = None
    if want_e2e:
        # e2e: canvases come from pinned host memory every step, the loss is read back
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            float(step(from_host=True).detach())
        barrier()
        e2e_s = (time.perf_counter() - t0) / steps
    if world > 1:
        t = torch.tensor([ms, e2e_s or 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(t[0]), (float(t[1]) if want_e2e else None)
    res = {
        "ms_per_step": ms, "images_per_s": args.global_batch / (ms * 1e-3), "batch_per_gpu": B,
        "launches_per_step": launches_per_step, "graph": graph is not None, "launch": graph_note,
        "allreduce": comm_kind, "bucket_floats": bucket.numel, "e2e_s": e2e_s, "clocks": clocks,
        "h2d_bytes_per_step": x_host.numel() * 4,
        "kernels": {k: {"launches": v[0], "avg_ms": v[1] / max(v[0], 1)} for k, v in prof.items()},
        "engine_ms_per_step": sum(v[1] for v in prof.values()),   # of the profiled eager step
    }
    del graph
    if comm is not None:
        barrier()
        comm.close()
    return res


def run_detector(args):
    """--workload detector: BASELINE configs[4] as its own bench line (see measure_detector)."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    r = measure_detector(args, world, rank, local_rank, dev, args.steps, args.warmup)
    if rank == 0:
        line = {
            "metric": "DeformConv2d fwd+bwd images/sec", "value": r["images_per_s"], "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": DETECTOR_DESC, "variant": args.variant, "global_batch": args.global_batch,
                       "batch_per_gpu": r["batch_per_gpu"], "parallelism": f"dp{world}",
                       "launch": r["launch"],
                       "post_op": ("framework BatchNorm2d + ReLU (cuDNN)" if args.stock_bn else
                                   "relu(bn(x)) on the engine (dcn_bn_relu_forward / _backward)" if args.nchw_between_layers
                                   else "relu(bn(x)) on the engine, writing the next DCN layer's staged channels-last input "
                                        "and reading its channels-last grad_x (dcn_bn_relu_*_staged): no layout pass "
                                        "between the layers"),
                       "allreduce": r["allreduce"],
                       "l2": "per-step activations (%.0f MB for conv2's input alone) exceed the 126 MB L2" %
                             (r["batch_per_gpu"] * 16 * 128 * 128 * 4 / 1e6)},
            "kernels": r["kernels"],
            "dcn_engine_ms_per_step": r["engine_ms_per_step"], "roofline": None, "cpu_baseline": None,
            "e2e": {"value": args.global_batch / r["e2e_s"], "unit": "images/s",
                    "h2d_bytes_per_step": r["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": 4, "ms_per_step": r["e2e_s"] * 1e3,
                    "api": "EDNetDetection (4 x jittor_dcn_b200.TorchDeformConv2d) train step"},
            "gpu_launches": r["launches_per_step"] * args.steps, "clocks": r["clocks"],
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_stack(args):
    """BASELINE configs[3]: every step runs the 13 layers of STACK_ORDER forward + backward through the C ABI
    (inputs resident in HBM); images/s = batch / time of the whole stack."""
    import ctypes

    import torch
    import torch.distributed as dist
    import jittor_dcn_b200 as dcn
    from jittor_dcn_b200 import _lib
    from jittor_dcn_b200.functional import staged_workspace

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    lib = dcn.load()
    variant = dcn.VARIANT_TORCH if args.variant == "torch" else dcn.VARIANT_JITTOR
    operand = dcn.OPERAND_BF16 if args.operand == "bf16" else dcn.OPERAND_FP32
    act = torch.bfloat16 if operand == dcn.OPERAND_BF16 else torch.float32
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    roles = ("fwd", "bwd_data", "bwd_weight", "bwd")
    layers, paths, work = {}, {}, {r: {"bytes": 0, "flops": 0} for r in roles}
    for name in sorted(set(STACK_ORDER)):
        _, B, C, O, H, W, k, s, p = WORKLOADS[name]
        N = k * k
        shp = dcn.make_shape(B, C, O, H, W, k, s, p, variant, operand=operand)
        Ho, Wo = _lib.output_hw(shp)
        x = torch.randn(B, C, H, W, device=dev, generator=gen).to(act)
        off = torch.randn(B, 2 * N, Ho, Wo, device=dev, generator=gen) * args.offset_sigma
        wt = (torch.randn(O, C, k, k, device=dev, generator=gen) * (2.0 / (C * N)) ** 0.5).to(act)
        bias = torch.randn(O, device=dev, generator=gen) * 0.1
        gout = torch.randn(B, O, Ho, Wo, device=dev, generator=gen).to(act)
        ws = staged_workspace(x, wt, k, s, p, variant, operand, 0)
        layers[name] = (x, off, wt, bias, gout, ws, (k, s, p))
        paths[name] = [lib.dcn_path_name(ctypes.byref(shp), ph).decode() for ph in (0, 1)]
        w1 = layer_bytes_flops(B, C, O, H, W, Ho, Wo, N, act_bytes=x.element_size())
        for ph in roles:
            for q in ("bytes", "flops"):
                work[ph][q] += w1[ph][q] * STACK_ORDER.count(name)
    B = WORKLOADS["c3"][1]
    stream = torch.cuda.current_stream(dev)

    def step():
        for name in STACK_ORDER:
            x, off, wt, bias, gout, ws, (k, s, p) = layers[name]
            dcn.dcn_forward(x, off, wt, bias, k, s, p, variant, operand=operand, ws=ws)
            dcn.dcn_backward(x, off, wt, gout, True, k, s, p, variant, operand=operand, ws=ws,
                             xt_staged=ws is not None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    lib.dcn_launch_count_reset()
    _lib.profile_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    launches = int(lib.dcn_launch_count())
    prof = _lib.profile_end()
    clocks = sampler.stop() if sampler else None
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    pk = peaks()
    kernels = {n: {"launches": c, "ms_per_step": tot / args.steps, "share": tot / max(elapsed_ms, 1e-9)}
               for n, (c, tot) in prof.items()}
    roofline = None
    ranked = sorted((n for n in prof if n in KERNEL_ROLE), key=lambda n: -prof[n][1])
    if ranked:
        top = ranked[0]
        role = KERNEL_ROLE[top]
        if top == "umma_bwd_data_kernel" and "umma_bwd_weight_kernel" not in prof and "bwd_weight_kernel" not in prof:
            role = "bwd"
        # all launches of the dominant kernel in one step, against the work of all 13 layers in that role
        tot_s = prof[top][1] / args.steps * 1e-3
        ach = work[role]["flops"] / tot_s / 1e12
        traffic, limiter = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            key = f"stack:{args.variant}:{args.operand}:{top}"
            traffic = tj.get(key)          # DRAM bytes of all launches of this kernel in one step (ncu --set full)
            limiter = tj.get("_limiter", {}).get(key)
        roofline = {"bound": "tensor", "achieved": ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                    "frac": ach / pk["bf16_sustained"], "traffic": traffic, "measured_limiter": limiter, "kernel": top,
                    "avg_ms": tot_s * 1e3 / len(STACK_ORDER), "peak_source": pk["source"],
                    "algorithmic_bytes": work[role]["bytes"], "algorithmic_flops": work[role]["flops"],
                    "note": "sum over the 13 layers' launches of this kernel in one step"}
    if rank == 0:
        emit({
            "metric": "DeformConv2d fwd+bwd images/sec", "value": world * B / (ms_per_step * 1e-3),
            "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if operand == dcn.OPERAND_BF16 else "f32", "data": "synthetic",
            "config": {"workload": STACK_DESC, "variant": args.variant, "operand": args.operand,
                       "batch_per_gpu": B, "global_batch": world * B, "offset_sigma_px": args.offset_sigma,
                       "paths_fwd_bwd": paths, "order": STACK_ORDER,
                       "l2": "layers interleaved; every layer's inputs are evicted by the others' traffic "
                             "(1.4 GB of operands per step)", "allreduce": "none", "parallelism": f"dp{world}"},
            "roofline": roofline, "kernels": kernels, "cpu_baseline": None, "e2e": None,
            "gpu_launches": launches, "clocks": clocks})
    if world > 1:
        dist.destroy_process_group()
    return 0


def measure_other_configs(args, dev, variant):
    """The other BASELINE configs next to the headline, so that the driver's default run sees them (N = 1 only):
    configs[2] (cfg3: 256 -> 256 @ 28 x 28, batch 64, fp32) and configs[3] (the 13-layer ResNet-50 C3-C5 stack, batch 128,
    bf16 operands), each fwd+bwd through the C ABI with inputs resident in HBM, W = 3 warm-up and K = 5 timed steps, an
    L2 flush (512 MB write) before every timed step.  Compact: images/s, ms/step, the dominant kernel and its share."""
    import torch
    import jittor_dcn_b200 as dcn
    from jittor_dcn_b200 import _lib
    from jittor_dcn_b200.functional import staged_workspace
    out = {}
    stream = torch.cuda.current_stream(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev).manual_seed(4321)

    def make(name, operand):
        _, B, C, O, H, W, k, s, p = WORKLOADS[name]
        act = torch.bfloat16 if operand == dcn.OPERAND_BF16 else torch.float32
        shp = dcn.make_shape(B, C, O, H, W, k, s, p, variant, operand=operand)
        Ho, Wo = _lib.output_hw(shp)
        x = torch.randn(B, C, H, W, device=dev, generator=gen).to(act)
        off = torch.randn(B, 2 * k * k, Ho, Wo, device=dev, generator=gen) * args.offset_sigma
        wt = (torch.randn(O, C, k, k, device=dev, generator=gen) * (2.0 / (C * k * k)) ** 0.5).to(act)
        bias = torch.randn(O, device=dev, generator=gen) * 0.1
        gout = torch.randn(B, O, Ho, Wo, device=dev, generator=gen).to(act)
        ws = staged_workspace(x, wt, k, s, p, variant, operand, 0)
        return (x, off, wt, bias, gout, ws, (k, s, p), operand)

    def run(layer):
        x, off, wt, bias, gout, ws, (k, s, p), operand = layer
        dcn.dcn_forward(x, off, wt, bias, k, s, p, variant, operand=operand, ws=ws)
        dcn.dcn_backward(x, off, wt, gout, True, k, s, p, variant, operand=operand, ws=ws, xt_staged=ws is not None)

    def timed(step, batch, label, steps=5, warmup=3):
        for _ in range(warmup):
            step()
        torch.cuda.synchronize(dev)
        _lib.profile_begin()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            flush.fill_(1)
            a.record(stream)
            step()
            b.record(stream)
        torch.cuda.synchronize(dev)
        ms = sum(a.elapsed_time(b) for a, b in ev) / steps
        prof = _lib.profile_end()
        top = max(prof, key=lambda n: prof[n][1]) if prof else None
        return {"workload": label, "images_per_s": batch / (ms * 1e-3), "ms_per_step": ms, "steps": steps, "warmup": warmup,
                "l2": "flushed (512 MB write) before every timed step",
                "top_kernel": top, "top_kernel_share": (prof[top][1] / steps / ms) if top else None,
                "kernel_ms_per_step": {n: v[1] / steps for n, v in prof.items() if v[1] / steps >= 0.05}}

    cfg3 = make("cfg3", dcn.OPERAND_FP32)
    out["cfg3"] = timed(lambda: run(cfg3), WORKLOADS["cfg3"][1], "cfg3: " + WORKLOADS["cfg3"][0] + ", fp32, variant " + args.variant)
    del cfg3
    layers = {n: make(n, dcn.OPERAND_BF16) for n in sorted(set(STACK_ORDER))}

    def stack_step():
        for n in STACK_ORDER:
            run(layers[n])
    out["stack_bf16"] = timed(stack_step, WORKLOADS["c3"][1], STACK_DESC + ", bf16 operands, variant " + args.variant)
    del layers, flush
    torch.cuda.empty_cache()
    return out


def main():
    args = parse_args()
    claim_stdout()
    if args.dump_outputs and (args.workload in ("stack", "detector") or args.impl == "reference"):
        raise SystemExit("--dump-outputs supports the single-layer workloads of --impl ours")
    if args.workload == "stack":
        if args.impl == "reference":
            raise SystemExit("--impl reference supports the single-layer workloads")
        return run_stack(args)
    if args.workload == "detector":
        if args.impl == "reference":
            raise SystemExit("--impl reference supports the single-layer workloads")
        return run_detector(args)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import jittor_dcn_b200 as dcn
    from jittor_dcn_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the ONE JSON line: NCCL's own banner / debug lines go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    lib = dcn.load()

    desc, B, C, O, H, W, k, s, p = WORKLOADS[args.workload]
    variant = dcn.VARIANT_TORCH if args.variant == "torch" else dcn.VARIANT_JITTOR
    flags = dcn.FLAG_FORCE_SIMT if args.force_simt else 0
    operand = dcn.OPERAND_BF16 if args.operand == "bf16" else dcn.OPERAND_FP32
    act = torch.bfloat16 if operand == dcn.OPERAND_BF16 else torch.float32
    N = k * k
    shp = dcn.make_shape(B, C, O, H, W, k, s, p, variant, operand=operand, flags=flags)
    Ho, Wo = _lib.output_hw(shp)

    # ---- synthetic data, resident in HBM (seeded per rank) ---------------------------
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.randn(B, C, H, W, device=dev, generator=gen).to(act)
    off = torch.randn(B, 2 * N, Ho, Wo, device=dev, generator=gen) * args.offset_sigma
    wt = (torch.randn(O, C, k, k, device=dev, generator=gen) * (2.0 / (C * N)) ** 0.5).to(act)
    bias = torch.randn(O, device=dev, generator=gen) * 0.1
    gout = torch.randn(B, O, Ho, Wo, device=dev, generator=gen).to(act)
    # flat gradient bucket: [grad_weight | grad_bias], plus [offset_conv.weight.grad | offset_conv.bias.grad] when the
    # whole layer is timed (--scope layer); every slot is written by the step before the all-reduce
    n_w, n_b, n_ow, n_ob = O * C * N, O, 2 * N * C * N, 2 * N
    bucket = torch.zeros(n_w + n_b + (n_ow + n_ob if args.scope == "layer" else 0), device=dev)

    comm = None
    allreduce_kind = "none"
    if world > 1:
        from jittor_dcn_b200 import dp
        comm = dp.DcnComm(rank, world, dev)       # NCCL communicator behind the C ABI
        allreduce_kind = "dcn_allreduce_sum_f32 (NCCL, one flat bucket)"

    import ctypes
    stream = torch.cuda.current_stream(dev)

    # one scratch buffer for both phases of the step: the backward pass reuses the staged
    # channels-last copy of x that the forward pass left at its head (DCN_FLAG_XT_STAGED)
    from jittor_dcn_b200.functional import staged_workspace
    ws = staged_workspace(x, wt, k, s, p, variant, operand, flags)

    layer_scope = args.scope == "layer"
    if layer_scope:
        from jittor_dcn_b200.functional import dcn_layer_backward, dcn_layer_forward, layer_supported, layer_workspace
        if operand != dcn.OPERAND_FP32 or not layer_supported(x.shape, O, k, s, p, variant, operand, flags):
            raise SystemExit("--scope layer: the whole-layer entry points do not cover this shape / operand mode")
        w_off = torch.randn(2 * N, C, k, k, device=dev, generator=gen) * 0.01
        b_off = torch.randn(2 * N, device=dev, generator=gen) * args.offset_sigma
        ws = layer_workspace(x, wt, k, s, p, variant, flags)

    def step():
        """-> {name: tensor} of what the caller of the timed path receives"""
        if layer_scope:
            off_l, out = dcn_layer_forward(x, w_off, b_off, wt, bias, k, s, p, variant, flags, ws=ws)
            gx, gwo, gbo, gw, gb = dcn_layer_backward(x, off_l, w_off, wt, gout, True, True, k, s, p, variant, flags,
                                                      ws=ws, xt_staged=True)
            res = {"offset": off_l, "out": out, "grad_x": gx, "grad_offset_weight": gwo, "grad_offset_bias": gbo}
        else:
            out = dcn.dcn_forward(x, off, wt, bias, k, s, p, variant, operand=operand, flags=flags, ws=ws)
            gx, goff, gw, gb = dcn.dcn_backward(x, off, wt, gout, True, k, s, p, variant, operand=operand, flags=flags,
                                                ws=ws, xt_staged=ws is not None)
            res = {"out": out, "grad_x": gx, "grad_offset": goff}
        if comm is not None:
            bucket[:n_w].copy_(gw.view(-1))
            bucket[n_w:n_w + n_b].copy_(gb)
            if layer_scope:
                bucket[n_w + n_b:n_w + n_b + n_ow].copy_(gwo.view(-1))
                bucket[n_w + n_b + n_ow:].copy_(gbo)
            comm.allreduce_mean_(bucket)
        res.update(grad_weight=gw, grad_bias=gb)
        return res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    lib.dcn_launch_count_reset()
    _lib.profile_begin()
    # L2 hygiene: workloads whose inputs fit in the 126 MB L2 get it flushed (a 512 MB write)
    # between timed iterations; the flush is outside the per-step event pairs.
    needs_flush = (x.numel() + gout.numel()) * x.element_size() < 400e6
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device=dev) if needs_flush else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps if needs_flush else 1)]
    # the last step's results are kept for --dump-outputs; every step first drops its predecessor's, so that the
    # allocator reuses the same buffers as in the warm-up steps
    barrier()
    if needs_flush:
        for a, b in ev:
            outs = None
            flush_buf.fill_(1)
            a.record(stream)
            outs = step()
            b.record(stream)
    else:
        ev[0][0].record(stream)
        for _ in range(args.steps):
            outs = None
            outs = step()
        ev[0][1].record(stream)
    barrier()
    elapsed_ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = int(lib.dcn_launch_count())
    prof = _lib.profile_end()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs)
    del outs
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)

    # ---- forward only (BASELINE configs[1] is quoted "fwd only"): same inputs, K timed calls --
    fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    fe0.record(stream)
    for _ in range(args.steps):
        dcn.dcn_forward(x, off, wt, bias, k, s, p, variant, operand=operand, flags=flags)
    fe1.record(stream)
    barrier()
    fwd_ms = fe0.elapsed_time(fe1) / args.steps
    if world > 1:
        t = torch.tensor([fwd_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        fwd_ms = float(t.item())
    fwd_only = {"value": world * B / (fwd_ms * 1e-3), "unit": "images/s", "ms_per_step": fwd_ms}

    # ---- roofline of the dominant kernel ------------------------------------------------
    pk = peaks()
    work = layer_bytes_flops(B, C, O, H, W, Ho, Wo, N, act_bytes=x.element_size())
    roofline, kernels = None, {}
    for name, (cnt, tot_ms) in prof.items():
        kernels[name] = {"launches": cnt, "avg_ms": tot_ms / max(cnt, 1), "share": tot_ms / max(elapsed_ms, 1e-9)}
    # the layout-staging passes are pure data movement: report them against the HBM copy peak too
    eb = x.element_size()
    stage_bytes = {"nchw_to_nhwc_kernel": 2 * x.numel() * eb,                    # read x, write the framed copy
                   "nhwc_to_nchw_kernel": 2 * x.numel() * 4,                     # read grad copy, write grad_x
                   "gout_tiles_kernel": gout.numel() * eb + gout.numel() * (4 if eb == 4 else 2),
                   "bias_grad_kernel": gout.numel() * eb}
    for name, nbytes in stage_bytes.items():
        if name in kernels and kernels[name]["avg_ms"] > 0:
            gbs = nbytes / (kernels[name]["avg_ms"] * 1e-3) / 1e9
            kernels[name].update({"bytes": nbytes, "GB/s": gbs, "hbm_frac": gbs / pk["hbm"]})
    ranked = sorted((n for n in prof if n in KERNEL_ROLE), key=lambda n: -prof[n][1])
    if ranked:
        top = ranked[0]
        role = KERNEL_ROLE[top]
        if top == "umma_bwd_data_kernel" and "umma_bwd_weight_kernel" not in prof and "bwd_weight_kernel" not in prof:
            role = "bwd"   # fused backward: this launch also produces grad_weight (SURVEY 8d backward total)
        avg_s = prof[top][1] / prof[top][0] * 1e-3
        hbm_floor = work[role]["bytes"] / (pk["hbm"] * 1e9)
        tc_floor = work[role]["flops"] / (pk["bf16_sustained"] * 1e12)
        traffic, limiter = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic = tj.get(f"{args.workload}:{args.variant}:{top}")
            # what the counters of the committed ncu capture say actually bounds this kernel
            limiter = tj.get("_limiter", {}).get(f"{args.workload}:{args.variant}:{top}")
        if hbm_floor >= tc_floor:
            ach = work[role]["bytes"] / avg_s / 1e9
            roofline = {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s",
                        "frac": ach / pk["hbm"], "traffic": traffic}
        else:
            ach = work[role]["flops"] / avg_s / 1e12
            roofline = {"bound": "tensor", "achieved": ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                        "frac": ach / pk["bf16_sustained"], "traffic": traffic}
        roofline.update({"kernel": top, "avg_ms": avg_s * 1e3, "peak_source": pk["source"], "measured_limiter": limiter,
                         "algorithmic_bytes": work[role]["bytes"], "algorithmic_flops": work[role]["flops"]})

    # ---- e2e: module API, host input buffers ----------------------------------------------
    e2e = None
    if not args.no_e2e:
        torch.manual_seed(99 + rank)
        cls = dcn.TorchDeformConv2d if args.variant == "torch" else dcn.TorchDeformConv2dJittorSemantics
        layer = cls(C, O, k, s, p).to(dev)
        layer.engine_flags = flags
        layer.operand = operand
        layer.keep_staged_input = True
        with torch.no_grad():
            layer.offset_conv.weight.normal_(0, 0.01)
            layer.offset_conv.bias.normal_(0, 1.0)
        # input pipeline as a training loop runs it: two pinned host batches, two device buffers and a
        # copy stream, so the H2D copy of step i+1 overlaps the compute of step i (both inside the
        # timed region; every step still copies its own input and reads its own result back)
        x_host = [torch.randn(B, C, H, W).pin_memory() for _ in range(2)]
        x_dev = [torch.empty(B, C, H, W, device=dev) for _ in range(2)]
        copy_stream = torch.cuda.Stream(dev)
        copied = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        params = [q for q in layer.parameters()]
        n_par = sum(q.numel() for q in params)
        g_host = torch.empty(n_par, dtype=torch.float32).pin_memory()
        e_steps = max(3, min(args.steps, 10))

        def prefetch(i):
            buf = i & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[buf])             # the step that used this buffer is done
                x_dev[buf].copy_(x_host[buf], non_blocking=True)  # H2D of step i's input
                copied[buf].record(copy_stream)

        def e2e_step(i):
            buf = i & 1
            stream.wait_event(copied[buf])
            prefetch(i + 1)
            xi = x_dev[buf].detach().requires_grad_(True)
            out = layer(xi)
            torch.autograd.backward(out, gout)
            consumed[buf].record(stream)
            flat = torch.cat([q.grad.reshape(-1) for q in params])
            if world > 1:
                dist.all_reduce(flat)
            g_host.copy_(flat, non_blocking=True)                   # D2H of the step's result
            for q in params:
                q.grad = None
            stream.synchronize()

        for buf in range(2):
            consumed[buf].record(stream)
        prefetch(0)
        for i in range(2):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(2, 2 + e_steps):
            e2e_step(i)
        barrier()
        dt = (time.perf_counter() - t0) / e_steps
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": world * B / dt, "unit": "images/s", "h2d_bytes_per_step": x_host[0].numel() * 4,
               "d2h_bytes_per_step": n_par * 4, "ms_per_step": dt * 1e3, "steps": e_steps,
               "api": f"jittor_dcn_b200.{cls.__name__}.forward + autograd backward (offset conv included); "
                      "H2D of step i+1 overlapped with step i on a copy stream"}
        del layer, x_host, x_dev

    # ---- CPU baseline (rank 0, N = 1 only) ---------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        micro_b = 8 if args.workload == "cfg2" else 16
        fn = cpu_reference_step(WORKLOADS[args.workload], args.variant, micro_b, with_offset_conv=False)
        med, runs = time_cpu(fn, budget_s=20.0)
        cpu = {"value": micro_b / med, "unit": "images/s", "cores": cores, "kind": "port",
               "sample": f"median of {runs} fwd+bwd passes over a {micro_b}-sample micro-batch of the same layer "
                         f"(reference op chain restated with torch CPU ops, offsets supplied)"}

    # ---- BASELINE configs[4] next to the headline, at this N: the data-parallel detector training step, global
    # batch 1024 sharded over the ranks (STRONG scaling; the headline above is weak scaling of one layer)
    detector_dp = None
    l2_note = ("L2 flushed (512 MB write) between timed iterations" if needs_flush else
               "inputs (x %.0f MB + gout %.0f MB) exceed the 126 MB L2; no flush needed"
               % (x.numel() * x.element_size() / 1e6, gout.numel() * gout.element_size() / 1e6))
    staging_note = ("backward reuses the forward pass's staged copy of x (DCN_FLAG_XT_STAGED, one scratch buffer for "
                    "both phases)" if ws is not None else "re-staged per phase")
    if args.workload == "cfg2" and not args.no_detector_dp:
        del x, off, gout, ws, flush_buf
        torch.cuda.empty_cache()
        try:
            r = measure_detector(args, world, rank, local_rank, dev, steps=10, warmup=3, want_e2e=False,
                                 sample_clocks=False)
            detector_dp = {"global_batch": args.global_batch, "batch_per_gpu": r["batch_per_gpu"],
                           "ms_per_step": r["ms_per_step"], "images_per_s": r["images_per_s"], "scaling": "strong",
                           "launches": r["launches_per_step"], "graph": r["graph"], "launch": r["launch"],
                           "allreduce": r["allreduce"], "dcn_engine_ms_per_step": r["engine_ms_per_step"],
                           "steps": 10, "warmup": 3}
        except Exception as e:  # noqa: BLE001 - the headline line must still be printed
            detector_dp = {"error": f"{type(e).__name__}: {e}"[:300]}
    other_configs = None
    if args.workload == "cfg2" and world == 1 and not args.no_detector_dp:
        try:
            other_configs = measure_other_configs(args, dev, variant)
        except Exception as e:  # noqa: BLE001
            other_configs = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        line = {
            "metric": "DeformConv2d fwd+bwd images/sec", "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if operand == dcn.OPERAND_BF16 else "f32",
            "data": "synthetic",
            "config": {"workload": args.workload + ": " + desc, "variant": args.variant, "operand": args.operand,
                       "scope": ("whole layer on the engine: companion offset conv + DCN span, forward and backward "
                                 "(dcn_layer_forward / dcn_layer_backward)" if layer_scope else
                                 "DCN span with offsets supplied (dcn_forward + dcn_backward); the offset conv is not in "
                                 "the timed region"),
                       "batch_per_gpu": B, "global_batch": world * B, "offset_sigma_px": args.offset_sigma,
                       "path_fwd": lib.dcn_path_name(ctypes.byref(shp), 0).decode(),
                       "path_bwd": lib.dcn_path_name(ctypes.byref(shp), 1).decode(),
                       "l2": l2_note, "staging": staging_note,
                       "allreduce": allreduce_kind, "parallelism": f"dp{world}"},
            "roofline": roofline, "kernels": kernels, "fwd_only": fwd_only, "cpu_baseline": cpu, "e2e": e2e,
            "detector_dp": detector_dp, "other_configs": other_configs, "gpu_launches": launches, "clocks": clocks,
        }
        emit(line)
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
