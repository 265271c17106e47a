#!/usr/bin/env python
"""BASELINE config 5: detector forward + backward (+ DDP-style gradient all-reduce) at growing cloud sizes.

    python tools/bench_train.py [--points 40000,80000,120000,200000] [--scenes 4] [--iters 5] [--ref]
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/bench_train.py
    python -m torch.distributed.run --nproc-per-node 8 tools/bench_train.py --points 40000 --sync-bn fused

Training mode: autograd through the unfused sm_100a kernels (FPS, ball query, grouping, three_nn,
interpolate and their backward passes) + cuDNN convolutions, exactly the reference's op sequence
(pointnet2_modules.py:227-276).  The loss is a surrogate (mean square of every head output): the
reference's loss (lib/loss_helper.py) is outside the hot path.  SA npoint is scaled with the cloud
(x1, x2, x3, x5 -> 2048..8192+, SURVEY 8d config 5).  `--ref` also times the reference's own CUDA
extension (oracle/_ref) driving the same modules on rank 0.  One JSON line per cloud size.

`--sync-bn` sets how BatchNorm statistics are taken across ranks: `off` (the default, per rank), `fused`
(nn.SyncBatchNorm.convert_sync_batchnorm: the fused BatchNorm + ReLU kernels with one exchange in the forward and one
in the backward of each block, torch's SyncBatchNorm for the voting and proposal heads) or `torch` (the converted
model with the fused kernels switched off: torch's SyncBatchNorm everywhere).  Each line records the GPU's name and
power limit.

`--amp` runs the step without autocast (`off`) or under torch.autocast("cuda", dtype=torch.bfloat16) (`bf16`: bf16
activations through the bf16 twins of the grouping, interpolation and fused BatchNorm kernels); `--amp off,bf16`
times both for every cloud size, alternating them `--repeats` times, eager and graphed (captured with
cache_enabled=False, so no cast of a weight is cached across replays).  Each line also records the peak memory of the
eager steps (torch.cuda.max_memory_allocated).
"""
import contextlib
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def build_model(scale, device, sync_bn="off"):
    from spacap3d_b200.detector import VoteNetDetector
    torch.manual_seed(0)
    model = VoteNetDetector(input_feature_dim=1)
    bb = model.backbone_net
    for sa, base in ((bb.sa1, 2048), (bb.sa2, 1024), (bb.sa3, 512), (bb.sa4, 256)):
        sa.npoint = base * scale
    if sync_bn != "off":
        model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)
    return model.to(device).train()


def gpu_info(index):
    """Name and power limit of the GPU the numbers were measured on."""
    info = {"gpu": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"] = out or None
    except (OSError, subprocess.SubprocessError):
        info["power_limit"] = None
    return info


def surrogate_loss(out):
    """Mean square of every head output (the reference's loss, lib/loss_helper.py, is outside the hot path)."""
    return sum((out[k].float() ** 2).mean() for k in ("objectness_scores", "center", "sem_cls_scores",
                                                      "size_scores", "size_residuals", "vote_xyz"))


def step(model, pc, world):
    out = model({"point_clouds": pc})
    loss = surrogate_loss(out)
    loss.backward()
    if world > 1:
        from spacap3d_b200.dist import allreduce_gradients
        allreduce_gradients(model)
    return loss


def amp_context(amp):
    """The autocast region of one step: nothing for `off`, bf16 autocast for `bf16`."""
    if amp == "bf16":
        return torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False)
    return contextlib.nullcontext()


def time_steps(fn, iters, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def measure(args, amp, n, scale, pc, dev, rank, world, ref, info, pytorch_utils, max_over_ranks):
    """One JSON record: eager (and graphed, on one GPU) ms per step of a fresh model in autocast mode `amp`."""
    model = build_model(scale, dev, args.sync_bn)

    def ours():
        model.zero_grad(set_to_none=True)
        with amp_context(amp):
            step(model, pc, world)

    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    ms = time_steps(ours, args.iters)
    peak = torch.cuda.max_memory_allocated(dev)
    ms = max_over_ranks(ms, device=dev) if world > 1 else ms
    rec = {"config": "fwd+bwd, %d scenes/GPU x %d pts, SA npoint x%d" % (args.scenes, n, scale), "n_gpus": world,
           "ms_per_step": round(ms, 3), "scenes_per_s": round(world * args.scenes / ms * 1e3, 2),
           "sync_bn": args.sync_bn, "amp": amp,
           "peak_mem_gb": round(peak / 1e9, 3), **info}
    if world == 1 and not args.no_graph:
        # the step has no host synchronisation (box decode stays on the device), so forward + backward can be
        # captured once and replayed: removes the ~3 ms/step of Python/launch overhead of ~600 small launches
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            ours()
        torch.cuda.current_stream().wait_stream(side)
        model.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph), amp_context(amp):
            step(model, pc, 1)
        gms = time_steps(graph.replay, args.iters)
        rec["graphed_ms_per_step"] = round(gms, 3)
        rec["graphed_scenes_per_s"] = round(args.scenes / gms * 1e3, 2)
        del graph
    if ref is not None:
        import bench

        def theirs():      # reference extension + the plain cuDNN BatchNorm / ReLU / max_pool2d sequence
            model.zero_grad(set_to_none=True)
            pytorch_utils.FUSED_BN_RELU_TRAINING = False
            try:
                with bench.swapped_ops(ref, host_decode=False), amp_context(amp):
                    step(model, pc, 1)
            finally:
                pytorch_utils.FUSED_BN_RELU_TRAINING = args.sync_bn != "torch"

        try:
            rms = time_steps(theirs, max(2, args.iters // 2), warmup=1)
            rec["reference_ext_ms_per_step"] = round(rms, 3)
            rec["speedup_vs_reference_ext"] = round(rms / ms, 2)
        except Exception as e:   # the reference FPS kernel has a fixed 512-thread block; very large N still works, but be safe
            rec["reference_ext_error"] = str(e)[:200]
    del model
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", default="40000,80000,120000,200000")
    ap.add_argument("--scenes", type=int, default=4, help="scenes per GPU")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--ref", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--sync-bn", choices=("off", "fused", "torch"), default="off",
                    help="BatchNorm statistics per rank (off) or across ranks with the fused kernels or torch's")
    ap.add_argument("--amp", default="off",
                    help="comma-separated autocast modes to time, alternated: off, bf16 (e.g. off,bf16)")
    ap.add_argument("--repeats", type=int, default=1, help="rounds of the --amp modes per cloud size")
    args = ap.parse_args()
    amps = args.amp.split(",")
    assert all(a in ("off", "bf16") for a in amps), args.amp
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    from spacap3d_b200 import pytorch_utils
    from spacap3d_b200.dist import max_over_ranks
    if args.sync_bn == "torch":
        pytorch_utils.FUSED_BN_RELU_TRAINING = False
    info = gpu_info(local)
    from spacap3d_b200.scenes import make_scene
    ref = None
    if args.ref and rank == 0:
        from oracle.build_ref import load_ref
        ref = load_ref()
    for n in [int(x) for x in args.points.split(",")]:
        scale = max(1, round(n / 40000))
        pc = torch.from_numpy(np.stack([make_scene(5000 + rank * 100 + i, n) for i in range(args.scenes)], 0)).to(dev)
        for _ in range(args.repeats):
            for amp in amps:
                rec = measure(args, amp, n, scale, pc, dev, rank, world, ref, info, pytorch_utils, max_over_ranks)
                if rank == 0:
                    print(json.dumps(rec), flush=True)
        del pc
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
