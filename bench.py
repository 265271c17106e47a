#!/usr/bin/env python
"""bench.py -- detector scenes/s @40k points on N B200s (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one full detector forward (PointNet++ backbone SA1-4 + FP1-2, Hough voting, vote
aggregation + proposal head + on-device box decode) over one batch of synthetic 40k-point
ScanNet-shaped scenes per GPU.  --config selects the BASELINE.json workload:
  2 (default, the config the metric is quoted on)  xyz+height, 8 scenes per GPU, weak scaling
  3  xyz+rgb+normal+height (C=7), 32 scenes in total sharded over the ranks (strong scaling); detector
     only -- the captioner is a non-target PyTorch path
  4  xyz+multiview+normal+height (C=132), 8 scenes per GPU (64 on 8 GPUs), weak scaling
  5  training sweep: forward + backward + one NCCL gradient all-reduce, 4 scenes per GPU,
     --points N (40k..200k) with the SA npoint scaled by N/40k
Inference is embarrassingly parallel over scenes: no data-path collective.

  value   : scenes/s with the batch already resident in HBM (CUDA-event time, max over ranks); the
            K-step timed region is repeated REPEATS times and the MEDIAN region is reported
  e2e     : same, through the public API from PINNED HOST buffers, host->device copy and
            device->host read of the detections inside the timed region
  roofline: the dominant roofline-bounded kernel of the step, timed live with CUDA events
  dominant: the kernel with the largest share of the step's time, whatever bounds it
  cpu_baseline: the CPU oracle port (oracle/, C + torch CPU MLP) on a bounded sample (rank 0, N=1)
  --impl reference: the reference's UNMODIFIED Python stack (baseline/_ref: lib/pointnet2/*.py, models/*.py,
            SpaCapNet detection branch incl. its host-side box decode) on the reference's own CUDA ops
            (oracle/_ref, unmodified sources rebuilt for sm_100a), one replica per rank; falls back to the CPU
            port when they are not loadable.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POINTS = 40000
REPEATS = 15             # the K-step timed region is repeated this often; the median region is reported
N_STREAMS = 32           # CUDA-graph replay streams (batches in flight; the sampler is latency-bound, 4 ms per call)
L2_BYTES = 126e6

CONFIGS = {
    2: dict(feature_dim=1, scene_kw=dict(use_height=True), scenes_per_gpu=8, scenes_total=None, scaling="weak",
            workload="SpaCap3D xyz: batch 8 scenes x 40k pts per GPU, full detector forward "
                     "(SA 2048/1024/512/256, FP1-2, voting, 256 proposals, box decode)"),
    3: dict(feature_dim=7, scene_kw=dict(use_color=True, use_normal=True, use_height=True), scenes_per_gpu=None,
            scenes_total=32, scaling="strong",
            workload="SpaCap3D xyz+rgb+normal: 32 scenes x 40k pts in total, 7 feature channels, sharded over the "
                     "ranks, full detector forward (captioner = non-target PyTorch path, not run)"),
    4: dict(feature_dim=132, scene_kw=dict(use_multiview=True, use_normal=True, use_height=True), scenes_per_gpu=8,
            scenes_total=None, scaling="weak",
            workload="SpaCap3D xyz+multiview+normal: batch 8 scenes x 40k pts per GPU (64 on 8 GPUs), 132 feature "
                     "channels (128-d multiview), full detector forward"),
    5: dict(feature_dim=1, scene_kw=dict(use_height=True), scenes_per_gpu=4, scenes_total=None, scaling="weak",
            workload="SpaCap3D training sweep: 4 scenes per GPU, forward + backward + NCCL gradient all-reduce, "
                     "SA npoint scaled with the cloud size"),
}
CFG = dict(CONFIGS[2], id=2)


def scenes_per_gpu(world):
    return CFG["scenes_per_gpu"] or max(1, CFG["scenes_total"] // world)


def n_input_sets(world):
    """Distinct batches rotated through the timed loops so that their total size exceeds the L2."""
    batch_bytes = scenes_per_gpu(world) * N_POINTS * (3 + CFG["feature_dim"]) * 4
    return max(3, int(math.ceil(1.06 * L2_BYTES / batch_bytes)))


def workload_config(world):
    """The part of `config` both arms print identically."""
    return {"workload": CFG["workload"], "baseline_config": CFG["id"], "scenes_per_gpu": scenes_per_gpu(world),
            "points": N_POINTS, "input_feature_dim": CFG["feature_dim"], "weights": weights_note()}


# ------------------------------------------------------------------------------------------------
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d.get("bf16_tflops", 1590.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(tag, source):
    """(dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, where it comes from), from
    this round's committed ncu capture (bench.py cannot run under a profiler).  The capture records the sha256 of the
    kernel source it was taken from; when csrc/<source> has changed since, the figure is stale and None is reported."""
    import hashlib
    path = os.path.join(ROOT, "profiles", "r2_%s_traffic.json" % tag)
    try:
        with open(path) as f:
            d = json.load(f)
        h = hashlib.sha256()
        for src in source.split(","):                      # the kernels of one op may live in several files
            with open(os.path.join(ROOT, "spacap3d_b200", "csrc", src), "rb") as f:
                h.update(f.read())
        sha = h.hexdigest()
        if d.get("source_sha256") != sha:
            return None, "profiles/r2_%s_traffic.json is stale (csrc/%s changed since the capture)" % (tag, source)
        return int(d["dram_bytes_per_launch_avg"]), ("profiles/r2_%s_traffic.json (ncu --set full, dram read+write per "
                                                     "launch, kernel %s)" % (tag, d.get("kernel", "?")))
    except (OSError, KeyError, ValueError):
        return None, "no capture committed"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def count(self):
        """Samples written so far."""
        try:
            with open(self.f.name) as f:
                return sum(1 for line in f if line.count(",") >= 8)
        except OSError:
            return 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons),
                       samples=len(sm))
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def make_host_batches(rank, world):
    """n_input_sets pinned (scenes, 40000, 3+C) float32 batches; seeds differ per rank and per set."""
    from spacap3d_b200.scenes import make_scene
    sets = []
    for s in range(n_input_sets(world)):
        scenes = [make_scene(1000 * CFG["id"] + 100 * rank + 10 * s + i, N_POINTS, **CFG["scene_kw"])
                  for i in range(scenes_per_gpu(world))]
        t = torch.from_numpy(np.stack(scenes, 0))
        sets.append(t.pin_memory() if torch.cuda.is_available() else t)
    return sets


def checkpoint_file():
    """The reference's pretrained VoteNet weights for this config's channel count, when staged (a data file)."""
    names = {1: "PRETRAIN_VOTENET_XYZ", 7: "PRETRAIN_VOTENET_XYZ_COLOR_NORMAL",
             132: "PRETRAIN_VOTENET_XYZ_MULTIVIEW_NORMAL"}
    p = os.path.join(ROOT, "baseline", "_ref", "pretrained", names.get(CFG["feature_dim"], "-"), "model.pth")
    return p if os.path.exists(p) else None


def weights_note():
    p = checkpoint_file()
    return ("reference checkpoint pretrained/%s/model.pth" % os.path.basename(os.path.dirname(p))) if p else \
        "random init (seed 0)"


def make_detector(device):
    from spacap3d_b200.detector import VoteNetDetector
    torch.manual_seed(0)
    model = VoteNetDetector(input_feature_dim=CFG["feature_dim"])
    p = checkpoint_file()
    if p:
        missing, unexpected = model.load_state_dict(torch.load(p, map_location="cpu"), strict=False)
        assert not missing and not unexpected, (missing, unexpected)
    return model.to(device).eval()


RESULT_KEYS = ("objectness_scores", "center", "size_scores", "size_residuals", "sem_cls_scores",
               "bbox_corner", "aggregated_vote_inds")
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: what the timed path computed in its last step, one <out_dir>/<name>.npy per array, so that two
    builds can be compared output for output (the inputs depend only on the arguments).  float64 stays float64,
    integers (indices) become float64, which holds them exactly; everything else is stored as float32."""
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        host[name] = a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind in "iub" else np.float32)
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs of one step take %d bytes, more than --dump-outputs stores" % total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class L2Flusher:
    def __init__(self, device):
        self.buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)  # > 126 MB L2

    def __call__(self):
        self.buf.fill_(1)


# ------------------------------------------------------------------------------------------------
# per-kernel accounting: every call through the C ABI is timed with CUDA events on torch's current
# stream (the stream the kernels are launched on)
ALGO_BYTES = {
    # SURVEY 8(d) per-scene formulas x B; args are the ctypes call arguments after the name
    "spc_group_points": lambda a: 4 * a[2] * (a[3] * a[4] + a[5] * a[6] + a[3] * a[5] * a[6]),
    "spc_group_points_grad": lambda a: 4 * a[2] * (a[3] * a[5] * a[6] + a[5] * a[6] + a[3] * a[4]),
    "spc_three_interpolate": lambda a: 4 * a[3] * (a[4] * a[5] + 6 * a[6] + a[4] * a[6]),
    "spc_three_interpolate_grad": lambda a: 4 * a[3] * (a[4] * a[5] + 6 * a[5] + a[4] * a[6]),
    "spc_gather_points": lambda a: 4 * a[2] * (a[5] + 2 * a[3] * a[5]),
    "spc_ball_query": lambda a: a[2] * (12 * a[3] + 12 * a[4] + 4 * a[4] * a[6]),
    "spc_three_nn": lambda a: a[2] * (12 * (a[3] + a[4]) + 24 * a[3]),
    "spc_furthest_point_sampling": lambda a: a[1] * (12 * a[2] + 4 * a[3] + (12 * a[3] if a[5] else 0)),
    # fused SA fwd = 12n + 4*C*n + 4*np*ns + 4*C_out*np per scene (C = table width actually read)
    "spc_sa_fused_forward": lambda a: a[13] * (12 * a[14] + (2 * a[17] if a[3] else 4 * a[7]) * a[14]
                                               + 4 * a[15] * a[16] + 4 * a[19] * a[15]),
    # _ex = same arguments with (W0_host, b0_host) inserted after b0: everything from Cf on moves by two
    "spc_sa_fused_forward_ex": lambda a: a[15] * (12 * a[16] + (2 * a[19] if a[3] else 4 * a[9]) * a[16]
                                                  + 4 * a[17] * a[18] + 4 * a[21] * a[17]),
}
# algorithmic FLOPs (SURVEY 8d: 2 * sum_l C_l*C_{l+1} * np*ns) of the MLP a fused launch replaces;
# C_0 = 3 + input channels is not known to the projected form, so only layers 1,2 (the tcgen05
# part) plus the in-line layer 0 are counted -- a lower bound on the replaced work
ALGO_FLOPS = {
    "spc_sa_fused_forward": lambda a: 2 * a[13] * a[15] * a[16] * (
        a[17] * a[18] + a[18] * a[19] + (3 if a[3] else 3 + a[7]) * a[17]),
    "spc_sa_fused_forward_ex": lambda a: 2 * a[15] * a[17] * a[18] * (
        a[19] * a[20] + a[20] * a[21] + (3 if a[3] else 3 + a[9]) * a[19]),
}
ROOFLINE_BOUNDED = ("spc_group_points", "spc_three_interpolate", "spc_gather_points", "spc_sa_fused_forward",
                    "spc_sa_fused_forward_ex")


class KernelMeter:
    """Wraps spacap3d_b200._lib.call: counts launches, optionally records event pairs."""

    def __init__(self):
        from spacap3d_b200 import _lib
        self._lib = _lib
        self._orig = _lib.call
        self.launches = 0
        self.records = []      # (name, bytes, ev0, ev1, extra)
        self.timing = False

    def install(self):
        def call(name, *args):
            self.launches += 1
            if not self.timing:
                return self._orig(name, *args)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self._orig(name, *args)
            e1.record()
            fn, ff = ALGO_BYTES.get(name), ALGO_FLOPS.get(name)
            self.records.append((name, fn(args) if fn else 0, e0, e1, args, ff(args) if ff else 0))
        self._lib.call = call

    def uninstall(self):
        self._lib.call = self._orig

    def summary(self, steps):
        """per-op: launches/step, ms/step, algorithmic GB/s (aggregated over the step)."""
        agg = {}
        for name, nbytes, e0, e1, args, flops in self.records:
            ms = e0.elapsed_time(e1)
            d = agg.setdefault(name, {"launches": 0, "ms": 0.0, "bytes": 0, "flops": 0, "max": (0.0, 0, None)})
            d["launches"] += 1
            d["ms"] += ms
            d["bytes"] += nbytes
            d["flops"] += flops
            if ms > d["max"][0]:
                d["max"] = (ms, nbytes, args)
        return agg


# ------------------------------------------------------------------------------------------------
def forward_resident(model, pc):
    with torch.no_grad():
        return model({"point_clouds": pc})


def timed_loop(step_fn, steps, warmup, flush, barrier, sampler=None):
    """W warm-up steps, then exactly K timed steps; each step is bracketed by CUDA events on the
    launching stream with an L2 flush in between (outside the events).  Returns per-step ms."""
    for i in range(warmup):
        flush()
        step_fn(i)
    torch.cuda.synchronize()
    barrier()
    if sampler:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t0 = time.perf_counter()
    for k in range(steps):
        flush()
        ev[k][0].record()
        step_fn(warmup + k)
        ev[k][1].record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop() if sampler else None
    return [a.elapsed_time(b) for a, b in ev], wall, clocks


def hbm_bound_ops(pc, flush, hbm_peak):
    """The HBM-bound point ops the north_star sets a roofline target for, timed live on BASELINE shapes (they are not
    launched by the eval forward, where the fused SA kernel replaces grouping): grouping forward at config 4's SA1
    shape (132 channels) and at SA2's, three_interpolate at FP2's and at config 5's x4 shape.  Graph-timed with an L2
    flush before every call (see `timed`); algorithmic bytes = SURVEY 8(d) formulas."""
    from spacap3d_b200 import _ext
    xyz = pc[:, :, :3].contiguous()
    B, N = xyz.shape[0], xyz.shape[1]
    out = []

    def timed(fn, reps=8):
        """Launch-overhead-free time of one call: [L2 flush, fn] x reps captured in one CUDA graph, minus the same graph
        without fn (these ops take 5-150 us; an eager launch adds ~5 us of host gap to every one of them)."""
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        side = torch.cuda.Stream()

        def capture(with_fn):
            g = torch.cuda.CUDAGraph()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.graph(g, stream=side):
                for _ in range(reps):
                    flush()
                    if with_fn:
                        fn()
            return g

        def run(g):
            ts = []
            for _ in range(7):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                g.replay()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            return statistics.median(ts)

        ga, gb = capture(True), capture(False)
        run(ga), run(gb)
        return max(run(ga) - run(gb), 1e-6) / reps

    _, c1 = _ext.furthest_point_sampling_with_xyz(xyz, 2048)
    _, c2 = _ext.furthest_point_sampling_with_xyz(c1, 1024)
    for name, pts, ctr, r, ns, C in (("group_points SA1 multiview (config 4)", xyz, c1, 0.2, 64, 132),
                                     ("group_points SA2", c1, c2, 0.4, 32, 128)):
        n, npnt = pts.shape[1], ctr.shape[1]
        idx = _ext.ball_query(ctr, pts, r, ns)
        feats = torch.randn(B, C, n, device=pc.device)
        ms = timed(lambda: _ext.group_points(feats, idx))
        nbytes = 4 * B * (C * n + npnt * ns + C * npnt * ns)
        out.append({"op": name, "shape": [B, C, n, npnt, ns], "ms": round(ms, 4), "algo_bytes": nbytes,
                    "gbs": round(nbytes / ms / 1e6, 1), "frac_of_hbm_peak": round(nbytes / ms / 1e6 / hbm_peak, 3)})
        del feats
    _, c3 = _ext.furthest_point_sampling_with_xyz(c2, 512)
    d2, idx3 = _ext.three_nn(c2, c3)
    w = torch.rand(B, 1024, 3, device=pc.device)
    feats = torch.randn(B, 256, 512, device=pc.device)
    ms = timed(lambda: _ext.three_interpolate(feats, idx3, w))
    nbytes = 4 * B * (256 * 512 + 6 * 1024 + 256 * 1024)
    out.append({"op": "three_interpolate FP2", "shape": [B, 256, 512, 1024], "ms": round(ms, 4), "algo_bytes": nbytes,
                "gbs": round(nbytes / ms / 1e6, 1), "frac_of_hbm_peak": round(nbytes / ms / 1e6 / hbm_peak, 3),
                "note": "12.8 MB per call: a few microseconds, latency-bound at the detector's own size"})
    # config 5's x4 cloud: 4096 unknown <- 2048 known points per scene
    _, u4 = _ext.furthest_point_sampling_with_xyz(xyz, 4096)
    k4 = u4[:, :2048].contiguous()
    _, idx4 = _ext.three_nn(u4, k4)
    w4 = torch.rand(B, 4096, 3, device=pc.device)
    feats4 = torch.randn(B, 256, 2048, device=pc.device)
    ms = timed(lambda: _ext.three_interpolate(feats4, idx4, w4))
    nbytes = 4 * B * (256 * 2048 + 6 * 4096 + 256 * 4096)
    out.append({"op": "three_interpolate config-5 x4 shape", "shape": [B, 256, 2048, 4096], "ms": round(ms, 4),
                "algo_bytes": nbytes, "gbs": round(nbytes / ms / 1e6, 1),
                "frac_of_hbm_peak": round(nbytes / ms / 1e6 / hbm_peak, 3)})
    return out


def gpu_local_cores(local):
    """Host cores NVML reports as local to GPU `local` (its NUMA node), restricted to the cores this process may use."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local])
                                              if os.environ.get("CUDA_VISIBLE_DEVICES", "").replace(",", "").isdigit()
                                              else local)
        n = os.cpu_count() or 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cores = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        return sorted(cores & set(os.sched_getaffinity(0)))
    except Exception:  # noqa: BLE001  (no NVML, no permission, exotic topology: fall back to an even split)
        return []


def bind_rank_cpus(local, world):
    """One disjoint core set per local rank, taken from the cores NVML reports as local to the rank's GPU, BEFORE the
    pinned host buffers are allocated (first touch => NUMA-local staging memory).  The ranks of one box otherwise
    share every core, the submit / copy threads of 8 ranks migrate over each other and half of the pinned buffers sit
    on the wrong socket: e2e scaled 0.886 at 8 GPUs in round 1."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
        if world <= 1 or len(allowed) < 2 * world:
            return None
        near = gpu_local_cores(local)
        # ranks whose GPUs share a NUMA node split that node's cores by their order among the local ranks
        per = max(2, len(allowed) // world)
        if len(near) >= per:
            peers = world if len(near) == len(allowed) else max(1, world * len(near) // len(allowed))
            slot = local % peers
            share = max(2, len(near) // peers)
            mine = near[slot * share:(slot + 1) * share] or near[-share:]
        else:
            mine = allowed[local * per:(local + 1) * per]
        os.sched_setaffinity(0, mine)
        torch.set_num_threads(max(1, min(len(mine), 4)))
        return mine
    except (AttributeError, OSError):
        return None


def init_dist(local, device, world):
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
        return dist, (lambda: dist.barrier(device_ids=[local]))
    return None, (lambda: None)


def region_stats(regions_ms):
    return {"repeats": len(regions_ms), "median_ms": round(statistics.median(regions_ms), 4),
            "min_ms": round(min(regions_ms), 4), "max_ms": round(max(regions_ms), 4)}


def run_ours(args):
    rank, world, local = dist_env()
    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    cpus = bind_rank_cpus(local, world)
    dist, barrier = init_dist(local, device, world)
    from spacap3d_b200 import _lib
    _lib.load()
    if CFG["id"] == 5:
        return run_train(args, rank, world, local, device, dist, barrier)
    meter = KernelMeter()
    meter.install()
    model = make_detector(device)
    host = make_host_batches(rank, world)
    n_sets = len(host)
    spg = scenes_per_gpu(world)
    resident = [h.to(device) for h in host]
    flush = L2Flusher(device)
    batch_mb = host[0].numel() * host[0].element_size() / 1e6

    # ---- (1) eager single-stream pass: inputs resident in HBM, L2 flushed between steps -------------
    out_holder = {}

    def step_resident(i):
        out_holder["o"] = forward_resident(model, resident[i % n_sets])

    meter.launches = 0
    eager_steps = args.steps if args.mode == "eager" else min(args.steps, 60)
    eager_warm = args.warmup if args.mode == "eager" else min(args.warmup, 12)
    per_step, wall, clocks = timed_loop(step_resident, eager_steps, eager_warm, flush, barrier,
                                        ClockSampler(local) if args.mode == "eager" else None)
    last_step = {k: out_holder["o"][k] for k in RESULT_KEYS}
    launches_per_step = meter.launches // (eager_steps + eager_warm)
    dev_s = sum(per_step) / 1e3
    regions = None

    eager = {"ms_per_step": round(dev_s / eager_steps * 1e3, 4),
             "scenes_per_s_per_gpu": round(spg * eager_steps / dev_s, 2),
             "note": "no CUDA graph, single stream, 256 MiB L2 flush between steps (excluded from the timing)"}
    graph_info = None
    if args.mode == "graph":
        # ---- (1b) headline: CUDA-graph replay, N_STREAMS batches in flight ------------------------
        from spacap3d_b200.pipeline import GraphedDetector
        tune = {k: v for k, v in (("pm_n_tile", args.pm_n_tile), ("sa_min_tiles", args.sa_min_tiles),
                                        ("pm_tiles_per_cta", args.pm_tiles_per_cta)) if v is not None}
        runner = GraphedDetector(model, resident[0], n_streams=N_STREAMS, result_keys=RESULT_KEYS, **tune)

        def timed_graph(submit, steps, warmup, repeats, sampler=None, after_regions=None):
            """`repeats` timed regions of exactly `steps` submits each, every region bracketed by a barrier +
            synchronize on both sides and timed with CUDA events (start event forked into every stream, end
            event after joining them).  nvidia-smi needs ~0.2 s for its first sample, so the sampler runs from
            the first warm-up step on and, if it still has fewer than 4 samples when the regions are done, the
            SAME workload keeps running untimed until it has (reported as extra untimed steps).
            `after_regions` is called once the last region has finished, before any untimed step."""
            if sampler:
                sampler.start()
            for i in range(warmup):
                submit(i)
            runner.wait_all()
            cur = torch.cuda.current_stream()
            out, n = [], warmup
            t0 = time.perf_counter()
            for _ in range(repeats):
                torch.cuda.synchronize()
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(cur)
                runner.fork_from(e0)
                for k in range(steps):
                    submit(n + k)
                n += steps
                runner.join_into(cur)
                e1.record(cur)
                torch.cuda.synchronize()
                barrier()
                out.append(e0.elapsed_time(e1))
            wall_ = time.perf_counter() - t0
            if after_regions:
                after_regions()
            clk = None
            if sampler:
                extra, t_end = 0, time.perf_counter() + 3.0
                while sampler.count() < 4 and time.perf_counter() < t_end:
                    for q in range(50):
                        submit(n + extra + q)
                    extra += 50
                    runner.wait_all()
                clk = sampler.stop()
                clk["window"] = ("warm-up + %d timed regions + %d extra untimed steps of the same workload"
                                 % (repeats, extra))
            return out, wall_, clk

        def keep_last_step():
            """Results of the last timed step, from its slot (the steps that follow reuse the slots)."""
            out = runner.outputs[(runner._next - 1) % runner.n]
            last_step.update({k: out[k].clone() for k in RESULT_KEYS})

        regions, wall, clocks = timed_graph(lambda i: runner.submit(resident[i % n_sets]),
                                            args.steps, args.warmup, REPEATS, ClockSampler(local), keep_last_step)

        def submit_e2e(i):
            slot = runner._next
            if runner.busy(slot):
                runner.wait(slot)                     # results of the previous use of this slot are on the host
            runner.submit(host[i % n_sets], to_host=True)

        e2e_regions, _, _ = timed_graph(submit_e2e, args.steps, args.warmup, REPEATS)
        graph_info = {"streams": N_STREAMS, "e2e_regions": e2e_regions}
        runner.close()

    # ---- (2) eager e2e: pinned host -> device -> forward -> device -> host ----------------------
    d2h_bytes = [0]

    def step_e2e(i):
        pc = host[i % n_sets].to(device, non_blocking=True)
        o = forward_resident(model, pc)
        res = [o[k].to("cpu", non_blocking=False) for k in RESULT_KEYS]
        d2h_bytes[0] = sum(r.numel() * r.element_size() for r in res)

    e2e_steps, e2e_wall, _ = timed_loop(step_e2e, args.steps if graph_info is None else min(args.steps, 5),
                                        args.warmup if graph_info is None else 3, flush, barrier)
    eager["e2e_ms_per_step"] = round(sum(e2e_steps) / len(e2e_steps), 4)
    h2d_bytes = host[0].numel() * host[0].element_size()

    # ---- (3) per-kernel event timing (separate pass so the events do not perturb (1)) ----------
    prof_steps = min(args.steps, 5)
    meter.timing = True
    for i in range(prof_steps):
        flush()
        step_resident(i)
    torch.cuda.synchronize()
    meter.timing = False
    agg = meter.summary(prof_steps)
    meter.uninstall()

    # ---- reduce over ranks: every region's time is the max over ranks, then the median region -------
    if graph_info is not None:
        t = torch.tensor([regions, graph_info["e2e_regions"]], device=device, dtype=torch.float64)
    else:
        t = torch.tensor([[dev_s * 1e3], [sum(e2e_steps)]], device=device, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_regions, e2e_regions = t[0].tolist(), t[1].tolist()
    steps_in_region = args.steps if graph_info is not None else eager_steps
    dev_s = statistics.median(dev_regions) / 1e3
    e2e_s = statistics.median(e2e_regions) / 1e3
    e2e_steps_in_region = args.steps if graph_info is not None else len(e2e_steps)
    total_scenes = spg * world * steps_in_region
    hbm_peak, tf_peak, peak_src = peaks()

    ops = {}
    step_ms_kernels = 0.0
    for name, d in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        ms = d["ms"] / prof_steps
        step_ms_kernels += ms
        ops[name.replace("spc_", "")] = {
            "launches_per_step": d["launches"] // prof_steps, "ms_per_step": round(ms, 4),
            "algo_gbs": round(d["bytes"] / prof_steps / (ms * 1e-3) / 1e9, 1) if ms > 0 else None}
    dom = None
    for name, d in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        if name in ROOFLINE_BOUNDED:
            dom = (name, d)
            break
    roofline = None
    if dom is not None:
        name, d = dom
        avg_ms = d["ms"] / d["launches"]
        avg_bytes = d["bytes"] / d["launches"]
        achieved = avg_bytes / (avg_ms * 1e-3) / 1e9
        avg_flops = d["flops"] / d["launches"]
        tensor_bound = avg_flops / (tf_peak * 1e12) > avg_bytes / (hbm_peak * 1e9)
        if tensor_bound:
            achieved = avg_flops / (avg_ms * 1e-3) / 1e12
        traffic, traffic_src = ncu_traffic("sa_fused", "sa_common.cuh,sa_fused.cu,sa_inline.cu")
        roofline = {"kernel": name.replace("spc_", "").replace("_ex", ""), "bound": "tensor" if tensor_bound else "hbm",
                    "achieved": round(achieved, 2),
                    "peak": tf_peak if tensor_bound else hbm_peak,
                    "unit": "TFLOP/s" if tensor_bound else "GB/s",
                    "frac": round(achieved / (tf_peak if tensor_bound else hbm_peak), 4),
                    "algo_flops_per_launch": int(avg_flops),
                    "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peak_src,
                    "launches_per_step": d["launches"] // prof_steps,
                    "avg_launch_us": round(avg_ms * 1e3, 2), "algo_bytes_per_launch": int(avg_bytes),
                    "share_of_step": round(d["ms"] / prof_steps / eager["ms_per_step"], 4),
                    "share_of": "eager single-stream step (kernels of different batches overlap in graph mode)"}
        if name == "spc_sa_fused_forward_ex":
            # what actually bounds the fused kernels (profiles/r2_sa_fused_limits.md): every fp32 accumulator element
            # is read out of TMEM once by the epilogue warps (tcgen05.ld), at ~64 B/clk per SM
            # (B300_MICROARCH.md, "TMEM-read 64 B/cyc"): 4 B x rows x (C1 if layer 0 is a UMMA) + C2 + C3)
            recs = [r for r in meter.records if r[0] == name]
            acc = sum(4 * r[4][15] * r[4][17] * r[4][18] * ((0 if r[4][3] else r[4][19]) + r[4][20] + r[4][21])
                      for r in recs) / max(len(recs), 1)
            floor_us = acc / (148 * 64 * 1.965e9) * 1e6
            roofline["tmem_read"] = {"accumulator_bytes_per_launch": int(acc), "rate": "64 B/clk/SM x 148 SMs x 1.965 GHz",
                                     "floor_us": round(floor_us, 2), "frac_of_floor": round(floor_us / (avg_ms * 1e3), 4)}
    # the kernel with the largest time share, whatever bounds it.  For the sequential sampler of the raw cloud (SA1;
    # args = (xyz, B, N, npoint, ...)) the meaningful figures are us per round and the SM-time a scene occupies; the
    # later FPS calls run on FPS-ordered inputs and mostly take the verified shortcut, so they are not "rounds"
    dominant = None
    if agg:
        name, d = max(agg.items(), key=lambda kv: kv[1]["ms"])
        dominant = {"kernel": name.replace("spc_", ""), "ms_per_step": round(d["ms"] / prof_steps, 4),
                    "launches_per_step": d["launches"] // prof_steps,
                    "share_of_step": round(d["ms"] / prof_steps / eager["ms_per_step"], 4),
                    "share_of": "eager single-stream step"}
        fps_recs = [r for r in meter.records if r[0].startswith("spc_furthest_point_sampling")]
        if name.startswith("spc_furthest_point_sampling") and fps_recs:
            n_max = max(r[4][2] for r in fps_recs)
            big = [r for r in fps_recs if r[4][2] == n_max]
            ms = sum(r[2].elapsed_time(r[3]) for r in big)
            rounds = sum(max(r[4][3] - 1, 0) for r in big)
            dominant.update({
                "bound": "latency (each round depends on the previous pick; no HBM traffic inside the rounds)",
                "what": "furthest_point_sampling N=%d -> %d" % (n_max, big[0][4][3]),
                "us_per_round": round(ms * 1e3 / max(rounds, 1), 4),
                "sequential_rounds_per_step": rounds // prof_steps,
                "single_call_ms": round(ms / len(big), 4),
                "note": "timed with the single-call sampler (thread-block-cluster kernel); the graph pipeline asks for the "
                        "bucketed sampler, see `pipeline_sampler`"})
            # the sampler the graph pipeline uses, timed alone on the same batch
            from spacap3d_b200 import _ext
            xyz0 = resident[0][..., :3].contiguous()
            with _ext.launch_options(fps_algo=_ext.FPS_BUCKET):
                for _ in range(2):
                    _ext.furthest_point_sampling_with_xyz(xyz0, big[0][4][3])
                ts = []
                for _ in range(5):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    _ext.furthest_point_sampling_with_xyz(xyz0, big[0][4][3])
                    e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
            dominant["pipeline_sampler"] = {
                "algo": "bucketed (Hilbert-sorted points parked in L2, one 512-thread CTA per scene)",
                "single_call_ms": round(statistics.median(ts), 4),
                "us_per_round": round(statistics.median(ts) * 1e3 / max(big[0][4][3] - 1, 1), 4),
                "why": "2.5x the latency of the cluster kernel but 1/5 of its instructions and 1/3 of its SM-time "
                       "(profiles/r2_fps_ncu.txt): with 32 batches in flight the pipeline is bound by issue slots, not by "
                       "one call's latency"}

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_baseline(model)
    hbm_ops = hbm_bound_ops(resident[0], flush, hbm_peak) if rank == 0 and world == 1 else None

    if rank == 0:
        cfg = workload_config(world)
        cfg.update({
            "precision": "shared-MLP 1x1 convs in fp16 on tcgen05 with fp32 accumulation; point ops fp32/int32",
            "l2": ("inputs larger than L2: %d distinct batches (%.0f MB) rotated; " % (n_sets, n_sets * batch_mb)) +
                  ("CUDA-graph replay on %d streams (batches overlap, no flush possible between them)" % N_STREAMS
                   if graph_info is not None else "256 MiB L2 flush between timed steps"),
            "execution": ("cuda-graph x %d streams" % N_STREAMS) if graph_info is not None else "eager, 1 stream",
            "parallelism": "scenes sharded by batch, %d rank(s), no collective" % world,
            "cpu_affinity": ("%d cores per rank, local to the rank's GPU when NVML says which are" % len(cpus))
                            if cpus else "inherited"})
        line = {
            "metric": "detector scenes/s @40k pts", "value": round(total_scenes / dev_s, 3),
            "unit": "scenes/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dev_s / steps_in_region * 1e3, 4), "higher_is_better": True,
            "scaling": CFG["scaling"], "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": cfg,
            "timed_regions": {"what": "%d regions of exactly %d steps, each bracketed by barrier + synchronize; "
                                      "value = median region" % (len(dev_regions), steps_in_region),
                              "device": region_stats(dev_regions), "e2e": region_stats(e2e_regions)},
            "e2e": {"value": round(spg * world * e2e_steps_in_region / e2e_s, 3), "unit": "scenes/s",
                    "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes[0]),
                    "ms_per_step": round(e2e_s / e2e_steps_in_region * 1e3, 4)},
            "gpu_launches": int(launches_per_step * args.steps),
            "gpu_launches_per_step": int(launches_per_step),
            "fast_path_check": {
                "fused_sa_launches_per_step": ops.get("sa_fused_forward_ex", {}).get("launches_per_step", 0),
                "expected": 5, "pm_linear_launches_per_step": ops.get("pm_linear", {}).get("launches_per_step", 0),
                "note": "5 fused set-abstraction launches (SA1-4 + vote aggregation) and 14 pm_linear layers per forward: "
                        "anything less means a layer fell back to the unfused kernels (a RuntimeWarning says which)"},
            "roofline": roofline, "dominant": dominant, "hbm_ops": hbm_ops, "ops": ops,
            "kernel_ms_per_step": round(step_ms_kernels, 4),
            "eager": eager,
            "cpu_baseline": cpu_base, "clocks": clocks,
            "wall_s_timed_region": round(wall, 4),
        }
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_step)
    if dist is not None:
        dist.destroy_process_group()


def run_train(args, rank, world, local, device, dist, barrier):
    """BASELINE config 5: forward + backward of the detector in training mode (autograd through the unfused
    sm_100a kernels and their backward passes + cuDNN convolutions + the fused BN/ReLU/max-pool training kernels)
    and ONE flat NCCL all-reduce of the gradients per step (the reference: nn.DataParallel, scripts/train.py:198-200).
    The loss is a surrogate (mean square of the head outputs): lib/loss_helper.py is outside the path.
    Forward + backward are captured once into a CUDA graph (the step has no host synchronisation: the box decode
    stays on the device) and replayed on a static input; the all-reduce runs after the replay."""
    from tools import bench_train
    from spacap3d_b200.dist import allreduce_gradients
    from spacap3d_b200.scenes import make_scene
    n, spg = args.points, scenes_per_gpu(world)
    scale = max(1, round(n / 40000))
    model = bench_train.build_model(scale, device)
    n_sets = 3
    host = [torch.from_numpy(np.stack([make_scene(5000 + 100 * rank + 10 * s + i, n, **CFG["scene_kw"])
                                       for i in range(spg)], 0)).pin_memory() for s in range(n_sets)]
    resident = [h.to(device) for h in host]
    flush = L2Flusher(device)
    static_in = torch.empty_like(resident[0])
    launches = [0]
    from spacap3d_b200 import _lib
    orig = _lib.call

    def counting(name, *a):
        launches[0] += 1
        return orig(name, *a)

    def fwd_bwd():
        out = model({"point_clouds": static_in})
        loss = bench_train.surrogate_loss(out)
        loss.backward()
        return loss.detach()

    static_in.copy_(resident[0])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):                                     # lazy initialisations outside the capture
            model.zero_grad(set_to_none=True)
            fwd_bwd()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    model.zero_grad(set_to_none=True)
    _lib.call = counting
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_loss = fwd_bwd()
    _lib.call = orig
    launches_per_step = launches[0]
    ar_events = []

    def step(pc, timed_ar=False):
        static_in.copy_(pc, non_blocking=True)
        graph.replay()
        if world > 1:
            if timed_ar:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                allreduce_gradients(model)
                e1.record()
                ar_events.append((e0, e1))
            else:
                allreduce_gradients(model)
        return static_loss

    per_step, wall, clocks = timed_loop(lambda i: step(resident[i % n_sets], True), args.steps, args.warmup, flush,
                                        barrier, ClockSampler(local))
    last_step = {"loss": static_loss.clone(),
                 "gradients": torch.cat([p.grad.reshape(-1) for p in model.parameters() if p.grad is not None])}
    loss_holder = {}

    def step_e2e(i):
        loss_holder["l"] = float(step(host[i % n_sets]))       # pinned host -> device ... device -> host read of the loss

    e2e_steps, _, _ = timed_loop(step_e2e, args.steps, args.warmup, flush, barrier)
    t = torch.tensor([sum(per_step), sum(e2e_steps)], device=device, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_s, e2e_s = float(t[0]) / 1e3, float(t[1]) / 1e3
    ar_us = [a.elapsed_time(b) * 1e3 for a, b in ar_events[-args.steps:]] if ar_events else []
    n_params = sum(p.numel() for p in model.parameters())
    # the collective alone: the same flat buffer, ranks aligned by a barrier, 20 back-to-back all-reduces
    iso_us = None
    if dist is not None:
        flat = torch.zeros(n_params, device=device)
        for _ in range(5):
            dist.all_reduce(flat)
        torch.cuda.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            dist.all_reduce(flat)
        e1.record()
        torch.cuda.synchronize()
        iso_us = e0.elapsed_time(e1) * 1e3 / 20
    if rank == 0:
        cfg = workload_config(world)
        cfg.update({"points": n, "sa_npoint_scale": scale, "mode": "training: forward + backward + gradient all-reduce",
                    "weights": "random init (seed 0), train mode",
                    "l2": "256 MiB L2 flush between timed steps",
                    "execution": "forward + backward as one CUDA graph, 1 stream; all-reduce after the replay",
                    "parallelism": "scenes sharded by batch, %d rank(s), one flat NCCL all-reduce of %d gradients "
                                   "(%.1f MB) per step" % (world, n_params, n_params * 4 / 1e6)})
        line = {"metric": "detector training scenes/s (fwd+bwd+allreduce)", "value": round(spg * world * args.steps / dev_s, 3),
                "unit": "scenes/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(dev_s / args.steps * 1e3, 4), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
                "e2e": {"value": round(spg * world * args.steps / e2e_s, 3), "unit": "scenes/s",
                        "h2d_bytes_per_step": int(host[0].numel() * 4), "d2h_bytes_per_step": 4,
                        "ms_per_step": round(e2e_s / args.steps * 1e3, 4)},
                "allreduce": {"in_step_median_us": round(statistics.median(ar_us), 1) if ar_us else None,
                              "isolated_us": round(iso_us, 1) if iso_us is not None else None,
                              "bytes": n_params * 4,
                              "note": "in_step: CUDA events around dist.allreduce_gradients on rank 0 (flatten + NCCL "
                                      "all-reduce + scatter back; includes waiting for the slowest rank's backward); "
                                      "isolated: the NCCL all-reduce of the same flat buffer alone, ranks aligned"},
                "gpu_launches": int(launches_per_step * args.steps), "gpu_launches_per_step": int(launches_per_step),
                "roofline": None, "cpu_baseline": None, "clocks": clocks, "wall_s_timed_region": round(wall, 4)}
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_step)
    if dist is not None:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# reference-structured pipeline on an arbitrary op provider (reference CUDA ext or the CPU oracle)
class OracleOps:
    """The nine `_ext` entry points on CPU torch tensors, backed by the C oracle (port)."""

    def __init__(self):
        import oracle
        self.o = oracle

    @staticmethod
    def _t(a):
        return torch.from_numpy(a)

    def furthest_point_sampling(self, p, n):
        return self._t(self.o.furthest_point_sampling(p.numpy(), n))

    def gather_points(self, p, i):
        return self._t(self.o.gather_points(p.numpy(), i.numpy()))

    def ball_query(self, q, p, r, ns):
        return self._t(self.o.ball_query(q.numpy(), p.numpy(), r, ns))

    def group_points(self, p, i):
        return self._t(self.o.group_points(p.numpy(), i.numpy()))

    def three_nn(self, u, k):
        d, i = self.o.three_nn(u.numpy(), k.numpy())
        return [self._t(d), self._t(i)]

    def three_interpolate(self, p, i, w):
        return self._t(self.o.three_interpolate(p.numpy(), i.numpy(), w.numpy()))

    def gather_points_grad(self, g, i, n):
        return self._t(self.o.gather_points_grad(g.numpy(), i.numpy(), n))

    def group_points_grad(self, g, i, n):
        return self._t(self.o.group_points_grad(g.numpy(), i.numpy(), n))

    def three_interpolate_grad(self, g, i, w, m):
        return self._t(self.o.three_interpolate_grad(g.numpy(), i.numpy(), w.numpy(), m))


class swapped_ops:
    """Route pointnet2_utils / pointnet2_modules to another op provider and force the
    reference's unfused op sequence (FPS -> gather -> ball query -> 2x grouping -> cat -> MLP)."""

    def __init__(self, provider, host_decode):
        self.provider, self.host_decode = provider, host_decode

    def __enter__(self):
        from spacap3d_b200 import detector, pointnet2_modules, pointnet2_utils
        self.mods = (pointnet2_utils, pointnet2_modules)
        self.saved = [(m, m._ext) for m in self.mods]
        for m in self.mods:
            m._ext = self.provider
        self.saved_fast = pointnet2_modules.FAST_PATHS
        pointnet2_modules.FAST_PATHS = False
        self.saved_decode = detector.ProposalModule.decode_pred_box
        if self.host_decode:
            detector.ProposalModule.decode_pred_box = reference_host_decode
        return self

    def __exit__(self, *exc):
        from spacap3d_b200 import detector, pointnet2_modules
        for m, e in self.saved:
            m._ext = e
        pointnet2_modules.FAST_PATHS = self.saved_fast
        detector.ProposalModule.decode_pred_box = self.saved_decode


def reference_host_decode(self, data_dict):
    """The reference's decode_pred_box (models/proposal_module.py:81-104): device->host, numpy,
    Python loop over the batch, host->device.  Used by the reference arm only."""
    center = data_dict["center"].detach().cpu().numpy()
    size_class = torch.argmax(data_dict["size_scores"], -1)
    residual = torch.gather(data_dict["size_residuals"], 2,
                            size_class.unsqueeze(-1).unsqueeze(-1).repeat(1, 1, 1, 3))
    size_class = size_class.detach().cpu().numpy()
    residual = residual.squeeze(2).detach().cpu().numpy()
    signs = np.array([[1, 1, 1], [1, -1, 1], [-1, -1, 1], [-1, 1, 1],
                      [1, 1, -1], [1, -1, -1], [-1, -1, -1], [-1, 1, -1]], np.float64)
    boxes = []
    for i in range(center.shape[0]):
        size = self.mean_size_arr[size_class[i]] + residual[i]
        corners = signs[None] * (size / 2)[:, None, :] + center[i][:, None, :].astype(np.float64)
        boxes.append(torch.from_numpy(corners).to(data_dict["center"].device).unsqueeze(0))
    return torch.cat(boxes, 0)


def cpu_baseline(model_gpu, budget_s=12.0):
    """BASELINE.json configs[0]: one 40k-point scene, batch 1, full detector forward with the CPU
    oracle ops (C port of the reference kernels, OpenMP) + torch CPU MLPs, on the host cores."""
    import copy
    from spacap3d_b200.scenes import make_scene
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = copy.deepcopy(model_gpu).to("cpu").eval()
    scenes = [torch.from_numpy(make_scene(1000 + i, N_POINTS, **CFG["scene_kw"])[None]) for i in range(2)]
    n, t0 = 0, time.perf_counter()
    with swapped_ops(OracleOps(), host_decode=False), torch.no_grad():
        model({"point_clouds": scenes[0]})          # warm-up (page-in, thread pools)
        t0 = time.perf_counter()
        while True:
            model({"point_clouds": scenes[n % 2]})
            n += 1
            el = time.perf_counter() - t0
            if el > budget_s or n >= 200:        # a bounded sample of ~12 s of CPU work
                break
    return {"value": round(n / el, 4), "unit": "scenes/s", "cores": cores, "kind": "port",
            "sample": "%d forward(s) of one 40k-pt scene, batch 1 (configs[0]), %.1f s; oracle C ops "
                      "(OpenMP) + torch CPU MLP" % (n, el)}


def run_reference(args):
    """Reference arm: the reference's UNMODIFIED Python stack (SpaCapNet detection branch, models/*.py,
    lib/pointnet2/*.py staged under baseline/_ref) on its own CUDA extension (oracle/_ref), one replica per rank,
    same workload config, same weights; timed like the eager pass of our arm (CUDA events per step, L2 flush between
    steps).  Falls back to the CPU oracle port when the stack or the extension is not loadable."""
    rank, world, local = dist_env()
    stack, why = None, ""
    if CFG["id"] == 5:
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "config 5 (training sweep) has no reference arm in "
                              "bench.py; tools/bench_train.py --ref times the reference extension on the same step"}))
        return
    if torch.cuda.is_available():
        try:
            from oracle import refstack
            stack = refstack.load_stack("reference")
        except Exception as e:  # noqa: BLE001
            why = "reference stack not loadable (%s: %s); CPU port used" % (type(e).__name__, str(e)[:80])
    else:
        why = "no GPU; CPU port used"
    config = workload_config(world)
    spg = scenes_per_gpu(world)
    if stack is not None:
        from oracle import refstack
        torch.cuda.set_device(local)
        device = torch.device("cuda", local)
        dist, barrier = init_dist(local, device, world)
        model = refstack.build_detector(stack, CFG["feature_dim"], device, pretrained=checkpoint_file() is not None)
        if checkpoint_file() is None:
            ours = make_detector("cpu")                   # same random weights as our arm
            model.load_state_dict(ours.state_dict(), strict=True)
        host = make_host_batches(rank, world)
        n_sets = len(host)
        resident = [h.to(device) for h in host]
        flush = L2Flusher(device)

        out_holder = {}

        def step(i):
            out_holder["o"] = forward_resident(model, resident[i % n_sets])
        per_step, wall, clocks = timed_loop(step, args.steps, args.warmup, flush, barrier, ClockSampler(local))
        t = torch.tensor([sum(per_step)], device=device, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        s = float(t[0]) / 1e3
        val = spg * world * args.steps / s
        if rank == 0:
            line = {"impl": "reference", "metric": "detector scenes/s @40k pts", "value": round(val, 3),
                    "unit": "scenes/s", "n_gpus": world, "ranks_used": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": round(s / args.steps * 1e3, 4), "higher_is_better": True,
                    "scaling": CFG["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": config, "device": "cuda",
                    "arm": "UNMODIFIED reference stack (baseline/_ref: models/SpaCapNet.py detection branch, "
                           "backbone/voting/proposal modules, lib/pointnet2/*.py, host-side box decode) on the "
                           "reference's CUDA ops rebuilt for sm_100a (oracle/_ref); torch defaults (TF32 convs); "
                           "eager, one replica per rank, 256 MiB L2 flush between timed steps",
                    "cpu_baseline": {"value": round(val, 3), "unit": "scenes/s", "cores": 0, "kind": "reference",
                                     "sample": "%d steps x %d scenes per GPU on the GPU (the reference has no CPU "
                                               "path: 'CPU not supported', sampling.cpp:33-35)" % (args.steps, spg)},
                    "e2e": {"value": round(val, 3), "unit": "scenes/s", "h2d_bytes_per_step": 0,
                            "d2h_bytes_per_step": 0},
                    "clocks": clocks}
            print(json.dumps(line))
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, {k: out_holder["o"][k] for k in RESULT_KEYS})
        if dist is not None:
            dist.destroy_process_group()
        return
    if rank != 0:
        return
    # CPU port: bounded sample = `steps` single-scene forwards
    model = make_detector("cpu")
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    from spacap3d_b200.scenes import make_scene
    scene = torch.from_numpy(make_scene(1000, N_POINTS, **CFG["scene_kw"])[None])
    steps = max(1, min(args.steps, 5))
    with swapped_ops(OracleOps(), host_decode=True), torch.no_grad():
        for _ in range(min(args.warmup, 1)):
            model({"point_clouds": scene})
        t0 = time.perf_counter()
        for _ in range(steps):
            out = model({"point_clouds": scene})
        el = time.perf_counter() - t0
    val = steps / el
    line = {"impl": "reference", "metric": "detector scenes/s @40k pts", "value": round(val, 4),
            "unit": "scenes/s", "n_gpus": world, "ranks_used": 1, "steps": steps, "warmup": min(args.warmup, 1),
            "ms_per_step": round(el / steps * 1e3, 3), "higher_is_better": True, "scaling": CFG["scaling"],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "device": "cpu", "arm": "CPU oracle port, batch 1 per step; " + why,
            "cpu_baseline": {"value": round(val, 4), "unit": "scenes/s", "cores": cores, "kind": "port",
                             "sample": "%d single-scene forwards" % steps},
            "e2e": {"value": round(val, 4), "unit": "scenes/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: out[k] for k in RESULT_KEYS})


def main():
    global N_STREAMS, CFG, N_POINTS
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="K, timed steps per measured region.  Graph mode (headline): %d regions of exactly K steps "
                         "each, on device-resident and on host inputs; its secondary passes time min(K, 60) eager "
                         "steps, min(K, 5) eager host-to-host steps and min(K, 5) steps of per-kernel events.  "
                         "Eager mode and config 5: exactly K steps.  --impl reference: K steps on the reference's "
                         "CUDA stack, min(K, 5) forwards on the CPU port" % REPEATS)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json workload")
    ap.add_argument("--points", type=int, default=N_POINTS, help="points per scene (config 5: 40000..200000)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streams", type=int, default=N_STREAMS, help="graph replay streams (batches in flight)")
    ap.add_argument("--pm-n-tile", type=int, default=None, help="tuning: pm_linear output channels per CTA in the graphs")
    ap.add_argument("--sa-min-tiles", type=int, default=None, help="tuning: fused-SA tiles per CTA in the graphs")
    ap.add_argument("--pm-tiles-per-cta", type=int, default=None, help="tuning: pm_linear row tiles per CTA in the graphs")
    ap.add_argument("--mode", default="graph", choices=["graph", "eager"],
                    help="graph: CUDA-graph replay on %d streams (headline); eager: plain launches" % N_STREAMS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path computed in its last step (rank 0) as "
                         "DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    N_STREAMS = max(1, args.streams)
    CFG = dict(CONFIGS[args.config], id=args.config)
    if args.config != 5:
        N_POINTS = args.points
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
