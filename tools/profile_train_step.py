#!/usr/bin/env python
"""torch.profiler table of three training steps (4 scenes x 40 k points, forward + backward): where a step's GPU time goes.

    python tools/profile_train_step.py [--amp off|bf16] [--rows 28]

--amp bf16 runs the steps under torch.autocast("cuda", dtype=torch.bfloat16), for a kernel table to set beside the
fp32 one (profiles/r2_train_step_profile.txt)."""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tools')]
import bench_train
from spacap3d_b200.scenes import make_scene

ap = argparse.ArgumentParser()
ap.add_argument("--amp", choices=("off", "bf16"), default="off")
ap.add_argument("--rows", type=int, default=28)
args = ap.parse_args()
dev = torch.device("cuda", 0)
model = bench_train.build_model(1, dev)
pc = torch.from_numpy(np.stack([make_scene(5000 + i, 40000) for i in range(4)], 0)).to(dev)


def one_step():
    model.zero_grad(set_to_none=True)
    with bench_train.amp_context(args.amp):
        bench_train.step(model, pc, 1)


for _ in range(3):
    one_step()
torch.cuda.synchronize()
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(3):
        one_step()
    torch.cuda.synchronize()
print("amp=%s on %s" % (args.amp, torch.cuda.get_device_name(0)))
print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=args.rows, max_name_column_width=90))
