#!/usr/bin/env python
"""Device time of wbc_sample_trajectory by batch size; the sizes cover all three instances-per-warp shapes of the sampler
kernel (2 / 8 / 32): python tools/sweep_sampler.py  -> one line per size."""
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np
import torch
from quadruped_drake_b200 import planner as pl
from quadruped_drake_b200.controller import BatchedController

ctl = BatchedController("mini_cheetah", device=0)
s = pl.TrajectorySampler(ctl, [pl.make_gait_plan("mini_cheetah", g) for g in range(4)])
dev = torch.device("cuda:0")
rng = np.random.default_rng(0)
for n in (1, 256, 4096, 16384, 65536, 262144, 1 << 20):
    t = torch.from_numpy(rng.uniform(0, 2.5, n)).to(dev)
    pi = torch.from_numpy(rng.integers(0, 4, n).astype(np.int32)).to(dev)
    for _ in range(5):
        s.sample(t, pi)
    torch.cuda.synchronize()
    reps = 200 if n <= 65536 else 30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        s.sample(t, pi)
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    print("n %8d  %9.2f us per call  %8.1f M samples/s" % (n, us, n / us))
