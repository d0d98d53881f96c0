"""The fused Adam step with and without the EMA update, alternated: device time per step (CUDA events over 500 steps,
median of 11 rounds each) on the model's 1 170 646 parameters.  python scratch/adam_ema_time.py"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arreau_b200.training import FlatParams, FusedAdam  # noqa: E402

dev = torch.device("cuda")
p = FlatParams(164, 4, 90, dev)
p.data.normal_()
p.grad.normal_()
opts = {"no EMA": FusedAdam(p, lr=1e-12), "EMA": FusedAdam(p, lr=1e-12, ema_decay=0.999)}
times = {k: [] for k in opts}
for k, o in opts.items():                       # warm-up (module load, first EMA copy)
    for _ in range(20):
        o.step()
for _ in range(11):
    for k, o in opts.items():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(500):
            o.step()
        b.record()
        b.synchronize()
        times[k].append(a.elapsed_time(b) / 500 * 1e3)
for k, t in times.items():
    print(f"{k}: {np.median(t):.2f} us per step (arreau_moments + arreau_adam_step), rounds {np.round(t, 2).tolist()}")
print(f"EMA adds {np.median(times['EMA']) - np.median(times['no EMA']):.2f} us; "
      f"bytes per step: {p.total * 4 * 2 / 1e6:.1f} MB more traffic")
