"""Cost of sample-quality monitoring and of keyed sampling noise, with the card name and power limit:

    python scratch/sample_quality_time.py [crystals in the synthetic data set]

1. The wall time of one monitoring pass of train.fit (SampleMonitor.run: 1024 crystals, atom counts drawn from a
   synthetic Alexandria-shaped training split, fp16 sampling twin, CUDA-graph trajectory of T = 1000, crystal_metrics,
   summary against the validation split).  The first pass also builds the twin and the reference metrics; the next
   passes are the steady cost per monitored epoch.  The weights are the golden seed-0 weights with the length read-out
   calibrated (quirk B7) for the data's mean cell, so the graph stays populated as in a trained model.
2. Keyed (arreau_sample_noise_keyed) against per-batch (arreau_step_noise) step noise on the headline C2 step (1024
   crystals x 40 atoms, fp16, max_neighbors 8): the noise launch alone and noise + arreau_denoise_step, alternated
   within this one command, CUDA events, 5 rounds of 50 steps each."""
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from arreau_b200.diffusion.lattice_dataset import CrystalDataset, CrystalSubset, save_dataset_npz, split_indices  # noqa: E402
from arreau_b200.engine import DenoiseEngine  # noqa: E402
from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION  # noqa: E402
from arreau_b200.synthetic import calibrate_length_readout, make_crystals, make_training_batch  # noqa: E402
from arreau_b200.tables import build_tables  # noqa: E402
from arreau_b200.train import SampleMonitor, default_args, format_quality  # noqa: E402
from arreau_b200.weights import PonitaWeights  # noqa: E402

n_cryst = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
dev = torch.device("cuda")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
w = np.load(os.path.join(ROOT, "tests", "golden", "weights_seed0.npz"))

# ---- 1. one monitoring pass ------------------------------------------------------------------------------------------
cr = make_training_batch(n_cryst, seed=5)
off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
zs = [cr.types[off[i]:off[i + 1]] % 89 + 1 for i in range(n_cryst)]
path = save_dataset_npz(os.path.join(tempfile.mkdtemp(), "synthetic"), zs,
                        np.stack([np.diag(cr.lengths[i]) for i in range(n_cryst)]),
                        [cr.frac[off[i]:off[i + 1]] for i in range(n_cryst)])
ds = CrystalDataset([path])
tr_idx, va_idx = split_indices(len(ds), [0.9, 0.1], seed=0)
tr, va = CrystalSubset(ds, tr_idx), CrystalSubset(ds, va_idx)
print(f"dataset {len(ds)} crystals ({int(cr.num_atoms.sum())} atoms), valid split {len(va)}", flush=True)
torch.manual_seed(0)
model = PONITA_DIFFUSION(default_args(), ds.z_table, ori_grid=w["ori_grid"])
n_states = len(ds.z_table)
sd = {k: torch.as_tensor(v) for k, v in w.items() if k not in ("ori_grid", "fourier_w")}
own = model.model.state_dict()
if all(k in own and tuple(own[k].shape) == tuple(v.shape) for k, v in sd.items()):
    sd = calibrate_length_readout(sd, int(round(float(cr.num_atoms.mean()))), first_row=n_states + 1)
    model.model.load_state_dict(sd)
    with torch.no_grad():
        model.t_emb.gaussian_fourier_proj_w.copy_(torch.as_tensor(w["fourier_w"]))
    print("weights: golden seed-0, length read-out calibrated", flush=True)
else:
    print(f"weights: random initialisation (the golden weights are for 90 states, the data has {n_states})", flush=True)
model.to(dev)
flat = model.model.flatten_parameters(dev)
mon = SampleMonitor(model, flat, tr, va, 1024, 0, dev)
print(f"monitoring pass: 1024 crystals, {int(mon.num_atoms.sum())} atoms (mean {mon.num_atoms.mean():.2f}, max "
      f"{mon.num_atoms.max()}), T = {model.diffusion_loss.T}", flush=True)
for i in range(4):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = mon.run(i)                       # ends in device -> host reads
    dt = time.perf_counter() - t0
    print(f"pass {i}: {dt * 1e3:.0f} ms{' (builds the twin and the reference metrics)' if i == 0 else ''}; "
          f"{format_quality(rec)}", flush=True)
torch.cuda.synchronize()
t0 = time.perf_counter()
mon.local_metrics()
print(f"sampling + crystal_metrics only: {(time.perf_counter() - t0) * 1e3:.0f} ms", flush=True)
del mon, model
torch.cuda.empty_cache()

# ---- 2. keyed against per-batch step noise on the C2 step ----------------------------------------------------------------
c2 = make_crystals(1024, 40, None, seed=0)
sd = calibrate_length_readout({k: w[k] for k in w.files if k not in ("ori_grid", "fourier_w")}, 40)
eng = DenoiseEngine(PonitaWeights(sd, w["ori_grid"], device=dev), build_tables(1000, 90), w["fourier_w"], c2.num_atoms,
                    5.0, 8, precision="fp16", device=dev)
eng.set_crystal_ids(torch.arange(1024))
print(f"C2 step: {eng.G} crystals, {eng.N} atoms, fp16, max_neighbors 8", flush=True)
draws = {"per-batch": lambda k: eng.draw_noise(7, k), "keyed": lambda k: eng.draw_noise_keyed(7, k)}


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(iters):
        fn(k)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


res = {(n, what): [] for n in draws for what in ("noise", "noise+step")}
for rnd in range(6):                       # round 0 is warm-up
    for name, draw in draws.items():
        ms = timed(draw, 200)
        eng.set_state(c2.frac, c2.types, c2.lengths, c2.angles)

        def one(k):
            draw(k)
            eng.step(999 - k)

        ms_step = timed(one, 50)
        if rnd:
            res[(name, "noise")].append(ms)
            res[(name, "noise+step")].append(ms_step)
for (name, what), v in res.items():
    v = np.asarray(v)
    print(f"{name:9s} {what:10s}: median {np.median(v) * 1e3:8.1f} us  (min {v.min() * 1e3:.1f}, max {v.max() * 1e3:.1f}, "
          f"5 rounds)", flush=True)
