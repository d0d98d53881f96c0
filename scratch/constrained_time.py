"""Cost of chemical-system-constrained sampling on the headline C2 shape (1024 crystals x 40 atoms, fp16, radius 5,
max_neighbors 8), with the card name and power limit:

    python scratch/constrained_time.py [rounds, default 3]

1. One C2 denoise step (arreau_denoise_step) unconstrained and with every crystal in the Li-Fe-P-O system (the
   allowed-state reverse step), CUDA events over 50 steps at t = 500, the two alternated round by round.
2. One whole C2 trajectory (T = 1000: 999 replays of the captured step, keyed noise, PONITA_DIFFUSION.sample with
   cuda_graph) without and with `elements`, host clock around work that ends in the device-to-host copy of the result,
   alternated round by round.  The golden seed-0 weights with the length read-out calibrated for 40 atoms (quirk B7)."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION  # noqa: E402
from arreau_b200.synthetic import calibrate_length_readout  # noqa: E402
from arreau_b200.tools.atomic_number_table import AtomicNumberTable, allowed_states_of_elements  # noqa: E402

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
G, A, Z, SYSTEM = 1024, 40, 90, ["Li", "Fe", "P", "O"]
dev = torch.device("cuda")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
w = np.load(os.path.join(ROOT, "tests", "golden", "weights_seed0.npz"))
args = argparse.Namespace(dataset="synthetic", lr=1e-3, weight_decay=0.0, epochs=1, warmup=0, layer_scale=1e-6,
                          train_augm=False, hidden_dim=128, layers=5, radius=5.0, num_ori=16, basis_dim=256, degree=3,
                          widening_factor=4, multiple_readouts=True, num_timesteps=1000, max_neighbors=8)
zt = AtomicNumberTable(list(range(1, Z)) + [2001])
m = PONITA_DIFFUSION(args, zt, ori_grid=w["ori_grid"], precision="fp16")
sd = calibrate_length_readout({k: w[k] for k in w.files if k not in ("ori_grid", "fourier_w")}, A)
m.model.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})
with torch.no_grad():
    m.t_emb.gaussian_fourier_proj_w.copy_(torch.as_tensor(w["fourier_w"]))
m.to(dev)
ids = torch.arange(G, dtype=torch.int64)
mask = allowed_states_of_elements(zt, SYSTEM, G)

# ---- 1. one step --------------------------------------------------------------------------------------------------
m.sample(A, G, crystal_ids=ids, seed=0, device=dev, cuda_graph=True)      # builds the engine (and warms it)
eng = m.diffusion_loss._engine
print(f"C2 step: {G} crystals, {eng.N} atoms, fp16, max_neighbors 8", flush=True)
state = [t.clone() for t in (eng.frac, eng.types, eng.lengths)]


def steps(constrained, n=50):
    for dst, src in zip((eng.frac, eng.types, eng.lengths), state):
        dst.copy_(src)
    eng.set_allowed_states(mask if constrained else None)
    eng.draw_noise_keyed(0, 499)
    for _ in range(5):
        eng.step(500)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        eng.step(500)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3


res = {False: [], True: []}
for r in range(rounds + 1):
    for c in (False, True):
        us = steps(c)
        if r:                    # round 0 is warm-up
            res[c].append(us)
for c in (False, True):
    v = np.asarray(res[c])
    print(f"step {'elements   ' if c else 'unconstrained'}: median {np.median(v):8.1f} us  (min {v.min():.1f}, "
          f"max {v.max():.1f}, {len(v)} rounds of 50 steps)", flush=True)
eng.set_allowed_states(None)

# ---- 2. whole trajectory ------------------------------------------------------------------------------------------
res = {False: [], True: []}
for r in range(rounds):
    for c in (False, True):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = m.sample(A, G, crystal_ids=ids, seed=1, device=dev, cuda_graph=True, elements=SYSTEM if c else None)
        res[c].append(time.perf_counter() - t0)
        if c:
            assert set(np.unique(out.atomic_numbers).tolist()) <= {3, 26, 15, 8}
for c in (False, True):
    v = np.asarray(res[c])
    print(f"trajectory {'--elements Li Fe P O' if c else 'unconstrained      '}: median {np.median(v):.3f} s  (min "
          f"{v.min():.3f}, max {v.max():.3f}, {len(v)} rounds; {G / np.median(v):.1f} crystals/s)", flush=True)
