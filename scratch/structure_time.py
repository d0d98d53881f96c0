"""Cost of structure-conditioned sampling on the headline C2 shape (1024 crystals x 40 atoms, fp16, radius 5,
max_neighbors 8), with the card name and power limit:

    python scratch/structure_time.py [rounds, default 3]

The crystals are a synthetic data set (Li-Fe-P-O compositions, random cells of 9-11 A, random positions) drawn as
`generate --structures_from D` draws them.
1. One C2 denoise step (arreau_denoise_step, type update on, so all three known-row reverse kernels run) unconditioned
   and with known lattices and the non-Li atoms known, CUDA events over 50 steps at t = 500, the two alternated round
   by round.
2. One whole C2 trajectory (T = 1000: 999 replays of the captured step, keyed noise, PONITA_DIFFUSION.sample with
   cuda_graph) with the drawn compositions, without and with `--fix_lattice --free_elements Li` (lattices and sites of
   the same draws), host clock around work that ends in the device-to-host copy of the result, alternated round by
   round.  The golden seed-0 weights with the length read-out calibrated for 40 atoms (quirk B7)."""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from arreau_b200.diffusion.lattice_dataset import CrystalDataset, save_dataset_npz  # noqa: E402
from arreau_b200.generate import draw_compositions, known_structures  # noqa: E402
from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION, known_lattice_array, known_site_arrays  # noqa: E402
from arreau_b200.synthetic import calibrate_length_readout  # noqa: E402
from arreau_b200.tools.atomic_number_table import AtomicNumberTable  # noqa: E402

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
G, A, Z = 1024, 40, 90
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

rng = np.random.default_rng(0)
zs = [rng.choice([3, 26, 15, 8], A) for _ in range(2 * G)]
with tempfile.TemporaryDirectory() as tmp:
    path = save_dataset_npz(os.path.join(tmp, "lfpo.npz"), zs,
                            np.stack([np.diag(rng.uniform(9, 11, 3)) + rng.uniform(-1, 1, (3, 3)) for _ in zs]),
                            [rng.random((A, 3)) for _ in zs])
    data = CrystalDataset([path])
    idx, _ = draw_compositions(data, G, seed=0)
    comps, lattices, sites = known_structures(data, idx, True, ["Li"])
ids = torch.arange(G, dtype=torch.int64)
known = sum(0 if s is None else len(s[0]) for s in sites)
print(f"C2: {G} crystals x {A} atoms, fp16, max_neighbors 8; {known} of {G * A} atoms known, every lattice known",
      flush=True)

# ---- 1. one step --------------------------------------------------------------------------------------------------
m.sample(None, G, compositions=comps, crystal_ids=ids, seed=0, device=dev, cuda_graph=True)   # builds the engine
eng = m.diffusion_loss._engine
kf, _ = known_site_arrays(sites, [A] * G, comps)
kl = known_lattice_array(lattices, G)
state = [t.clone() for t in (eng.frac, eng.types, eng.lengths, eng.angles, eng.angle_trig)]


def steps(conditioned, n=50):
    for dst, src in zip((eng.frac, eng.types, eng.lengths, eng.angles, eng.angle_trig), state):
        dst.copy_(src)
    eng.set_known(kf, kl) if conditioned else eng.set_known()
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
    print(f"step {'known part   ' if c else 'unconditioned'}: median {np.median(v):8.1f} us  (min {v.min():.1f}, "
          f"max {v.max():.1f}, {len(v)} rounds of 50 steps)", flush=True)
eng.set_known()

# ---- 2. whole trajectory ------------------------------------------------------------------------------------------
res = {False: [], True: []}
for r in range(rounds):
    for c in (False, True):
        kw = dict(lattices=lattices, sites=sites) if c else {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = m.sample(None, G, compositions=comps, crystal_ids=ids, seed=1, device=dev, cuda_graph=True, **kw)
        res[c].append(time.perf_counter() - t0)
for c in (False, True):
    v = np.asarray(res[c])
    print(f"trajectory {'--fix_lattice --free_elements Li' if c else 'compositions only              '}: median "
          f"{np.median(v):.3f} s  (min {v.min():.3f}, max {v.max():.3f}, {len(v)} rounds; {G / np.median(v):.1f} "
          f"crystals/s)", flush=True)
