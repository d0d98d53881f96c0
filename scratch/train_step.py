"""A few C5 training steps (TF32 backward) for ncu launch lists: python scratch/train_step.py [steps]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arreau_b200.diffusion.lattice_helpers import lattice_from_params  # noqa: E402
from arreau_b200.synthetic import make_training_batch  # noqa: E402
from arreau_b200.tables import build_tables  # noqa: E402
from arreau_b200.training import FlatParams, FusedAdam, TrainEngine  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
dev = torch.device("cuda")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
w = np.load(os.path.join(ROOT, "tests", "golden", "weights_seed0.npz"))
sd = {k: w[k] for k in w.files if k not in ("ori_grid", "fourier_w")}
p = FlatParams(164, 4, 90, dev)
p.load_state_dict(sd)
cr = make_training_batch(270, seed=100)
G, N = cr.num_crystals, cr.total_atoms
te = TrainEngine(p, build_tables(1000, 90), w["fourier_w"], w["ori_grid"], cr.num_atoms, 5.0, 8, device=dev, backward_precision="tf32")
opt = FusedAdam(p, lr=3e-4, max_grad_norm=0.5)
lat0 = lattice_from_params(torch.as_tensor(cr.lengths).to(dev), torch.as_tensor(cr.angles).to(dev))
g = torch.Generator(device=dev).manual_seed(7)
frac0, types0 = torch.as_tensor(cr.frac).to(dev), torch.as_tensor(cr.types).to(dev)
times = []
for i in range(steps):
    ts = torch.randint(1, 1001, (G,), device=dev, generator=g)
    eps_x = torch.randn(N, 3, device=dev, dtype=torch.float64, generator=g)
    u = torch.rand(N, 90, device=dev, dtype=torch.float64, generator=g)
    eps_l = torch.randn(G, 3, device=dev, dtype=torch.float64, generator=g)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    te.loss_and_grads(frac0, types0, lat0, ts, eps_x, u, eps_l)
    opt.step()
    e1.record()
    torch.cuda.synchronize()
    times.append(e0.elapsed_time(e1))
print("G", G, "N", N, "E", te.eng.num_edges(), "ms per step", np.round(times, 3).tolist(), "loss", te.loss.tolist()[0])
