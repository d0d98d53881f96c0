"""Validation throughput of the forward-only evaluation path (evaluation.evaluate_dataset) on a synthetic
Alexandria-shaped split (C5-shaped crystals, 89 element states + mask), fp32 and fp16, at C5-sized GPU batches (270
crystals) and at a large GPU batch; then the extra wall time train.fit spends per epoch on a 10 % validation split.
Prints the card name and power limit with the numbers:  python scratch/eval_throughput.py [crystals]"""
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arreau_b200.diffusion.lattice_dataset import CrystalDataset, CrystalSubset, save_dataset_npz, split_indices  # noqa: E402
from arreau_b200.evaluation import evaluate_dataset  # noqa: E402
from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION  # noqa: E402
from arreau_b200.synthetic import make_training_batch  # noqa: E402
from arreau_b200.train import default_args, fit  # noqa: E402

n_cryst = int(sys.argv[1]) if len(sys.argv) > 1 else 27000
dev = torch.device("cuda")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
cr = make_training_batch(n_cryst, seed=5)
off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
zs = [cr.types[off[i]:off[i + 1]] % 89 + 1 for i in range(n_cryst)]
path = save_dataset_npz(os.path.join(tempfile.mkdtemp(), "synthetic"), zs,
                        np.stack([np.diag(cr.lengths[i]) for i in range(n_cryst)]),
                        [cr.frac[off[i]:off[i + 1]] for i in range(n_cryst)])
ds = CrystalDataset([path])
tr_idx, va_idx = split_indices(len(ds), [0.9, 0.1], seed=0)
tr, va = CrystalSubset(ds, tr_idx), CrystalSubset(ds, va_idx)
print(f"dataset {len(ds)} crystals ({int(cr.num_atoms.sum())} atoms), {len(ds.z_table)} states; valid split {len(va)}",
      flush=True)

for precision in ("fp32", "fp16"):
    torch.manual_seed(0)
    model = PONITA_DIFFUSION(default_args(), ds.z_table, precision=precision).to(dev)
    for gb in (270, 2700):
        evaluate_dataset(model, va, 270, dev, gpu_batch=gb)              # warm-up: engine build, first launches
        torch.cuda.synchronize()
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            res = evaluate_dataset(model, va, 270, dev, gpu_batch=gb)    # ends in a device -> host read
            times.append(time.perf_counter() - t0)
        best = min(times)
        print(f"{precision} gpu_batch {gb}: {len(va) / best:,.0f} valid crystals/s (best of 3: {best * 1e3:.1f} ms for "
              f"{len(va)} crystals; valid loss {res['loss']:.6f})", flush=True)

for val in (None, va):
    torch.manual_seed(0)
    model = PONITA_DIFFUSION(default_args(epochs=2), ds.z_table)
    marks = []

    def log(msg):
        torch.cuda.synchronize()
        marks.append(time.perf_counter())
        print(msg, flush=True)

    t0 = time.perf_counter()
    fit(model, tr, epochs=2, batch_size=270, device=dev, log=log, val_dataset=val)
    print(f"fit {'with' if val is not None else 'without'} a 10 % validation split: epoch 2 took "
          f"{(marks[1] - marks[0]) * 1e3:.0f} ms", flush=True)
