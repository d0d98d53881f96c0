"""Training throughput through the PUBLIC API (`train.fit`: dataset reader -> shuffled batches -> collate -> H2D ->
DiffusionLoss.__call__ -> backward -> fused Adam) on a synthetic Alexandria-shaped dataset written to the .npz twin of
the reference's HDF5 format: python scratch/fit_throughput.py [crystals] [batch] [epochs] [ema_decay]

With ema_decay the optimizer keeps the EMA of the weights (FusedAdam).  Every epoch writes last.ckpt (and its -EMA twin)
to a temporary checkpoint directory; the time of each write is printed."""
import os
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arreau_b200.diffusion.lattice_dataset import CrystalDataset, save_dataset_npz  # noqa: E402
from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION  # noqa: E402
from arreau_b200.synthetic import make_training_batch  # noqa: E402
from arreau_b200.train import default_args, fit  # noqa: E402

n_cryst = int(sys.argv[1]) if len(sys.argv) > 1 else 8100
batch = int(sys.argv[2]) if len(sys.argv) > 2 else 270
epochs = int(sys.argv[3]) if len(sys.argv) > 3 else 3
ema_decay = float(sys.argv[4]) if len(sys.argv) > 4 else None
dev = torch.device("cuda")
cr = make_training_batch(n_cryst, seed=5)
off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
zs = [cr.types[off[i]:off[i + 1]] % 89 + 1 for i in range(n_cryst)]
frac = [cr.frac[off[i]:off[i + 1]] for i in range(n_cryst)]
lat = np.stack([np.diag(cr.lengths[i]) for i in range(n_cryst)])
path = save_dataset_npz(os.path.join(tempfile.mkdtemp(), "synthetic"), zs, lat, frac)
t0 = time.time()
ds = CrystalDataset([path])
print(f"dataset: {len(ds)} crystals, {int(cr.num_atoms.sum())} atoms, {len(ds.z_table)} states, loaded in {time.time() - t0:.1f} s", flush=True)
torch.manual_seed(0)
model = PONITA_DIFFUSION(default_args(lr=3e-4, epochs=epochs, warmup=0, batch_size=batch), ds.z_table)
marks = []
writes = []
_save = PONITA_DIFFUSION.save_checkpoint


def timed_save(self, path, training_state=None):
    t = time.time()
    _save(self, path, training_state)
    writes.append((os.path.basename(path), time.time() - t))


PONITA_DIFFUSION.save_checkpoint = timed_save


def log(msg):
    torch.cuda.synchronize()
    marks.append(time.time())
    print(msg, flush=True)


torch.cuda.synchronize()
marks.append(time.time())
fit(model, ds, epochs, batch, dev, backward_precision="tf32", log=log, checkpoint_dir=tempfile.mkdtemp(),
    ema_decay=ema_decay)
steps = (n_cryst + batch - 1) // batch
# the log line of epoch e comes before its checkpoint writes: epochs after the first include the previous epoch's writes
per_epoch = len(writes) // epochs
for e in range(epochs):
    dt = marks[e + 1] - marks[e] - (sum(w for _, w in writes[(e - 1) * per_epoch:e * per_epoch]) if e else 0.0)
    print(f"epoch {e} (ema_decay {ema_decay}): {dt:.3f} s = {dt / steps * 1e3:.2f} ms per step, {n_cryst / dt:.0f} crystals/s")
for name, dt in writes:
    print(f"write {name}: {dt * 1e3:.1f} ms")
dl = model.diffusion_loss
print("train engines built:", dl.train_engine_builds)
