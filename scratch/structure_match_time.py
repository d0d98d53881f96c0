"""Time arreau_structure_match on one GPU: 10 000 Alexandria-shaped pairs (make_training_batch statistics, up to 236
atoms, five elements), half of them transformed and displaced copies of their source (sigma 0.05 (V/n)^(1/3), which
match) and half the same compositions at random positions (which mostly do not).  Kernel time from CUDA events (5
launches after 1 warm-up, median of 3 rounds), end-to-end structure_match() from host memory, the kernel against the
numpy oracle of tests/test_structure_match_host.py on a subset, and that oracle's own time on the host CPU.

    python scratch/structure_match_time.py        (profiles/structure_match.txt holds a run)"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from arreau_b200 import _lib  # noqa: E402
from arreau_b200.inference.structure_match import _sorted_by_z, structure_match  # noqa: E402
from arreau_b200.synthetic import make_training_batch  # noqa: E402
from oracle import restatement as R  # noqa: E402
from test_structure_match_host import match_pairs, transformed_copy  # noqa: E402

dev = torch.device("cuda", 0)
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())

G = 10_000
ELEMENTS = np.array([3, 8, 12, 26, 29])
cr = make_training_batch(G, seed=3)
lat = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles)).numpy()
off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
rng = np.random.default_rng(0)
gen, ref = [], []
for g in range(G):
    c = (cr.frac[off[g]:off[g + 1]], lat[g], ELEMENTS[cr.types[off[g]:off[g + 1]] % 5])
    ref.append(c)
    if g % 2 == 0:
        gen.append(transformed_copy(*c, rng, sigma=0.05))
    else:
        n = len(c[2])
        gen.append((rng.random((n, 3)), c[1], c[2][rng.permutation(n)]))


def pack(cs):
    return (np.concatenate([c[0] for c in cs]), np.stack([c[1] for c in cs]), np.concatenate([c[2] for c in cs]),
            np.array([len(c[2]) for c in cs], np.int64))


gi, ri = pack(gen), pack(ref)
print(f"{G} pairs, {int(gi[3].sum())} atoms per set, largest {int(gi[3].max())}, mean {gi[3].mean():.2f}")

# kernel time
bufs = []
for inp in (gi, ri):
    f, L, z, na = _sorted_by_z(inp)
    o = np.concatenate([[0], np.cumsum(na)]).astype(np.int32)
    bufs.append([torch.as_tensor(a).to(dev) for a in (f, L, z, o)])
outs = [torch.empty(G, dtype=torch.float64, device=dev) for _ in range(2)] + \
       [torch.empty(G, dtype=torch.int32, device=dev) for _ in range(2)]
stream = torch.cuda.current_stream(dev).cuda_stream
N = int(gi[3].sum())


def launch():
    _lib.call("arreau_structure_match", *[t.data_ptr() for t in bufs[0]], *[t.data_ptr() for t in bufs[1]], N, N, G,
              0.5, 0.3, 10.0, *[t.data_ptr() for t in outs], stream)


launch()
torch.cuda.synchronize()
rounds = []
for _ in range(3):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        launch()
    b.record()
    b.synchronize()
    rounds.append(a.elapsed_time(b) / 5)
ms = float(np.median(rounds))
flags = outs[3].cpu().numpy()
nm = outs[2].cpu().numpy()
print(f"flags: matched {int((flags & 1).sum())}, composition {int(((flags & 2) != 0).sum())}, degenerate "
      f"{int(((flags & 4) != 0).sum())}, search limit {int(((flags & 8) != 0).sum())}, too large "
      f"{int(((flags & 16) != 0).sum())}; matched among copies {int((flags[0::2] & 1).sum())} of {G // 2}, among "
      f"random positions {int((flags[1::2] & 1).sum())} of {G // 2}; mappings per pair mean {nm.mean():.1f}, max {nm.max()}")
print(f"kernel {ms:.2f} ms per launch ({G / ms * 1e3:.0f} pairs/s; median of 3 rounds of 5 launches, rounds "
      f"{np.round(rounds, 2).tolist()})")

t = []
for _ in range(3):
    t0 = time.perf_counter()
    m = structure_match(gi, ri, device=dev)      # ends with the device->host read of the results
    t.append(time.perf_counter() - t0)
print(f"end to end structure_match() from host memory: {np.median(t) * 1e3:.1f} ms (median of 3: "
      f"{np.round(np.array(t) * 1e3, 1).tolist()}), {G / np.median(t):.0f} pairs/s")
assert m.flags.tobytes() == flags.tobytes()

sub = np.arange(0, G, 25)        # 400 pairs, every 25th: half copies, half random
gs, rs = pack([gen[i] for i in sub]), pack([ref[i] for i in sub])
t0 = time.perf_counter()
expect = match_pairs(gs, rs)
dt = time.perf_counter() - t0
assert np.array_equal(expect["flags"], flags[sub]) and np.array_equal(expect["num_mappings"], nm[sub])
fin = np.isfinite(expect["rms"])
err = np.abs(m.rms[sub][fin] - expect["rms"][fin]).max(initial=0)
print(f"oracle agrees on {len(sub)} pairs (flags and num_mappings equal, max |rms diff| {err:.1e})")
print(f"numpy oracle on the host CPU: {dt:.2f} s for {len(sub)} pairs ({dt / len(sub) * 1e3:.2f} ms per pair, "
      f"{len(sub) / dt:.0f} pairs/s; {os.cpu_count()} logical CPUs, one used)")
