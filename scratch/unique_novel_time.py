"""Time uniqueness and novelty on one GPU: 10 000 generated Alexandria-shaped crystals against a 100 000-crystal
synthetic reference, both drawing their compositions from one pool of 2 000 (make_training_batch statistics, 1-71
atoms, five elements).  The reference crystals are pool compositions at random positions in the pool crystal's cell,
perturbed by 5 % per axis.  Of the generated crystals 30 % are transformed copies of a random reference crystal
(sigma 0.02 (V/n)^(1/3): not novel), 20 % transformed copies of an earlier generated crystal (sigma 0.02: not
unique), and 50 % pool compositions at random positions.  Reports the fit kernel's time on each pair list (CUDA
events, median of 3 rounds), unique_novel() end to end from host memory (median of 3), the pair counts, the summary,
and the kernel against the numpy fit oracle of tests/test_unique_novel_host.py on a subset of the pairs.

    python scratch/unique_novel_time.py        (profiles/unique_novel.txt holds a run)"""
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
from arreau_b200.inference.crystal_metrics import _check_inputs, crystal_metrics  # noqa: E402
from arreau_b200.inference.structure_match import (_upload_used, unique_novel, unique_novel_summary)  # noqa: E402
from arreau_b200.synthetic import make_training_batch  # noqa: E402
from oracle import restatement as R  # noqa: E402
from test_structure_match_host import transformed_copy  # noqa: E402
from test_unique_novel_host import fit_pairs  # noqa: E402

dev = torch.device("cuda", 0)
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())

POOL, NREF, NGEN = 2_000, 100_000, 10_000
ELEMENTS = np.array([3, 8, 12, 26, 29])
cr = make_training_batch(POOL, seed=3)
lat = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles)).numpy()
off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
pool = [(lat[k], ELEMENTS[cr.types[off[k]:off[k + 1]] % 5]) for k in range(POOL)]
rng = np.random.default_rng(0)


def random_structure(k):
    L, z = pool[k]
    return rng.random((len(z), 3)), L @ np.diag(1 + 0.05 * rng.standard_normal(3)), z


ref = [random_structure(int(k)) for k in rng.integers(0, POOL, NREF)]
gen, kind = [], []
for i in range(NGEN):
    u = rng.random()
    if u < 0.3:
        gen.append(transformed_copy(*ref[int(rng.integers(0, NREF))], rng, sigma=0.02))
        kind.append("ref copy")
    elif u < 0.5 and i > 0:
        gen.append(transformed_copy(*gen[int(rng.integers(0, i))], rng, sigma=0.02))
        kind.append("gen copy")
    else:
        gen.append(random_structure(int(rng.integers(0, POOL))))
        kind.append("random")
kind = np.array(kind)


def pack(cs):
    return (np.concatenate([c[0] for c in cs]), np.stack([c[1] for c in cs]), np.concatenate([c[2] for c in cs]),
            np.array([len(c[2]) for c in cs], np.int64))


gi, ri = pack(gen), pack(ref)
print(f"pool {POOL} compositions; reference {NREF} crystals ({int(ri[3].sum())} atoms); generated {NGEN} "
      f"({int(gi[3].sum())} atoms, largest {int(gi[3].max())}, mean {gi[3].mean():.2f}): "
      + ", ".join(f"{k} {int((kind == k).sum())}" for k in ("ref copy", "gen copy", "random")))

metrics = crystal_metrics(*gi, device=dev)
un = unique_novel(gi, metrics, ri, device=dev)            # warm-up, and the pair lists for the kernel timing
torch.cuda.synchronize()
s = unique_novel_summary(un)
print("summary: " + ", ".join(f"{k} {v:.4f}" if isinstance(v, float) else f"{k} {v}" for k, v in s.items()))
for name, fit in (("uniqueness", un.uniqueness_fit), ("novelty", un.novelty_fit)):
    m = fit.matched
    print(f"{name}: {len(m)} pairs, {int(m.sum())} matched; mappings visited mean {fit.num_mappings.mean():.1f} "
          f"(matched {fit.num_mappings[m].mean() if m.any() else 0:.1f}, unmatched "
          f"{fit.num_mappings[~m].mean() if (~m).any() else 0:.1f}); flags search limit "
          f"{int(((fit.flags & 8) != 0).sum())}, degenerate {int(((fit.flags & 4) != 0).sum())}, too large "
          f"{int(((fit.flags & 16) != 0).sum())}")
for k in ("ref copy", "gen copy", "random"):
    sel = (kind == k) & un.considered
    print(f"  {k}: considered {int(sel.sum())}, unique {int(un.unique[sel].sum())}, novel {int(un.novel[sel].sum())}")

# kernel time per pair list
stream = torch.cuda.current_stream(dev).cuda_stream
for name, (i1, i2), s2 in (("uniqueness", un.uniqueness_pairs, gi), ("novelty", un.novelty_pairs, ri)):
    P = len(i1)
    t1, n1, c1, x1 = _upload_used(gi, *_check_inputs(*gi), i1, dev)
    t2, n2, c2, x2 = _upload_used(s2, *_check_inputs(*s2), i2, dev)
    x1, x2 = torch.as_tensor(x1).to(dev), torch.as_tensor(x2).to(dev)
    outs = [torch.empty(P, dtype=torch.float64, device=dev), torch.empty(P, dtype=torch.int32, device=dev),
            torch.empty(P, dtype=torch.int32, device=dev)]

    def launch():
        _lib.call("arreau_structure_fit_pairs", *[t.data_ptr() for t in t1], n1, c1, *[t.data_ptr() for t in t2], n2,
                  c2, x1.data_ptr(), x2.data_ptr(), P, 0.3, 0.2, 5.0, *[t.data_ptr() for t in outs], stream)

    launch()
    torch.cuda.synchronize()
    rounds = []
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            launch()
        b.record()
        b.synchronize()
        rounds.append(a.elapsed_time(b) / 3)
    ms = float(np.median(rounds))
    fit = un.uniqueness_fit if name == "uniqueness" else un.novelty_fit
    assert outs[2].cpu().numpy().tobytes() == fit.flags.tobytes()
    m = fit.matched
    print(f"fit kernel, {name} pairs: {ms:.2f} ms per launch, {P / ms * 1e3:.0f} pairs/s ({int(m.sum())} matched, "
          f"{int((~m).sum())} not; median of 3 rounds of 3 launches, rounds {np.round(rounds, 2).tolist()})")

t = []
for _ in range(3):
    t0 = time.perf_counter()
    u2 = unique_novel(gi, metrics, ri, device=dev)        # ends with the device->host reads of the results
    t.append(time.perf_counter() - t0)
print(f"end to end unique_novel() from host memory (metrics given): {np.median(t) * 1e3:.0f} ms (median of 3: "
      f"{np.round(np.array(t) * 1e3).tolist()}), {NGEN / np.median(t):.0f} generated crystals/s against {NREF}")
assert u2.group.tobytes() == un.group.tobytes() and u2.novel.tobytes() == un.novel.tobytes()

sub = rng.choice(len(un.novelty_pairs[0]), 150, replace=False)
t0 = time.perf_counter()
expect = fit_pairs(gi, ri, un.novelty_pairs[0][sub], un.novelty_pairs[1][sub])
dt = time.perf_counter() - t0
fit = un.novelty_fit
same = np.array_equal(expect["flags"], fit.flags[sub])
un_sub = (fit.flags[sub] & 1) == 0
nm = np.array_equal(expect["num_mappings"][un_sub], fit.num_mappings[sub][un_sub])
print(f"numpy fit oracle on {len(sub)} novelty pairs: flags equal {same}, num_mappings of the unmatched equal {nm}; "
      f"{dt / len(sub) * 1e3:.2f} ms per pair on one host core")
