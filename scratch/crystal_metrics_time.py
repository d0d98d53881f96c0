"""Time arreau_crystal_metrics on one GPU: kernel time from CUDA events (20 launches after 3 warm-up launches, median
of 5 rounds) for 65 536 sampler-shaped 40-atom crystals and 100 000 Alexandria-shaped crystals (make_training_batch
statistics, up to 236 atoms); the pair-image evaluation rate; end-to-end crystal_metrics() on a SampleResult from host
memory, copies included; and the numpy oracle of tests/test_crystal_metrics.py on a subsample, for scale.

    python scratch/crystal_metrics_time.py        (profiles/crystal_metrics.txt holds a run)"""
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
from arreau_b200.diffusion.diffusion_loss import SampleResult  # noqa: E402
from arreau_b200.diffusion.lattice_helpers import lattice_from_params  # noqa: E402
from arreau_b200.inference.crystal_metrics import _mass_table, crystal_metrics, sample_inputs  # noqa: E402
from arreau_b200.synthetic import make_crystals, make_training_batch  # noqa: E402

dev = torch.device("cuda", 0)
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())


def workload(name):
    if name == "sampler 65536 x 40":
        cr = make_crystals(65536, 40, seed=1)
        rng = np.random.default_rng(2)      # the sampler's [90, U(90, 180), 90] degrees, consumed as radians
        angles = np.stack([np.full(65536, 90.0), rng.uniform(90, 180, 65536), np.full(65536, 90.0)], 1)
    else:
        cr = make_training_batch(100_000, seed=3)
        angles = cr.angles
    lat = lattice_from_params(torch.as_tensor(cr.lengths).to(dev), torch.as_tensor(angles).to(dev)).cpu().numpy()
    return cr.frac, lat, cr.types + 1, cr.num_atoms


def kernel_time(frac, lat, z, na):
    G, N = len(na), len(z)
    off = np.concatenate([[0], np.cumsum(na)]).astype(np.int32)
    f, L = torch.as_tensor(frac).to(dev), torch.as_tensor(lat).to(dev)
    zt, o = torch.as_tensor(z).to(dev), torch.as_tensor(off).to(dev)
    out = [torch.empty(G, dtype=torch.float64, device=dev) for _ in range(3)] + \
          [torch.empty(G, dtype=torch.int32, device=dev) for _ in range(2)]
    mass = _mass_table(dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def launch():
        _lib.call("arreau_crystal_metrics", f.data_ptr(), L.data_ptr(), zt.data_ptr(), o.data_ptr(), N, G,
                  mass.data_ptr(), mass.shape[0] - 1, 0.5, 0.1, *[t.data_ptr() for t in out], stream)

    for _ in range(3):
        launch()
    rounds = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            launch()
        b.record()
        b.synchronize()
        rounds.append(a.elapsed_time(b) / 20)
    flags = out[4].cpu().numpy()
    return float(np.median(rounds)), rounds, flags


for name in ("sampler 65536 x 40", "alexandria-shaped 100k"):
    frac, lat, z, na = workload(name)
    ms, rounds, flags = kernel_time(frac, lat, z, na)
    searched = ((flags & 4) == 0) & (na >= 2)
    pairs = na * (na - 1) // 2
    evals = 27 * int(pairs[searched].sum())
    ext = (flags & 8) != 0
    print(f"\n[{name}] {len(na)} crystals, {int(na.sum())} atoms, {int(pairs.sum())} pairs; "
          f"valid {int((flags & 1).sum())}, degenerate {int(((flags & 4) != 0).sum())}, "
          f"extended search {int(ext.sum())} ({int(pairs[ext].sum())} pairs)")
    print(f"  kernel {ms:.3f} ms (median of 5 rounds of 20 launches; rounds {np.round(rounds, 3).tolist()})")
    print(f"  first-pass pair-image evaluations {evals / 1e9:.3f} G -> {evals / ms / 1e6:.1f} G/s; at 8 fp64 flops "
          f"each (3 add, 1 mul, 2 fma) {evals * 8 / ms / 1e9:.2f} TFLOP/s (extended-search images not counted)")
    if name.startswith("sampler"):
        res = SampleResult(frac_x=frac, lattice=lat, atomic_numbers=z, num_atoms=na)
        crystal_metrics(*sample_inputs(res), device=dev)
        t = []
        for _ in range(3):
            t0 = time.perf_counter()
            crystal_metrics(*sample_inputs(res), device=dev)     # ends with the device->host read of the results
            t.append(time.perf_counter() - t0)
        print(f"  end to end crystal_metrics(SampleResult) from host memory: {np.median(t) * 1e3:.1f} ms "
              f"(median of 3: {np.round(np.array(t) * 1e3, 1).tolist()})")
        from test_crystal_metrics import oracle
        sub = 200
        t0 = time.perf_counter()
        oracle(frac[:sub * 40], lat[:sub], z[:sub * 40], na[:sub])
        dt = time.perf_counter() - t0
        print(f"  numpy oracle: {dt:.2f} s for {sub} crystals ({dt / sub * 1e3:.2f} ms per crystal; "
              f"{dt / sub * len(na):.0f} s for all {len(na)} by extrapolation)")
