#!/usr/bin/env python
"""Benchmark of the Arreau denoising step (BASELINE.json: crystals/sec over a full 999-step denoise
trajectory, and ms per denoise step).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision fp32|fp16] [--impl ours|reference]
                    [--dump-outputs DIR]

A "step" is one denoise step (graph + Ponita forward + VE/VP/D3PM update) of one batch of synthetic crystals;
the N=1 workload is BASELINE.json configs[1] (C2: 1024 crystals x 40 atoms, 5 A cutoff, max_neighbors 8 as in the
reference's Makefile:7).  value = crystals / (999 * step time): the whole-job trajectory throughput with the state
resident in HBM, from --steps timed steps.  e2e = ONE WHOLE 999-step trajectory of the same batch through the public
API a user calls (PONITA_DIFFUSION.sample, the mirror of lightning_wrappers/diffusion.py:220-253: host RNG draws of
the initial state -> upload -> 999 x arreau_denoise_step -> SampleResult as numpy arrays on the host), everything
inside the clock; e2e.step_api is the older per-step measurement (state + noise uploaded from pinned host memory and
the result read back EVERY step).  N>1: one process per GPU (torchrun), each rank owns its own batch of independent
crystals (weak scaling, no data-path collective), time = max over ranks.

--impl reference times the reference's algorithm on the host cores (the oracle port; the reference itself is
Python that needs /root/reference and cannot travel) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# NCCL writes its version banner to stdout (NCCL_DEBUG=VERSION in this image); stdout must carry the ONE JSON line
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

T_STEPS = 1000          # Makefile:7 num_timesteps -> 999 denoise steps per trajectory
Z = 90
RADIUS = 5.0
O, C, D, L, MONO = 16, 128, 256, 5, 83
DUMP_LIMIT = 64_000_000  # bytes of --dump-outputs in all, .npy headers included


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as out_dir/<name>.npy, float32 and float64 arrays as they are, any other dtype as float64.  Above
    DUMP_LIMIT bytes in all, the arrays of each row count that holds more than 1 MB keep one seeded sample of their rows
    (per-atom arrays the same atoms, per-crystal arrays the same crystals), so the dumps of two builds run with the same
    arguments compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    host = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        host[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    total = sum(a.nbytes + 4096 for a in host.values())            # 4 KB per .npy header is ample
    per_rows = {}
    for a in host.values():
        if a.ndim:
            per_rows[a.shape[0]] = per_rows.get(a.shape[0], 0) + a.nbytes
    big = {n: b for n, b in per_rows.items() if b > 1 << 20}
    large = sum(big.values())
    budget = DUMP_LIMIT - (total - large)                           # left for the rows of the sampled arrays
    rows = ({n: np.sort(np.random.default_rng(n).choice(n, max(1, n * budget // large), replace=False)) for n in big}
            if total > DUMP_LIMIT else {})
    for name, a in host.items():
        if a.ndim and a.shape[0] in rows:
            a = a[rows[a.shape[0]]]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_weights(atoms_per_crystal: int):
    from arreau_b200.synthetic import calibrate_length_readout
    w = np.load(os.path.join(ROOT, "tests", "golden", "weights_seed0.npz"))
    sd = {k: w[k] for k in w.files if k not in ("ori_grid", "fourier_w")}
    # quirk B7: random-init length read-out would blow the cells up and empty the graph; calibrate it
    return calibrate_length_readout(sd, atoms_per_crystal), w["ori_grid"], w["fourier_w"]


def sampler_init(G: int, n: int, seed: int):
    """The reference sampler's initial state (diffusion_loss.py:294-316)."""
    rng = np.random.default_rng(seed)
    angles = np.stack([np.full(G, 90.0), rng.uniform(90, 180, G), np.full(G, 90.0)], 1)
    lengths = rng.standard_normal((G, 3))
    frac = rng.standard_normal((G * n, 3))
    types = np.full(G * n, Z - 1, dtype=np.int64)
    return frac, types, lengths, angles


def teacher_state(G: int, n: int, seed: int, t: int):
    """Teacher-forced state at timestep t (SURVEY 8d): synthetic Alexandria-shaped crystals pushed through the
    reference's forward noising (VE on frac helpers:43-46, VP on lengths :156-163, D3PM mask chain d3pm.py:140-143),
    so that E/N is realistic for per-step timing at any t."""
    from arreau_b200.synthetic import make_crystals
    from arreau_b200.tables import build_tables
    tb = build_tables(T_STEPS, Z)
    cr = make_crystals(G, n, None, seed=seed)
    rng = np.random.default_rng(seed + 7)
    sig = float(tb.ve_sigmas[t])
    frac = (cr.frac + sig * rng.standard_normal(cr.frac.shape)) % 1.0
    ab = float(tb.vp_alpha_bars[t])
    lengths = np.sqrt(ab) * cr.lengths + np.sqrt(1 - ab) * rng.standard_normal(cr.lengths.shape)
    keep = float(tb.q_keep[t - 1])
    types = np.where(rng.random(cr.types.shape) < keep, cr.types, Z - 1).astype(np.int64)
    return frac, types, lengths, cr.angles


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        self.mark0 = self.mark1 = 0

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def summary(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [l.split(", ") for t, l in self.lines if self.t0 - 0.05 <= t <= self.t1 + 0.15]
        if not rows:
            rows = [l.split(", ") for _, l in self.lines[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def oracle_step_time(G_s: int, n: int, steps: int, warmup: int, cap: int, threads: int, radius: float = RADIUS):
    """Times the CPU restatement of the reference step (oracle/restatement.py, fp64 like the reference) on
    G_s crystals x n atoms.  Returns (seconds per step, edges per atom)."""
    import torch
    from arreau_b200.synthetic import make_crystals
    from oracle import restatement as R
    torch.set_num_threads(threads)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        sd, ori, fw = load_weights(n)
        T64 = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float64)  # noqa: E731
        W = R.PonitaWeights({k: T64(v) for k, v in sd.items()}, T64(ori), radius)
        tabs = R.DiffusionTables.build(T_STEPS, Z)
        cr = make_crystals(G_s, n, None, seed=0)       # Alexandria-shaped cells: E/N = cap like the GPU run
        frac, types, lengths, angles = T64(cr.frac), torch.as_tensor(cr.types), T64(cr.lengths), T64(cr.angles)
        na = torch.as_tensor(cr.num_atoms)
        N = cr.total_atoms
        g = torch.Generator().manual_seed(0)
        times, epa = [], 0.0
        for it in range(warmup + steps):
            t = T_STEPS - 1 - it
            z_len = torch.randn(G_s, 3, generator=g); z_frac = torch.randn(N, 3, generator=g); u = torch.rand(N, Z, generator=g)
            t0 = time.perf_counter()
            out = R.denoise_step(W, tabs, T64(fw), frac, types, lengths, angles, na, t, z_len, z_frac, u, radius, cap)
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
        lat = R.lattice_from_params(lengths, angles)
        ei = R.radius_graph_pbc(R.frac_to_cart_coords(frac, lat, na), lat, na, radius, cap)[0]
        epa = ei.shape[1] / N
        return float(np.mean(times)), epa
    finally:
        torch.set_default_dtype(prev)


def build_public_model(dev, atoms_per_crystal: int, precision: str):
    """The reference-facing module (arreau_b200.lightning_wrappers.diffusion.PONITA_DIFFUSION, constructor arguments of
    main_diffusion.py:88-120 / Makefile:7) carrying the benchmark weights."""
    import torch
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    from arreau_b200.tools.atomic_number_table import AtomicNumberTable
    a = argparse.Namespace(dataset="synthetic", lr=3e-4, weight_decay=0.0, epochs=1, warmup=0, layer_scale=1e-6,
                           train_augm=False, hidden_dim=C, layers=L, radius=RADIUS, num_ori=O, basis_dim=D, degree=3,
                           widening_factor=4, multiple_readouts=True, num_timesteps=T_STEPS, max_neighbors=8)
    sd, ori, fw = load_weights(atoms_per_crystal)
    m = PONITA_DIFFUSION(a, AtomicNumberTable(list(range(1, Z)) + [2001]), ori_grid=ori, precision=precision)
    m.model.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})
    with torch.no_grad():
        m.t_emb.gaussian_fourier_proj_w.copy_(torch.as_tensor(fw))
    return m.to(dev)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    G_s = args.ref_crystals
    t_step, epa = oracle_step_time(G_s, args.atoms, args.steps, args.warmup, args.cap, cores, args.radius)
    value = G_s / ((T_STEPS - 1) * t_step)
    sample = f"{G_s} crystals x {args.atoms} atoms, {args.steps} denoise steps (+{args.warmup} warm-up), E/N={epa:.2f}"
    line = {"impl": "reference", "metric": "crystals_per_sec_full_trajectory", "value": value, "unit": "crystals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(config_dict(args), cpu_sample=f"{G_s} of the {args.crystals} crystals per step (the reference "
                           f"costs ~1.4 s per step at 64 x 40 atoms; crystals are independent, cost is linear in them)",
                           cpu_sample_crystals=G_s),
            "cpu_baseline": {"value": value, "unit": "crystals/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "crystals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "ms_per_step is for the bounded sample; crystals/s = sample crystals / (999 * step time)"}
    print(json.dumps(line))


def config_dict(args):
    tag = "C2" if (args.crystals, args.atoms) == (1024, 40) else ("C3" if args.atoms >= 200 else "custom")
    return {"workload": f"{tag}: full-trajectory sampling, {args.crystals} crystals x {args.atoms} atoms per GPU "
                        f"(Alexandria-shaped), {args.radius:g} A PBC cutoff, max_neighbors {args.cap}, T={T_STEPS} "
                        f"(999 denoise steps per trajectory)",
            "model": "random-init reference architecture, 1 170 678 params (hidden 128, basis 256, 5 layers, 16 ori), "
                     "length read-out calibrated (SURVEY B7)",
            "crystals_per_gpu": args.crystals, "atoms_per_crystal": args.atoms, "max_neighbors": args.cap,
            "state": ("free-running from the reference sampler init (t=999)" if args.state == "sampler" else
                      f"teacher-forced at t={args.t0} (reference forward noising of the synthetic crystals)"),
            "l2": "inputs larger than L2 (per-layer kernel slabs >= 1.3 GB, node features 335 MB)",
            "parallelism": f"crystal-sharded x{args.gpus}, no per-step collective"}


def run_train(args):
    """--workload train: BASELINE.json configs[4] (C5): one training step = noising + predict_scores + 3-term loss +
    backward + gradient all-reduce (N>1) + Adam on a synthetic 270-crystal batch per GPU.  Not the headline metric;
    prints its own JSON line (train_crystals_per_sec) with a per-phase breakdown."""
    import torch
    import torch.distributed as dist
    from arreau_b200 import _lib
    from arreau_b200.distributed import allreduce_gradients, broadcast_parameters
    from arreau_b200.synthetic import make_training_batch
    from arreau_b200.tables import build_tables
    from arreau_b200.training import FlatParams, FusedAdam, TrainEngine
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    w = np.load(os.path.join(ROOT, "tests", "golden", "weights_seed0.npz"))
    sd = {k: w[k] for k in w.files if k not in ("ori_grid", "fourier_w")}
    p = FlatParams(164, 4, Z, dev)
    p.load_state_dict(sd)
    broadcast_parameters(p.data)
    cr = make_training_batch(args.crystals if args.crystals != 1024 else 270, seed=100 + rank)
    G, N = cr.num_crystals, cr.total_atoms
    bwd_prec = "fp32" if args.precision == "fp32" else "tf32"
    te = TrainEngine(p, build_tables(T_STEPS, Z), w["fourier_w"], w["ori_grid"], cr.num_atoms, args.radius, args.cap, device=dev,
                     backward_precision=bwd_prec)
    opt = FusedAdam(p, lr=3e-4, max_grad_norm=0.5)
    from arreau_b200.diffusion.lattice_helpers import lattice_from_params
    lat0 = lattice_from_params(torch.as_tensor(cr.lengths).to(dev), torch.as_tensor(cr.angles).to(dev))
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    phases = ["noise", "forward", "loss", "backward", "allreduce", "adam"]
    frac0, types0 = torch.as_tensor(cr.frac).to(dev), torch.as_tensor(cr.types).to(dev)

    def step(timed):
        ts = torch.randint(1, T_STEPS + 1, (G,), device=dev, generator=g)
        eps_x = torch.randn(N, 3, device=dev, dtype=torch.float64, generator=g)
        u = torch.rand(N, Z, device=dev, dtype=torch.float64, generator=g)
        eps_l = torch.randn(G, 3, device=dev, dtype=torch.float64, generator=g)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(phases) + 1)] if timed else None
        mark = (lambda i: evs[i].record()) if timed else (lambda i: None)
        mark(0)
        te.repack(); te.set_batch(frac0, types0, lat0, ts, eps_x, u, eps_l); te.noise_batch(); mark(1)
        te.predict(); mark(2)
        te.compute_loss(); mark(3)
        te.backward(); mark(4)
        allreduce_gradients(p.grad); mark(5)
        opt.step(); mark(6)
        return evs

    for _ in range(max(args.warmup, 3)):
        step(False)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step(False)
    e1.record()
    torch.cuda.synchronize(dev)
    launches = _lib.launch_count() - l0
    if args.dump_outputs and rank == 0:        # before the breakdown steps below train further
        dump_outputs(args.dump_outputs, {"loss": te.loss, "grad": p.grad, "params": p.data})
    ms = e0.elapsed_time(e1) / args.steps
    if world > 1:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
    br = {k: 0.0 for k in phases}
    for _ in range(3):
        evs = step(True)
        torch.cuda.synchronize(dev)
        for i, k in enumerate(phases):
            br[k] += evs[i].elapsed_time(evs[i + 1]) / 3
    if rank == 0:
        E = te.eng.num_edges()
        print(json.dumps({"metric": "train_crystals_per_sec", "value": world * G / (ms * 1e-3), "unit": "crystals/s",
                          "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f32" if bwd_prec == "fp32" else "tf32 GEMMs (tcgen05, fp32 accumulate) in forward and backward; fp32 elsewhere",
                          "data": "synthetic", "impl": "ours",
                          "config": {"workload": f"C5: training step (score-matching + D3PM + lattice loss), {G} crystals "
                                                 f"/ {N} atoms / {E} edges per GPU, max_neighbors {args.cap}, "
                                                 f"{'DDP x' + str(world) if world > 1 else 'single GPU'}",
                                     "parallelism": f"data parallel x{world}: one all-reduce of the flat 4.7 MB gradient"},
                          "loss": te.loss.tolist(), "gpu_launches": int(launches),
                          "breakdown_ms_per_step": {k: round(v, 4) for k, v in br.items()}}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="sample", choices=["sample", "train"])
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 10)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("ARREAU_PRECISION", "fp16"), choices=["fp32", "fp16"],
                    help="fp16: tcgen05 tensor-core path (fp16 operands, fp32 accumulate; stated tolerance 5e-3 of "
                         "max|ref| -- tests/conftest.py TOL_FP16_MODEL, measured 3e-5..4e-3); fp32: FFMA2 SIMT path "
                         "(<= 1e-4, measured 2e-6)")
    ap.add_argument("--crystals", type=int, default=1024)
    ap.add_argument("--atoms", type=int, default=40)
    ap.add_argument("--cap", type=int, default=8)
    ap.add_argument("--radius", type=float, default=RADIUS)
    ap.add_argument("--ref-crystals", type=int, default=64)
    ap.add_argument("--state", default="sampler", choices=["sampler", "teacher"],
                    help="sampler: free-running from the reference sampler's init at t=999 (the headline); teacher: "
                         "teacher-forced state at --t0 (needed for uncapped graphs, whose 1 A initial cells are all images)")
    ap.add_argument("--t0", type=int, default=500)
    ap.add_argument("--trajectory", action="store_true",
                    help="time ONE WHOLE trajectory (every denoise step from the sampler init at t=T-1 down to t=1, "
                         "state re-initialised after the warm-up) instead of --steps steps; value = crystals / that time")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="run the timed steps as replays of ONE captured CUDA graph of the step (arreau_denoise_step_replay: "
                         "device-resident step counter, Philox noise inside the graph): one launch per step instead of 26")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e-trajectory", action="store_true", help="skip the whole-trajectory e2e leg (~7 s at C2)")
    ap.add_argument("--no-other-precision", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0's "
                         "batch): the sampler state and model outputs, or with --workload train the loss, gradient and "
                         "updated parameters; a seeded sample of rows above 64 MB in all")
    args = ap.parse_args()
    if args.trajectory and args.steps is not None:
        ap.error("--trajectory times every step of one trajectory; it takes no --steps")
    if args.steps is None:
        args.steps = 10
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "train":
        return run_train(args)

    import torch
    import torch.distributed as dist
    from arreau_b200 import _lib
    from arreau_b200.engine import DenoiseEngine
    from arreau_b200.tables import build_tables
    from arreau_b200.weights import PonitaWeights

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: arreau_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    G, n = args.crystals, args.atoms
    N = G * n
    sd, ori, fw = load_weights(n)
    eng = DenoiseEngine(PonitaWeights(sd, ori, device=dev), build_tables(T_STEPS, Z), fw, [n] * G, args.radius, args.cap,
                        precision=args.precision, device=dev)
    if args.state == "teacher":
        frac, types, lengths, angles = teacher_state(G, n, 1234 + rank, args.t0)
        t_start = args.t0
    else:
        frac, types, lengths, angles = sampler_init(G, n, seed=1234 + rank)
        t_start = T_STEPS - 1
    eng.set_state(frac, types, lengths, angles)
    seed = 99 + rank

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- device-resident trajectory steps -------------------------------------------------------------
    t = t_start
    for i in range(max(args.warmup, 3)):
        eng.draw_noise(seed, i)
        eng.step(t); t -= 1
    if args.trajectory:
        eng.set_state(frac, types, lengths, angles)
        t = t_start
        args.steps = t_start
    barrier()
    epa_first = eng.num_edges() / N
    graph = eng.capture_trajectory_graph(t, seed) if args.cuda_graph else None      # state and counter are restored
    clocks = ClockSampler(local)
    time.sleep(0.25)
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.begin()
    ev0.record()
    if graph is not None:
        for i in range(args.steps):
            graph.replay()
    else:
        for i in range(args.steps):
            eng.draw_noise(seed, 1000 + i)
            eng.step(t); t = max(t - 1, 1)
    ev1.record()
    barrier()
    clocks.end()
    launches = _lib.launch_count() - l0
    if graph is not None:
        launches = 26 * args.steps          # kernels inside the replayed graph (the library counts launches at capture only)
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
    ms_per_step = ms / args.steps
    value = world * G / ((T_STEPS - 1) * ms_per_step * 1e-3)
    epa_last = eng.num_edges() / N
    overflow = int(eng.overflow_flag.item())
    clk = clocks.summary()
    if args.dump_outputs and rank == 0:        # before the legs below overwrite the engine's state
        dump_outputs(args.dump_outputs, {"frac": eng.frac, "types": eng.types, "lengths": eng.lengths,
                                         "lattice": eng.lattice, "score": eng.score, "logits": eng.logits,
                                         "len0": eng.len0})

    # ---- end to end: state + noise from pinned host memory every step, result read back --------------
    pin = lambda a: torch.as_tensor(a).pin_memory()  # noqa: E731
    g = torch.Generator().manual_seed(5 + rank)
    if args.state == "teacher":
        h_in = [pin(torch.as_tensor(frac)), pin(torch.as_tensor(types)), pin(torch.as_tensor(lengths)),
                pin(torch.as_tensor(angles))]
    else:
        h_in = [pin(torch.randn(N, 3, generator=g, dtype=torch.float64)), pin(torch.as_tensor(types)),
                pin(torch.as_tensor(np.abs(lengths) + 5.0)), pin(torch.as_tensor(angles))]
    h_noise = [pin(torch.randn(G, 3, generator=g, dtype=torch.float64)), pin(torch.randn(N, 3, generator=g, dtype=torch.float64)),
               pin(torch.rand(N, Z, generator=g, dtype=torch.float64))]
    h_out = [torch.empty(N, 3, dtype=torch.float64).pin_memory(), torch.empty(N, dtype=torch.int64).pin_memory(),
             torch.empty(G, 3, dtype=torch.float64).pin_memory(), torch.empty(G, 3, 3, dtype=torch.float64).pin_memory()]
    h2d = sum(x.numel() * x.element_size() for x in h_in + h_noise)
    d2h = sum(x.numel() * x.element_size() for x in h_out)

    def e2e_step(tt):
        # the step's state and noise come from pinned host memory, its result goes back to the host; the noise of
        # step k+1 does not depend on step k, so its upload is staged on a side stream under step k's kernels
        # (engine.stage_noise) -- every byte is still copied inside the timed region, once per step
        eng.set_state(*h_in)
        eng.use_staged_noise()
        eng.step(tt)
        eng.release_noise()
        eng.stage_noise(*h_noise)                          # next step's draws
        for dst_, src_ in zip(h_out, (eng.frac, eng.types, eng.lengths, eng.lattice)):
            dst_.copy_(src_, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()      # the caller holds the step's result on the host

    eng.stage_noise(*h_noise)
    for i in range(2):
        e2e_step(500)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_steps = min(args.steps, 20)
    for i in range(e2e_steps):
        e2e_step(500 - i)
    e1.record()
    barrier()
    ems = e0.elapsed_time(e1)
    if world > 1:
        tmax = torch.tensor([ems], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ems = float(tmax.item())
    e2e_step_value = world * G / ((T_STEPS - 1) * (ems / e2e_steps) * 1e-3)

    # ---- end to end, the call a user makes: ONE whole trajectory through PONITA_DIFFUSION.sample -------
    # (host RNG draws + upload of the initial state, 999 denoise steps with in-kernel Philox noise -- the default of
    # generate_n_crystals --, result back on the host as the reference's SampleResult; capped graphs only: the
    # reference sampler's ~1 A initial cells are all images without the cap)
    e2e_traj = None
    if args.cap > 0 and args.state == "sampler" and not args.no_e2e_trajectory:
        model = build_public_model(dev, n, args.precision)
        model.diffusion_loss.max_neighbors, model.diffusion_loss.cutoff = args.cap, args.radius
        dl = model.diffusion_loss
        model.model._packed = eng.w                       # same packed weights; the engine below is this topology's
        model.model._packed_version = (0, 0)
        dl._engine, dl._engine_key = eng, (id(model.model), tuple([n] * G), str(dev), False, args.precision)
        np.random.seed(17 + rank)
        torch.manual_seed(17 + rank)
        barrier()
        clocks2 = ClockSampler(local)
        time.sleep(0.25)
        clocks2.begin()
        tw0 = time.perf_counter()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        res = model.sample(num_atoms_per_sample=n, num_samples_in_batch=G, device=dev, device_noise=True, seed=31 + rank)
        t1e.record()
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - tw0
        clocks2.end()
        tsec = max(t0e.elapsed_time(t1e) * 1e-3, wall)    # the host work before the first launch counts too
        if world > 1:
            tmax = torch.tensor([tsec], device=dev, dtype=torch.float64)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            tsec = float(tmax.item())
        assert res.frac_x.shape == (N, 3) and np.isfinite(res.frac_x).all() and np.isfinite(res.lattice).all()
        up = N * 3 * 8 + N * 8 + G * 3 * 8 * 2 + G * 6 * 8                 # frac, types, lengths, angles, angle factors
        down = N * 3 * 8 + N * 8 + G * 9 * 8                               # frac, types, lattice
        e2e_traj = {"value": world * G / tsec, "seconds": tsec, "steps": T_STEPS - 1, "ms_per_step": tsec * 1e3 / (T_STEPS - 1),
                    "h2d_bytes": up, "d2h_bytes": down, "clocks": clocks2.summary(),
                    "final_edges_per_atom": eng.num_edges() / N,
                    "api": "PONITA_DIFFUSION.sample(num_atoms_per_sample, num_samples_in_batch, device_noise=True)"}

    # ---- final gather of a trajectory's result (the only collective of the sampling path) -------------
    gather_ms = None
    if world > 1:
        outs = [torch.empty_like(eng.frac) for _ in range(world)]
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        dist.all_gather(outs, eng.frac)
        dist.all_gather([torch.empty_like(eng.types) for _ in range(world)], eng.types)
        dist.all_gather([torch.empty_like(eng.lattice) for _ in range(world)], eng.lattice)
        g1.record()
        barrier()
        gather_ms = g0.elapsed_time(g1)

    # ---- per-kernel breakdown and the roofline of the dominant kernel (rank 0) -------------------------
    line = None
    if rank == 0:
        eng.set_state(*h_in)
        br = eng.timed_breakdown(400, iters=3)
        E = eng.num_edges()
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            pk = json.load(open(peaks_path)); peak_src = "measured (MEASURED_PEAKS.json)"
            peak_tf, peak_bw = pk["bf16_tflops_sustained"], pk["hbm_gbs"]
        else:
            peak_tf, peak_bw, peak_src = 1590.0, 6650.0, "fallback (B200_PROFILING.md)"
        top = max(br, key=lambda k: br[k]["ms_per_step"])
        flops_edge = 2.0 * E * O * (MONO * C + C * D + L * D * C) + 2.0 * L * 0   # SURVEY 8d: 6.63 MFLOP/edge
        flops_mlp = 2.0 * 2 * C * 4 * C * N * O                                   # per layer
        kbytes = 2 if args.precision == "fp16" else 4
        # per layer (SURVEY 8d): the gather streams the layer's kernel slab once, reads h once (compulsory) and the
        # edge list, and writes the message sums; the fiber conv + LayerNorm reads them and writes y
        alg = {"edge_kernels": ("tensor", flops_edge / 1e12, peak_tf, "TFLOP/s"),
               "convnext_mlp": ("tensor", flops_mlp / 1e12, peak_tf, "TFLOP/s")}
        if args.precision == "fp16":
            # fused gather + fiber conv + LayerNorm: kernel slab + h (compulsory) + edge list in, y out
            bytes_fused = E * O * C * 2 + 4 * N * O * C + 12 * E + 2 * N * O * C
            alg["message_fiber_norm"] = ("hbm", bytes_fused / 1e9, peak_bw, "GB/s")
        else:
            bytes_gather = E * O * C * 4 + 4 * N * O * C + 12 * E + 4 * N * O * C
            bytes_fiber = 4 * N * O * C + 4 * N * O * C
            alg["message_gather"] = ("hbm", bytes_gather / 1e9, peak_bw, "GB/s")
            alg["fiber_norm"] = ("hbm", bytes_fiber / 1e9, peak_bw, "GB/s")
        kernels = {}
        for name, (bound, work, peak, unit) in alg.items():
            sec = br[name]["ms_per_launch"] * 1e-3
            if name == "message_fiber_norm":      # work is per layer; long rows run two launches per layer (gather + fiber conv)
                sec = br[name]["ms_per_step"] * 1e-3 / L
            ach = work / sec
            kernels[name] = {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                             "ms_per_launch": sec * 1e3, "launches_per_step": br[name]["launches_per_step"]}
        dom = top if top in kernels else "edge_kernels"
        # measured DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full`
        # capture of this workload, profiles/r1_traffic.json); only valid for the configuration it was captured on
        traffic = None
        import glob
        for tpath in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")), reverse=True):   # newest round first
            tj = json.load(open(tpath))
            if tj.get("workload") == [args.crystals, args.atoms, args.cap, args.radius, args.precision]:
                traffic = tj["bytes_per_launch"].get(dom)
                for kname, kv in kernels.items():
                    kv["traffic"] = tj["bytes_per_launch"].get(kname)
                break
        roof = dict(kernels[dom]); roof.update({"kernel": dom, "traffic": traffic, "peak_source": peak_src,
                                                "share_of_step": br[dom]["ms_per_step"] / sum(v["ms_per_step"] for v in br.values())})
        line = {"metric": "crystals_per_sec_full_trajectory", "value": value, "unit": "crystals/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "f16",
                "data": "synthetic", "config": config_dict(args), "clocks": clk,
                "e2e": ({"value": e2e_traj["value"], "unit": "crystals/s", "ms_per_step": e2e_traj["ms_per_step"],
                         "h2d_bytes_per_step": e2e_traj["h2d_bytes"] / (T_STEPS - 1),
                         "d2h_bytes_per_step": e2e_traj["d2h_bytes"] / (T_STEPS - 1), "trajectory": e2e_traj,
                         "what": "one whole 999-step trajectory through PONITA_DIFFUSION.sample: host draws + upload of the "
                                 "initial state, every step, SampleResult back on the host; bytes are per trajectory / 999",
                         "step_api": {"value": e2e_step_value, "ms_per_step": ems / e2e_steps, "h2d_bytes_per_step": h2d,
                                      "d2h_bytes_per_step": d2h,
                                      "what": "engine API, state + noise from pinned host memory and result read back EVERY step"}}
                        if e2e_traj is not None else
                        {"value": e2e_step_value, "unit": "crystals/s", "ms_per_step": ems / e2e_steps,
                         "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                         "what": "engine API, state + noise from pinned host memory and result read back EVERY step"}),
                "gpu_launches": int(launches), "roofline": roof, "kernels": kernels,
                "breakdown_ms_per_step": {k: round(v["ms_per_step"], 4) for k, v in br.items()},
                "edges_per_atom": {"first_timed_step": epa_first, "last_timed_step": epa_last, "breakdown": E / N},
                "edge_overflow": overflow, "final_gather_ms": gather_ms, "impl": "ours", "precision": args.precision,
                "cuda_graph": bool(args.cuda_graph)}
        if args.trajectory:
            line["trajectory"] = {"steps_run": args.steps, "t_from": t_start, "t_to": 1, "seconds": ms * 1e-3,
                                  "crystals": world * G, "note": "value = crystals / seconds of this one whole trajectory"}
        if world == 1 and not args.no_other_precision:
            other = "fp32" if args.precision == "fp16" else "fp16"
            del eng
            torch.cuda.empty_cache()
            eng2 = DenoiseEngine(PonitaWeights(sd, ori, device=dev), build_tables(T_STEPS, Z), fw, [n] * G, args.radius, args.cap,
                                 precision=other, device=dev)
            eng2.set_state(frac, types, lengths, angles)
            t2 = t_start
            for i in range(3):
                eng2.draw_noise(seed, i); eng2.step(t2); t2 -= 1
            torch.cuda.synchronize(dev)
            o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            o0.record()
            o_steps = min(args.steps, 20)
            for i in range(o_steps):
                eng2.draw_noise(seed, 1000 + i); eng2.step(t2); t2 -= 1
            o1.record()
            torch.cuda.synchronize(dev)
            oms = o0.elapsed_time(o1) / o_steps
            line["other_precision_path"] = {"precision": other, "ms_per_step": oms, "value": G / ((T_STEPS - 1) * oms * 1e-3),
                                            "unit": "crystals/s"}
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            t_cpu, epa = oracle_step_time(args.ref_crystals, n, 3, 1, args.cap, cores, args.radius)
            line["cpu_baseline"] = {"value": args.ref_crystals / ((T_STEPS - 1) * t_cpu), "unit": "crystals/s", "cores": cores,
                                    "kind": "port", "ms_per_step_sample": t_cpu * 1e3,
                                    "sample": f"{args.ref_crystals} crystals x {n} atoms, 3 denoise steps (+1 warm-up), "
                                              f"fp64 torch CPU restatement of the reference step, E/N={epa:.2f}"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
