"""Dump the keyed draws of arreau_eval_noise, arreau_sample_init_keyed and arreau_sample_noise_keyed (odd Z, step
ordinals 0, 7 and 2^28 - 1) and one keyed trajectory on the replayed CUDA-graph step, for a bitwise comparison of two
trees:   python scratch/keyed_draws_dump.py OUT.npz    (run from the tree under test)"""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from arreau_b200 import _lib  # noqa: E402

dev = torch.device("cuda")
s = torch.cuda.current_stream().cuda_stream
rng = np.random.default_rng(0)
counts = rng.integers(1, 30, 50)
ids = rng.choice(1 << 30, 50, replace=False).astype(np.int64) + (np.int64(1) << 40)
G, N = len(counts), int(counts.sum())
off = torch.tensor(np.concatenate([[0], np.cumsum(counts)]), dtype=torch.int32, device=dev)
coa = torch.tensor(np.repeat(np.arange(G), counts), dtype=torch.int32, device=dev)
cid = torch.tensor(ids, device=dev)
f64 = lambda *sh: torch.full(sh, float("nan"), dtype=torch.float64, device=dev)  # noqa: E731
out = {}
for seed in (1, 0xDEADBEEFCAFEF00D):
    for Z in (7, 91):
        t = torch.zeros(G, dtype=torch.int32, device=dev)
        eps_x, u, eps_l = f64(N, 3), f64(N, Z), f64(G, 3)
        _lib.call("arreau_eval_noise", C.c_uint64(seed), G, N, Z, 1000, cid.data_ptr(), off.data_ptr(), coa.data_ptr(),
                  t.data_ptr(), eps_x.data_ptr(), u.data_ptr(), eps_l.data_ptr(), s)
        out.update({f"eval_{seed}_{Z}_{k}": v.cpu().numpy() for k, v in (("t", t), ("eps_x", eps_x), ("u", u), ("eps_l", eps_l))})
        for step in (0, 7, (1 << 28) - 1):
            z_len, z_frac, u = f64(G, 3), f64(N, 3), f64(N, Z)
            _lib.call("arreau_sample_noise_keyed", C.c_uint64(seed), step, G, N, Z, cid.data_ptr(), off.data_ptr(),
                      coa.data_ptr(), z_len.data_ptr(), z_frac.data_ptr(), u.data_ptr(), s)
            out.update({f"noise_{seed}_{Z}_{step}_{k}": v.cpu().numpy() for k, v in (("z_len", z_len), ("z_frac", z_frac), ("u", u))})
    angles, lengths, frac = f64(G, 3), f64(G, 3), f64(N, 3)
    _lib.call("arreau_sample_init_keyed", C.c_uint64(seed), G, N, cid.data_ptr(), off.data_ptr(), coa.data_ptr(), 0.7,
              angles.data_ptr(), lengths.data_ptr(), frac.data_ptr(), s)
    out.update({f"init_{seed}_{k}": v.cpu().numpy() for k, v in (("angles", angles), ("lengths", lengths), ("frac", frac))})

from test_gpu_wrapper import _model  # noqa: E402
w = np.load(os.path.join(ROOT, "tests", "golden", "weights_seed0.npz"))
for precision in ("fp32", "fp16"):
    m = _model(dev, w, T=11, precision=precision)
    res = m.sample(None, G, num_atoms=torch.as_tensor(counts), crystal_ids=torch.as_tensor(ids), seed=5, device=dev,
                   cuda_graph=True)
    out.update({f"graph_{precision}_frac": np.asarray(res.frac_x), f"graph_{precision}_types": np.asarray(res.atomic_numbers),
                f"graph_{precision}_lattice": np.asarray(res.lattice)})
os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
np.savez(sys.argv[1], **out)
print(f"{len(out)} arrays -> {sys.argv[1]}")
