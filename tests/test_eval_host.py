"""Host side of the evaluation path (no GPU): dataset splits, the virtual-batch loss metric, its reduction over ranks
(gloo, world size 2) and the argument validation of arreau_eval_noise / arreau_eval_loss."""
import argparse
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def test_split_indices_is_seeded_disjoint_and_complete():
    from arreau_b200.diffusion.lattice_dataset import split_indices
    for n, fr in ((1000, [0.7, 0.2, 0.1]), (37, [0.5, 0.5]), (10, [0.9, 0.1, 0.0]), (5, [1.0])):
        a, b = split_indices(n, fr, seed=3), split_indices(n, fr, seed=3)
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
        allidx = np.concatenate(a)
        assert np.array_equal(np.sort(allidx), np.arange(n))                     # disjoint and complete
        for part, f in zip(a, fr):
            assert abs(len(part) - n * f) <= 1.0
            assert np.array_equal(part, np.sort(part))
    assert not np.array_equal(split_indices(1000, [0.5, 0.5], 3)[0], split_indices(1000, [0.5, 0.5], 4)[0])
    with pytest.raises(ValueError):
        split_indices(10, [0.5, 0.4])
    with pytest.raises(ValueError):
        split_indices(10, [1.2, -0.2])


def test_crystal_subset_collates_the_parents_crystals(tmp_path):
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset, CrystalSubset, save_dataset_npz
    from arreau_b200.synthetic import make_crystals
    cr = make_crystals(12, 1, 6, seed=2)
    off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
    ds = CrystalDataset([save_dataset_npz(str(tmp_path / "d"), [cr.types[off[i]:off[i + 1]] % 5 + 1 for i in range(12)],
                                          np.stack([np.diag(cr.lengths[i]) for i in range(12)]),
                                          [cr.frac[off[i]:off[i + 1]] for i in range(12)])])
    sub = CrystalSubset(ds, [7, 2, 9])
    assert len(sub) == 3 and sub.z_table is ds.z_table and list(sub.crystal_ids) == [7, 2, 9]
    assert np.array_equal(sub.atom_counts(), ds.atom_counts()[[7, 2, 9]])
    a, b = sub.collate_indices([2, 0]), ds.collate_indices([9, 7])
    for k in ("X0", "A0", "L0", "num_atoms"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
    assert np.array_equal(sub[1]["X0"], ds[2]["X0"])


def _loss_finish(frac, vb, ce, len0, lengths, num_atoms, coeff):
    """numpy statement of loss_finish_kernel (csrc/train_ops.cu) on one batch's per-atom terms."""
    N, G = frac.shape[0], num_atoms.shape[0]
    lat = ((len0 - lengths / num_atoms[:, None]) ** 2).sum() / (3.0 * G)
    e_frac, e_vb, e_ce = frac.sum() / N, vb.sum() / N, ce.sum() / N
    return np.array([e_frac + (e_vb * coeff + e_ce) + lat, e_frac, e_vb, e_ce, lat])


def test_virtual_batch_metric_against_loss_finish():
    from arreau_b200.evaluation import LOSS_PARTS, batch_metric
    from arreau_b200.training import HYBRID_LOSS_COEFF
    rng = np.random.default_rng(5)
    G, bs = 23, 5                                                               # last batch ragged (3 crystals)
    na = rng.integers(1, 9, G)
    frac, vb, ce = (rng.random(int(na.sum())) for _ in range(3))
    len0, lengths = rng.random((G, 3)) + 1, rng.random((G, 3)) * 10
    off = np.concatenate([[0], np.cumsum(na)])
    terms = np.stack([[frac[off[g]:off[g + 1]].sum(), vb[off[g]:off[g + 1]].sum(), ce[off[g]:off[g + 1]].sum(),
                       ((len0[g] - lengths[g] / na[g]) ** 2).sum()] for g in range(G)])
    got = batch_metric(na, terms, bs)
    want = np.zeros(5)
    for s in range(0, G, bs):
        e = min(s + bs, G)
        a = slice(off[s], off[e])
        want += _loss_finish(frac[a], vb[a], ce[a], len0[s:e], lengths[s:e], na[s:e], HYBRID_LOSS_COEFF)
    want /= G                                                                   # reduce_loss_metric: sum / crystals
    for i, k in enumerate(LOSS_PARTS):
        assert abs(got[k] - want[i]) <= 1e-13 * abs(want[i]), k


class _FakeLoss:
    """Stands in for DiffusionLoss.evaluate: per-crystal terms that depend on the crystal id only."""

    def evaluate(self, model, batch, t_emb, crystal_ids, seed=0, capacity=None):
        from arreau_b200.evaluation import EvalResult
        ids = torch.as_tensor(np.asarray(crystal_ids), dtype=torch.float64)
        terms = torch.stack([ids.sin() + 1, ids.cos() + 1, (ids * 0.37).sin() + 2, ids * 1e-3], 1) * (seed + 1)
        return EvalResult(t=(ids.long() % 1000 + 1).int(), num_atoms=batch.num_atoms.clone(), terms=terms)


def _fake_model():
    return argparse.Namespace(diffusion_loss=_FakeLoss(), t_emb=None)


def _split(tmp_path):
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset, CrystalSubset, save_dataset_npz, split_indices
    rng = np.random.default_rng(1)
    n = 41
    na = rng.integers(1, 7, n)
    path = save_dataset_npz(str(tmp_path / "d"), [rng.integers(1, 9, k) for k in na], np.tile(np.eye(3) * 4, (n, 1, 1)),
                            [rng.random((k, 3)) for k in na])
    ds = CrystalDataset([path])
    return CrystalSubset(ds, split_indices(n, [0.3, 0.7], seed=2)[1])


def _eval_worker(rank, world, port, tmp_path, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from arreau_b200.evaluation import evaluate_dataset
        res = evaluate_dataset(_fake_model(), _split(tmp_path), 4, "cpu", seed=1, gpu_batch=3)
        np.savez(os.path.join(out, f"e{rank}.npz"), terms=res["terms"], t=res["t"], loss=res["loss"], vb=res["vb"])
    finally:
        dist.destroy_process_group()


def test_evaluate_dataset_reduction_is_independent_of_world_and_grouping(tmp_path):
    """The per-crystal terms are all-gathered in dataset order and every rank rebuilds the same metric: world 2 (gloo)
    gives exactly what world 1 gives, whatever the GPU grouping."""
    from arreau_b200.evaluation import batch_metric, evaluate_dataset
    sub = _split(tmp_path)
    ref = evaluate_dataset(_fake_model(), sub, 4, "cpu", seed=1)
    assert ref["terms"].shape == (len(sub), 4) and np.array_equal(ref["crystal_ids"], sub.crystal_ids)
    assert ref["loss"] == batch_metric(sub.atom_counts(), ref["terms"], 4)["loss"]
    for gb in (1, 5, 100):
        r = evaluate_dataset(_fake_model(), sub, 4, "cpu", seed=1, gpu_batch=gb)
        assert np.array_equal(r["terms"], ref["terms"]) and r["loss"] == ref["loss"]
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_eval_worker, args=(2, port, tmp_path, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        z = np.load(tmp_path / f"e{r}.npz")
        assert np.array_equal(z["terms"], ref["terms"]) and np.array_equal(z["t"], ref["t"])
        assert float(z["loss"]) == ref["loss"] and float(z["vb"]) == ref["vb"]


def test_eval_entry_points_validate_arguments():
    from arreau_b200 import _lib
    lib = _lib.load()
    buf = (C.c_double * 64)()
    p = C.cast(buf, C.c_void_p)
    # arreau_eval_noise(seed, G, N, Z, T, ids, atom_offset, crystal_of_atom, t, eps_x, u, eps_l, stream)
    assert lib.arreau_eval_noise(0, 0, 0, 90, 1000, None, None, None, None, None, None, None, None) == 0   # empty batch
    assert lib.arreau_eval_noise(0, 2, 5, 90, 1000, None, p, p, p, p, p, p, None) == -4
    assert lib.arreau_eval_noise(0, 2, 5, 90, 1000, p, p, None, p, p, p, p, None) == -4
    assert lib.arreau_eval_noise(0, -1, 5, 90, 1000, p, p, p, p, p, p, p, None) == -1
    assert lib.arreau_eval_noise(0, 2, 5, 129, 1000, p, p, p, p, p, p, p, None) == -1                    # Z > 128
    assert lib.arreau_eval_noise(0, 2, 5, 1, 1000, p, p, p, p, p, p, p, None) == -1
    assert lib.arreau_eval_noise(0, 2, 5, 90, 0, p, p, p, p, p, p, p, None) == -1                        # T < 1
    # arreau_eval_loss(score, logits, len0, target, types0, types_t, t, lengths, offset, q_keep, q_to_mask, k1, m1, T,
    #                  N, G, Z, terms, per_crystal, stream)
    ok = [p] * 11
    assert lib.arreau_eval_loss(*([None] + ok[1:]), 0.98, 0.02, 1000, 5, 2, 90, p, p, None) == -4
    assert lib.arreau_eval_loss(*ok, 0.98, 0.02, 1000, 5, 2, 90, p, None, None) == -4
    assert lib.arreau_eval_loss(*ok, 0.98, 0.02, 1000, 5, 2, 129, p, p, None) == -1                     # Z > 128
    assert lib.arreau_eval_loss(*ok, 0.98, 0.02, 1000, 0, 2, 90, p, p, None) == -1
    assert lib.arreau_eval_loss(*ok, 0.98, 0.02, 1000, 5, 0, 90, p, p, None) == -1
    assert lib.arreau_eval_loss(*ok, 0.98, 0.02, 0, 5, 2, 90, p, p, None) == -1
    with pytest.raises(RuntimeError, match="ARREAU_ERR_BAD_SHAPE"):
        _lib.call("arreau_eval_loss", *ok, 0.98, 0.02, 1000, 5, 2, 200, p, p, None)
