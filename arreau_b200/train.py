"""Mirror of the training entry point (main_diffusion.py:284-307, SURVEY 3.2) without Lightning:

    python -m arreau_b200.train --data out/alexandria_ps_000.npz --epochs 2 --batch_size 270
    torchrun --nproc-per-node 8 -m arreau_b200.train ...        # data parallel: one all-reduce of the flat gradient per step

Per step: DiffusionLoss.__call__ (noising, predict_scores, loss, hand-written backward -> flat gradient buffer),
gradient all-reduce (mean) across ranks, fused Adam with global-norm clip 0.5 and the cosine-warmup schedule per epoch;
the first batch runs the one-time `callibrate` pass (ponita/nn/conv.py:122-123) like the reference's first train-mode
forward.  The loss metric is reduced like DiffusionLossMetric (sum of losses / number of crystals over all ranks).

With a validation split (--val_fraction) every epoch ends with a forward-only evaluation of it (arreau_b200/evaluation.py)
logged as "valid loss"; --checkpoint_dir receives last.ckpt every epoch and best.ckpt whenever the valid loss improves
(the reference keeps the top 3 by "valid loss"; here only the best).  A test split (--test_fraction) is evaluated once at
the end with the best.ckpt weights (the final weights without a validation split)."""
from __future__ import annotations

import argparse
import os
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from .diffusion.lattice_dataset import CrystalDataset, CrystalSubset, batches, split_indices
from .distributed import allreduce_gradients, broadcast_parameters, reduce_loss_metric
from .evaluation import evaluate_dataset
from .lightning_wrappers.diffusion import PONITA_DIFFUSION


def default_args(**over):
    """argparse defaults of main_diffusion.py:88-120 + Makefile:7."""
    a = argparse.Namespace(dataset="alexandria", lr=3e-4, weight_decay=0.0, epochs=1, warmup=0, layer_scale=1e-6,
                           train_augm=False, hidden_dim=128, layers=5, radius=5.0, num_ori=16, basis_dim=256, degree=3,
                           widening_factor=4, multiple_readouts=True, num_timesteps=1000, max_neighbors=8, batch_size=270)
    for k, v in over.items():
        setattr(a, k, v)
    return a


def fit(model: PONITA_DIFFUSION, dataset: CrystalDataset, epochs: int, batch_size: int, device, seed: int = 0,
        backward_precision: str = "tf32", calibrate: bool = True, log=print, val_dataset=None,
        checkpoint_dir: Optional[str] = None, metrics: Optional[dict] = None):
    """Trains `model` for `epochs` and returns the per-epoch train loss.  val_dataset: evaluated after every epoch
    (evaluate_dataset with the same batch_size and seed; logged as "valid loss").  checkpoint_dir: rank 0 writes
    last.ckpt every epoch and, with a validation set, best.ckpt whenever the valid loss improves.  metrics (optional
    dict): receives metrics["valid"], one evaluate_dataset result per epoch."""
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    model.to(device)
    model.diffusion_loss.backward_precision = backward_precision
    opt = model.configure_optimizers(device)
    flat = model.model.flat
    broadcast_parameters(flat.data)
    history = []
    best = float("inf")
    if checkpoint_dir is not None and rank == 0:
        os.makedirs(checkpoint_dir, exist_ok=True)
    for epoch in range(epochs):
        opt.set_epoch(epoch, model.warmup, max(model.epochs, 1))
        total_loss = torch.zeros((), dtype=torch.float64, device=device)
        total_samples = torch.zeros((), dtype=torch.float64, device=device)
        for batch in batches(dataset, batch_size, shuffle=True, seed=seed + epoch, device=device, rank=rank, world=world):
            loss = model.training_step(batch)          # the step's kernels have filled flat.grad
            if calibrate:
                # ponita/nn/conv.py:122-123: the reference's FIRST train-mode forward -- the noised batch of the first
                # training step at its random timesteps -- re-initialises the kernel / fiber_kernel scales from its own
                # activations AFTER using the old weights, and that same forward's loss is then back-propagated: the
                # first gradient belongs to the un-rescaled weights and is applied to the rescaled ones.  Same here:
                # statistics from the step that has just run, rescale, then the optimizer step.  (Under DDP every
                # reference rank rescales from its own shard and the replicas silently diverge; here rank 0's scales
                # are broadcast -- the one deliberate deviation.)
                te = model.diffusion_loss.train_engine_for(model.model, model.t_emb, getattr(batch, "num_atoms_cpu", batch.num_atoms), device)
                te.calibrate_from_last_forward()
                broadcast_parameters(flat.data)
                for layer in model.model.interaction_layers:
                    layer.conv.callibrated.fill_(True)
                calibrate = False
            allreduce_gradients(flat.grad)
            opt.step()
            total_loss += loss.detach().double()
            total_samples += batch.num_atoms.shape[0]
        metric = reduce_loss_metric(total_loss, total_samples)
        history.append(float(metric))
        valid = None
        if val_dataset is not None:
            valid = evaluate_dataset(model, val_dataset, batch_size, device, seed=seed)
            if metrics is not None:
                metrics.setdefault("valid", []).append(valid)
        if rank == 0:
            log(f"epoch {epoch}: train loss {history[-1]:.6f}" + (f", valid loss {valid['loss']:.6f}" if valid is not None else "")
                + f" (lr {opt.lr:.3e})")
            if checkpoint_dir is not None:
                model.save_checkpoint(os.path.join(checkpoint_dir, "last.ckpt"))
                if valid is not None and valid["loss"] < best:
                    best = valid["loss"]
                    model.save_checkpoint(os.path.join(checkpoint_dir, "best.ckpt"))
    return history


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--data", nargs="+", required=True, help="dataset files (.h5 as written by prep_datasets.py, or .npz)")
    ap.add_argument("--epochs", type=int, default=1)
    ap.add_argument("--batch_size", type=int, default=270)
    ap.add_argument("--lr", type=float, default=3e-4)
    ap.add_argument("--warmup", type=int, default=0)
    ap.add_argument("--backward_precision", default="tf32", choices=["fp32", "tf32"])
    ap.add_argument("--out", default="out/model.ckpt")
    ap.add_argument("--val_fraction", type=float, default=0.0, help="share of the data held out for the valid loss")
    ap.add_argument("--test_fraction", type=float, default=0.0, help="share of the data held out for the test loss")
    ap.add_argument("--checkpoint_dir", default=None, help="last.ckpt every epoch, best.ckpt by valid loss")
    args = ap.parse_args()
    if args.val_fraction < 0 or args.test_fraction < 0 or args.val_fraction + args.test_fraction >= 1:
        ap.error("--val_fraction and --test_fraction must be >= 0 and leave a training split")
    if args.val_fraction > 0 and args.test_fraction > 0 and args.checkpoint_dir is None:
        ap.error("a test split with a validation split is evaluated with best.ckpt: give --checkpoint_dir")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        dist.init_process_group("nccl", device_id=device)
    ds = CrystalDataset(args.data)
    rank0 = not dist.is_initialized() or dist.get_rank() == 0
    train_ds, val_ds, test_ds = ds, None, None
    if args.val_fraction > 0 or args.test_fraction > 0:
        parts = split_indices(len(ds), [1.0 - args.val_fraction - args.test_fraction, args.val_fraction,
                                        args.test_fraction], seed=0)
        train_ds, val_ds, test_ds = (CrystalSubset(ds, p) if len(p) else None for p in parts)
    torch.manual_seed(0)
    model = PONITA_DIFFUSION(default_args(lr=args.lr, epochs=args.epochs, warmup=args.warmup, batch_size=args.batch_size), ds.z_table)
    fit(model, train_ds, args.epochs, args.batch_size, device, backward_precision=args.backward_precision,
        val_dataset=val_ds, checkpoint_dir=args.checkpoint_dir)
    if rank0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)) or ".", exist_ok=True)
        model.save_checkpoint(args.out)
    if test_ds is not None:
        if val_ds is not None:           # the weights of the best epoch, as every rank reads them from rank 0's file
            if dist.is_initialized():
                dist.barrier()
            model = PONITA_DIFFUSION.load_from_checkpoint(os.path.join(args.checkpoint_dir, "best.ckpt"))
        res = evaluate_dataset(model, test_ds, args.batch_size, device)
        if rank0:
            print(f"test loss {res['loss']:.6f} (e_frac {res['e_frac']:.6f}, vb {res['vb']:.6f}, ce {res['ce']:.6f}, "
                  f"e_lat {res['e_lat']:.6f}) over {len(test_ds)} crystals")
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
