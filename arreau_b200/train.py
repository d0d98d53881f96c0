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
the end with the best.ckpt weights (the final weights without a validation split).

last.ckpt also carries the training state (Adam moments and step, epoch, loss history, best valid loss, every rank's
CUDA generator, the EMA), so `--resume out/ckpt/last.ckpt` with the same data, batch size, fractions and --epochs
continues the run exactly where it stopped.  --ema_decay D keeps an exponential moving average of the weights (the NeMo
EMA callback the reference carries): the EMA weights are the ones validated and tested, and last.ckpt, best.ckpt and
--out each get a twin *-EMA.ckpt holding them (a plain model checkpoint, e.g. for `generate --model_path`).

--sample_every K --sample_count M tracks sample quality during training: after the validation of every K-th and of the
last epoch, M crystals (atom counts drawn once from the training split, noise keyed per crystal, so every pass samples
the same crystals) are generated at fp16 with the validated weights, each GPU its shard; their structural validity,
density and element-count distances to the validation split (the training split without one) and min-distance
percentiles are logged on the epoch line and kept in last.ckpt (SampleMonitor).  best.ckpt stays chosen by the valid
loss, and the training itself is the same with and without monitoring."""
from __future__ import annotations

import argparse
import os
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from .diffusion.lattice_dataset import CrystalDataset, CrystalSubset, batches, split_indices
from .distributed import (allreduce_gradients, broadcast_parameters, gather_rng_states, rank_rng_state,
                          reduce_loss_metric, shard_range)
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


def ema_path(path: str) -> str:
    """The EMA twin of a checkpoint path: out/ckpt/last.ckpt -> out/ckpt/last-EMA.ckpt (NeMo's naming)."""
    root, ext = os.path.splitext(path)
    return f"{root}-EMA{ext}"


def ema_model(model: PONITA_DIFFUSION, device) -> PONITA_DIFFUSION:
    """A second model whose trainable tensors are views of the EMA buffer of `model`'s optimizer (FusedAdam with
    ema_decay; the buffer is not written): evaluating or saving it reads the EMA, while the training weights, moments
    and engines are not touched.  Its buffers (the `callibrated` flags) and time embedding are copies of `model`'s.
    Every optimizer step bumps the EMA buffer's version, so its packed kernel weights are rebuilt when used.  The CPU
    random generator is left as it was."""
    opt = model._optimizer
    if opt is None or opt.ema is None:
        raise ValueError("the model's optimizer keeps no EMA: configure_optimizers(ema_decay=...) first")
    with torch.random.fork_rng(devices=[]):
        m = PONITA_DIFFUSION(model.hparams.args, model.hparams.z_table, ori_grid=model.model.ori_grid.detach().cpu(),
                             precision=model.model.precision)
    m.load_state_dict(model.state_dict(), strict=False)
    m.to(device)
    m.model.flatten_parameters(device, into=opt.ema)
    return m


def sampling_model(model: PONITA_DIFFUSION, device, flat=None) -> PONITA_DIFFUSION:
    """A twin of `model` for sampling, built like `ema_model`'s: fp16 (generate's default precision), its trainable
    tensors views of `flat` (a FlatParams; default the model's own weight buffer, or e.g. its optimizer's EMA buffer),
    which is only read.  It has its own DiffusionLoss, so its sampling engine is neither the train nor the eval engine.
    Its buffers and time embedding are copies of `model`'s.  The CPU random generator is left as it was."""
    flat = model.model.flat if flat is None else flat
    if flat is None:
        raise ValueError("the model has no flat weight buffer: flatten_parameters / configure_optimizers first")
    with torch.random.fork_rng(devices=[]):
        m = PONITA_DIFFUSION(model.hparams.args, model.hparams.z_table, ori_grid=model.model.ori_grid.detach().cpu(),
                             precision="fp16")
    m.load_state_dict(model.state_dict(), strict=False)
    m.to(device)
    m.model.flatten_parameters(device, into=flat)
    return m


# crystals per sampling batch of a sample-quality pass (the batch bounds the device memory, not the result)
SAMPLE_BATCH = 1024


class SampleMonitor:
    """Sample quality inside `fit`: `count` crystals with ids 0..count-1, their atom counts drawn once per run from the
    training split (draw_num_atoms with the run's seed) and their noise keyed by (seed, id), so every pass samples the
    same crystals with the same noise and a change between passes comes from the weights only.  Each rank samples its
    shard_range of the ids with the fp16 sampling twin (the CUDA-graph trajectory when max_neighbors > 0), computes
    crystal_metrics on the device, and the rows are all-gathered once; rank 0 summarizes them against a reference
    computed once from `reference_dataset`.  No torch RNG, and neither the training weights nor the train / eval
    engines are written."""

    def __init__(self, model: PONITA_DIFFUSION, flat, train_dataset, reference_dataset, count: int, seed: int, device):
        from .generate import draw_num_atoms
        self.model, self.flat, self.device, self.seed = model, flat, torch.device(device), int(seed)
        self.num_atoms = draw_num_atoms(train_dataset.atom_counts(), int(count), self.seed)
        self.reference_dataset = reference_dataset
        self.reference = None
        self.twin = None

    def local_metrics(self):
        """crystal_metrics of this rank's shard of the crystals (its SampleResults never leave the rank)."""
        from .inference.crystal_metrics import concat_metrics, crystal_metrics, sample_inputs
        rank = dist.get_rank() if dist.is_initialized() else 0
        world = dist.get_world_size() if dist.is_initialized() else 1
        if self.twin is None:
            self.twin = sampling_model(self.model, self.device, self.flat)
        lo, hi = shard_range(len(self.num_atoms), rank, world)
        graph = self.twin.diffusion_loss.max_neighbors > 0
        parts = []
        for b0 in range(lo, hi, SAMPLE_BATCH):
            b1 = min(b0 + SAMPLE_BATCH, hi)
            res = self.twin.sample(None, b1 - b0, num_atoms=torch.from_numpy(self.num_atoms[b0:b1].copy()),
                                   crystal_ids=torch.arange(b0, b1, dtype=torch.int64), seed=self.seed,
                                   device=self.device, cuda_graph=graph)
            parts.append(crystal_metrics(*sample_inputs(res), device=self.device))
        return concat_metrics(parts)

    def run(self, epoch: int) -> Optional[dict]:
        """One pass (a collective): the quality_record of `epoch` on rank 0, None on the other ranks."""
        from .distributed import gather_crystal_metrics
        from .inference.crystal_metrics import crystal_metrics, dataset_inputs, quality_record, summarize
        local = self.local_metrics()
        comm = self.device if dist.is_initialized() and dist.get_backend() == "nccl" else None
        rows = gather_crystal_metrics(local, device=comm)
        if dist.is_initialized() and dist.get_rank() != 0:
            return None
        if self.reference is None:
            self.reference = crystal_metrics(*dataset_inputs(self.reference_dataset), device=self.device)
        return quality_record(summarize(rows, self.reference), epoch)


def _fmt(v) -> str:
    return "n/a" if v is None else f"{v:.4g}"


def format_quality(rec: dict) -> str:
    """The sample-quality part of fit's epoch line."""
    return (f"samples: valid {_fmt(rec['frac_valid'])}, w1 density {_fmt(rec['w1_density'])}, w1 elements "
            f"{_fmt(rec['w1_num_elements'])}, min dist p1/p5/p25/p50 "
            + "/".join(_fmt(rec[f"min_dist_p{p}"]) for p in (1, 5, 25, 50)))


def check_monitoring(sample_every: int, sample_count: int) -> None:
    """ValueError unless sample_every >= 0 (0: off) and sample_count >= 1."""
    if int(sample_every) != sample_every or sample_every < 0:
        raise ValueError(f"sample_every must be an integer >= 0 (0 turns sample monitoring off), got {sample_every}")
    if int(sample_count) != sample_count or sample_count < 1:
        raise ValueError(f"sample_count must be an integer >= 1, got {sample_count}")


def check_resume(ckpt, *, epochs: int, batch_size: int, world_size: int, backward_precision: str, num_train: int,
                 num_valid: int, seed: int = 0, ema_decay: Optional[float] = None, sample_every: int = 0,
                 sample_count: int = 1024) -> dict:
    """The checkpoint (a path or the loaded dict) if it is a resume point of the run these arguments describe; a
    ValueError naming every mismatch otherwise.  Reads the file only (no device work).  A checkpoint written before
    sample monitoring existed is a run with sample_every 0; with monitoring off the sample count is not compared."""
    from .lightning_wrappers.diffusion import load_checkpoint_file
    name = ckpt if isinstance(ckpt, (str, os.PathLike)) else "checkpoint"
    if not isinstance(ckpt, dict):
        ckpt = load_checkpoint_file(ckpt)
    fs = ckpt.get("fit_state")
    if not isinstance(fs, dict) or "optimizer_states" not in ckpt or "epoch" not in ckpt:
        raise ValueError(f"{name} holds no training state written by train.fit (a model-only checkpoint such as "
                         "best.ckpt, or a Lightning checkpoint): resume from the last.ckpt of a fit run")
    saved_ema = ckpt.get("ema")
    have = {"batch_size": fs["batch_size"], "world size": fs["world_size"],
            "backward_precision": fs["backward_precision"], "train split size": fs["num_train"],
            "valid split size": fs["num_valid"], "seed": fs["seed"],
            "ema_decay": None if saved_ema is None else float(saved_ema["decay"]),
            "epochs": getattr(ckpt["hyper_parameters"]["args"], "epochs", None)}
    saved_every = int(fs.get("sample_every", 0))
    have.update({"sample_every": saved_every, "sample_count": fs.get("sample_count") if saved_every else None})
    want = {"batch_size": batch_size, "world size": world_size, "backward_precision": backward_precision,
            "train split size": num_train, "valid split size": num_valid, "seed": seed,
            "ema_decay": None if ema_decay is None else float(ema_decay), "epochs": epochs,
            "sample_every": int(sample_every), "sample_count": int(sample_count) if sample_every else None}
    bad = [f"{k}: checkpoint {have[k]}, this run {want[k]}" for k in want if have[k] != want[k]]
    if bad:
        raise ValueError(f"{name} is not a resume point of this run: " + "; ".join(bad))
    return ckpt


def fit(model: PONITA_DIFFUSION, dataset: CrystalDataset, epochs: int, batch_size: int, device, seed: int = 0,
        backward_precision: str = "tf32", calibrate: bool = True, log=print, val_dataset=None,
        checkpoint_dir: Optional[str] = None, metrics: Optional[dict] = None, resume_from: Optional[str] = None,
        ema_decay: Optional[float] = None, sample_every: int = 0, sample_count: int = 1024):
    """Trains `model` for `epochs` and returns the per-epoch train loss.  val_dataset: evaluated after every epoch
    (evaluate_dataset with the same batch_size and seed; logged as "valid loss").  checkpoint_dir: rank 0 writes
    last.ckpt every epoch -- the weights plus the training state a resume needs -- and, with a validation set, best.ckpt
    whenever the valid loss improves.  metrics (optional dict): receives metrics["valid"], one evaluate_dataset result
    per epoch of this call, and (rank 0, with sample monitoring) metrics["samples"], one record per pass of this call,
    and metrics["sample_quality"], the run's whole history of them.

    sample_every K > 0: after the validation of every K-th epoch and of the last epoch, `sample_count` crystals are
    sampled with the weights that are validated (the EMA when there is one) and their quality is measured on the
    device (SampleMonitor: keyed noise, so every pass samples the same crystals with the same noise).  Rank 0 appends a
    compact record -- epoch, valid fraction, w1_density, w1_num_elements, min-distance percentiles (quality_record),
    against the validation split, or the training split without one -- to the run's `sample_quality` history, which
    last.ckpt carries and a resume restores; it is logged on the epoch line.  best.ckpt is still chosen by the valid
    loss, and training is bit-identical with and without monitoring.  K < 0 or sample_count < 1 is a ValueError,
    raised before any device work.

    resume_from: a last.ckpt of a run with the same data splits, batch_size, world size, backward_precision, seed and
    ema_decay, whose model was built with `epochs` epochs (checked before any device work, ValueError otherwise).  The
    weights, the Adam state, the EMA, every rank's CUDA generator, the loss history and the best valid loss are
    restored, calibration is skipped, and epochs epoch+1 .. epochs-1 run; the returned history starts at epoch 0, so
    a resumed run returns what the uninterrupted run returns.

    ema_decay: the optimizer keeps an EMA of the weights (FusedAdam).  The EMA weights are the ones validated (and
    best.ckpt is chosen by their loss), and last.ckpt / best.ckpt each get a twin *-EMA.ckpt, a model checkpoint of
    the EMA weights.  Training itself is the same as without EMA."""
    check_monitoring(sample_every, sample_count)
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    ckpt = None
    if resume_from is not None:
        ckpt = check_resume(resume_from, epochs=epochs, batch_size=batch_size, world_size=world,
                            backward_precision=backward_precision, num_train=len(dataset),
                            num_valid=0 if val_dataset is None else len(val_dataset), seed=seed, ema_decay=ema_decay,
                            sample_every=sample_every, sample_count=sample_count)
    model.to(device)
    model.diffusion_loss.backward_precision = backward_precision
    opt = model.configure_optimizers(device, ema_decay=ema_decay)
    flat = model.model.flat
    history, valid_losses, quality = [], [], []
    best = float("inf")
    first = 0
    if ckpt is not None:
        sd = ckpt["state_dict"]
        own = model.state_dict()
        model.load_state_dict({k: v for k, v in sd.items() if k in own}, strict=False)   # parameters are views of flat
        flat.version += 1
        model.model._packed = None
        opt.load_state_dict(ckpt["optimizer_states"][0])
        fs = ckpt["fit_state"]
        history, valid_losses, best = list(fs["train_losses"]), list(fs["valid_losses"]), float(fs["best_valid"])
        quality = [dict(r) for r in fs.get("sample_quality", [])]
        first = int(ckpt["epoch"]) + 1
        calibrate = False
    broadcast_parameters(flat.data)
    twin = ema_model(model, device) if ema_decay is not None else None
    if ckpt is not None:
        if twin is not None:
            opt.ema.load_state_dict({k[len("model."):]: v for k, v in ckpt["ema"]["state_dict"].items()})
        torch.cuda.set_rng_state(rank_rng_state(ckpt["fit_state"]["cuda_rng"]), device)
    monitor = None
    if sample_every > 0:
        monitor = SampleMonitor(model, opt.ema if twin is not None else flat, dataset,
                                val_dataset if val_dataset is not None else dataset, sample_count, seed, device)
    comm = device if dist.is_initialized() and dist.get_backend() == "nccl" else None
    if checkpoint_dir is not None and rank == 0:
        os.makedirs(checkpoint_dir, exist_ok=True)
    for epoch in range(first, epochs):
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
                for m in (model,) if twin is None else (model, twin):
                    for layer in m.model.interaction_layers:
                        layer.conv.callibrated.fill_(True)
                calibrate = False
            allreduce_gradients(flat.grad)
            opt.step()                                 # with ema_decay: the EMA is initialised at the first step
            total_loss += loss.detach().double()
            total_samples += batch.num_atoms.shape[0]
        metric = reduce_loss_metric(total_loss, total_samples)
        history.append(float(metric))
        valid = None
        if val_dataset is not None:
            valid = evaluate_dataset(model if twin is None else twin, val_dataset, batch_size, device, seed=seed)
            valid_losses.append(valid["loss"])
            if metrics is not None:
                metrics.setdefault("valid", []).append(valid)
        improved = valid is not None and valid["loss"] < best
        if improved:
            best = valid["loss"]
        sampled = None
        if monitor is not None and ((epoch + 1) % sample_every == 0 or epoch == epochs - 1):
            sampled = monitor.run(epoch)              # a collective; the record on rank 0 only
            if sampled is not None:
                quality.append(sampled)
                if metrics is not None:
                    metrics.setdefault("samples", []).append(sampled)
        state = None
        if checkpoint_dir is not None:                 # every rank's generator (a collective), then rank 0 writes
            rng = gather_rng_states(torch.cuda.get_rng_state(device), device=comm)
            if rank == 0:
                state = {"epoch": epoch, "global_step": opt.step_count, "optimizer_states": [opt.state_dict()],
                         "ema": None if twin is None else {
                             "decay": opt.ema_decay,
                             "state_dict": {"model." + k: v.detach().cpu() for k, v in opt.ema.views().items()}},
                         "fit_state": {"seed": seed, "batch_size": batch_size, "world_size": world,
                                       "backward_precision": backward_precision, "num_train": len(dataset),
                                       "num_valid": 0 if val_dataset is None else len(val_dataset),
                                       "train_losses": list(history), "valid_losses": list(valid_losses),
                                       "best_valid": best, "cuda_rng": rng, "sample_every": int(sample_every),
                                       "sample_count": int(sample_count),
                                       "sample_quality": [dict(r) for r in quality]}}
        if rank == 0:
            shown = "" if valid is None else f", valid loss {valid['loss']:.6f}" + (" (EMA weights)" if twin is not None else "")
            if sampled is not None:
                shown += ", " + format_quality(sampled)
            log(f"epoch {epoch}: train loss {history[-1]:.6f}{shown} (lr {opt.lr:.3e})")
            if checkpoint_dir is not None:
                saves = [("last.ckpt", state)] + ([("best.ckpt", None)] if improved else [])
                for name, extra in saves:
                    model.save_checkpoint(os.path.join(checkpoint_dir, name), training_state=extra)
                    if twin is not None:
                        twin.save_checkpoint(ema_path(os.path.join(checkpoint_dir, name)))
    if metrics is not None and monitor is not None and rank == 0:
        metrics["sample_quality"] = [dict(r) for r in quality]
    return history


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--data", nargs="+", required=True, help="dataset files (.h5 as written by prep_datasets.py, or .npz)")
    ap.add_argument("--epochs", type=int, default=1)
    ap.add_argument("--batch_size", type=int, default=270)
    ap.add_argument("--lr", type=float, default=None, help="default 3e-4 (on --resume: the checkpoint's)")
    ap.add_argument("--warmup", type=int, default=None, help="default 0 (on --resume: the checkpoint's)")
    ap.add_argument("--backward_precision", default="tf32", choices=["fp32", "tf32"])
    ap.add_argument("--out", default="out/model.ckpt")
    ap.add_argument("--val_fraction", type=float, default=0.0, help="share of the data held out for the valid loss")
    ap.add_argument("--test_fraction", type=float, default=0.0, help="share of the data held out for the test loss")
    ap.add_argument("--checkpoint_dir", default=None, help="last.ckpt every epoch, best.ckpt by valid loss")
    ap.add_argument("--resume", default=None, metavar="PATH",
                    help="continue the run whose last.ckpt this is; --data, --batch_size, the fractions, --epochs, "
                         "--backward_precision and --ema_decay must be the run's")
    ap.add_argument("--ema_decay", type=float, default=None,
                    help="keep an EMA of the weights (e.g. 0.999): it is validated and saved as *-EMA.ckpt twins")
    ap.add_argument("--sample_every", type=int, default=0, metavar="K",
                    help="every K-th and the last epoch, sample --sample_count crystals with the validated weights and "
                         "log their quality (0: off)")
    ap.add_argument("--sample_count", type=int, default=1024, metavar="M", help="crystals per sample-quality pass")
    args = ap.parse_args(argv)
    try:
        check_monitoring(args.sample_every, args.sample_count)
    except ValueError as e:
        ap.error(str(e))
    if args.val_fraction < 0 or args.test_fraction < 0 or args.val_fraction + args.test_fraction >= 1:
        ap.error("--val_fraction and --test_fraction must be >= 0 and leave a training split")
    if args.val_fraction > 0 and args.test_fraction > 0 and args.checkpoint_dir is None:
        ap.error("a test split with a validation split is evaluated with best.ckpt: give --checkpoint_dir")
    if args.ema_decay is not None and not 0.0 <= args.ema_decay <= 1.0:
        ap.error("--ema_decay must be in [0, 1]")
    ds = CrystalDataset(args.data)
    train_ds, val_ds, test_ds = ds, None, None
    if args.val_fraction > 0 or args.test_fraction > 0:
        parts = split_indices(len(ds), [1.0 - args.val_fraction - args.test_fraction, args.val_fraction,
                                        args.test_fraction], seed=0)
        train_ds, val_ds, test_ds = (CrystalSubset(ds, p) if len(p) else None for p in parts)
    if args.resume is not None:         # refused before any device work
        try:
            hp = check_resume(args.resume, epochs=args.epochs, batch_size=args.batch_size,
                              world_size=int(os.environ.get("WORLD_SIZE", "1")),
                              backward_precision=args.backward_precision, num_train=len(train_ds),
                              num_valid=0 if val_ds is None else len(val_ds), ema_decay=args.ema_decay,
                              sample_every=args.sample_every,
                              sample_count=args.sample_count)["hyper_parameters"]["args"]
        except ValueError as e:
            ap.error(str(e))
        for k in ("lr", "warmup"):
            if getattr(args, k) is not None and getattr(args, k) != getattr(hp, k):
                ap.error(f"--{k} {getattr(args, k)} differs from the resumed run's {getattr(hp, k)}")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        dist.init_process_group("nccl", device_id=device)
    rank0 = not dist.is_initialized() or dist.get_rank() == 0
    if args.resume is not None:
        model = PONITA_DIFFUSION.load_from_checkpoint(args.resume)
    else:
        torch.manual_seed(0)
        model = PONITA_DIFFUSION(default_args(lr=3e-4 if args.lr is None else args.lr, epochs=args.epochs,
                                              warmup=args.warmup or 0, batch_size=args.batch_size), ds.z_table)
    fit(model, train_ds, args.epochs, args.batch_size, device, backward_precision=args.backward_precision,
        val_dataset=val_ds, checkpoint_dir=args.checkpoint_dir, resume_from=args.resume, ema_decay=args.ema_decay,
        sample_every=args.sample_every, sample_count=args.sample_count)
    twin = ema_model(model, device) if args.ema_decay is not None else None
    if rank0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)) or ".", exist_ok=True)
        model.save_checkpoint(args.out)
        if twin is not None:
            twin.save_checkpoint(ema_path(args.out))
    if test_ds is not None:
        model = model if twin is None else twin
        if val_ds is not None:           # the weights of the best epoch, as every rank reads them from rank 0's file
            if dist.is_initialized():
                dist.barrier()
            best = os.path.join(args.checkpoint_dir, "best.ckpt")
            model = PONITA_DIFFUSION.load_from_checkpoint(best if twin is None else ema_path(best))
        res = evaluate_dataset(model, test_ds, args.batch_size, device)
        if rank0:
            print(f"test loss {res['loss']:.6f} (e_frac {res['e_frac']:.6f}, vb {res['vb']:.6f}, ce {res['ce']:.6f}, "
                  f"e_lat {res['e_lat']:.6f}) over {len(test_ds)} crystals")
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
