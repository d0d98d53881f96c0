"""Mirror of lightning_wrappers/diffusion.py: PONITA_DIFFUSION (wiring only -- model, time embedding, diffusion loss,
z_table buffer) with the reference's constructor, `sample`, `training_step`, `configure_optimizers`, and checkpoint
ingestion.  pytorch_lightning is not required: this is a plain nn.Module whose state_dict keys equal the Lightning
module's (`model.*`, `t_emb.*`, `z_table_zs`), so a reference .ckpt loads by name."""
from __future__ import annotations

import argparse
import io
import os
import pickle
from typing import Optional

import numpy as np
import torch
import torch.nn as nn

from ..diffusion.diffusion_helpers import GaussianFourierProjection
from ..diffusion.diffusion_loss import DiffusionLoss, SampleResult
from ..ponita.models.ponita import PonitaFiberBundle
from ..tools.atomic_number_table import AtomicNumberTable, atomic_symbols_to_indices

t_emb_dim = 64          # lightning_wrappers/diffusion.py:22-23
fourier_scale = 16


class PONITA_DIFFUSION(nn.Module):
    """lightning_wrappers/diffusion.py:29-106,220-253."""

    def __init__(self, args, z_table: AtomicNumberTable, ori_grid=None, precision: str = "fp32"):
        super().__init__()
        self.hparams = argparse.Namespace(args=args, z_table=z_table)
        self.register_buffer("z_table_zs", torch.tensor(list(z_table.zs), dtype=torch.int64))
        self.dataset = getattr(args, "dataset", "synthetic")
        Z = len(z_table)
        self.lr, self.weight_decay = getattr(args, "lr", 3e-4), getattr(args, "weight_decay", 0.0)
        self.epochs, self.warmup = getattr(args, "epochs", 1), getattr(args, "warmup", 0)
        if getattr(args, "layer_scale", None) == 0.0:
            args.layer_scale = None
        self.train_augm = getattr(args, "train_augm", False)
        if self.train_augm:
            raise NotImplementedError("rotation augmentation (train_augm) is outside the accelerated path")
        self.t_emb = GaussianFourierProjection(t_emb_dim // 2, fourier_scale)
        self.diffusion_loss = DiffusionLoss(args, Z, precision=precision)
        in_scalar = Z + t_emb_dim + 1 + 3 + 3 + 3                       # :69-76
        self.model = PonitaFiberBundle(in_scalar + 4, args.hidden_dim, Z, 3, 0, 0, args.layers, output_dim_vec=1,
                                       radius=args.radius, num_ori=args.num_ori, basis_dim=args.basis_dim,
                                       degree=args.degree, widening_factor=args.widening_factor,
                                       layer_scale=args.layer_scale, multiple_readouts=args.multiple_readouts,
                                       ori_grid=ori_grid, precision=precision)
        self._optimizer = None

    def forward(self, graph):
        return self.model(graph)

    # ---- training (lightning_wrappers/diffusion.py:107-118,154-216) ------------------------------------------------
    def training_step(self, graph, timestep=None):
        return self.diffusion_loss(self, graph, self.t_emb, timestep)

    def validation_step(self, graph, crystal_ids, seed: int = 0):
        """Forward-only loss of a batch per crystal (DiffusionLoss.evaluate -> EvalResult); `evaluation.evaluate_dataset`
        reduces a whole split to the reference's "valid loss"."""
        return self.diffusion_loss.evaluate(self, graph, self.t_emb, crystal_ids, seed=seed)

    test_step = validation_step

    def configure_optimizers(self, device="cuda", ema_decay=None):
        """torch.optim.Adam with the two weight-decay groups of :161-207 as ONE fused kernel over the flat parameter
        buffer, plus the trainer's gradient_clip_val=0.5 (main_diffusion.py:297); the cosine-warmup factor of
        scheduler.py is applied per epoch with `optimizer.set_epoch(epoch, self.warmup, self.epochs)`.  ema_decay: the
        optimizer also keeps an EMA of the weights (FusedAdam)."""
        from ..training import FusedAdam
        flat = self.model.flat if self.model.flat is not None else self.model.flatten_parameters(device)
        self._optimizer = FusedAdam(flat, lr=self.lr, weight_decay=self.weight_decay, max_grad_norm=0.5,
                                    ema_decay=ema_decay)
        return self._optimizer

    # ---- sampling (:220-253) ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def sample(self, num_atoms_per_sample: int, num_samples_in_batch: int, visualization_setting=None,
               show_bonds: bool = False, use_constant_atomic_symbols: Optional[list] = None, **kw) -> SampleResult:
        z_table = AtomicNumberTable(self.z_table_zs.tolist())
        constant_atoms = None
        if use_constant_atomic_symbols is not None:
            constant_atoms = torch.as_tensor(np.repeat(atomic_symbols_to_indices(z_table, use_constant_atomic_symbols).numpy(),
                                                       num_samples_in_batch))
        return self.diffusion_loss.sample(model=self, z_table=z_table, t_emb_weights=self.t_emb,
                                          num_atoms_per_sample=num_atoms_per_sample,
                                          num_samples_in_batch=num_samples_in_batch, constant_atoms=constant_atoms, **kw)

    # ---- checkpoint ingestion (SURVEY 8f-2) --------------------------------------------------------------------------
    @classmethod
    def load_from_checkpoint(cls, path, ori_grid=None, strict: bool = True, map_location="cpu", **kw):
        """A Lightning .ckpt of the reference: {"state_dict": {model.*, t_emb.*, z_table_zs, diffusion_loss.* ...},
        "hyper_parameters": {"args": Namespace, "z_table": AtomicNumberTable}}.  The pickled z_table refers to the
        reference's module path; it is resolved to this package's class.  The orientation grid is NOT in a reference
        checkpoint (quirk B2: it is rebuilt randomly at construction): pass the grid the model was trained with via
        `ori_grid=` (a checkpoint written by `save_checkpoint` below carries it as `ori_grid`); without one the
        deterministic Fibonacci grid is used and a warning is raised.  `strict` (default True): every `model.*` /
        `t_emb.*` tensor of this module must be in the checkpoint with the same shape, otherwise KeyError -- the
        reference passes strict=False to Lightning only to tolerate ITS extra keys (metrics, zero-width edge
        read-outs), which are ignored here in either mode; a checkpoint that does not fit never samples from
        random weights silently."""
        ckpt = load_checkpoint_file(path, map_location)
        hp = ckpt.get("hyper_parameters", {})
        args, z_table = hp["args"], hp["z_table"]
        if not isinstance(z_table, AtomicNumberTable):
            z_table = AtomicNumberTable(list(z_table.zs))
        grid = ori_grid if ori_grid is not None else ckpt.get("ori_grid")
        if grid is None:
            import warnings
            warnings.warn("checkpoint carries no orientation grid (reference quirk B2): using the Fibonacci grid; "
                          "outputs will differ from the training-time model unless ori_grid= is given")
        m = cls(args, z_table, ori_grid=grid, **kw)
        sd = ckpt["state_dict"]
        own = m.state_dict()
        picked = {k: v for k, v in sd.items() if k in own and tuple(v.shape) == tuple(own[k].shape)}
        missing = [k for k in own if k not in picked and own[k].numel() > 0 and not k.endswith("callibrated")
                   and not k.startswith("diffusion_loss.")]
        if missing:
            bad_shape = {k: (tuple(sd[k].shape), tuple(own[k].shape)) for k in missing if k in sd}
            msg = f"checkpoint {path} lacks {len(missing)} tensors of the model: {missing[:8]}{' ...' if len(missing) > 8 else ''}"
            if bad_shape:
                msg += f"; shape mismatches (checkpoint, model): {bad_shape}"
            if strict:
                raise KeyError(msg)
            import warnings
            warnings.warn(msg + " -- they keep their random initialisation")
        m.load_state_dict(picked, strict=False)
        m.model._packed = None
        return m

    def save_checkpoint(self, path, training_state: Optional[dict] = None) -> None:
        """Lightning-shaped checkpoint (same keys) plus the orientation grid.  training_state: further top-level keys
        that make the file a resume point (`train.fit` writes epoch, global_step, optimizer_states, ema and fit_state
        into last.ckpt); `load_from_checkpoint` ignores them.  The file is written to a temporary name in the same
        directory and renamed over `path`, so an interrupted write leaves the previous file intact."""
        sd = {k: v.detach().cpu() for k, v in self.state_dict().items()}
        ckpt = {"state_dict": sd, "hyper_parameters": {"args": self.hparams.args, "z_table": self.hparams.z_table},
                "ori_grid": self.model.ori_grid.detach().cpu()}
        ckpt.update(training_state or {})
        save_atomic(ckpt, path)


class _RefUnpickler(pickle.Unpickler):
    """Resolves the reference's module paths inside a checkpoint pickle to this package."""
    MAP = {("diffusion.tools.atomic_number_table", "AtomicNumberTable"): AtomicNumberTable}

    def find_class(self, module, name):
        if (module, name) in self.MAP:
            return self.MAP[(module, name)]
        return super().find_class(module, name)


class _PickleModule:
    __name__ = "arreau_b200_ckpt_pickle"
    Unpickler = _RefUnpickler
    load = staticmethod(lambda f, **kw: _RefUnpickler(f, **kw).load())
    loads = staticmethod(lambda b, **kw: _RefUnpickler(io.BytesIO(b), **kw).load())


def save_atomic(obj, path) -> None:
    """torch.save to a temporary file next to `path`, then os.replace: readers see the old file or the new one."""
    path = os.fspath(path)
    tmp = f"{path}.{os.getpid()}.tmp"
    try:
        with open(tmp, "wb") as f:
            torch.save(obj, f)
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.unlink(tmp)
        raise


def load_checkpoint_file(path, map_location="cpu") -> dict:
    """torch.load of a (trusted) Lightning checkpoint with the reference's class paths remapped."""
    return torch.load(path, map_location=map_location, weights_only=False, pickle_module=_PickleModule)
