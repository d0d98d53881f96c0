"""Training step of the Arreau diffusion model on the GPU (SURVEY 8a rows a19-a23).

Host logic only: buffer ownership and the launch sequence of one step
    noising (VE / D3PM / VP)  ->  predict_scores (graph + fp32 forward, per-layer buffers kept)
    ->  three-term loss + output gradients  ->  hand-written backward  ->  flat gradient buffer
mirroring DiffusionLoss.__call__ (diffusion/diffusion_loss.py:204-274) followed by loss.backward().  Every
computation is a kernel of libarreau_b200.so (csrc/train_ops.cu, csrc/train_net.cu, and the forward kernels).
Parameters and gradients live in ONE flat fp32 buffer each (arreau_train_layout_t order) whose slices are exposed
under the reference's state_dict names, so an optimizer / all-reduce sees a single tensor.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Mapping, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .engine import DenoiseEngine
from .tables import DiffusionTables
from .weights import BASIS, HIDDEN, LAYERS, WIDEN, PonitaWeights, monomial_fold_table

HYBRID_LOSS_COEFF = 0.001    # diffusion/d3pm.py:15


class FlatParams:
    """The model's trainable tensors as slices of one flat fp32 device buffer (+ a gradient buffer of the same
    layout), keyed like the reference's state_dict."""

    def __init__(self, num_scalar: int, num_vec: int, num_states: int, device):
        self.device = torch.device(device)
        self.layout = _lib.TrainLayout()
        _lib.call("arreau_train_layout", num_scalar, num_vec, num_states, C.byref(self.layout))
        self.num_scalar, self.num_vec, self.num_states = num_scalar, num_vec, num_states
        self.total = int(self.layout.total)
        self.data = torch.zeros(self.total, dtype=torch.float32, device=self.device)
        self.grad = torch.zeros(self.total, dtype=torch.float32, device=self.device)
        # bumped by everything that changes `data` in place (optimizer step, load_state_dict, callibrate), so that
        # cached kernel-layout copies of the weights (PonitaWeights of a sampling engine) know they are stale
        self.version = 0
        R, FV, L, Cc, D, W = num_states + 4, num_scalar + num_vec, LAYERS, HIDDEN, BASIS, WIDEN * HIDDEN
        lay = self.layout
        self.specs = {   # name -> (offset, shape)
            "basis_fn.1.weight": (lay.basis_w1, (Cc, 258)), "basis_fn.1.bias": (lay.basis_b1, (Cc,)),
            "basis_fn.3.weight": (lay.basis_w2, (D, Cc)), "basis_fn.3.bias": (lay.basis_b2, (D,)),
            "fiber_basis_fn.1.weight": (lay.fiber_w1, (Cc, 3)), "fiber_basis_fn.1.bias": (lay.fiber_b1, (Cc,)),
            "fiber_basis_fn.3.weight": (lay.fiber_w2, (D, Cc)), "fiber_basis_fn.3.bias": (lay.fiber_b2, (D,)),
            "x_embedder.weight": (lay.embed_w, (Cc, FV)),
        }
        per_layer = {"layer_scale": (lay.layer_scale, (Cc,)), "conv.bias": (lay.conv_bias, (Cc,)),
                     "conv.kernel.weight": (lay.conv_kernel_w, (Cc, D)),
                     "conv.fiber_kernel.weight": (lay.conv_fiber_w, (Cc, D)),
                     "linear_1.weight": (lay.lin1_w, (W, Cc)), "linear_1.bias": (lay.lin1_b, (W,)),
                     "linear_2.weight": (lay.lin2_w, (Cc, W)), "linear_2.bias": (lay.lin2_b, (Cc,)),
                     "norm.weight": (lay.norm_w, (Cc,)), "norm.bias": (lay.norm_b, (Cc,))}
        for l in range(L):
            for name, (off, shape) in per_layer.items():
                self.specs[f"interaction_layers.{l}.{name}"] = (off + l * int(np.prod(shape)), shape)
            self.specs[f"read_out_layers.{l}.weight"] = (lay.readout_w + l * R * Cc, (R, Cc))
            self.specs[f"read_out_layers.{l}.bias"] = (lay.readout_b + l * R, (R,))
        assert sum(int(np.prod(s)) for _, s in self.specs.values()) == self.total

    def decay_mask(self) -> torch.Tensor:
        """1 for the elements torch.optim.Adam decays in the reference (lightning_wrappers/diffusion.py:161-186: the
        `weight` of every nn.Linear), 0 for biases, LayerNorm weights and layer_scale."""
        mask = torch.zeros(self.total, dtype=torch.uint8)
        for k, (off, shape) in self.specs.items():
            if k.endswith(".weight") and ".norm." not in k:
                mask[off:off + int(np.prod(shape))] = 1
        return mask.to(self.device)

    def _views(self, buf: torch.Tensor) -> Dict[str, torch.Tensor]:
        return {k: buf[off:off + int(np.prod(shape))].view(shape) for k, (off, shape) in self.specs.items()}

    def views(self) -> Dict[str, torch.Tensor]:
        return self._views(self.data)

    def grad_views(self) -> Dict[str, torch.Tensor]:
        return self._views(self.grad)

    def load_state_dict(self, sd: Mapping[str, object]) -> None:
        for k, v in self.views().items():
            v.copy_(torch.as_tensor(np.asarray(sd[k].detach().cpu()) if isinstance(sd[k], torch.Tensor) else np.asarray(sd[k]),
                                    dtype=torch.float32).reshape(v.shape))
        self.version += 1

    def state_dict(self) -> Dict[str, torch.Tensor]:
        return {k: v.clone() for k, v in self.views().items()}


def cosine_warmup_factor(epoch: int, warmup: int, max_iters: int) -> float:
    """lightning_wrappers/scheduler.py:14-18."""
    f = 0.5 * (1 + np.cos(np.pi * epoch / max_iters))
    if epoch <= warmup:
        f *= (epoch + 1e-6) * 1.0 / (warmup + 1e-6)
    return float(f)


class FusedAdam:
    """torch.optim.Adam over the flat buffers as one kernel (arreau_adam_step) with the reference's two weight-decay
    groups and the trainer's global-norm clip (gradient_clip_val=0.5, main_diffusion.py:297).

    ema_decay: keep an exponential moving average of the weights in `self.ema` (a FlatParams of the same layout), the
    rule of the NeMo EMA callback the reference carries (lightning_wrappers/callbacks.py): the EMA is set to the weights
    as they are just before the first optimizer step (device copy), and every step updates it from the post-step weights,
    ema = decay * ema + (1 - decay) * p, inside the Adam kernel."""

    def __init__(self, params: FlatParams, lr: float = 3e-4, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0, max_grad_norm: float = 0.5, ema_decay: Optional[float] = None):
        self.p, self.base_lr, self.lr = params, lr, lr
        self.betas, self.eps, self.weight_decay, self.max_grad_norm = betas, eps, weight_decay, max_grad_norm
        self.exp_avg, self.exp_avg_sq = torch.zeros_like(params.data), torch.zeros_like(params.data)
        self.mask = params.decay_mask()
        self.step_count = 0
        self.scratch = torch.zeros(512, dtype=torch.float64, device=params.device)
        self.moments = torch.zeros(2, dtype=torch.float64, device=params.device)
        if ema_decay is not None and not 0.0 <= float(ema_decay) <= 1.0:
            raise ValueError(f"ema_decay must be in [0, 1], got {ema_decay}")
        self.ema_decay = None if ema_decay is None else float(ema_decay)
        self.ema = None if ema_decay is None else FlatParams(params.num_scalar, params.num_vec, params.num_states,
                                                              params.device)
        self.ema_initialized = False

    def set_epoch(self, epoch: int, warmup: int, max_epochs: int) -> None:
        self.lr = self.base_lr * cosine_warmup_factor(epoch, warmup, max_epochs)

    def step(self) -> None:
        p = self.p
        s = torch.cuda.current_stream(p.device).cuda_stream
        self.step_count += 1
        p.version += 1
        if self.ema is not None:
            if not self.ema_initialized:
                self.ema.data.copy_(p.data)
                self.ema_initialized = True
            self.ema.version += 1
        _lib.call("arreau_moments", p.grad.data_ptr(), None, p.total, self.scratch.data_ptr(), self.moments.data_ptr(), s)
        _lib.call("arreau_adam_step", p.data.data_ptr(), p.grad.data_ptr(), self.exp_avg.data_ptr(),
                  self.exp_avg_sq.data_ptr(), self.mask.data_ptr(), p.total, self.lr, self.betas[0], self.betas[1],
                  self.eps, self.weight_decay, self.step_count, self.max_grad_norm, self.moments.data_ptr(),
                  _lib.ptr(None if self.ema is None else self.ema.data), self.ema_decay or 0.0, s)

    def grad_norm(self) -> float:
        """Global L2 norm of the last step's (unclipped) gradient (host synchronisation)."""
        return float(np.sqrt(self.moments[1].item()))

    # -- state (the layout of torch.optim.Adam.state_dict) ------------------------------------------------------------
    def param_groups(self):
        """The two groups of the reference's configure_optimizers as (weight_decay, [names]): the decayed Linear
        weights, then everything else, each in FlatParams.specs order (the names of FlatParams.decay_mask)."""
        decayed = [k for k in self.p.specs if k.endswith(".weight") and ".norm." not in k]
        rest = [k for k in self.p.specs if not (k.endswith(".weight") and ".norm." not in k)]
        return [(self.weight_decay, decayed), (0.0, rest)]

    def state_dict(self) -> dict:
        """torch.optim.Adam.state_dict() of the same named groups: state[i] = {step, exp_avg, exp_avg_sq} in each
        parameter's shape (host copies), param_groups with the hyper-parameters, `params` and `param_names` -- it loads
        into a torch.optim.Adam built from those groups.  `ema`: the EMA's bookkeeping {decay, initialized} (its
        weights are saved with the model's names by the checkpoint)."""
        m, v = self.p._views(self.exp_avg), self.p._views(self.exp_avg_sq)
        state, groups, i = {}, [], 0
        for wd, names in self.param_groups():
            idx = list(range(i, i + len(names)))
            for j, k in zip(idx, names):
                state[j] = {"step": torch.tensor(float(self.step_count), dtype=torch.float32),
                            "exp_avg": m[k].detach().cpu().clone(), "exp_avg_sq": v[k].detach().cpu().clone()}
            groups.append({"param_names": list(names), "weight_decay": wd, "lr": self.lr, "initial_lr": self.base_lr,
                           "betas": tuple(self.betas), "eps": self.eps, "amsgrad": False, "maximize": False,
                           "foreach": None, "capturable": False, "differentiable": False, "fused": None,
                           "decoupled_weight_decay": False, "params": idx})
            i += len(names)
        return {"state": state, "param_groups": groups,
                "ema": {"decay": self.ema_decay, "initialized": bool(self.ema_initialized)}}

    def load_state_dict(self, sd: Mapping) -> None:
        """Restores the step count, both moments and the EMA bookkeeping from `state_dict()`'s layout, matched by
        parameter NAME (not position).  The hyper-parameters stay this optimizer's.  Refuses a state without
        `param_names` (e.g. a Lightning checkpoint of the reference), with other names or shapes, or with a different
        EMA decay.  The EMA weights themselves are restored with `self.ema.load_state_dict`.  Bumps the flat buffers'
        versions like every other in-place load."""
        groups = sd.get("param_groups", [])
        if not groups or any("param_names" not in g for g in groups):
            raise ValueError("optimizer state has no param_names: it was not written by this project's FusedAdam "
                             "state_dict (a Lightning optimizer state cannot be mapped onto the parameters)")
        by_name = {}
        for g in groups:
            if len(g["param_names"]) != len(g["params"]):
                raise ValueError("optimizer state: param_names and params differ in length")
            for k, i in zip(g["param_names"], g["params"]):
                by_name[k] = sd["state"][i]
        if set(by_name) != set(self.p.specs):
            diff = sorted(set(by_name) ^ set(self.p.specs))
            raise ValueError(f"optimizer state does not name this model's parameters: {diff[:8]}")
        steps = {int(float(st["step"])) for st in by_name.values()}
        if len(steps) != 1:
            raise ValueError(f"optimizer state: parameters are at different steps {sorted(steps)}")
        ema = sd.get("ema") or {"decay": None, "initialized": False}
        if (ema["decay"] is None) != (self.ema_decay is None) or (ema["decay"] is not None and float(ema["decay"]) != self.ema_decay):
            raise ValueError(f"optimizer state has EMA decay {ema['decay']}, this optimizer {self.ema_decay}")
        m, v = self.p._views(self.exp_avg), self.p._views(self.exp_avg_sq)
        for k, st in by_name.items():
            for dst, key in ((m[k], "exp_avg"), (v[k], "exp_avg_sq")):
                src = torch.as_tensor(st[key])
                if tuple(src.shape) != tuple(dst.shape):
                    raise ValueError(f"optimizer state {key} of {k}: shape {tuple(src.shape)}, parameter {tuple(dst.shape)}")
                dst.copy_(src.to(torch.float32))
        self.step_count = steps.pop()
        self.ema_initialized = bool(ema["initialized"])
        self.p.version += 1
        if self.ema is not None:
            self.ema.version += 1


def noising_buffers(N: int, G: int, Z: int, dev) -> Dict[str, tuple]:
    """Capacity buffers of a clean batch, its random draws and the noising outputs: name -> (leading extent kind,
    buffer), the layout `noise_into` reads."""
    f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)  # noqa: E731
    return {"frac0": ("N", f64(N, 3)), "types0": ("N", torch.zeros(N, dtype=torch.int64, device=dev)),
            "lattice0": ("G", f64(G, 3, 3)), "lengths0": ("G", f64(G, 3)), "angles0": ("G", f64(G, 3)),
            "target_eps": ("N", f64(N, 3)), "eps_x": ("N", f64(N, 3)), "u": ("N", f64(N, Z)), "eps_l": ("G", f64(G, 3)),
            "t_crystal": ("G", torch.ones(G, dtype=torch.int32, device=dev)),
            "t_atom": ("N", torch.ones(N, dtype=torch.int32, device=dev)), "terms": ("3N", f64(3 * N))}


def noise_into(e: DenoiseEngine, b) -> None:
    """VE_pbc.forward, D3PM.get_xt, matrix_to_params + VP_lattice.forward (diffusion_loss.py:218-237) of the clean
    batch held by `b` (the `noising_buffers` of a training or evaluation engine, bound to e's topology) into the forward
    engine's state."""
    s = e.stream
    _lib.call("arreau_matrix_to_params", b.lattice0.data_ptr(), e.G, b.lengths0.data_ptr(), b.angles0.data_ptr(), s)
    _lib.call("arreau_ve_pbc_forward", b.frac0.data_ptr(), b.eps_x.data_ptr(), b.t_atom.data_ptr(),
              e.d_ve_sigmas.data_ptr(), b.lattice0.data_ptr(), e.crystal_of_atom.data_ptr(), e.N,
              e.frac.data_ptr(), b.target_eps.data_ptr(), s)
    _lib.call("arreau_d3pm_q_sample", b.types0.data_ptr(), b.u.data_ptr(), b.t_atom.data_ptr(),
              e.d_q_keep.data_ptr(), e.d_q_to_mask.data_ptr(), e.N, e.Z, e.types.data_ptr(), s)
    _lib.call("arreau_vp_lattice_forward", b.lengths0.data_ptr(), b.eps_l.data_ptr(), b.t_crystal.data_ptr(),
              b.d_alpha_bars.data_ptr(), e.G, e.lengths.data_ptr(), s)
    e.angles.copy_(b.angles0)


class BatchEngine:
    """A DenoiseEngine plus per-batch buffers (`_bufs`: name -> (leading extent kind, capacity buffer)) sized for a
    CAPACITY and re-bound in place to every batch topology."""

    def _bind(self) -> None:
        e = self.eng
        ext = {"N": e.N, "G": e.G, "3N": 3 * e.N}
        for name, (kind, buf) in self._bufs.items():
            setattr(self, name, buf[: ext[kind]])

    def fits(self, num_atoms) -> bool:
        na = np.asarray(num_atoms, dtype=np.int64).reshape(-1)
        return int(na.sum()) <= self.eng.N_cap and int(na.shape[0]) <= self.eng.G_cap

    def set_topology(self, num_atoms) -> None:
        """Bind the next batch's atoms-per-crystal vector (no allocation)."""
        self.eng.set_topology(num_atoms)
        self._bind()


class TrainEngine(BatchEngine):
    """The training step's buffers on one GPU, sized for a CAPACITY (atoms, crystals) and re-bound in place to every
    batch topology (`set_topology`): a shuffled epoch of variable-size batches (lattice_dataset.py:96-113,
    main_diffusion.py:221-230) runs through one engine without reallocating (SURVEY 8f-4)."""

    def __init__(self, params: FlatParams, tables: DiffusionTables, fourier_w, ori_grid, num_atoms: Sequence[int],
                 radius: float, max_neighbors: int, device="cuda", backward_precision: str = "fp32",
                 node_capacity: Optional[int] = None, crystal_capacity: Optional[int] = None):
        """backward_precision: "fp32" (FFMA GEMMs: the parity path) or "tf32" (tensor-core GEMMs with fp32
        accumulation in the backward pass; the forward stays fp32).  node_capacity / crystal_capacity: room for
        larger batches than `num_atoms` (default: exactly that topology)."""
        if backward_precision not in ("fp32", "tf32"):
            raise ValueError("backward_precision must be 'fp32' or 'tf32'")
        self.backward_precision = _lib.PRECISION_TF32 if backward_precision == "tf32" else _lib.PRECISION_FP32
        self.p, self.tabs = params, tables
        self.device = dev = torch.device(device)
        self.ori = (ori_grid.detach() if isinstance(ori_grid, torch.Tensor) else torch.as_tensor(np.asarray(ori_grid))) \
            .to(dev, torch.float32).contiguous()
        self.w = PonitaWeights.from_flat(params, self.ori)
        self.eng = DenoiseEngine(self.w, tables, fourier_w, num_atoms, radius, max_neighbors, precision="fp32",
                                 debug=True, device=dev, node_capacity=node_capacity, crystal_capacity=crystal_capacity)
        e = self.eng
        N, G, Z = e.N_cap, e.G_cap, e.Z
        f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)  # noqa: E731
        f32 = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)  # noqa: E731
        self._bufs = noising_buffers(N, G, Z, dev)
        self._bufs.update({"dscore": ("N", f32(N, 3)), "dlogits": ("N", f32(N, Z)), "dlen0": ("G", f32(G, 3))})
        self.loss = f64(5)
        self.d_alpha_bars = tables.vp_alpha_bars.to(torch.float32).to(dev)
        self.fold = torch.as_tensor(monomial_fold_table(), dtype=torch.int32).to(dev)
        self.mom_scratch, self.mom_out = f64(512), f64(2)
        self._bwd_ws = None
        self._bind()

    # ------------------------------------------------------------------ pieces (each = the mirrored reference call)
    def repack(self) -> None:
        """Kernel layouts of the current flat parameters (after an optimizer step)."""
        self.w = PonitaWeights.from_flat(self.p, self.ori)
        self.eng.w = self.w

    def set_batch(self, frac0, types0, lattice0, timestep, eps_x, u, eps_l) -> None:
        """Batch{X0, A0, L0} and the step's random draws (diffusion_loss.py:205-237).  timestep: [G] or [G,1]."""
        e = self.eng
        self.frac0.copy_(torch.as_tensor(frac0).reshape(e.N, 3), non_blocking=True)
        self.types0.copy_(torch.as_tensor(types0).reshape(e.N), non_blocking=True)
        self.lattice0.copy_(torch.as_tensor(lattice0).reshape(e.G, 3, 3), non_blocking=True)
        self.t_crystal.copy_(torch.as_tensor(timestep).reshape(e.G).to(torch.int32), non_blocking=True)
        # one gather through the engine's atom -> crystal map (repeat_interleave would upload the counts and synchronise)
        torch.index_select(self.t_crystal, 0, e.crystal_of_atom[: e.N], out=self.t_atom)
        self.eps_x.copy_(torch.as_tensor(eps_x).reshape(e.N, 3), non_blocking=True)
        self.u.copy_(torch.as_tensor(u).reshape(e.N, e.Z), non_blocking=True)
        self.eps_l.copy_(torch.as_tensor(eps_l).reshape(e.G, 3), non_blocking=True)

    def noise_batch(self) -> None:
        """VE_pbc.forward, D3PM.get_xt, matrix_to_params + VP_lattice.forward into the forward engine's state."""
        noise_into(self.eng, self)

    def _workspace(self) -> torch.Tensor:
        e = self.eng
        need = int(_lib.load().arreau_ponita_backward_workspace_bytes(e.N, e.edge_capacity, e.F, 4))
        if need < 0:
            _lib.check(need, "arreau_ponita_backward_workspace_bytes")
        if self._bwd_ws is None or self._bwd_ws.numel() * 4 < need:
            self._bwd_ws = None
            self._bwd_ws = torch.empty((need + 3) // 4, dtype=torch.float32, device=self.device)
        return self._bwd_ws

    def predict(self) -> None:
        """DiffusionLoss.predict_scores (diffusion_loss.py:112-197) on the noised batch; per-layer buffers kept.
        backward_precision "tf32": the forward's dense contractions run on the tcgen05 TF32 GEMM as well and keep their
        activations for the backward (arreau_ponita_forward_train); "fp32": the plain fp32 forward (the parity path),
        the backward recomputes what it needs."""
        e = self.eng
        e.prepare_inputs(self.t_atom, from_trig=False)
        e._ensure_capacity()
        e.build_graph()
        self._forward_kept = 0
        if self.backward_precision == _lib.PRECISION_TF32:
            ws = self._workspace()
            _lib.call("arreau_ponita_forward_train", self.p.data.data_ptr(), C.byref(self.p.layout), self.w.ref(), C.byref(e.ws),
                      self.fold.data_ptr(), e.x.data_ptr(), e.vec.data_ptr(), e.row_ptr.data_ptr(), e.src.data_ptr(),
                      e.dist.data_ptr(), e.dir.data_ptr(), e.lattice.data_ptr(), e.atom_offset.data_ptr(),
                      e.crystal_of_atom.data_ptr(), e.N, e.G, e.radius, ws.data_ptr(), ws.numel() * 4, self.backward_precision,
                      e.logits.data_ptr(), e.score.data_ptr(), e.len0.data_ptr(), e.stream)
            self._forward_kept = 1
        else:
            e.forward()

    def compute_loss(self) -> torch.Tensor:
        e, tb = self.eng, self.tabs
        _lib.call("arreau_training_loss", e.score.data_ptr(), e.logits.data_ptr(), e.len0.data_ptr(),
                  self.target_eps.data_ptr(), self.types0.data_ptr(), e.types.data_ptr(), self.t_atom.data_ptr(),
                  self.lengths0.data_ptr(), e.atom_offset.data_ptr(), e.d_q_keep.data_ptr(), e.d_q_to_mask.data_ptr(),
                  tb.onestep_keep, tb.onestep_to_mask, tb.T, e.N, e.G, e.Z, HYBRID_LOSS_COEFF, self.terms.data_ptr(),
                  self.loss.data_ptr(), self.dscore.data_ptr(), self.dlogits.data_ptr(), self.dlen0.data_ptr(), e.stream)
        return self.loss

    def backward(self, dlogits: Optional[torch.Tensor] = None, dscore: Optional[torch.Tensor] = None,
                 dlen0: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Parameter gradients of the last predict() for the given output gradients (default: the loss's)."""
        e = self.eng
        dlogits = self.dlogits if dlogits is None else dlogits
        dscore = self.dscore if dscore is None else dscore
        dlen0 = self.dlen0 if dlen0 is None else dlen0
        self._workspace()
        _lib.call("arreau_ponita_backward", self.p.data.data_ptr(), C.byref(self.p.layout), self.w.ref(), C.byref(e.ws),
                  self.fold.data_ptr(), e.x.data_ptr(), e.vec.data_ptr(), e.row_ptr.data_ptr(), e.src.data_ptr(),
                  e.dst.data_ptr(), e.dist.data_ptr(), e.dir.data_ptr(), e.lattice.data_ptr(), e.atom_offset.data_ptr(),
                  e.crystal_of_atom.data_ptr(), e.N, e.G, e.radius, dlogits.data_ptr(), dscore.data_ptr(),
                  dlen0.data_ptr(), self._bwd_ws.data_ptr(), self._bwd_ws.numel() * 4, self.p.grad.data_ptr(),
                  self.backward_precision, int(getattr(self, "_forward_kept", 0)), e.stream)
        return self.p.grad

    # ------------------------------------------------------------------ the step
    def loss_and_grads(self, frac0, types0, lattice0, timestep, eps_x, u, eps_l):
        """DiffusionLoss.__call__ + loss.backward(): returns (loss[5] f64 device = {total, frac, vb, ce, lattice},
        flat gradient buffer)."""
        self.repack()
        self.set_batch(frac0, types0, lattice0, timestep, eps_x, u, eps_l)
        self.noise_batch()
        self.predict()
        self.compute_loss()
        self.backward()
        return self.loss, self.p.grad

    # ------------------------------------------------------------------ callibrate (conv.py:122-123,140-146)
    def _std(self, x: torch.Tensor, sub_cols: Optional[torch.Tensor] = None) -> float:
        n = x.numel()
        _lib.call("arreau_moments", x.data_ptr(), _lib.ptr(sub_cols), n, self.mom_scratch.data_ptr(),
                  self.mom_out.data_ptr(), self.eng.stream)
        s, q = self.mom_out.tolist()
        return float(np.sqrt(max(q - s * s / n, 0.0) / (n - 1)))      # torch.std: unbiased

    def calibrate(self, frac, types, lengths, angles, t) -> None:
        """The one-time re-initialisation of the reference's first train-mode forward on a GIVEN state: runs
        predict_scores at timestep(s) t, then `calibrate_from_last_forward`."""
        e = self.eng
        e.set_state(frac, types, lengths, angles)
        e.predict_scores(t)
        self.calibrate_from_last_forward()

    def calibrate_from_last_forward(self) -> None:
        """conv.py:122-123,140-146 with the tensors of the forward that has just run (`predict` of a training step or
        `calibrate`): per layer kernel.weight *= std(x) / std(x1) and fiber_kernel.weight *= std(x1) / std(x2), x2
        before the bias, all three taken from that ONE forward with the weights as they were (the reference rescales
        a layer's weights after the layer has produced its output, so later layers see un-rescaled activations).
        The statistics are reduced on the device (arreau_moments)."""
        e = self.eng
        v = self.p.views()
        for l in range(LAYERS):
            s_in, s_1 = self._std(e.h_debug[l]), self._std(e.x1_debug[l])
            s_2 = self._std(e.x2_debug[l], v[f"interaction_layers.{l}.conv.bias"])
            v[f"interaction_layers.{l}.conv.kernel.weight"].mul_(s_in / s_1)
            v[f"interaction_layers.{l}.conv.fiber_kernel.weight"].mul_(s_1 / s_2)
        self.p.version += 1
        self.repack()
